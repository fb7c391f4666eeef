"""The reach masks the forward blend records for the backward, under the SIMT emulator of tests/simt.

``csrc/blend_fwd.cu`` writes, for every key it stages, the mask of the 8 patches of the tile (8x4 pixels, one per warp)
that the splat can reach; ``csrc/blend_bwd_transposed.cu`` reads nothing else to decide which splats a warp visits.
Checked here on the kernel sources compiled as host C++ (``tests/simt/emu_patch_masks.cpp``):
  (a) every byte the forward writes is the one ``splat_patch_mask`` (common.cuh) gives, the written keys of a tile are
      whole staging batches from its start, and they cover every key below the tile's deepest ``last_effective``;
  (b) the backward fed with the forward's own masks reproduces the butterfly kernel (blend_bwd.cu), which runs its own
      reach tests, within the tolerance of test_simt_blend_cpu.py.
The scenes between them have empty tiles, tiles that saturate before their list ends, patch lists longer than one
32-key window, chunks that take their splats from two windows and short last chunks; each run asserts what its scene
has to exercise."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from helpers import oracle_forward
from simt_helpers import SIMT, c
from taichi_3d_gaussian_splatting_b200.synthetic import make_scene

TILE, BATCH, WINDOW, CHUNK = 16, 256, 32, 16

# (points, H, W, sigma, seed): a dense frame, a frame of large splats where two of the six tiles saturate, a sparse frame;
# and what each has to exercise: "empty" tiles, tiles "saturated" before their list ends,
# patch lists "long"er than one window, chunks "spanning" two windows, "short" last chunks
SCENES = [((9000, 32, 32, 0.06, 4), {"long", "spanning", "short"}),
          ((3000, 48, 32, 0.4, 5), {"saturated", "long", "spanning", "short"}),
          ((40, 64, 64, 0.03, 6), {"empty", "short"})]


@pytest.fixture(scope="module")
def emu(tmp_path_factory):
    """tests/simt/emu_patch_masks.cpp built like the emulator library of simt_helpers, into a temporary directory."""
    out = str(tmp_path_factory.mktemp("simt") / "libsimt_patch_masks.so")
    cuda_inc = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "include")
    subprocess.run(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-fPIC", "-shared", "-I", cuda_inc, "-o", out,
                    os.path.join(SIMT, "emu_patch_masks.cpp")], check=True)
    L = ctypes.CDLL(out)
    L.emu_blend_forward_masks.restype = ctypes.c_longlong
    L.emu_blend_backward_masks.restype = ctypes.c_longlong
    return L


def _scene(num_points, H, W, sigma, seed):
    scene = make_scene(num_points, H, W, sigma, seed, sh_degree=3)
    _, fwd, _ = oracle_forward(scene)
    M = fwd.point_id_in_camera_list.shape[0]
    rec = np.zeros((M, 12), np.float32)  # u v a b | c rescale opacity depth | r g b radius
    rec[:, 0:2] = fwd.point_uv
    rec[:, 2:6] = fwd.point_uv_conic_and_rescale
    rec[:, 6] = fwd.point_alpha_after_activation
    rec[:, 7] = fwd.point_in_camera[:, 2]
    rec[:, 8:11] = fwd.point_color
    rec[:, 11] = fwd.point_radii
    start = np.ascontiguousarray(fwd.tile_points_start, dtype=np.int32)
    end = np.ascontiguousarray(fwd.tile_points_end, dtype=np.int32)
    vals = np.ascontiguousarray(fwd.point_offset_with_sort_key, dtype=np.int32)
    g = np.random.default_rng(seed + 1).standard_normal((H, W, 3)).astype(np.float32)
    return H, W, start, end, vals, rec, g


def _forward(emu, H, W, start, end, vals, rec, exact, fill):
    K = max(int(end.max()), 1)
    masks = np.full(K, fill, np.uint8)
    image, depth = np.zeros((H, W, 3), np.float32), np.zeros((H, W), np.float32)
    acc, last, cnt = np.zeros((H, W), np.float32), np.zeros((H, W), np.int32), np.zeros((H, W), np.int32)
    assert emu.emu_blend_forward_masks(0, int(exact), H, W, c(start), c(end), c(vals), c(rec), c(image), c(depth), c(acc),
                                       c(last), c(cnt), c(masks)) > 0
    return masks, acc, last


def _backward(emu, H, W, start, end, vals, rec, masks, g, acc, last, transposed, exact):
    accum = np.zeros((rec.shape[0], 12), np.float32)
    mag = np.full((H, W, 2), -1.0, np.float32)
    assert emu.emu_blend_backward_masks(int(transposed), int(exact), 1, H, W, c(start), c(end), c(vals), c(rec), c(masks),
                                        c(g), c(acc), c(last), c(accum), c(mag)) > 0
    return accum, mag


def _close(got, exp, rtol, floor):
    exp = np.asarray(exp, np.float64)
    tol = rtol * np.abs(exp) + floor * max(np.abs(exp).max(), 1e-30)
    bad = np.abs(got - exp) > tol
    return not bad.any(), int(bad.sum()), float((np.abs(got - exp) / tol).max())


def _patch_lists(start, end, last, masks, W):
    """Per (tile, patch): the deepest last_effective of the patch and the keys the backward visits, back to front."""
    tiles_x = W // TILE
    for t in range(start.shape[0]):
        tu, tv = t % tiles_x, t // tiles_x
        for w in range(8):
            x0, y0 = tu * TILE + (w & 1) * 8, tv * TILE + (w >> 1) * 4
            warp_last = int(last[y0:y0 + 4, x0:x0 + 8].max())
            keys = [i for i in range(warp_last - 1, int(start[t]) - 1, -1) if (masks[i] >> w) & 1]
            yield t, warp_last, keys


@pytest.mark.parametrize("exact", [True, False])
@pytest.mark.parametrize("scene,features", SCENES)
def test_forward_records_the_reach_masks_and_the_backward_follows_them(emu, scene, features, exact):
    H, W, start, end, vals, rec, g = _scene(*scene)
    # two runs over differently pre-filled arrays: a byte the forward writes is the same in both, one it leaves differs
    m0, acc, last = _forward(emu, H, W, start, end, vals, rec, exact, 0x00)
    m1, acc1, last1 = _forward(emu, H, W, start, end, vals, rec, exact, 0xFF)
    assert np.array_equal(acc, acc1) and np.array_equal(last, last1)
    written = m0 == m1
    expected = np.zeros_like(m0)
    emu.emu_patch_masks(H, W, c(start), c(end), c(vals), c(rec), c(expected))

    # (a) the bytes, and which keys get them
    assert np.array_equal(m0[written], expected[written])
    tiles_x = W // TILE
    cov = dict(empty=0, saturated=0, long=0, spanning=0, short=0)
    for t in range(start.shape[0]):
        s, e = int(start[t]), int(end[t])
        tu, tv = t % tiles_x, t // tiles_x
        deepest = int(last[tv * TILE:(tv + 1) * TILE, tu * TILE:(tu + 1) * TILE].max())
        n = int(written[s:e].sum())
        assert written[s:s + n].all(), t  # a prefix of the tile's list ...
        assert n == e - s or n % BATCH == 0, (t, n)  # ... of whole staging batches
        assert n >= deepest - s, (t, n, deepest)  # every key the backward can read
        cov["empty"] += e == s
        cov["saturated"] += n < e - s
    for _, warp_last, keys in _patch_lists(start, end, last, m0, W):
        idx = np.asarray(keys, np.int64)
        cov["long"] += len(keys) > WINDOW
        cov["short"] += len(keys) % CHUNK != 0
        for k in range(0, len(keys), CHUNK):
            win = (warp_last - 1 - idx[k:k + CHUNK]) // WINDOW
            cov["spanning"] += int(win.min() != win.max())
    print(scene, "exact" if exact else "fast", cov)
    assert all(cov[f] > 0 for f in features), cov

    # (b) the backward on the forward's own masks against the butterfly kernel (its own reach tests), same forward state
    ref, ref_img = _backward(emu, H, W, start, end, vals, rec, m0, g, acc, last, False, exact)
    got, got_img = _backward(emu, H, W, start, end, vals, rec, m0, g, acc, last, True, exact)
    assert ref[:, 10].max() > 0 or int(end.max()) == 0
    assert np.array_equal(got[:, 10], ref[:, 10])
    for cols in (slice(0, 2), slice(2, 5), slice(5, 8), slice(8, 9), slice(9, 10)):
        ok, nbad, worst = _close(got[:, cols], ref[:, cols], 1e-4, 2e-6)
        assert ok, (cols, nbad, worst)
    if exact:
        assert np.array_equal(got_img, ref_img)
    else:
        assert np.allclose(got_img, ref_img, rtol=2e-6, atol=1e-7 * float(np.abs(ref_img).max()))

