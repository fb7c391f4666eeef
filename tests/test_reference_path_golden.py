"""The whole hot path against vectors produced by the REFERENCE's own kernels.

``tests/golden/make_reference_path_golden.py`` imports the reference rasteriser from /root/reference and executes its
unmodified ``@ti.kernel`` / ``@ti.func`` source under ``tests/golden/taichi_shim.py`` (float32 numpy arithmetic, by-value
``ti.func`` arguments, lock-step SIMT emulation of the two shared-memory kernels), forward + backward through the
reference's ``torch.autograd.Function``, for the scenes of ``tests/golden/reference_path_scenes.py``; the outputs are
committed in ``reference_path_vectors.npz``.  This pins, against the reference source itself, what its unit tests do
not: multi-splat ordering and ties, the alpha cut-off / clamp / saturation rule, depth and count outputs, the
w-recursion of the backward, SH colour and its gradient with band masking, the in-place quaternion normalisation, the
off-screen bounding-box quirk, multi-object poses and every tensor handed to the backward hook.

* CPU: the oracle must reproduce the vectors to float32 rounding (it is a strict-IEEE restatement of the same arithmetic).
* GPU (``-m gpu``): the CUDA operator must reproduce them within the path's tolerances (RGB 1e-4, gradients 1e-3).
"""
import os
import sys
from types import SimpleNamespace

import numpy as np
import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "golden"))
from reference_path_scenes import scenes  # noqa: E402

from helpers import grad_close, oracle_backward, oracle_forward  # noqa: E402
from taichi_3d_gaussian_splatting_b200 import CameraInfo  # noqa: E402

SCENES = scenes()
GOLDEN = np.load(os.path.join(HERE, "golden", "reference_path_vectors.npz"))


def _golden(name):
    prefix = name + "/"
    return SimpleNamespace(**{k[len(prefix):]: GOLDEN[k] for k in GOLDEN.files if k.startswith(prefix)})


def _as_scene(sc, device="cpu"):
    return SimpleNamespace(
        point_cloud=sc["point_cloud"].clone().to(device), point_cloud_features=sc["point_cloud_features"].clone().to(device),
        point_invalid_mask=sc["point_invalid_mask"].to(device), point_object_id=sc["point_object_id"].to(device),
        camera_info=CameraInfo(camera_intrinsics=sc["camera_intrinsics"].clone().to(device), camera_height=sc["camera_height"],
                               camera_width=sc["camera_width"], camera_id=0),
        q_pointcloud_camera=sc["q_pointcloud_camera"].to(device), t_pointcloud_camera=sc["t_pointcloud_camera"].to(device))


def _grad_image(sc):
    shape = (sc["camera_height"], sc["camera_width"], 3)
    return torch.randn(shape, generator=torch.Generator().manual_seed(sc["grad_seed"]))


def _close(a, b, rtol, floor):
    ok, worst, nviol = grad_close(a, b, rtol=rtol, floor_frac=floor)
    return ok, (worst, nviol)


def test_scenes_exercise_what_they_claim():
    b = _golden("B_dense_saturating")
    sc = SCENES["B_dense_saturating"]
    _, fwd, _ = oracle_forward(_as_scene(sc), near_plane=sc["near_plane"], far_plane=sc["far_plane"],
                               depth_to_sort_key_scale=sc["depth_to_sort_key_scale"])
    lengths = fwd.tile_points_end - fwd.tile_points_start
    assert lengths.min() > 256                                     # more than one shared-memory group per tile
    assert (fwd.pixel_offset_of_last_effective_point < fwd.tile_points_end[0]).any()  # early termination happens
    assert b.count.max() >= 50 and float(fwd.pixel_accumulated_alpha.max()) > 0.999
    d = _golden("D_borders_band0")
    assert d.hook_point_id_in_camera_list.shape[0] < 80             # frustum rejections
    assert (d.hook_num_overlap_tiles == 0).any()                    # right / bottom off-screen: no tile
    c = _golden("C_two_objects_band1_ties")
    assert float(np.abs(c.grad_pointcloud_features[:, 12:24]).max()) == 0.0  # band 1: coefficients 4..15 masked
    assert float(np.abs(c.grad_pointcloud_features[:, 9:12]).max()) > 0.0


@pytest.mark.parametrize("name", list(SCENES))
def test_oracle_reproduces_the_reference_kernels(name):
    sc, ref = SCENES[name], _golden(name)
    scene = _as_scene(sc)
    o, fwd, feats = oracle_forward(scene, near_plane=sc["near_plane"], far_plane=sc["far_plane"],
                                   depth_to_sort_key_scale=sc["depth_to_sort_key_scale"])
    assert np.array_equal(fwd.point_id_in_camera_list, ref.hook_point_id_in_camera_list)
    assert np.array_equal(fwd.num_overlap_tiles, ref.hook_num_overlap_tiles)
    assert np.array_equal(fwd.pixel_valid_point_count, ref.count)
    assert np.abs(fwd.image - ref.image).max() <= 5e-7
    assert np.abs(fwd.depth - ref.depth).max() <= 1e-5 * max(1.0, float(np.abs(ref.depth).max()))
    assert np.array_equal(fwd.point_uv, ref.hook_point_uv_in_camera) and np.array_equal(fwd.point_in_camera[:, 2], ref.hook_point_depth)
    # per-stage tensors written by the reference kernels: integer stages exactly, per-point floats to float32 rounding
    assert np.array_equal(fwd.point_in_camera_sort_key, ref.stage_point_in_camera_sort_key)     # sorted 64-bit keys
    assert np.array_equal(fwd.point_offset_with_sort_key, ref.stage_point_offset_with_sort_key)  # incl. the tie order
    assert np.array_equal(fwd.tile_points_start, ref.stage_tile_points_start)
    assert np.array_equal(fwd.tile_points_end, ref.stage_tile_points_end)
    assert np.array_equal(fwd.pixel_offset_of_last_effective_point, ref.stage_pixel_offset_of_last_effective_point)
    # The per-point stage is BIT-IDENTICAL: the shim follows Taichi's own definitions (Matrix.sum in element order,
    # normalized() = (1 / norm) * v, elementary functions correctly rounded) and the oracle restates the same operation
    # order, so projection, covariance, conic, rescale, opacity, SH colour, radius and the in-place normalised quaternion
    # agree to the last bit.
    for got, exp in ((fwd.point_uv, ref.stage_point_uv), (fwd.point_in_camera, ref.stage_point_in_camera),
                     (fwd.point_uv_conic_and_rescale, ref.stage_point_uv_conic_and_rescale),
                     (fwd.point_alpha_after_activation, ref.stage_point_alpha_after_activation),
                     (fwd.point_color, ref.stage_point_color), (fwd.point_radii, ref.stage_point_radii),
                     (feats, ref.features_after_forward)):
        assert np.array_equal(got, exp), (name, float(np.abs(got - exp).max()))
    # the blend evaluates exp() per (pixel, splat): libm expf here, correctly rounded in the shim -- last-bit differences
    assert np.abs(fwd.pixel_accumulated_alpha - ref.stage_pixel_accumulated_alpha).max() <= 2e-6
    assert (fwd.image == ref.image).mean() >= 0.99
    bwd = oracle_backward(o, fwd, scene, feats, _grad_image(sc).numpy(), sc["color_max_sh_band"])
    for got, exp in ((bwd.grad_pointcloud, ref.grad_pointcloud), (bwd.grad_pointcloud_features, ref.grad_pointcloud_features),
                     (bwd.grad_point_in_camera, ref.hook_grad_point_in_camera),
                     (bwd.grad_pointfeatures_in_camera, ref.hook_grad_pointfeatures_in_camera),
                     (bwd.grad_viewspace, ref.hook_grad_viewspace), (bwd.magnitude_grad_viewspace, ref.hook_magnitude_grad_viewspace),
                     (bwd.magnitude_grad_viewspace_on_image, ref.hook_magnitude_grad_viewspace_on_image)):
        # the reference sums its per-pixel contributions in float32 (thread order under the shim), the oracle in
        # double: with ~80 blended splats per pixel and ~500 pixels per splat that is worth a few 1e-5 on scene B
        rtol, floor = (3e-4, 3e-5) if name == "B_dense_saturating" else (2e-5, 2e-6)
        ok, info = _close(got, exp, rtol=rtol, floor=floor)
        assert ok, (name, info)
    assert np.array_equal(bwd.num_affected_pixels, ref.hook_num_affected_pixels)


@pytest.mark.gpu
@pytest.mark.parametrize("exact_exp", [True, False], ids=["exact_exp", "default_fast_path"])
@pytest.mark.parametrize("name", list(SCENES))
def test_cuda_operator_reproduces_the_reference_kernels(name, exact_exp):
    from gpu_helpers import make_op, n, run_forward
    sc, ref = SCENES[name], _golden(name)
    scene = _as_scene(sc, "cuda")
    scene.point_cloud.requires_grad_(True)
    scene.point_cloud_features.requires_grad_(True)
    hook = {}
    op = make_op(hook=lambda h: hook.update(h=h), exact_exp=exact_exp, near_plane=sc["near_plane"], far_plane=sc["far_plane"],
                 depth_to_sort_key_scale=sc["depth_to_sort_key_scale"])
    image, depth, count = run_forward(op, scene, band=sc["color_max_sh_band"])
    assert np.abs(n(image) - ref.image).max() <= 1e-4
    assert np.abs(n(depth) - ref.depth).max() <= 1e-3 * max(1.0, float(np.abs(ref.depth).max()))
    assert (n(count) != ref.count).sum() <= 2  # a (pixel, splat) pair within an ulp of the alpha cut-off may flip
    # the preprocess kernel evaluates the oracle's operation order (-fmad=false, exp rounded once from double), and the
    # oracle is bit-identical to the reference kernels here: so is the CUDA per-point stage
    frame = op.last_frame
    for got, exp in ((frame.point_uv, ref.stage_point_uv), (frame.point_in_camera, ref.stage_point_in_camera),
                     (frame.point_uv_conic_and_rescale, ref.stage_point_uv_conic_and_rescale),
                     (frame.point_alpha_after_activation, ref.stage_point_alpha_after_activation),
                     (frame.point_color, ref.stage_point_color), (frame.point_radii, ref.stage_point_radii)):
        assert np.array_equal(n(got), exp), name
    assert np.array_equal(n(scene.point_cloud_features), ref.features_after_forward)
    image.backward(_grad_image(sc).cuda())
    h = hook["h"]
    assert np.array_equal(n(h.point_id_in_camera_list), ref.hook_point_id_in_camera_list)
    assert np.array_equal(n(h.num_overlap_tiles), ref.hook_num_overlap_tiles)
    assert (n(h.num_affected_pixels) != ref.hook_num_affected_pixels).sum() <= 2
    for got, exp in ((scene.point_cloud.grad, ref.grad_pointcloud), (scene.point_cloud_features.grad, ref.grad_pointcloud_features),
                     (h.grad_point_in_camera, ref.hook_grad_point_in_camera),
                     (h.grad_pointfeatures_in_camera, ref.hook_grad_pointfeatures_in_camera),
                     (h.grad_viewspace, ref.hook_grad_viewspace), (h.magnitude_grad_viewspace, ref.hook_magnitude_grad_viewspace),
                     (h.magnitude_grad_viewspace_on_image, ref.hook_magnitude_grad_viewspace_on_image)):
        got = n(got)
        ok, (worst, nviol) = _close(got, exp, rtol=1e-3, floor=1e-5)
        # float32 atomics over ~500 pixels x ~80 blended splats (scene B): as in the full-size parity test, a few
        # entries in a thousand may leave the per-entry tolerance, none by more than 1e-3 of the largest entry
        assert ok or (nviol <= 2e-3 * exp.size and np.abs(got - exp).max() <= 1e-3 * np.abs(exp).max()), (name, worst, nviol)


# ---------------------------------------------------------------- BASELINE config 1 through the reference's kernels
# reference_path_c1.npz: the same generator, run with --with-c1 (5 minutes in the interpreter), on SURVEY 8(d) C1 =
# BASELINE config 1 (1e4 Gaussians, 256 x 256, SH deg 0).  Stored within 1 MB: ids, tile counts, pixel counts and tile
# ranges whole, every other array that must be bit-equal as a SHA-256, the floats as samples (a quarter of the pixels
# and of the in-frustum rows) beside per-tile image sums and each hook gradient's L1 norm.  The dense gradients are the
# hook tensors on the in-frustum rows and zero elsewhere (checked when the file was made).
def _digest(a):
    import hashlib
    return np.frombuffer(hashlib.sha256(np.ascontiguousarray(a).tobytes()).digest(), dtype=np.uint8)


def _tile_sums(image):
    h, w = image.shape[:2]
    return image.reshape(h // 16, 16, w // 16, 16, 3).astype(np.float64).sum(axis=(1, 3))


C1_PER_POINT_STAGE = ("point_uv", "point_in_camera", "point_uv_conic_and_rescale", "point_alpha_after_activation", "point_color",
                      "point_radii")


def _c1():
    from reference_path_scenes import baseline_config_1
    g = np.load(os.path.join(HERE, "golden", "reference_path_c1.npz"))
    return baseline_config_1(), SimpleNamespace(**{k: g[k] for k in g.files})


def _c1_sampled_gradients_close(ref, got_by_name, rtol, allow_few):
    """Each hook gradient on the stored rows (``got_by_name[name]``: all in-frustum rows) and its L1 norm over all of them."""
    for name, got in got_by_name.items():
        exp = getattr(ref, "rows_hook_" + name)
        sampled = got[ref.point_rows]
        ok, (worst, nviol) = _close(sampled, exp, rtol=rtol, floor=1e-5)
        # GPU / emulated CUDA: float32 atomics -- a few entries in a thousand may leave the per-entry tolerance, none by more
        # than 1e-3 of the largest entry
        assert ok or (allow_few and nviol <= 2e-3 * exp.size and np.abs(sampled - exp).max() <= 1e-3 * np.abs(exp).max()), \
            (name, worst, nviol)
        l1 = float(np.abs(got.astype(np.float64)).sum())
        assert abs(l1 - float(getattr(ref, "l1_hook_" + name)[0])) <= rtol * l1, name


def test_oracle_reproduces_the_reference_kernels_at_baseline_config_1():
    sc, ref = _c1()
    scene = _as_scene(sc)
    o, fwd, feats = oracle_forward(scene)
    assert np.array_equal(fwd.point_id_in_camera_list, ref.hook_point_id_in_camera_list) and fwd.point_id_in_camera_list.shape[0] == 9566
    assert np.array_equal(fwd.num_overlap_tiles, ref.hook_num_overlap_tiles)
    assert np.array_equal(_digest(fwd.point_in_camera_sort_key), ref.sha256_stage_point_in_camera_sort_key)
    assert np.array_equal(_digest(fwd.point_offset_with_sort_key), ref.sha256_stage_point_offset_with_sort_key)
    assert np.array_equal(fwd.tile_points_start, ref.stage_tile_points_start)
    assert np.array_equal(fwd.tile_points_end, ref.stage_tile_points_end)
    assert np.array_equal(fwd.pixel_valid_point_count, ref.count)
    assert np.array_equal(_digest(fwd.pixel_offset_of_last_effective_point), ref.sha256_stage_pixel_offset_of_last_effective_point)
    pix = ref.pixel_index
    image = fwd.image.reshape(-1, 3)[pix]
    assert np.abs(image - ref.pixel_image).max() <= 5e-7 and (image == ref.pixel_image).mean() >= 0.99
    assert np.abs(_tile_sums(fwd.image) - ref.tile_image_sum).max() <= 256 * 5e-7 + 1e-4  # + float32 rounding of the stored sums
    assert np.abs(fwd.depth.reshape(-1, 1)[pix] - ref.pixel_depth).max() <= 1e-4
    assert np.abs(fwd.pixel_accumulated_alpha.reshape(-1, 1)[pix] - ref.pixel_stage_pixel_accumulated_alpha).max() <= 2e-6
    for key in C1_PER_POINT_STAGE:  # the per-point stage is bit-identical (see above)
        assert np.array_equal(_digest(getattr(fwd, key)), getattr(ref, "sha256_stage_" + key)), key
    bwd = oracle_backward(o, fwd, scene, feats, _grad_image(sc).numpy(), 0)
    ids = ref.hook_point_id_in_camera_list.astype(np.int64)
    _c1_sampled_gradients_close(ref, {"grad_point_in_camera": bwd.grad_pointcloud[ids],
                                      "grad_pointfeatures_in_camera": bwd.grad_pointcloud_features[ids],
                                      "grad_viewspace": bwd.grad_viewspace, "magnitude_grad_viewspace": bwd.magnitude_grad_viewspace},
                                rtol=1e-4, allow_few=False)
    assert np.array_equal(bwd.num_affected_pixels, ref.hook_num_affected_pixels)


@pytest.mark.gpu
@pytest.mark.parametrize("exact_exp", [True, False], ids=["exact_exp", "default_fast_path"])
def test_cuda_operator_reproduces_the_reference_kernels_at_baseline_config_1(exact_exp):
    from gpu_helpers import make_op, n, run_forward
    sc, ref = _c1()
    scene = _as_scene(sc, "cuda")
    scene.point_cloud.requires_grad_(True)
    scene.point_cloud_features.requires_grad_(True)
    hook = {}
    op = make_op(hook=lambda h: hook.update(h=h), exact_exp=exact_exp)
    image, depth, count = run_forward(op, scene, band=0)
    pix = ref.pixel_index
    assert np.abs(n(image).reshape(-1, 3)[pix] - ref.pixel_image).max() <= 1e-4
    assert np.abs(_tile_sums(n(image)) - ref.tile_image_sum).max() <= 256 * 1e-4
    assert np.abs(n(depth).reshape(-1, 1)[pix] - ref.pixel_depth).max() <= 1e-3
    assert (n(count) != ref.count).sum() <= 3
    image.backward(_grad_image(sc).cuda())
    h = hook["h"]
    assert np.array_equal(n(h.point_id_in_camera_list), ref.hook_point_id_in_camera_list)
    assert np.array_equal(n(h.num_overlap_tiles), ref.hook_num_overlap_tiles)
    assert (n(h.num_affected_pixels) != ref.hook_num_affected_pixels).sum() <= 3
    ids = torch.from_numpy(ref.hook_point_id_in_camera_list.astype(np.int64)).cuda()
    _c1_sampled_gradients_close(ref, {"grad_point_in_camera": n(scene.point_cloud.grad[ids]),
                                      "grad_pointfeatures_in_camera": n(scene.point_cloud_features.grad[ids]),
                                      "grad_viewspace": n(h.grad_viewspace), "magnitude_grad_viewspace": n(h.magnitude_grad_viewspace)},
                                rtol=1e-3, allow_few=True)
    rest = torch.ones(scene.point_cloud.shape[0], dtype=torch.bool, device="cuda")
    rest[ids] = False
    assert float(scene.point_cloud.grad[rest].abs().max()) == 0.0 and float(scene.point_cloud_features.grad[rest].abs().max()) == 0.0


# ---------------------------------------------------------------- reduced BASELINE config 2 through the reference's kernels
# reference_path_c2_reduced.npz (generator option --with-c2r, more than two and a half hours in the interpreter): 4.3e4 Gaussians at
# 976 x 544 = 2074 tiles with C2's splat density per tile.  Everything that must be bit-equal is stored as a SHA-256,
# images and gradients as samples (6000 pixels, per-tile sums, 1500 in-frustum rows, global L1 norms).
def _c2r():
    from reference_path_scenes import reduced_config_2
    path = os.path.join(HERE, "golden", "reference_path_c2_reduced.npz")
    if not os.path.exists(path):
        pytest.skip("reference_path_c2_reduced.npz has not been generated")
    g = np.load(path)
    return reduced_config_2(), SimpleNamespace(**{k: g[k] for k in g.files}), _digest


def test_oracle_reproduces_the_reference_kernels_at_reduced_config_2():
    sc, ref, digest = _c2r()
    scene = _as_scene(sc)
    o, fwd, feats = oracle_forward(scene)
    assert (fwd.point_uv.shape[0], fwd.point_offset_with_sort_key.shape[0], int(fwd.pixel_valid_point_count.max())) == tuple(ref.sizes)
    lengths = fwd.tile_points_end - fwd.tile_points_start
    assert lengths.shape[0] == 61 * 34 and lengths.max() > 256
    for key, got in (("hook_point_id_in_camera_list", fwd.point_id_in_camera_list), ("hook_num_overlap_tiles", fwd.num_overlap_tiles),
                     ("count", fwd.pixel_valid_point_count), ("stage_point_in_camera_sort_key", fwd.point_in_camera_sort_key),
                     ("stage_point_offset_with_sort_key", fwd.point_offset_with_sort_key),
                     ("stage_tile_points_start", fwd.tile_points_start), ("stage_tile_points_end", fwd.tile_points_end),
                     ("stage_pixel_offset_of_last_effective_point", fwd.pixel_offset_of_last_effective_point),
                     ("stage_point_uv", fwd.point_uv), ("stage_point_in_camera", fwd.point_in_camera),
                     ("stage_point_uv_conic_and_rescale", fwd.point_uv_conic_and_rescale),
                     ("stage_point_alpha_after_activation", fwd.point_alpha_after_activation),
                     ("stage_point_color", fwd.point_color), ("stage_point_radii", fwd.point_radii),
                     ("features_after_forward", feats)):
        assert np.array_equal(digest(got), getattr(ref, "sha256_" + key)), key  # bit-identical arrays
    h, w = fwd.pixel_valid_point_count.shape
    pix = ref.pixel_index
    assert np.abs(fwd.image.reshape(h * w, 3)[pix] - ref.pixel_image).max() <= 5e-7
    assert np.abs(fwd.depth.reshape(h * w, 1)[pix] - ref.pixel_depth).max() <= 1e-4
    assert np.abs(fwd.pixel_accumulated_alpha.reshape(h * w, 1)[pix] - ref.pixel_stage_pixel_accumulated_alpha).max() <= 2e-6
    tiles = fwd.image.reshape(h // 16, 16, w // 16, 16, 3).astype(np.float64).sum(axis=(1, 3))
    assert np.abs(tiles - ref.tile_image_sum).max() <= 1e-4
    bwd = oracle_backward(o, fwd, scene, feats, _grad_image(sc).numpy(), 3)
    assert np.array_equal(digest(bwd.num_affected_pixels), ref.sha256_hook_num_affected_pixels)
    rows = ref.point_rows
    for got, key in ((bwd.grad_point_in_camera, "hook_grad_point_in_camera"),
                     (bwd.grad_pointfeatures_in_camera, "hook_grad_pointfeatures_in_camera"),
                     (bwd.grad_viewspace, "hook_grad_viewspace"), (bwd.magnitude_grad_viewspace, "hook_magnitude_grad_viewspace")):
        ok, info = _close(got[rows], getattr(ref, "rows_" + key), rtol=3e-4, floor=3e-5)
        assert ok, (key, info)
        l1 = float(np.abs(got.astype(np.float64)).sum())
        assert abs(l1 - float(getattr(ref, "l1_" + key)[0])) <= 1e-4 * l1, key


@pytest.mark.gpu
@pytest.mark.parametrize("exact_exp", [True, False], ids=["exact_exp", "default_fast_path"])
def test_cuda_operator_reproduces_the_reference_kernels_at_reduced_config_2(exact_exp):
    from gpu_helpers import make_op, n, run_forward
    sc, ref, digest = _c2r()
    scene = _as_scene(sc, "cuda")
    scene.point_cloud.requires_grad_(True)
    scene.point_cloud_features.requires_grad_(True)
    hook = {}
    op = make_op(hook=lambda h: hook.update(h=h), exact_exp=exact_exp, keep_all_tile_pairs=True)
    image, depth, count = run_forward(op, scene, band=3)
    frame = op.last_frame
    assert (frame.num_points_in_camera, frame.num_keys) == tuple(ref.sizes[:2])
    # integer stages: bit-identical to the reference kernels (SHA-256 of the arrays the reference produced)
    packed = n(frame.sorted_keys).astype(np.int64)
    bits = frame.layout.depth_bits
    keys64 = ((packed >> bits) << 32) | (packed & ((1 << bits) - 1))  # back to the reference's (tile << 32) + depth
    for key, got in (("hook_point_id_in_camera_list", frame.point_id_in_camera_list), ("hook_num_overlap_tiles", frame.num_overlap_tiles),
                     ("stage_point_offset_with_sort_key", frame.point_offset_with_sort_key),
                     ("stage_tile_points_start", frame.tile_points_start), ("stage_tile_points_end", frame.tile_points_end)):
        assert np.array_equal(digest(np.ascontiguousarray(n(got))), getattr(ref, "sha256_" + key)), key
    # per-point floats: equal to the oracle's (value equality, so that a signed zero cannot matter), and the oracle's are
    # equal to the reference kernels' bit for bit (the CPU test above compares their SHA-256)
    from test_gpu_parity import _check_stages
    _, fwd, _ = oracle_forward(_as_scene(sc))
    _check_stages(frame, fwd)
    assert np.array_equal(digest(keys64), ref.sha256_stage_point_in_camera_sort_key)
    h, w = count.shape
    pix = ref.pixel_index
    d_pix = np.abs(n(image).reshape(h * w, 3)[pix] - ref.pixel_image)
    assert (d_pix > 1e-4).sum() <= 3 and d_pix.max() <= 5e-3  # cut-off flips, see the tile sums below
    assert (n(count).reshape(h * w, 1)[pix] != ref.pixel_count).sum() <= 3
    tiles = n(image).reshape(h // 16, 16, w // 16, 16, 3).astype(np.float64).sum(axis=(1, 3))
    # 1.2e8 (pixel, splat) evaluations with CUDA's expf against the reference's correctly rounded exp: a handful of pairs within
    # an ulp of the alpha = 1/255 cut-off may fall on the other side (3 of 531k pixels at the full C2, DESIGN section 6), each
    # moving its pixel -- and so its tile sum -- by up to 1/255 * T * colour
    d_tiles = np.abs(tiles - ref.tile_image_sum)
    assert (d_tiles > 2e-3).sum() <= 4 and d_tiles.max() <= 1.2e-2, (int((d_tiles > 2e-3).sum()), float(d_tiles.max()))
    image.backward(_grad_image(sc).cuda())
    h_in = hook["h"]
    rows = ref.point_rows
    for got, key in ((h_in.grad_point_in_camera, "hook_grad_point_in_camera"),
                     (h_in.grad_pointfeatures_in_camera, "hook_grad_pointfeatures_in_camera"),
                     (h_in.grad_viewspace, "hook_grad_viewspace"), (h_in.magnitude_grad_viewspace, "hook_magnitude_grad_viewspace")):
        got = n(got)
        exp = getattr(ref, "rows_" + key)
        ok, (worst, nviol) = _close(got[rows], exp, rtol=1e-3, floor=1e-5)
        assert ok or (nviol <= 2e-3 * exp.size and np.abs(got[rows] - exp).max() <= 1e-3 * np.abs(exp).max()), (key, worst, nviol)
        l1 = float(np.abs(got.astype(np.float64)).sum())
        assert abs(l1 - float(getattr(ref, "l1_" + key)[0])) <= 1e-3 * l1, key
