"""Gradients of the object poses (``gsb200_backward_with_pose``) from the kernel sources under the SIMT emulator of tests/simt.

The emulated CUDA path (simt_helpers: preprocess -> sort -> forward blend -> loop A of the backward) feeds the per-point kernel
with its pose epilogue, ``backward_points_kernel<*, true>``, and ``pose_grad_finalize_kernel`` (``tests/simt/emu_pose_grad.cpp``,
built on its own).  Checked against float64 torch autograd of ``torch_reference.dense_render`` with the pose as the leaf
(``inverse_SE3_qt_torch(q, t)`` in front, as the forward builds W and t_c), on one- and three-object scenes, with the
per-object reduction over several CTAs, in COMPACT and dense modes, and for bit-identical dense outputs with and without the
pose epilogue.  Argument validation goes through the real ``libgsb200.so`` (no device needed: it fails before any launch)."""
import ctypes
import os
import subprocess

import numpy as np
import pytest
import torch

from simt_helpers import SIMT, build_emulator, c, emulated_forward
from taichi_3d_gaussian_splatting_b200 import _lib
from taichi_3d_gaussian_splatting_b200.synthetic import make_scene
from taichi_3d_gaussian_splatting_b200.utils import inverse_SE3_qt_torch
from torch_reference import dense_render, quat_to_rot, sh_basis

FACTORS = (1.0, 0.5, 20.0, 5.0, 1.0)


@pytest.fixture(scope="module")
def emu():
    return build_emulator()


@pytest.fixture(scope="module")
def emu_pose(tmp_path_factory):
    """tests/simt/emu_pose_grad.cpp built like the emulator library of simt_helpers, into a temporary directory."""
    out = str(tmp_path_factory.mktemp("simt") / "libsimt_pose_grad.so")
    cuda_inc = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "include")
    subprocess.run(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-fPIC", "-shared", "-I", cuda_inc, "-o", out,
                    os.path.join(SIMT, "emu_pose_grad.cpp")], check=True)
    L = ctypes.CDLL(out)
    L.emu_backward_points_pose.restype = ctypes.c_int
    return L


def _scene(seed, n=400, h=32, w=48, sigma=0.12, yaw=4.0, sh_degree=3, n_obj=1, q_scale=1.0, skew=0.0):
    """test_oracle_dense_crosscheck's scene; n_obj > 1 interleaves the rows over objects with their own poses."""
    sc = make_scene(n, h, w, sigma, seed, sh_degree=sh_degree, yaw_degrees=yaw)
    sc.point_cloud[:, 2] = sc.point_cloud[:, 2] * 0.5
    sc.point_cloud_features[:, 7] += 1.5
    sc.point_invalid_mask[::7] = 1
    g = torch.Generator().manual_seed(seed + 7)
    if n_obj > 1:
        sc.point_object_id = (torch.arange(n, dtype=torch.int32) * 7 // 3 % n_obj).to(torch.int32)
        q = torch.randn((n_obj, 4), generator=g) * 0.04 + torch.tensor([0.0, 0.0, 0.0, 1.0])
        q = q / q.norm(dim=-1, keepdim=True)
        t = torch.randn((n_obj, 3), generator=g) * 0.1
        sc.q_pointcloud_camera, sc.t_pointcloud_camera = q.float(), t.float()
    else:
        sc.t_pointcloud_camera = (torch.randn((1, 3), generator=g) * 0.1).float()
    sc.q_pointcloud_camera = (sc.q_pointcloud_camera * q_scale).contiguous()
    if skew:
        sc.camera_info.camera_intrinsics[0, 1] = skew
    return sc


def _backward(emu, emu_pose, st, grad_image, band=3, compact=False, pose=True, max_blocks=16 * 148):
    """Loop A, then the per-point kernel (with the pose epilogue if ``pose``) under the emulator."""
    pre, scene, M = st.pre, st.scene, st.M
    H, W = pre.H, pre.W
    g = np.ascontiguousarray(grad_image, dtype=np.float32)
    accum, mag = np.zeros((max(M, 1), 12), np.float32), np.zeros((H, W, 2), np.float32)
    if st.K:
        emu.emu_blend_backward(0, int(st.exact), 1, H, W, c(st.start), c(st.end), c(st.sorted_vals), c(pre.records), c(g),
                               c(st.acc_alpha), c(st.last_effective), c(accum), c(mag))
    N = pre.point_offset.shape[0]
    q = scene.q_pointcloud_camera.numpy().astype(np.float32).copy()
    t = scene.t_pointcloud_camera.numpy().astype(np.float32).copy()
    n_obj = q.shape[0]
    poses = np.zeros((n_obj, 20), np.float32)
    emu.emu_pose(n_obj, c(q), c(t), c(poses))
    xyz = scene.point_cloud.detach().numpy().astype(np.float32).copy()
    K = scene.camera_info.camera_intrinsics.numpy().astype(np.float32).copy()
    obj = scene.point_object_id.numpy().astype(np.int32).copy()
    ctl = [np.zeros(N, np.int32), np.zeros(N, np.int32), np.zeros(N, np.float32), np.zeros(N, np.float32),
           np.zeros((N, 3), np.float32), np.zeros(N, np.float32)]
    if compact:
        out = (None, None, np.full((N, 12), 7.0, np.float32), np.full((N, 3), 7.0, np.float32))
    else:
        out = (np.full((N, 3), 7.0, np.float32), np.full((N, 56), 7.0, np.float32), None, None)
    partials = np.full((4096, n_obj, 12), 7.0, np.float32)
    gq, gt = np.full((n_obj, 4), 7.0, np.float32), np.full((n_obj, 3), 7.0, np.float32)
    f = ctypes.c_float
    blocks = emu_pose.emu_backward_points_pose(
        ctypes.c_longlong(N), c(pre.point_offset), c(pre.records), c(pre.pic), c(accum), c(poses), c(xyz), c(pre.feats),
        c(obj), c(t), c(K), int(band), *(f(v) for v in FACTORS), *(None if a is None else c(a) for a in out),
        *(c(a) for a in ctl), max_blocks, int(pose), n_obj, c(q), c(partials), c(gq), c(gt))
    return dict(out=[a for a in out if a is not None], ctl=ctl, gq=gq, gt=gt, blocks=blocks,
                partials=partials[:blocks])


def _render_objects(xyz, feats, invalid, obj, K, q_cp, t_cp, H, W):
    """dense_render with one pose row per object (point_object_id indexes q_cp / t_cp), same surrogate."""
    Rc_o = quat_to_rot(q_cp.double())
    Rc, tc = Rc_o[obj.long()], t_cp.double()[obj.long()]
    # dense_render's body, per-point rotation / translation
    dt = torch.float64
    xyz, feats, K = xyz.to(dt), feats.to(dt), K.to(dt)
    pc = torch.einsum("nij,nj->ni", Rc, xyz) + tc
    z = pc[:, 2]
    uv = ((pc @ K.T) / z[:, None])[:, :2]
    inside = (invalid.to(torch.bool) == 0) & (z > 0.8) & (z < 1000.0) & (uv[:, 0] >= -48) & (uv[:, 0] < W + 48) & \
        (uv[:, 1] >= -48) & (uv[:, 1] < H + 48)
    ids = torch.nonzero(inside.detach()).reshape(-1)
    pc, uv, z, f, Rc, tcp = pc[ids], uv[ids], z[ids], feats[ids], Rc[ids], tc[ids]
    M = ids.shape[0]
    q, s, logit = f[:, 0:4], f[:, 4:7], f[:, 7]
    pcd = pc.detach()
    fx, fy = K[0, 0], K[1, 1]
    zeros = torch.zeros_like(pcd[:, 0])
    J = torch.stack([torch.stack([fx / pcd[:, 2], zeros, -fx * pcd[:, 0] / pcd[:, 2] ** 2], -1),
                     torch.stack([zeros, fy / pcd[:, 2], -fy * pcd[:, 1] / pcd[:, 2] ** 2], -1)], -2)
    R = quat_to_rot(q)
    Sigma = R @ torch.diag_embed(torch.exp(2 * s)) @ R.transpose(-1, -2)
    U = J @ Rc
    cov = U @ Sigma @ U.transpose(-1, -2)
    a0, b0, c0, d0 = cov[:, 0, 0], cov[:, 0, 1], cov[:, 1, 0], cov[:, 1, 1]
    det0 = a0 * d0 - b0 * c0
    a1, d1 = a0 + 0.3, d0 + 0.3
    det1 = a1 * d1 - b0 * c0
    rescale = torch.sqrt(torch.clamp(det0 / det1, min=0.0)).detach()
    ca, cb, cc = d1 / det1, -b0 / det1, a1 / det1
    opacity = torch.sigmoid(logit)
    cam_centre = -torch.einsum("nji,nj->ni", Rc, tcp)
    basis = sh_basis((xyz[ids] - cam_centre).detach())
    color = torch.sigmoid((f[:, 8:56].reshape(M, 3, 16) * basis[:, None, :]).sum(-1))
    lam = (a0 + d0 + torch.sqrt((a0 - d0) ** 2 + 4 * b0 * c0)) / 2
    radius = (3.0 * torch.sqrt(lam)).detach().to(torch.float32)
    uvf = uv.detach().to(torch.float32)
    r = torch.clamp(radius, min=1.0)
    tw, th = W // 16, H // 16
    min_tu = torch.clamp(torch.floor(torch.clamp(uvf[:, 0] - r, min=0.0) / 16).to(torch.int64), max=tw)
    max_tu = torch.clamp(torch.maximum(torch.floor((uvf[:, 0] + r) / 16).to(torch.int64) + 1, min_tu + 1), max=tw)
    min_tv = torch.clamp(torch.floor(torch.clamp(uvf[:, 1] - r, min=0.0) / 16).to(torch.int64), max=th)
    max_tv = torch.clamp(torch.maximum(torch.floor((uvf[:, 1] + r) / 16).to(torch.int64) + 1, min_tv + 1), max=th)
    depth_key = (z.detach().to(torch.float32) * torch.tensor(100.0, dtype=torch.float32)).to(torch.int32)
    order = torch.argsort(depth_key.to(torch.int64) * (M + 1) + torch.arange(M), stable=True)
    ys, xs = torch.meshgrid(torch.arange(H), torch.arange(W), indexing="ij")
    px, py = xs.to(dt) + 0.5, ys.to(dt) + 0.5
    ptu, ptv = xs // 16, ys // 16
    T = torch.ones((H, W), dtype=dt)
    C = torch.zeros((H, W, 3), dtype=dt)
    stopped = torch.zeros((H, W), dtype=torch.bool)
    for m in order.tolist():
        member = (ptu >= min_tu[m]) & (ptu < max_tu[m]) & (ptv >= min_tv[m]) & (ptv < max_tv[m])
        if not bool(member.any()):
            continue
        dx, dy = px - uv[m, 0], py - uv[m, 1]
        alpha = torch.exp(-0.5 * (dx * dx * ca[m] + dy * dy * cc[m]) - dx * dy * cb[m]) * rescale[m] * opacity[m]
        active = member & ~stopped & (alpha.detach() >= 1.0 / 255.0)
        alpha_c = alpha + (torch.clamp(alpha, max=0.99) - alpha).detach()
        nT = T * (1 - alpha_c)
        stop_now = active & (nT.detach() < 1e-4)
        stopped = stopped | stop_now
        blend = active & ~stop_now
        C = C + torch.where(blend[..., None], color[m][None, None, :] * (alpha_c * T)[..., None], torch.zeros_like(C))
        T = torch.where(blend, nT, T)
    return C, ids


def _autograd_pose(sc, feats_after_forward, grad_image):
    """float64 autograd of the dense evaluator with (q, t) as the leaves: (grad q, grad t, grad xyz)."""
    H, W = sc.camera_info.camera_height, sc.camera_info.camera_width
    q = sc.q_pointcloud_camera.clone().double().requires_grad_(True)
    t = sc.t_pointcloud_camera.clone().double().requires_grad_(True)
    xyz = sc.point_cloud.clone().double().requires_grad_(True)
    feats = torch.from_numpy(feats_after_forward).double()
    q_cp, t_cp = inverse_SE3_qt_torch(q, t)
    if q.shape[0] == 1:
        image, aux = dense_render(xyz, feats, sc.point_invalid_mask, sc.camera_info.camera_intrinsics, q_cp, t_cp, H, W)
        ids = aux["ids"]
    else:
        image, ids = _render_objects(xyz, feats, sc.point_invalid_mask, sc.point_object_id, sc.camera_info.camera_intrinsics,
                                     q_cp, t_cp, H, W)
    (image * torch.from_numpy(grad_image).double()).sum().backward()
    return q.grad.numpy(), t.grad.numpy(), xyz.grad.numpy(), ids.numpy()


def _rel(got, exp):
    exp = np.asarray(exp, np.float64)
    return float(np.abs(np.asarray(got, np.float64) - exp).max() / max(np.abs(exp).max(), 1e-30))


@pytest.mark.parametrize("seed,band,n_obj,q_scale,skew", [
    (11, 3, 1, 1.0, 0.0),   # band 3
    (12, 0, 1, 1.0, 0.0),   # band 0
    (13, 3, 1, 1.03, 0.0),  # non-unit pose quaternion
    (14, 3, 1, 1.0, 4.5),   # skewed K
    (15, 3, 3, 1.0, 0.0),   # three objects, rows interleaved
])
def test_pose_gradients_match_float64_autograd(emu, emu_pose, seed, band, n_obj, q_scale, skew):
    sc = _scene(seed, n_obj=n_obj, q_scale=q_scale, skew=skew)
    st = emulated_forward(emu, sc, exact=True)
    assert st.M > 100
    H, W = st.pre.H, st.pre.W
    grad_image = np.random.default_rng(seed + 100).standard_normal((H, W, 3)).astype(np.float32)
    r = _backward(emu, emu_pose, st, grad_image, band=band)
    gq_ref, gt_ref, gx_ref, ids = _autograd_pose(sc, st.pre.feats, grad_image)
    assert sorted(ids.tolist()) == sorted(st.pre.point_id[:st.M].tolist())
    assert np.abs(gq_ref).max() > 0 and np.abs(gt_ref).max() > 0
    for o in range(n_obj):
        assert _rel(r["gq"][o], gq_ref[o]) < 1e-3, (o, r["gq"][o], gq_ref[o])
        assert _rel(r["gt"][o], gt_ref[o]) < 1e-3, (o, r["gt"][o], gt_ref[o])
    if q_scale == 1.0:  # unit q: grad t of an object = -(sum of its rows' xyz gradients)
        gx = r["out"][0].astype(np.float64)
        obj = sc.point_object_id.numpy()
        for o in range(n_obj):
            assert _rel(r["gt"][o], -gx[obj == o].sum(0)) < 1e-4


def test_empty_frame_gives_zeros(emu, emu_pose):
    sc = _scene(16, n_obj=2)
    sc.point_cloud[:, 2] = -5.0  # everything behind the camera
    st = emulated_forward(emu, sc, exact=True)
    assert st.M == 0
    r = _backward(emu, emu_pose, st, np.ones((st.pre.H, st.pre.W, 3), np.float32))
    assert (r["gq"] == 0).all() and (r["gt"] == 0).all()


def test_several_ctas_interleaved_objects_compact_dense_and_determinism(emu, emu_pose):
    sc = _scene(17, n=2000, n_obj=3)
    st = emulated_forward(emu, sc, exact=True)
    grad_image = np.random.default_rng(5).standard_normal((st.pre.H, st.pre.W, 3)).astype(np.float32)
    # 16 rows x 3 objects interleaved in every warp; 3 CTAs over 16 row-blocks: the grid-stride loop runs several rounds
    r = _backward(emu, emu_pose, st, grad_image, max_blocks=3)
    assert r["blocks"] == 3
    obj = sc.point_object_id.numpy()
    assert all(len(set(obj[k:k + 32].tolist())) == 3 for k in range(0, 2000 - 32, 32))
    # every CTA saw every object, and the partials add up to what the finalisation took
    assert (np.abs(r["partials"][:, :, 0:3]).sum(-1) > 0).all()
    gx = r["out"][0].astype(np.float64)
    for o in range(3):
        assert _rel(r["gt"][o], -gx[obj == o].sum(0)) < 1e-4
    gq_ref, gt_ref, _, _ = _autograd_pose(sc, st.pre.feats, grad_image)
    assert _rel(r["gq"], gq_ref) < 1e-3 and _rel(r["gt"], gt_ref) < 1e-3
    # COMPACT: the same pose outputs, bit for bit
    rc = _backward(emu, emu_pose, st, grad_image, max_blocks=3, compact=True)
    assert np.array_equal(rc["gq"], r["gq"]) and np.array_equal(rc["gt"], r["gt"])
    assert np.array_equal(rc["partials"], r["partials"])
    # the dense / compact outputs and the controller accumulators do not depend on the pose epilogue
    for compact in (False, True):
        with_pose = _backward(emu, emu_pose, st, grad_image, max_blocks=3, compact=compact)
        without = _backward(emu, emu_pose, st, grad_image, max_blocks=3, compact=compact, pose=False)
        for a, b in zip(with_pose["out"] + with_pose["ctl"], without["out"] + without["ctl"]):
            assert np.array_equal(a, b)
    # two runs: bit-identical
    r2 = _backward(emu, emu_pose, st, grad_image, max_blocks=3)
    assert np.array_equal(r2["gq"], r["gq"]) and np.array_equal(r2["gt"], r["gt"])


def _args(n_obj):
    a = _lib.GsbBackwardArgs(num_points=0, num_objects=n_obj)
    buf = (ctypes.c_float * 64)()
    p = ctypes.addressof(buf)
    pose = _lib.GsbPoseGradArgs(q_pointcloud_camera=p, t_pointcloud_camera=p, grad_q_pointcloud_camera=p,
                                grad_t_pointcloud_camera=p, temp=(p + 15) // 16 * 16,
                                temp_bytes=_lib.load().gsb200_pose_grad_temp_bytes(n_obj))
    return a, pose, buf


def test_backward_with_pose_rejects_bad_arguments():
    lib = _lib.load()
    assert lib.gsb200_pose_grad_temp_bytes(1) == 4096 * 12 * 4
    assert lib.gsb200_pose_grad_temp_bytes(16) == 16 * lib.gsb200_pose_grad_temp_bytes(1)
    call = lambda a, p: lib.gsb200_backward_with_pose(ctypes.byref(a) if a is not None else None,  # noqa: E731
                                                      ctypes.byref(p) if p is not None else None)
    a, p, _keep = _args(17)
    assert call(a, p) == -4  # GSB_EUNSUPPORTED: more objects than GSB_POSE_MAX_OBJECTS
    assert "at most 16" in lib.gsb200_last_error().decode()
    a, p, _keep = _args(2)
    assert call(None, p) == -1 and call(a, None) == -1
    for field in ("q_pointcloud_camera", "t_pointcloud_camera", "grad_q_pointcloud_camera", "grad_t_pointcloud_camera", "temp"):
        a, p, _keep = _args(2)
        setattr(p, field, None)
        assert call(a, p) == -1, field
    a, p, _keep = _args(2)
    p.temp_bytes -= 4
    assert call(a, p) == -1 and "temp must hold" in lib.gsb200_last_error().decode()
    a, p, _keep = _args(0)
    assert call(a, p) == -1
