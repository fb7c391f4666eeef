"""-m gpu: gradients of the object poses through the public operator (``q_pointcloud_camera`` / ``t_pointcloud_camera`` with
``requires_grad``; ``gsb200_backward_with_pose``).

* small scenes (one and three objects, SH bands 0 and 3, a non-unit pose quaternion, a skewed K) against float64 torch
  autograd of the dense evaluator, on both arithmetic paths, within the gradient tolerance of the parity tests (1e-3 of
  the largest entry);
* at the full C2 / C3 sizes, with a unit pose quaternion: grad t = -(float64 sum of grad_pointcloud over the object's rows);
* a pose-only backward (scene frozen) calls no hook and returns no scene gradients;
* the scene gradients and hook tensors do not change when pose gradients are requested as well, and repeated backwards
  agree -- up to the float-atomic ordering of loop A, which already separates two backwards without pose gradients (the
  pose reduction itself is fixed-order: bit-identity is pinned on the kernel sources by test_simt_pose_gradients_cpu.py);
* a pose-recovery run: Adam on (q, t) alone brings a perturbed camera back to the pose the target was rendered at.
"""
import json
import math
import os

import numpy as np
import pytest
import torch

from taichi_3d_gaussian_splatting_b200.synthetic import CONFIGS, make_scene

from gpu_helpers import Input, make_op, n
from test_simt_pose_gradients_cpu import _autograd_pose, _rel, _scene

pytestmark = pytest.mark.gpu

# measured values (translation identity errors, repeatability, the pose-recovery trajectory) are written as JSON to
# $GSB200_TEST_RECORD_DIR/pose_gradients.json when that variable is set
RECORD_DIR = os.environ.get("GSB200_TEST_RECORD_DIR")


def _record(key, entry):
    if not RECORD_DIR:
        return
    os.makedirs(RECORD_DIR, exist_ok=True)
    RECORD = os.path.join(RECORD_DIR, "pose_gradients.json")
    data = {}
    if os.path.exists(RECORD):
        with open(RECORD) as f:
            data = json.load(f)
    data[key] = entry
    with open(RECORD, "w") as f:
        json.dump(data, f, indent=1, sort_keys=True)


def _inputs(sc, q, t, band=3):
    return Input(point_cloud=sc.point_cloud, point_cloud_features=sc.point_cloud_features, point_object_id=sc.point_object_id,
                 point_invalid_mask=sc.point_invalid_mask, camera_info=sc.camera_info, q_pointcloud_camera=q,
                 t_pointcloud_camera=t, color_max_sh_band=band)


def _pose_leaves(sc):
    return (sc.q_pointcloud_camera.clone().requires_grad_(True), sc.t_pointcloud_camera.clone().requires_grad_(True))


@pytest.mark.parametrize("exact", [False, True])
@pytest.mark.parametrize("seed,band,n_obj,q_scale,skew", [
    (11, 3, 1, 1.0, 0.0), (12, 0, 1, 1.0, 0.0), (13, 3, 1, 1.03, 0.0), (14, 3, 1, 1.0, 4.5), (15, 3, 3, 1.0, 0.0)])
def test_pose_gradients_match_float64_autograd(seed, band, n_obj, q_scale, skew, exact):
    scene = _scene(seed, n_obj=n_obj, q_scale=q_scale, skew=skew)
    sc = scene.to("cuda")
    q, t = _pose_leaves(sc)
    op = make_op(exact_exp=exact)
    image, _, _ = op(_inputs(sc, q, t, band))
    H, W = image.shape[:2]
    grad_image = np.random.default_rng(seed + 100).standard_normal((H, W, 3)).astype(np.float32)
    image.backward(torch.from_numpy(grad_image).cuda())
    scene.point_cloud_features = sc.point_cloud_features.cpu()  # q of the in-frustum rows normalised by the forward
    gq_ref, gt_ref, _, _ = _autograd_pose(scene, n(sc.point_cloud_features), grad_image)
    assert q.grad.shape == q.shape and t.grad.shape == t.shape
    for o in range(n_obj):
        assert _rel(n(q.grad)[o], gq_ref[o]) < 1e-3, (o, n(q.grad)[o], gq_ref[o])
        assert _rel(n(t.grad)[o], gt_ref[o]) < 1e-3, (o, n(t.grad)[o], gt_ref[o])


@pytest.mark.parametrize("name", ["C2", "C3"])
def test_translation_gradient_is_minus_the_sum_of_xyz_gradients_full_size(name):
    sc = make_scene(**CONFIGS[name]).to("cuda")
    assert float((sc.q_pointcloud_camera.norm(dim=-1) - 1).abs().max()) < 1e-6
    sc.point_cloud.requires_grad_(True)
    sc.point_cloud_features.requires_grad_(True)
    q, t = _pose_leaves(sc)
    image, _, _ = make_op()(_inputs(sc, q, t))
    g = torch.Generator().manual_seed(5)
    image.backward(torch.randn(image.shape, generator=g).cuda())
    gx = sc.point_cloud.grad.double()
    expected = -gx.sum(0)
    scale = gx.abs().sum(0)  # f32 sums in another order: error bounded by a small multiple of eps * sum |terms|
    err = (t.grad[0].double() - expected).abs()
    _record(f"translation_identity_{name}", dict(grad_t=n(t.grad[0]).tolist(), expected=n(expected).tolist(),
                                                 err_over_l1=n(err / scale).tolist()))
    assert bool((err <= 2e-5 * scale).all()), (n(t.grad[0]), n(expected), n(err / scale))
    assert bool(torch.isfinite(q.grad).all()) and float(q.grad.abs().max()) > 0


def test_pose_only_backward_calls_no_hook_and_returns_no_scene_gradients():
    calls = []
    scene = _scene(15, n_obj=3)
    sc = scene.to("cuda")
    q, t = _pose_leaves(sc)
    op = make_op(hook=calls.append)
    image, _, _ = op(_inputs(sc, q, t))
    image.sum().backward()
    assert calls == [] and sc.point_cloud.grad is None and sc.point_cloud_features.grad is None
    gq, gt = q.grad.clone(), t.grad.clone()
    assert float(gq.abs().max()) > 0 and float(gt.abs().max()) > 0
    # the same pose gradients when the scene is trained too (then the hook runs)
    sc2 = scene.to("cuda")
    sc2.point_cloud.requires_grad_(True)
    q2, t2 = _pose_leaves(sc2)
    image2, _, _ = op(_inputs(sc2, q2, t2))
    image2.sum().backward()
    assert len(calls) == 1 and sc2.point_cloud.grad is not None
    assert _rel(n(q2.grad), n(gq)) < 1e-5 and _rel(n(t2.grad), n(gt)) < 1e-5


def _close_to_noise(a, b, noise):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.abs(a - b).max()) <= max(2 * noise, 1e-6 * max(np.abs(b).max(), 1e-30))


def test_scene_gradients_and_hook_unchanged_and_repeatable():
    hooks = []
    scene = _scene(17, n=2000, n_obj=3)
    sc = scene.to("cuda")
    sc.point_cloud.requires_grad_(True)
    sc.point_cloud_features.requires_grad_(True)
    q, t = sc.q_pointcloud_camera.clone(), sc.t_pointcloud_camera.clone()
    op = make_op(hook=hooks.append)
    image, _, _ = op(_inputs(sc, q, t))
    g = torch.randn(image.shape, generator=torch.Generator().manual_seed(3)).cuda()
    outs = []
    for with_pose in (False, False, True, True):
        xyz = sc.point_cloud.detach().clone().requires_grad_(True)
        feats = sc.point_cloud_features.detach().clone().requires_grad_(True)
        qq, tt = q.clone().requires_grad_(with_pose), t.clone().requires_grad_(with_pose)
        image, _, _ = op(Input(point_cloud=xyz, point_cloud_features=feats, point_object_id=sc.point_object_id,
                               point_invalid_mask=sc.point_invalid_mask, camera_info=sc.camera_info,
                               q_pointcloud_camera=qq, t_pointcloud_camera=tt, color_max_sh_band=3))
        image.backward(g)
        h = hooks[-1]
        outs.append(dict(gx=n(xyz.grad), gf=n(feats.grad), ids=n(h.point_id_in_camera_list), hx=n(h.grad_point_in_camera),
                         hf=n(h.grad_pointfeatures_in_camera), vs=n(h.grad_viewspace), mag=n(h.magnitude_grad_viewspace),
                         img=n(h.magnitude_grad_viewspace_on_image), npix=n(h.num_affected_pixels),
                         gq=n(qq.grad) if with_pose else None, gt=n(tt.grad) if with_pose else None))
    a, b, c, d = outs
    assert np.array_equal(a["ids"], c["ids"]) and np.array_equal(a["npix"], c["npix"])
    for k in ("gx", "gf", "hx", "hf", "vs", "mag", "img"):
        noise = float(np.abs(a[k].astype(np.float64) - b[k]).max())
        assert _close_to_noise(c[k], a[k], noise), k
    assert _rel(d["gq"], c["gq"]) < 1e-5 and _rel(d["gt"], c["gt"]) < 1e-5
    _record("repeatability", dict(pose_q_rel=_rel(d["gq"], c["gq"]), pose_t_rel=_rel(d["gt"], c["gt"]),
                                  gx_noise=float(np.abs(a["gx"].astype(np.float64) - b["gx"]).max())))


def _angle_deg(q, q_ref):
    q, q_ref = q / q.norm(), q_ref / q_ref.norm()
    return math.degrees(2 * math.acos(min(1.0, abs(float((q * q_ref).sum())))))


def test_pose_recovery_with_adam():
    sc = make_scene(**CONFIGS["C1"]).to("cuda")
    q_true, t_true = sc.q_pointcloud_camera.clone(), sc.t_pointcloud_camera.clone()
    op = make_op()
    with torch.no_grad():
        target, _, _ = op(_inputs(sc, q_true, t_true))
    axis = torch.tensor([0.3, 0.8, -0.5], device="cuda")
    axis = axis / axis.norm()
    half = math.radians(2.0) / 2
    dq = torch.cat([axis * math.sin(half), torch.tensor([math.cos(half)], device="cuda")])
    x0, y0, z0, w0 = dq.unbind()
    x1, y1, z1, w1 = q_true[0].unbind()
    q0 = torch.stack([w0 * x1 + x0 * w1 + y0 * z1 - z0 * y1, w0 * y1 - x0 * z1 + y0 * w1 + z0 * x1,
                      w0 * z1 + x0 * y1 - y0 * x1 + z0 * w1, w0 * w1 - x0 * x1 - y0 * y1 - z0 * z1])[None]
    depth = float(sc.point_cloud[:, 2].median())
    t0 = t_true + torch.tensor([[0.02, -0.015, 0.03]], device="cuda") * depth
    q = q0.clone().requires_grad_(True)
    t = t0.clone().requires_grad_(True)
    opt = torch.optim.Adam([q, t], lr=2e-3)
    start = (_angle_deg(q0[0], q_true[0]), float((t0 - t_true).norm()))
    history = []
    for step in range(300):
        opt.zero_grad()
        image, _, _ = op(_inputs(sc, q, t, band=0))
        loss = (image - target).abs().mean()
        loss.backward()
        opt.step()
        if step % 25 == 0 or step == 299:
            history.append((step, float(loss), _angle_deg(q.detach()[0], q_true[0]), float((t.detach() - t_true).norm())))
    end = (_angle_deg(q.detach()[0], q_true[0]), float((t.detach() - t_true).norm()))
    _record("pose_recovery", dict(start_deg=start[0], start_t=start[1], end_deg=end[0], end_t=end[1], depth=depth,
                                  history=history, device=torch.cuda.get_device_name()))
    assert end[0] < 0.5 * start[0] and end[1] < 0.5 * start[1], (start, end, history)
