"""Cost of the pose gradients (gsb200_backward_with_pose) at a full-size configuration.

    python scripts/bench_pose_grad.py [--config C3] [--rounds 3] [--steps 50] [--warmup 10] [--profile-steps 10]

One training-style step is forward + image.backward(g) with the point cloud and the features requiring grad (the default
operator: transposed loop A, no hook).  Variant "scene" leaves the pose alone (gsb200_backward); variant "pose" also
differentiates q_pointcloud_camera / t_pointcloud_camera (gsb200_backward_with_pose).  The two are timed alternately,
``--rounds`` times each, with CUDA events around ``--steps`` steps.  A separate torch.profiler run afterwards gives the
device time per call of the per-point kernel in both instantiations and of the finalisation kernel.  Prints the card's
name and power limit first.  Needs a CUDA device."""
import argparse
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from taichi_3d_gaussian_splatting_b200 import GaussianPointCloudRasterisation as GPCR  # noqa: E402
from taichi_3d_gaussian_splatting_b200.synthetic import CONFIGS, make_scene  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", default="C3")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--profile-steps", type=int, default=10)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_pose_grad.py needs a CUDA device")
    print(subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"], capture_output=True,
                         text=True).stdout.strip(), flush=True)

    sc = make_scene(**CONFIGS[args.config]).to("cuda")
    xyz = sc.point_cloud.requires_grad_(True)
    feats = sc.point_cloud_features.requires_grad_(True)
    op = GPCR(GPCR.GaussianPointCloudRasterisationConfig())
    g = torch.randn((sc.camera_info.camera_height, sc.camera_info.camera_width, 3),
                    generator=torch.Generator().manual_seed(5)).cuda()
    q_leaf = sc.q_pointcloud_camera.clone().requires_grad_(True)
    t_leaf = sc.t_pointcloud_camera.clone().requires_grad_(True)

    def step(pose):
        q, t = (q_leaf, t_leaf) if pose else (sc.q_pointcloud_camera, sc.t_pointcloud_camera)
        image, _, _ = op(GPCR.GaussianPointCloudRasterisationInput(
            point_cloud=xyz, point_cloud_features=feats, point_object_id=sc.point_object_id,
            point_invalid_mask=sc.point_invalid_mask, camera_info=sc.camera_info, q_pointcloud_camera=q,
            t_pointcloud_camera=t, color_max_sh_band=3))
        image.backward(g)
        xyz.grad = feats.grad = q_leaf.grad = t_leaf.grad = None

    def timed(pose, steps):
        start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        start.record()
        for _ in range(steps):
            step(pose)
        end.record()
        end.synchronize()
        return start.elapsed_time(end) / steps

    for pose in (False, True):
        timed(pose, args.warmup)
    res = {False: [], True: []}
    for r in range(args.rounds):
        for pose in (False, True):
            ms = timed(pose, args.steps)
            res[pose].append(ms)
            print(f"round {r} {'pose ' if pose else 'scene'}: {ms:.4f} ms/step (forward + backward, {args.steps} steps)",
                  flush=True)
    for pose in (False, True):
        v = sorted(res[pose])
        print(f"{'pose ' if pose else 'scene'}: median {v[len(v) // 2]:.4f} ms/step  min {v[0]:.4f}  max {v[-1]:.4f}")
    print(f"added by the pose gradients (median difference): {1000 * (sorted(res[True])[args.rounds // 2] - sorted(res[False])[args.rounds // 2]):.1f} us/step")

    # kernel times: a separate profiled run
    from torch.profiler import ProfilerActivity, profile
    for pose in (False, True):
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(args.profile_steps):
                step(pose)
            torch.cuda.synchronize()
        totals = {}
        for ev in prof.events():
            if ev.device_type == torch.autograd.DeviceType.CUDA and (
                    "backward_points_kernel" in ev.name or "pose_grad_finalize" in ev.name):
                tot, cnt = totals.get(ev.name, (0.0, 0))
                totals[ev.name] = (tot + ev.time_range.elapsed_us(), cnt + 1)
        for name, (tot, cnt) in sorted(totals.items()):
            print(f"profile {'pose ' if pose else 'scene'}: {name[:90]}  {tot / cnt:.1f} us/call  ({cnt} calls)")


if __name__ == "__main__":
    main()
