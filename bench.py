#!/usr/bin/env python
"""bench.py -- headline benchmark of the rasteriser hot path (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W [--impl b200|reference] [--dump-outputs DIR]
    (N > 1: launched by torch.distributed.run, one rank per GPU)

A "step" is one pass of the hot path over one view: forward (GaussianPointCloudRasterisation,
full outputs) + backward (dense per-Gaussian gradients) at 1920x1072 with 1e6 Gaussians, SH deg 3
(SURVEY.md §8(d) config C3 = the configuration BASELINE.json's metric is quoted on).  With N ranks
every rank renders its own view of the replicated scene (view-parallel, weak scaling) and the per-Gaussian
gradients are summed over the ranks inside the operator's backward by the compact exchange of parallel.py
(all-reduce of 11 + all-gather of 3 floats per Gaussian instead of an all-reduce of 59, then
gsb200_expand_view_gradients).  At N = 8 the line also carries BASELINE config 4 (2.1e6 Gaussians, 8 views).

Output: ONE JSON line on rank 0 (see the task contract): metric/value/unit, ms_per_step, e2e (host
buffers in, loss scalar out, copies inside the timed region), roofline of the dominant kernel,
cpu_baseline (the CPU oracle on the host cores), clocks sampled during the timed region.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "rendered Mpix/sec fwd+bwd @1080p, 1e6 Gaussians"
UNIT = "Mpix/s"
WORKLOAD = "C3"


def workload_string(name):
    """The SAME text in both arms' config.workload (the driver compares the two strings)."""
    from taichi_3d_gaussian_splatting_b200.synthetic import CONFIGS
    c = CONFIGS[name]
    return (f"{name}: N={c['num_points']} Gaussians, {c['width']}x{c['height']}, SH deg {c['sh_degree']}, sigma_med {c['sigma_med']}, "
            f"seed {c['seed']}, fwd+bwd, 1 view per GPU per step")


def percentiles(ms_list):
    xs = sorted(ms_list)
    pick = lambda q: xs[min(len(xs) - 1, max(0, int(round(q * (len(xs) - 1)))))]  # noqa: E731
    return {"n": len(xs), "median_ms_per_step": round(statistics.median(xs), 4), "p10_ms_per_step": round(pick(0.1), 4),
            "p90_ms_per_step": round(pick(0.9), 4)}


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default=WORKLOAD)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--repeats", type=int, default=0,
                    help="extra timed regions of --steps steps each after the first; the headline is the median region")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step returned as DIR/<name>.npy (float32): image, "
                         "depth, valid point count and the gradient rows of a fixed, seeded sample of Gaussians")
    ap.add_argument("--exchange-streams", type=int, default=1, choices=[1, 2],
                    help="N > 1: 2 = the all-gather of the compact exchange on a second NCCL communicator, concurrent with the all-reduce")
    ap.add_argument("--exchange", default="auto", choices=["auto", "multimem", "nccl"],
                    help="N > 1: collectives of the compact exchange: multimem = the hand-written NVLS kernel (gsb200_exchange_multimem), "
                         "nccl = ncclAllReduce + ncclAllGather, auto = multimem where the group has multicast support, else nccl")
    ap.add_argument("--exchange-blocks", type=int, default=0, help="CTAs of the multimem exchange kernel (0 = two per SM)")
    ap.add_argument("--overlap-expansion-nccl", action="store_true",
                    help="NCCL exchange: gather first and expand the SH columns beside the all-reduce (measured slower at 2 ranks)")
    ap.add_argument("--overlap-expansion", action="store_true",
                    help="multimem exchange: expand the SH columns on a second stream while the all-reduce is on the wire instead of "
                         "one expansion pass behind it (measured slower at 8 GPUs: 1.809 vs 1.797 ms per step)")
    ap.add_argument("--serial-expansion", action="store_true", help="(default behaviour; kept so that older call scripts still parse)")
    ap.add_argument("--dense-exchange", action="store_true",
                    help="N > 1: one all-reduce of the dense gradients instead of the compact exchange (comparison)")
    return ap.parse_args()


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            d = json.load(f)
        return float(d.get("hbm_gbs", 6650.0)), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


# --------------------------------------------------------------------------- clocks
class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.rows = []
        self.proc = None
        self.thread = None
        self.gpu_index = gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits", "-lms", "50",
                 "-i", str(self.gpu_index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None
            return
        self.thread = threading.Thread(target=self._read, daemon=True)
        self.thread.start()

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            parts = [p.strip() for p in r.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0]))
                mx.append(float(parts[1]))
            except ValueError:
                continue
            for nme, val in zip(names, parts[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(nme)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# --------------------------------------------------------------------------- reference arm (CPU)
def oracle_step(scene, band=3):
    """One forward+backward of the CPU oracle (reference arithmetic restated in C, OpenMP)."""
    import numpy as np
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from helpers import oracle_backward, oracle_forward
    o, fwd, feats = oracle_forward(scene)
    g = np.ones(fwd.image.shape, np.float32)
    bwd = oracle_backward(o, fwd, scene, feats, g, band)
    return fwd, bwd


def pin_cpu_threads():
    """One OpenMP thread per PHYSICAL core, bound (the CPU arm varied 4x between boxes with unbound threads on all logical
    CPUs).  Must run before the oracle's OpenMP runtime starts."""
    try:
        import psutil
        physical = psutil.cpu_count(logical=False) or os.cpu_count()
    except Exception:  # pragma: no cover
        physical = os.cpu_count()
    os.environ.setdefault("OMP_PROC_BIND", "spread")
    os.environ.setdefault("OMP_PLACES", "cores")
    os.environ["OMP_NUM_THREADS"] = str(physical)
    return physical


def run_reference(args):
    """--impl reference: the reference's algorithm for this path on the HOST cores.  Taichi (the
    reference's only backend) is not installable in this image, so this is the oracle port
    (oracle/gs_oracle.c, OpenMP on all host cores), kind = "port"."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = pin_cpu_threads()
    from oracle import gs_oracle
    from taichi_3d_gaussian_splatting_b200.synthetic import CONFIGS, make_scene
    gs_oracle.set_num_threads(threads)
    cfg = CONFIGS[args.workload]
    scene = make_scene(**cfg)
    H, W = cfg["height"], cfg["width"]
    for _ in range(max(args.warmup, 0)):
        oracle_step(scene)
    per_step = []
    for _ in range(args.steps):
        t0 = time.perf_counter()
        fwd, bwd = oracle_step(scene)
        per_step.append((time.perf_counter() - t0) * 1e3)
    if args.dump_outputs:
        import torch
        dump_outputs(args.dump_outputs, *(torch.from_numpy(a) for a in (
            fwd.image, fwd.depth, fwd.pixel_valid_point_count, bwd.grad_pointcloud, bwd.grad_pointcloud_features)))
    dt = sum(per_step) / 1e3
    value = H * W * args.steps / dt / 1e6
    cores = gs_oracle.num_threads()
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "impl": "reference",
        "config": {"workload": workload_string(args.workload),
                   "threads": f"{cores} OpenMP threads, OMP_PROC_BIND={os.environ.get('OMP_PROC_BIND')} OMP_PLACES={os.environ.get('OMP_PLACES')} "
                              f"(one thread per physical core of the box: {os.cpu_count()} logical CPUs)"},
        "spread": percentiles(per_step),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": f"full {args.workload} frames, fwd+bwd, {args.steps} steps"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------- B200 arm
SM_CLOCK_HZ, NUM_SMS = 1.965e9, 148
ISSUE_PEAK = NUM_SMS * 4 * SM_CLOCK_HZ          # warp instructions / s (one per SMSP per cycle)
FP32_LANE_PEAK = NUM_SMS * 128 * SM_CLOCK_HZ    # FP32 lane operations / s (an FMA counts once)
MUFU_LANE_PEAK = NUM_SMS * 16 * SM_CLOCK_HZ     # MUFU (ex2 / rcp) lane operations / s
# SASS instructions per (warp, splat) visit of the inner loops (cuobjdump of this build, DESIGN section 3)
FWD_INSTR_PER_VISIT, BWD_INSTR_PER_VISIT = 29, 30 + 34
DUMP_BYTES = 60_000_000  # array data of --dump-outputs: the files stay under 64 MB with their headers


def dump_outputs(out_dir, image, depth, count, grad_xyz, grad_features):
    """Write one step's outputs as float32 .npy files so that two builds can be compared output for output.  The per-pixel
    outputs are written whole; the dense gradients of 1e6 Gaussians (236 MB) do not fit the budget, so the rows of a fixed,
    seeded sample of Gaussians (the same for the same workload) fill what the pixels leave of it."""
    import numpy as np
    import torch
    pixel_bytes = 4 * (image.numel() + depth.numel() + count.numel())
    n = grad_xyz.shape[0]
    num_rows = min(n, (DUMP_BYTES - pixel_bytes) // (4 * (grad_xyz.shape[1] + grad_features.shape[1])))
    rows = np.sort(np.random.default_rng(0).choice(n, num_rows, replace=False))
    idx = torch.from_numpy(rows).to(grad_xyz.device)
    os.makedirs(out_dir, exist_ok=True)
    for name, t in (("image", image), ("depth", depth), ("pixel_valid_point_count", count),
                    ("grad_pointcloud_sampled_rows", grad_xyz[idx]), ("grad_pointcloud_features_sampled_rows", grad_features[idx])):
        np.save(os.path.join(out_dir, name + ".npy"), t.detach().to(torch.float32).cpu().numpy())


def run_b200(args):
    import torch
    import torch.distributed as dist
    from taichi_3d_gaussian_splatting_b200 import CameraInfo
    from taichi_3d_gaussian_splatting_b200 import GaussianPointCloudRasterisation as GPCR
    from taichi_3d_gaussian_splatting_b200 import fused_l1_loss_with_grad, profiling
    from taichi_3d_gaussian_splatting_b200.parallel import (MulticastViewParallelExchange, ViewParallelExchange,
                                                          exchange_gradients)
    from taichi_3d_gaussian_splatting_b200.synthetic import C4_YAWS, CONFIGS, make_scene

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py --impl b200 needs a CUDA device (no CPU fallback exists)")
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=device)
    warmup = max(args.warmup, 3)
    steps = args.steps
    Input = GPCR.GaussianPointCloudRasterisationInput
    exchange, exchange_kind = None, "dense all-reduce"
    if world > 1 and not args.dense_exchange:
        # measured (profiles/r02_bench_n*_{multimem,nccl}.json): at 2 ranks the NCCL collectives win (1.69 vs 1.73 ms per step: two
        # barriers + two launches outweigh 60 MB of wire time), from 4 ranks on the hand-written NVLS kernel does (8 ranks: 1.90 vs 2.00)
        if args.exchange == "multimem" or (args.exchange == "auto" and world >= 4):
            try:
                exchange = MulticastViewParallelExchange(num_blocks=args.exchange_blocks, overlap_expansion=args.overlap_expansion and not args.serial_expansion)
                exchange.allocate(CONFIGS[args.workload]["num_points"], 1, device)  # the rendezvous is a collective: do it up front
                exchange_kind = "multimem"
            except Exception as e:  # no multicast support (or no symmetric-memory backend) on this box
                if args.exchange == "multimem":
                    raise
                exchange = None
                if rank == 0:
                    print(f"[bench] multicast exchange unavailable ({type(e).__name__}: {e}); using the NCCL collectives", file=sys.stderr)
        if exchange is None:
            exchange = ViewParallelExchange(gather_group=dist.new_group() if args.exchange_streams == 2 else None,
                                            overlap_expansion=args.overlap_expansion_nccl and not args.serial_expansion)
            exchange_kind = "nccl"

    def barrier():
        if world > 1:
            dist.barrier()

    def timed(fn, k, rewarm=2):
        """k calls of fn between barrier + synchronize on both sides, CUDA events on the launching stream, MAX over ranks.
        `rewarm` untimed calls run immediately before the region: rank 0 has just started the clock sampler / printed, the
        other ranks have been spinning in a barrier -- the first timed step must not pay for that (observed at 8 GPUs:
        a first region of 2.7 ms per step against a median of 1.9 ms without it)."""
        for _ in range(rewarm):
            fn()
        barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(k):
            fn()
        e1.record()
        torch.cuda.synchronize()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=device)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    class Workload:
        """One configuration resident on this rank: scene replica, this rank's view, the operator, a fixed dL/dimage."""

        def __init__(self, name):
            self.name = name
            self.cfg = dict(CONFIGS[name])
            self.H, self.W, self.N = self.cfg["height"], self.cfg["width"], self.cfg["num_points"]
            self.scene = make_scene(**self.cfg, yaw_degrees=C4_YAWS[rank % len(C4_YAWS)]).to(device)
            self.scene.point_cloud.requires_grad_(True)
            self.scene.point_cloud_features.requires_grad_(True)
            self.op = GPCR(GPCR.GaussianPointCloudRasterisationConfig(), gradient_exchange=exchange)
            g = torch.Generator(device="cpu").manual_seed(1234 + rank)
            self.grad_image = torch.randn((self.H, self.W, 3), generator=g, dtype=torch.float32).to(device)
            sc = self.scene
            self.dev_input = self.make_input(sc.q_pointcloud_camera, sc.t_pointcloud_camera, sc.camera_info.camera_intrinsics)

        def make_input(self, q, t, K):
            sc = self.scene
            return Input(point_cloud=sc.point_cloud, point_cloud_features=sc.point_cloud_features,
                         point_object_id=sc.point_object_id, point_invalid_mask=sc.point_invalid_mask,
                         camera_info=CameraInfo(K, self.H, self.W, 0), q_pointcloud_camera=q, t_pointcloud_camera=t,
                         color_max_sh_band=3)

        def finish_step(self):
            if world > 1 and exchange is None:  # --dense-exchange: one all-reduce of the dense (N,3)+(N,56) buffer
                exchange_gradients([self.scene.point_cloud.grad, self.scene.point_cloud_features.grad],
                                   fused_buffer=self.op.last_gradient_buffer)

        def step(self):
            sc = self.scene
            sc.point_cloud.grad = None
            sc.point_cloud_features.grad = None
            self.outputs = self.op(self.dev_input)  # (image, depth, valid point count): kept for --dump-outputs
            self.outputs[0].backward(self.grad_image)  # N > 1: the gradient exchange over NVLink happens inside this backward
            self.finish_step()

        def mpix(self, ms_per_step):
            return world * self.H * self.W / (ms_per_step * 1e-3) / 1e6

    wl = Workload(args.workload)
    H, W, N, cfg, op, scene = wl.H, wl.W, wl.N, wl.cfg, wl.op, wl.scene

    # ---- headline: inputs resident in HBM; one timed region of exactly `steps` steps, then `repeats` (default 0) more
    #      regions of the same length
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    for _ in range(warmup):
        wl.step()
    # the headline is the MEDIAN region (BASELINE.md's protocol: median with p10 / p90 beside it, which takes --repeats), the
    # first region is reported as well.  No event between the steps: one after every step costs 3-5 us per step (B200, 1000 W).
    regions = [timed(wl.step, steps) / steps for _ in range(1 + max(args.repeats, 0))]
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, *wl.outputs, scene.point_cloud.grad, scene.point_cloud_features.grad)
    first_region_ms = regions[0]
    ms_per_step = statistics.median(regions)
    value = wl.mpix(ms_per_step)
    frame = op.last_frame
    M, Kk = frame.num_points_in_camera, frame.num_keys
    K_ref = int(frame.num_overlap_tiles.sum())  # pairs of the reference's 3-sigma squares (before the reach filter)

    # ---- N > 1: the exchanged gradient against a dense all-reduce of the same step (untimed self-check)
    exchange_check = None
    if world > 1 and exchange is not None:
        wl.step()
        got_x, got_f = scene.point_cloud.grad.clone(), scene.point_cloud_features.grad.clone()
        dense_op = GPCR(GPCR.GaussianPointCloudRasterisationConfig())
        scene.point_cloud.grad = None
        scene.point_cloud_features.grad = None
        image, _, _ = dense_op(wl.dev_input)
        image.backward(wl.grad_image)
        exchange_gradients([scene.point_cloud.grad, scene.point_cloud_features.grad], fused_buffer=dense_op.last_gradient_buffer)
        ref_x, ref_f = scene.point_cloud.grad.clone(), scene.point_cloud_features.grad.clone()
        # the same dense step once more: the run-to-run noise of loop A's float atomics (the yardstick for the error above)
        scene.point_cloud.grad = None
        scene.point_cloud_features.grad = None
        image, _, _ = dense_op(wl.dev_input)
        image.backward(wl.grad_image)
        exchange_gradients([scene.point_cloud.grad, scene.point_cloud_features.grad], fused_buffer=dense_op.last_gradient_buffer)
        ag_x, ag_f = scene.point_cloud.grad, scene.point_cloud_features.grad
        err = torch.stack([(got_x - ref_x).abs().max() / ref_x.abs().max(), (got_f - ref_f).abs().max() / ref_f.abs().max(),
                           (ag_x - ref_x).abs().max() / ref_x.abs().max(), (ag_f - ref_f).abs().max() / ref_f.abs().max()])
        dist.all_reduce(err, op=dist.ReduceOp.MAX)
        exchange_check = {"max_abs_err_over_max_abs_grad_xyz": float(err[0]), "max_abs_err_over_max_abs_grad_features": float(err[1]),
                          "dense_rerun_noise_xyz": float(err[2]), "dense_rerun_noise_features": float(err[3]),
                          "what": "compact exchange vs one NCCL all-reduce of the dense gradients of another run of the same step, max "
                                  "over ranks; *_noise = two runs of the DENSE path against each other (float atomics of loop A land in "
                                  "a different order every run)"}
        # and the dense exchange timed the same way, for the comparison in the line
        def dense_step():
            scene.point_cloud.grad = None
            scene.point_cloud_features.grad = None
            im, _, _ = dense_op(wl.dev_input)
            im.backward(wl.grad_image)
            exchange_gradients([scene.point_cloud.grad, scene.point_cloud_features.grad], fused_buffer=dense_op.last_gradient_buffer)
        for _ in range(3):
            dense_step()
        dense_ms = timed(dense_step, steps) / steps
        exchange_check["dense_all_reduce_ms_per_step"] = round(dense_ms, 4)
        exchange_check["dense_all_reduce_Mpix_s"] = round(wl.mpix(dense_ms), 2)
        # the collectives of the compact exchange alone (no compute in front: every rank arrives at the same time), and this
        # rank's own fwd+bwd without any exchange -- what the exchange adds to a step is the difference to `ms_per_step`
        gs, bl = exchange.allocate(N, 1, device)
        def collectives_alone():
            exchange.rows_written(gs, bl)  # (the multicast variant pushes its block here, the NCCL variant gathers inside run)
            exchange.run(gs, bl)
        for _ in range(3):
            collectives_alone()
        exchange_check["compact_collectives_alone_ms"] = round(timed(collectives_alone, 20) / 20, 4)
        exchange_check["compact_payload_MB_per_rank"] = {"summed": round(48 * N / 1e6, 1), "gathered_from_each_rank": round(12 * N / 1e6, 1)}

        def local_step():
            scene.point_cloud.grad = None
            scene.point_cloud_features.grad = None
            im, _, _ = dense_op(wl.dev_input)
            im.backward(wl.grad_image)
        for _ in range(3):
            local_step()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            local_step()
        e1.record()
        torch.cuda.synchronize()
        mine = torch.tensor([e0.elapsed_time(e1) / steps], dtype=torch.float64, device=device)
        every = [torch.zeros_like(mine) for _ in range(world)]
        dist.all_gather(every, mine)
        exchange_check["fwd_bwd_without_exchange_ms_per_rank"] = [round(float(x), 4) for x in every]

    # ---- e2e: per-step inputs in pinned HOST memory (target image, pose, intrinsics), loss scalar back
    target_host = torch.rand((H, W, 3), dtype=torch.float32).pin_memory()
    q_host = scene.q_pointcloud_camera.detach().cpu().pin_memory()
    t_host = scene.t_pointcloud_camera.detach().cpu().pin_memory()
    K_host = scene.camera_info.camera_intrinsics.detach().cpu().pin_memory()
    h2d = target_host.numel() * 4 + q_host.numel() * 4 + t_host.numel() * 4 + K_host.numel() * 4

    # The step's host inputs are uploaded on a copy stream into double-buffered device slots, one step
    # ahead (what a DataLoader with pin_memory + non_blocking does); every step's copy is issued and
    # completed inside the timed region.
    copy_stream = torch.cuda.Stream(device=device)
    slots = [dict(target=torch.empty((H, W, 3), dtype=torch.float32, device=device),
                  q=torch.empty_like(scene.q_pointcloud_camera), t=torch.empty_like(scene.t_pointcloud_camera),
                  K=torch.empty((3, 3), dtype=torch.float32, device=device), pose_ready=torch.cuda.Event(),
                  ready=torch.cuda.Event())
             for _ in range(2)]

    def upload(slot):
        # pose and intrinsics (64 bytes) first: the forward needs only them; the 24.7 MB target image is needed by the loss,
        # so the forward of a step waits for `pose_ready` and only the loss kernel waits for `ready`
        with torch.cuda.stream(copy_stream):
            slot["q"].copy_(q_host, non_blocking=True)
            slot["t"].copy_(t_host, non_blocking=True)
            slot["K"].copy_(K_host, non_blocking=True)
            slot["pose_ready"].record(copy_stream)
            slot["target"].copy_(target_host, non_blocking=True)
            slot["ready"].record(copy_stream)

    # The step's loss goes to pinned host memory with an async copy and is read one step later (what a
    # training loop that logs its loss does); every step's loss is read inside the timed region.
    loss_host = [torch.zeros((), dtype=torch.float32).pin_memory() for _ in range(2)]
    loss_done = [torch.cuda.Event() for _ in range(2)]
    e2e_losses = []

    def run_e2e(k):
        e2e_losses.clear()
        upload(slots[0])
        for i in range(k):
            slot = slots[i % 2]
            torch.cuda.current_stream().wait_event(slot["pose_ready"])
            scene.point_cloud.grad = None
            scene.point_cloud_features.grad = None
            image, _, _ = op(wl.make_input(slot["q"], slot["t"], slot["K"]))
            # fused L1 loss + gradient (gsb200_l1_loss), then the operator's backward
            torch.cuda.current_stream().wait_event(slot["ready"])  # the target image of this step has arrived
            loss, grad = fused_l1_loss_with_grad(image, slot["target"])
            image.backward(grad)
            wl.finish_step()
            loss_host[i % 2].copy_(loss, non_blocking=True)
            loss_done[i % 2].record()
            if i > 0:  # D2H read of the previous step's result; also frees its input slot for the next upload
                loss_done[(i - 1) % 2].synchronize()
                e2e_losses.append(float(loss_host[(i - 1) % 2]))
            if i + 1 < k:
                upload(slots[(i + 1) % 2])  # overlaps with this step's compute
        loss_done[(k - 1) % 2].synchronize()
        e2e_losses.append(float(loss_host[(k - 1) % 2]))

    run_e2e(3)
    e2e_regions = [timed(lambda: run_e2e(steps), 1, rewarm=0) / steps for _ in range(1 + max(args.repeats, 0))]
    e2e_ms = statistics.median(e2e_regions)
    e2e_value = wl.mpix(e2e_ms)

    # ---- forward-only numbers (inference: torch.no_grad, full outputs and rgb_only)
    def fwd_only(o):
        def f():
            with torch.no_grad():
                o(wl.dev_input)
        return f
    op_rgb = GPCR(GPCR.GaussianPointCloudRasterisationConfig(rgb_only=True))
    for f in (fwd_only(op), fwd_only(op_rgb)):
        for _ in range(3):
            f()
    fwd_ms = timed(fwd_only(op), steps) / steps
    fwd_rgb_ms = timed(fwd_only(op_rgb), steps) / steps

    # inference THROUGHPUT with two frames in flight (parallel.render_views(..., streams=...)): consecutive frames on
    # alternating streams, so the latency-bound per-point stage and sort of frame i+1 run under the blend of frame i
    from taichi_3d_gaussian_splatting_b200.parallel import render_views
    side_streams = [torch.cuda.Stream(device=device) for _ in range(2)]

    def frames_in_flight(o, k):
        main = torch.cuda.current_stream(device)
        start = torch.cuda.Event()
        start.record(main)
        for st in side_streams:
            st.wait_event(start)
        render_views(o, lambda i: wl.dev_input, range(k), streams=side_streams)
        for st in side_streams:
            done = torch.cuda.Event()
            done.record(st)
            main.wait_event(done)
    frames_in_flight(op_rgb, 4)
    frames_in_flight(op, 4)
    fwd2_ms = timed(lambda: frames_in_flight(op, steps), 1, rewarm=0) / steps
    fwd2_rgb_ms = timed(lambda: frames_in_flight(op_rgb, steps), 1, rewarm=0) / steps

    # ---- inference e2e through the C ABI with HOST buffers (gsb200_render_host): pose + intrinsics H2D,
    #      forward (rgb_only), image D2H into pinned memory, every frame
    def render_host_e2e(k):
        import ctypes
        from taichi_3d_gaussian_splatting_b200 import _lib
        lib = _lib.load()
        fr = op_rgb.last_frame
        ws = torch.empty(fr.layout.total_bytes, dtype=torch.uint8, device=device)
        img_dev = torch.empty((H, W, 3), device=device)
        aux_f = torch.empty((H, W), device=device)
        aux_i = torch.empty((H, W), dtype=torch.int32, device=device)
        cfgr = op_rgb.config
        a = _lib.GsbForwardArgs(
            num_points=N, pointcloud=scene.point_cloud.data_ptr(), pointcloud_features=scene.point_cloud_features.data_ptr(),
            point_invalid_mask=scene.point_invalid_mask.data_ptr(), point_object_id=scene.point_object_id.data_ptr(),
            num_objects=1, camera_height=H, camera_width=W, near_plane=cfgr.near_plane, far_plane=cfgr.far_plane,
            depth_to_sort_key_scale=cfgr.depth_to_sort_key_scale, rgb_only=1, flags=fr.flags, workspace=ws.data_ptr(),
            workspace_bytes=fr.layout.total_bytes, key_capacity=fr.key_capacity, rasterized_image=img_dev.data_ptr(),
            rasterized_depth=aux_f.data_ptr(), pixel_accumulated_alpha=aux_f.data_ptr(),
            pixel_offset_of_last_effective_point=aux_i.data_ptr(), pixel_valid_point_count=aux_i.data_ptr(),
            stream=torch.cuda.current_stream(device).cuda_stream)
        staging = torch.empty(32, device=device)
        image_host = torch.empty((H, W, 3)).pin_memory()

        def one():
            _lib.check(lib.gsb200_render_host(ctypes.byref(a), q_host.data_ptr(), t_host.data_ptr(), K_host.data_ptr(),
                                              staging.data_ptr(), image_host.data_ptr(), None), "gsb200_render_host")
        for _ in range(3):
            one()
        ms = timed(one, k) / k
        return {"ms": round(ms, 4), "Mpix_s": round(wl.mpix(ms), 1),
                "h2d_bytes_per_frame": 64, "d2h_bytes_per_frame": H * W * 3 * 4,
                "what": "gsb200_render_host: host pose/intrinsics in, forward (rgb_only), image to pinned host memory"}
    render_host = render_host_e2e(steps)

    # ---- other BASELINE configurations as side numbers (fwd+bwd incl. the exchange at N > 1, and forward only)
    def side_config(name, k=10):
        w2 = Workload(name)

        def fw():
            with torch.no_grad():
                w2.op(w2.dev_input)
        for _ in range(5):
            w2.step()
        ms = min(timed(w2.step, k), timed(w2.step, k)) / k   # side number: best of two short runs
        fms = min(timed(fw, k), timed(fw, k)) / k
        return {"workload": workload_string(name), "fwd_bwd_ms": round(ms, 4), "fwd_bwd_Mpix_s": round(w2.mpix(ms), 1),
                "fwd_ms": round(fms, 4), "fwd_Mpix_s": round(w2.mpix(fms), 1),
                "M": w2.op.last_frame.num_points_in_camera, "K": w2.op.last_frame.num_keys}
    side = {}
    if args.workload == "C3":
        side["C2"] = side_config("C2")
        if world == 8:  # BASELINE config 4 as specified: 2.1e6 Gaussians, 8 views on 8 GPUs, gradient exchange every step
            side["C4"] = side_config("C4", k=steps)

    # clocks were sampled from the start of the headline region to here (all timed regions of this run)
    clocks = sampler.stop() if rank == 0 else None

    # ---- per-kernel device times (CUDA events recorded inside the library on the launching stream) and the blend
    #      kernels' work counted on the device (untimed diagnostics)
    stage_ms = profiling.stage_times(op, wl.dev_input, wl.grad_image, iters=min(steps, 10))
    work = profiling.blend_work(op, wl.dev_input, wl.grad_image)

    if world > 1:
        dist.barrier()
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peak, peak_src = measured_peaks()
    T = (H // 16) * (W // 16)
    alg_bytes = {  # SURVEY.md §8(d) algorithmic bytes per frame
        "preprocess": 17 * N + 296 * M + 32 * M + 12 * Kk,
        "sort": 24 * Kk,
        "tile_ranges": 8 * Kk + 8 * T,
        "blend_forward": 52 * Kk + 28 * H * W,
        "blend_backward": 88 * Kk + 28 * H * W,
        "backward_points": 512 * M,
    }
    per_stage = {}
    for name, ms in stage_ms.items():
        if name in alg_bytes and ms > 0:
            gbs = alg_bytes[name] / (ms * 1e-3) / 1e9
            per_stage[name] = {"ms": round(ms, 4), "alg_GB": round(alg_bytes[name] / 1e9, 4),
                               "GBps": round(gbs, 1), "frac_hbm": round(gbs / peak, 4)}
        else:
            per_stage[name] = {"ms": round(ms, 4)}
    dominant = max((k for k in stage_ms if k in alg_bytes), key=lambda k: stage_ms[k])
    dom_gbs = alg_bytes[dominant] / (stage_ms[dominant] * 1e-3) / 1e9

    def compute_side(kind, visits, contributing, ms, instr_per_visit, mufu_per_eval):
        evals = 32 * visits  # every lane of a visiting warp evaluates the splat
        s_ = ms * 1e-3
        return {"warp_splat_visits": visits, "pixel_splat_evaluations_E": evals, "contributing_evaluations": contributing,
                "contributing_fraction": round(contributing / max(evals, 1), 3),
                "evaluations_per_s": round(evals / s_, 1),
                "inner_loop_sass_instructions_per_visit": instr_per_visit,
                "inner_loop_issue_slot_fraction": round(visits * instr_per_visit / s_ / ISSUE_PEAK, 3),
                "mufu_fraction_of_peak": round(evals * mufu_per_eval / s_ / MUFU_LANE_PEAK, 3),
                "what": f"{kind}: counted on the device by the kernel's COUNT instantiation; issue peak = 148 SMs x 4 schedulers x "
                        f"1.965 GHz, MUFU peak = 16 lanes / SM / clk"}
    compute = {
        "blend_forward": compute_side("forward blend", work["forward_warp_splat_visits"], work["forward_contributing_evaluations"],
                                      stage_ms["blend_forward"], FWD_INSTR_PER_VISIT, 1),
        "blend_backward": compute_side("backward blend (phase 1 visits)", work["backward_warp_splat_visits"],
                                       work["backward_contributing_evaluations"], stage_ms["blend_backward"],
                                       BWD_INSTR_PER_VISIT, 2),
    }
    p84, p88, p164 = work["staged_patch_pairs_8x4"], work["staged_patch_pairs_8x8"], work["staged_patch_pairs_16x4"]
    compute["patch_shape_what_if"] = {
        "staged_patch_splat_pairs": {"8x4_one_pixel_per_thread": p84, "8x8_two_pixels_per_thread": p88, "16x4_two_pixels_per_thread": p164,
                                     "4x4_one_splat_per_half_warp": work["staged_patch_pairs_4x4"]},
        "relative_inner_loop_instructions": {"8x4": 1.0, "8x8": round(p88 * (4 + 2 * 25) / max(p84 * FWD_INSTR_PER_VISIT, 1), 3),
                                             "16x4": round(p164 * (4 + 2 * 25) / max(p84 * FWD_INSTR_PER_VISIT, 1), 3),
                                             "4x4_two_splats_per_warp_iteration_lower_bound": round(work["staged_patch_pairs_4x4"] / 2 / max(p84, 1), 3)},
        "what": "counted on the device at staging time: a two-pixels-per-thread warp (8x8 or 16x4 patch) visits a splat if either of its "
                "two 8x4 halves can be reached and then pays ~4 shared + 2 x 25 per-pixel instructions instead of 29 per 8x4 visit"}
    ncu = None
    npath = os.path.join(ROOT, "profiles", "r02_ncu_step_full.json")
    if args.workload == "C3" and os.path.exists(npath):  # committed ncu --set full capture of both blend kernels (not live)
        with open(npath) as f:
            ncu = json.load(f)
    traffic = (ncu or {}).get(dominant, {}).get("dram_bytes_per_launch")
    roofline = {
        "kernel": dominant,
        "bound": "issue (FP32/ALU instruction slots): the blend kernels reuse each 48-B record across up to 256 pixels, "
                 "so neither hbm nor tensor bounds them; the hbm figures below are the mandated algorithmic-bytes roofline, "
                 "`compute` is the one that explains the time",
        "achieved": round(dom_gbs, 2), "peak": peak, "unit": "GB/s",
        "frac": round(dom_gbs / peak, 5), "traffic": traffic, "peak_source": peak_src,
        "launch_ms": round(stage_ms[dominant], 4),
        "compute": compute,
        "ncu_committed_capture": ncu,
        "per_stage": per_stage,
    }

    cpu_baseline = None
    if world == 1 and not args.no_cpu_baseline:
        threads = pin_cpu_threads()
        from oracle import gs_oracle
        gs_oracle.set_num_threads(threads)
        cpu_scene = make_scene(**cfg)
        t0 = time.perf_counter()
        oracle_step(cpu_scene)
        dt = time.perf_counter() - t0
        cpu_baseline = {"value": H * W / dt / 1e6, "unit": UNIT, "cores": gs_oracle.num_threads(), "kind": "port",
                        "sample": f"1 full {args.workload} frame fwd+bwd ({dt:.1f} s), oracle/gs_oracle.c with OpenMP, one bound "
                                  f"thread per physical core"}

    launches_per_step = profiling.KERNELS_PER_FORWARD(frame.layout.sort_passes) + profiling.KERNELS_PER_BACKWARD + \
        (0 if exchange is None else                       # + gsb200_expand_view_gradients (two launches when split around the
         ((2 if args.overlap_expansion_nccl and not args.serial_expansion and args.exchange_streams == 1 else 1)
          if exchange_kind != "multimem" else              # all-reduce)
          (4 if args.overlap_expansion and not args.serial_expansion else 3)))  # + the two launches of gsb200_exchange_multimem
    if world == 1:
        parallelism = "single GPU"
    elif exchange is not None:
        how = ("one hand-written NVLS kernel, gsb200_exchange_multimem: multimem.ld_reduce / multimem.st over NVSwitch multicast memory"
               if exchange_kind == "multimem" else
               "NCCL all-reduce + all-gather" + (", concurrently on two communicators" if args.exchange_streams == 2 else ""))
        parallelism = (f"view-parallel x{world}: compact gradient exchange inside backward (sum of the (N,12) columns + gather of the "
                       f"(N,3) colour-argument gradients and camera centres: {how}), then gsb200_expand_view_gradients")
    else:
        parallelism = f"view-parallel x{world}: one NCCL all-reduce of the dense (N,59) gradients"
    line = {
        "metric": METRIC, "value": round(value, 2), "unit": UNIT, "n_gpus": world, "steps": steps,
        "warmup": warmup, "ms_per_step": round(ms_per_step, 4), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_string(args.workload),
                   "frame": f"M={M} in frustum, K={Kk} (tile,splat) pairs sorted and blended (of {K_ref} in the reference's "
                            f"3-sigma squares; the rest cannot reach alpha>=1/255)",
                   "parallelism": parallelism,
                   "l2": "inputs larger than L2 (scene 236 MB + 200 MB workspace per frame vs 126 MB L2)",
                   "backward_impl": op.backward_impl},
        "spread": dict(percentiles(regions), first_region_ms_per_step=round(first_region_ms, 4),
                       what=f"{len(regions)} timed regions of {steps} steps each; `value` / `ms_per_step` are the median region"),
        "e2e": {"value": round(e2e_value, 2), "unit": UNIT, "ms_per_step": round(e2e_ms, 4),
                "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4, "spread": percentiles(e2e_regions),
                "what": "per step: pinned host pose + intrinsics + target image -> device (copy stream, one step ahead; the forward waits for the pose, the loss kernel for the image), forward, fused L1 loss + gradient kernel, backward, loss -> pinned host (read one step later, all inside the timed region)"},
        "forward_only": {"Mpix_s": round(wl.mpix(fwd_ms), 2), "ms": round(fwd_ms, 4),
                         "rgb_only_Mpix_s": round(wl.mpix(fwd_rgb_ms), 2),
                         "rgb_only_ms": round(fwd_rgb_ms, 4),
                         "two_frames_in_flight": {"Mpix_s": round(wl.mpix(fwd2_ms), 2), "ms_per_frame": round(fwd2_ms, 4),
                                                  "rgb_only_Mpix_s": round(wl.mpix(fwd2_rgb_ms), 2),
                                                  "rgb_only_ms_per_frame": round(fwd2_rgb_ms, 4),
                                                  "what": "throughput of parallel.render_views(..., streams=2 streams): consecutive frames "
                                                          "on alternating streams (per-point stage + sort of frame i+1 under the blend of frame i)"}},
        "forward_e2e_c_abi": render_host,
        "other_configs": side,
        "gpu_launches": launches_per_step * steps,
        "clocks": clocks,
        "roofline": roofline,
    }
    if exchange_check is not None:
        line["exchange_check"] = exchange_check
    if cpu_baseline is not None:
        line["cpu_baseline"] = cpu_baseline
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
