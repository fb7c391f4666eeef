"""Work statistics of the two blend-backward kernels at a BASELINE workload, WITHOUT a GPU: the oracle renders the frame,
the unmodified kernel sources replay loop A under the SIMT emulator (tests/simt) on a sample of tiles, and the
emulation-only counters of csrc/blend_bwd.cuh report how many (warp, splat) visits, contributing pairs, chunks and rows the
kernels process.  With the SASS instruction counts per visit / per chunk (DESIGN.md section 8) this gives the expected
warp-instruction ratio of the transposed kernel over the butterfly kernel.  Not a measurement of time.

    python scripts/emu_work_stats.py C3 [tiles_sampled=400] [processes=6]
"""
import ctypes
import json
import os
import sys
from multiprocessing import Pool

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def _state(name):
    from helpers import oracle_forward
    from taichi_3d_gaussian_splatting_b200.synthetic import CONFIGS, make_scene
    scene = make_scene(**CONFIGS[name])
    o, fwd, feats = oracle_forward(scene)
    M = fwd.point_id_in_camera_list.shape[0]
    rec = np.zeros((M, 12), np.float32)
    rec[:, 0:2] = fwd.point_uv
    rec[:, 2:6] = fwd.point_uv_conic_and_rescale
    rec[:, 6] = fwd.point_alpha_after_activation
    rec[:, 7] = fwd.point_in_camera[:, 2]
    rec[:, 8:11] = fwd.point_color
    rec[:, 11] = fwd.point_radii
    H, W = fwd.image.shape[:2]
    g = np.random.default_rng(1).standard_normal((H, W, 3)).astype(np.float32)
    return dict(H=H, W=W, rec=rec, g=g, start=np.ascontiguousarray(fwd.tile_points_start, dtype=np.int32),
                end=np.ascontiguousarray(fwd.tile_points_end, dtype=np.int32),
                vals=np.ascontiguousarray(fwd.point_offset_with_sort_key, dtype=np.int32),
                acc=np.ascontiguousarray(fwd.pixel_accumulated_alpha, dtype=np.float32),
                last=np.ascontiguousarray(fwd.pixel_offset_of_last_effective_point, dtype=np.int32))


STATE = None


def _work_forward(tiles):
    from simt_helpers import build_emulator
    emu = build_emulator()
    s = STATE
    c = lambda a: a.ctypes.data_as(ctypes.c_void_p)  # noqa: E731
    H, W = s["H"], s["W"]
    image, depth, acc = np.zeros((H, W, 3), np.float32), np.zeros((H, W), np.float32), np.zeros((H, W), np.float32)
    last, cnt = np.zeros((H, W), np.int32), np.zeros((H, W), np.int32)
    total, out = np.zeros(16, np.int64), np.zeros(16, np.int64)
    for t in tiles:
        emu.emu_blend_forward_stats(H, W, int(t), int(t) + 1, c(s["start"]), c(s["end"]), c(s["vals"]), c(s["rec"]), c(image),
                                    c(depth), c(acc), c(last), c(cnt), c(out))
        total += out
    return total


def _work(args):
    transposed, tiles = args
    from simt_helpers import build_emulator
    emu = build_emulator()
    s = STATE
    c = lambda a: a.ctypes.data_as(ctypes.c_void_p)  # noqa: E731
    accum = np.zeros((s["rec"].shape[0], 12), np.float32)
    mag = np.zeros((s["H"], s["W"], 2), np.float32)
    total = np.zeros(8, np.int64)
    out = np.zeros(8, np.int64)
    for t in tiles:
        emu.emu_blend_backward_stats(int(transposed), 0, s["H"], s["W"], int(t), int(t) + 1, c(s["start"]), c(s["end"]), c(s["vals"]),
                                     c(s["rec"]), c(s["g"]), c(s["acc"]), c(s["last"]), c(accum), c(mag), c(out))
        total += out
    return transposed, total


def main():
    global STATE
    name = sys.argv[1] if len(sys.argv) > 1 else "C3"
    sample = int(sys.argv[2]) if len(sys.argv) > 2 else 400
    procs = int(sys.argv[3]) if len(sys.argv) > 3 else 6
    from simt_helpers import build_emulator
    build_emulator()
    STATE = _state(name)
    T = STATE["start"].shape[0]
    tiles = np.sort(np.random.default_rng(0).choice(T, min(sample, T), replace=False))
    pairs_sampled = int((STATE["end"] - STATE["start"])[tiles].sum())
    jobs = [(tr, tiles[k::procs // 2]) for tr in (0, 1) for k in range(procs // 2)]
    with Pool(procs) as pool:  # fork: the workers inherit STATE
        res = pool.map(_work, jobs)
    tot = {0: np.zeros(8, np.int64), 1: np.zeros(8, np.int64)}
    for tr, c in res:
        tot[tr] += c
    with Pool(procs) as pool:
        fw = sum(pool.map(_work_forward, [tiles[k::procs] for k in range(procs)]))
    bf, tb = tot[0], tot[1]
    # SASS instruction counts (cuobjdump, fast path without hook statistics; DESIGN.md section 8 item 3)
    BF_VISIT_ANY, BF_VISIT_NONE = 107, 55      # butterfly kernel per (warp, splat) visit: with / without the butterfly + RED
    TB_PHASE1, TB_CHUNK = 36, 548              # transposed kernel: per splat (phase 1), per chunk (fill + phase 2 + epilogue)
    est_bf = BF_VISIT_ANY * bf[1] + BF_VISIT_NONE * (bf[0] - bf[1])
    est_tb = TB_PHASE1 * tb[3] + TB_CHUNK * tb[4]
    print(json.dumps({
        "workload": name, "tiles_sampled": int(tiles.shape[0]), "of_tiles": int(T), "list_entries_sampled": pairs_sampled,
        "butterfly": {"visits": int(bf[0]), "visits_with_a_contributing_pixel": int(bf[1]), "contributing_pairs": int(bf[2]),
                      "contributing_lanes_per_visit": round(float(bf[2]) / max(int(bf[0]), 1), 2),
                      "visits_per_list_entry": round(float(bf[0]) / max(pairs_sampled, 1), 3)},
        "forward": {"visits": int(fw[7]), "pairs_with_alpha_above_cutoff_on_live_pixels": int(fw[8]),
                    "evaluated_pixel_splat_pairs": int(fw[7]) * 32, "scale_to_frame": round(float(T) / tiles.shape[0], 2)},
        "transposed": {"splat_visits": int(tb[3]), "chunks": int(tb[4]), "mean_chunk_fill": round(float(tb[3]) / max(int(tb[4]), 1), 2),
                       "rows_flushed": int(tb[5]), "windows": int(tb[6])},
        "estimated_warp_instructions_in_the_visit_loops": {"butterfly": int(est_bf), "transposed": int(est_tb),
                                                           "ratio": round(float(est_tb) / max(float(est_bf), 1.0), 3)},
        "note": "counts from the kernel sources under the CPU emulator; instruction weights from SASS; NOT a time measurement"}))


if __name__ == "__main__":
    main()
