"""Compare the outputs two builds wrote with ``bench.py --dump-outputs``.

    python scripts/compare_dumps.py PARENT_A PARENT_B NEW

PARENT_A and PARENT_B are two runs of the same (reference) build: their difference is the run-to-run noise of the float
atomics that add up the gradient rows.  The image, depth and valid point count have to be bit-identical between all
three; every gradient array of NEW has to differ from PARENT_A by no more than twice the largest of that noise."""
import os
import sys

import numpy as np

EXACT = ("image", "depth", "pixel_valid_point_count")
GRADS = ("grad_pointcloud_sampled_rows", "grad_pointcloud_features_sampled_rows")


def main(a_dir, b_dir, new_dir):
    load = lambda d, n: np.load(os.path.join(d, n + ".npy"))  # noqa: E731
    ok = True
    for name in EXACT:
        a, b, n = load(a_dir, name), load(b_dir, name), load(new_dir, name)
        same = np.array_equal(a.view(np.uint32), n.view(np.uint32)) and np.array_equal(a.view(np.uint32), b.view(np.uint32))
        print(f"{name}: shape {a.shape} bit-identical {same}")
        ok &= same
    for name in GRADS:
        a, b, n = (load(d, name).astype(np.float64) for d in (a_dir, b_dir, new_dir))
        scale = max(float(np.abs(a).max()), 1e-30)
        noise, diff = float(np.abs(b - a).max()), float(np.abs(n - a).max())
        within = diff <= 2.0 * noise or diff <= 1e-6 * scale
        print(f"{name}: shape {a.shape} max|x| {scale:.3e}  parent-vs-parent max|d| {noise:.3e} ({noise / scale:.2e} rel)  "
              f"new-vs-parent max|d| {diff:.3e} ({diff / scale:.2e} rel)  within noise {within}")
        ok &= within
    print("outputs agree" if ok else "OUTPUTS DIFFER")
    return 0 if ok else 1


if __name__ == "__main__":
    sys.exit(main(*sys.argv[1:4]))
