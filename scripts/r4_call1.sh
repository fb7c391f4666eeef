#!/bin/bash
# round 4, call 1 (1 GPU): cost of the pose gradients at C3 (alternated, then profiled); bench.py against the parent commit's
# library (built from the parent's sources as libgsb200_parent.so), alternated three times, and the outputs of both builds
# compared; the GPU suite and smoke().
set -u
OUT=${1:?usage: bash $0 OUTPUT_DIR}  # logs and output dumps go here
mkdir -p "$OUT"
export PYTHONUNBUFFERED=1
P=$PWD/taichi_3d_gaussian_splatting_b200/libgsb200_parent.so
BENCH="python bench.py --gpus 1 --steps 200 --warmup 20 --no-cpu-baseline"
DUMP="python bench.py --gpus 1 --steps 20 --warmup 5 --no-cpu-baseline"
{
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv
echo "== build + smoke"; timeout 900 python -c "import __graft_entry__ as g; g.build(); g.smoke()" 2>&1 | tail -3
echo "== pose gpu tests"; GSB200_TEST_RECORD_DIR="$OUT" timeout 900 python -m pytest tests/test_gpu_pose_gradients.py -q -m gpu -p no:cacheprovider 2>&1 | tail -15
cat "$OUT/pose_gradients.json"
echo "== pose gradient cost"; timeout 600 python scripts/bench_pose_grad.py --config C3 --rounds 3
for r in 1 2 3; do
  echo "== round $r parent"; GSB200_LIB_PATH=$P timeout 300 $BENCH | tail -1
  echo "== round $r new"; timeout 300 $BENCH | tail -1
done
echo "== output dumps"
GSB200_LIB_PATH=$P timeout 300 $DUMP --dump-outputs "$OUT/dump_parent_a" | tail -1
GSB200_LIB_PATH=$P timeout 300 $DUMP --dump-outputs "$OUT/dump_parent_b" | tail -1
timeout 300 $DUMP --dump-outputs "$OUT/dump_new" | tail -1
python scripts/compare_dumps.py "$OUT/dump_parent_a" "$OUT/dump_parent_b" "$OUT/dump_new"
echo "== gpu tests"; timeout 1800 python -m pytest tests -q -m gpu -p no:cacheprovider 2>&1 | tail -8
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv
} 2>&1 | tee "$OUT/r4_call1.log"
rm -rf "$OUT/dump_parent_a" "$OUT/dump_parent_b" "$OUT/dump_new"
