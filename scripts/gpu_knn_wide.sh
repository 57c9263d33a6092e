# knn at C > 64 (knn_tcgen05.cu): the wide-feature tests and the K1 benchmark in one call, with the card they ran on.
# usage: bash scripts/gpu_knn_wide.sh [output directory, default knn_wide_out]
OUT=${1:-knn_wide_out}
mkdir -p "$OUT"; rm -f "$OUT/rc.txt"
python -c "import __graft_entry__ as g; g.build(force=False)" > "$OUT/build.log" 2>&1; echo "build rc=$?" >> "$OUT/rc.txt"
{ python -c "import torch; print(torch.cuda.get_device_name())"; nvidia-smi --query-gpu=power.limit,clocks.max.sm --format=csv; } > "$OUT/device.txt" 2>&1
( time timeout 1200 python -m pytest tests/test_gpu_knn_wide.py -q -s -m gpu -p no:cacheprovider --durations=10 ) > "$OUT/tests.log" 2>&1; echo "tests rc=$?" >> "$OUT/rc.txt"
( time timeout 1200 python scripts/kbench_knn.py ) > "$OUT/bench.log" 2>&1; echo "bench rc=$?" >> "$OUT/rc.txt"
cat "$OUT/rc.txt" "$OUT/device.txt"; tail -25 "$OUT/tests.log"; cat "$OUT/bench.log"
