# The three validity sets in one PnP launch: the GPU tests of cp_pnp_ransac_sets and kbench_pnp_sets.py in one call, with
# the card's name and power limit.
# usage: bash scripts/gpu_pnp_sets.sh [output directory, default pnp_sets_out]
OUT=${1:-pnp_sets_out}
mkdir -p "$OUT"; rm -f "$OUT/rc.txt"
python -c "import __graft_entry__ as e; e.build(force=False)" > "$OUT/build.log" 2>&1; echo "build rc=$?" >> "$OUT/rc.txt"
timeout 900 python -m pytest tests/test_gpu_pnp_sets.py tests/test_cpu_pnp_sets.py -q -s -p no:cacheprovider --durations=6 > "$OUT/tests.log" 2>&1; echo "tests rc=$?" >> "$OUT/rc.txt"
timeout 1200 python scripts/kbench_pnp_sets.py > "$OUT/bench.log" 2>&1; echo "bench rc=$?" >> "$OUT/rc.txt"
cat "$OUT/rc.txt"; tail -15 "$OUT/tests.log"; cat "$OUT/bench.log"
