# ObjectBank: its GPU tests and kbench_object_bank.py in one call, with the card's name and power limit.
# usage: bash scripts/gpu_object_bank.sh [output directory, default object_bank_out]
OUT=${1:-object_bank_out}
mkdir -p "$OUT"; rm -f "$OUT/rc.txt"
python -c "import __graft_entry__ as e; e.build(force=False)" > "$OUT/build.log" 2>&1; echo "build rc=$?" >> "$OUT/rc.txt"
timeout 1500 python -m pytest tests/test_gpu_object_bank.py -q -s -p no:cacheprovider --durations=6 > "$OUT/tests.log" 2>&1; echo "tests rc=$?" >> "$OUT/rc.txt"
timeout 1200 python scripts/kbench_object_bank.py > "$OUT/bench.log" 2>&1; echo "bench rc=$?" >> "$OUT/rc.txt"
cat "$OUT/rc.txt"; tail -15 "$OUT/tests.log"; cat "$OUT/bench.log"
