# PCB quantile search tests: build, smoke, the new test file, the whole GPU suite, get_pcb_vectors of another build of
# the library (e.g. the parent commit's) vs this one (K = 8 BLaIR-base, alternated in one process, checksums), and the
# default bench line.
set -u
OUT=${1:?usage: bash tools/runs/run49.sh OUTPUT_DIR [OTHER_LIB.so]}
OTHER=${2:-}
mkdir -p "$OUT"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > "$OUT"/r49_gpu.txt 2>&1; cat "$OUT"/r49_gpu.txt
python -c "import __graft_entry__ as g; g.build()" > "$OUT"/r49_build.log 2>&1; echo "build rc=$?"
python -c "import __graft_entry__ as g; g.smoke()" > "$OUT"/r49_smoke.log 2>&1; echo "smoke rc=$?"
python -m pytest tests/test_pcb_search_gpu.py -m gpu -q -s -rxXfE --durations=10 > "$OUT"/r49_pytest_new.log 2>&1; echo "new tests rc=$?"
grep -E "FAILED|XPASS|XFAIL|passed|failed|BLaIR-base K=8" "$OUT"/r49_pytest_new.log | tail -20
[ -n "$OTHER" ] && { python tools/pcb_lib_compare.py "$OTHER" > "$OUT"/r49_compare.json 2> "$OUT"/r49_compare.err; echo "compare rc=$?"; cat "$OUT"/r49_compare.json; }
python bench.py --gpus 1 --steps 10 --warmup 3 > "$OUT"/r49_bench.json 2> "$OUT"/r49_bench.err; echo "bench rc=$?"; tail -c 800 "$OUT"/r49_bench.json
python -m pytest tests -m gpu -q --ignore=tests/test_pcb_search_gpu.py > "$OUT"/r49_pytest_gpu.log 2>&1; echo "gpu suite rc=$?"; tail -5 "$OUT"/r49_pytest_gpu.log
