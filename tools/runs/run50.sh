# Items left out of the ranking (evaluator `exclude`): build, smoke, the new test files, the exclusion benchmark at
# BASELINE config 5 (4 cases alternated in one process), the default bench line (its topk_ids checksum must stay
# 165473006011287), and the whole GPU suite.
set -u
OUT=${1:?usage: bash tools/runs/run50.sh OUTPUT_DIR}
mkdir -p "$OUT"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > "$OUT"/r50_gpu.txt 2>&1; cat "$OUT"/r50_gpu.txt
python -c "import __graft_entry__ as g; g.build()" > "$OUT"/r50_build.log 2>&1; echo "build rc=$?"
python -c "import __graft_entry__ as g; g.smoke()" > "$OUT"/r50_smoke.log 2>&1; echo "smoke rc=$?"
python -m pytest tests/test_exclude_gpu.py tests/test_exclude_host.py -q -rxXfE --durations=10 > "$OUT"/r50_pytest_new.log 2>&1; echo "new tests rc=$?"
grep -E "FAILED|Error|passed|failed" "$OUT"/r50_pytest_new.log | tail -20
python tools/exclude_bench.py --iters 5 --warmup 2 > "$OUT"/r50_exclude_bench.json 2> "$OUT"/r50_exclude_bench.err; echo "exclude bench rc=$?"
cat "$OUT"/r50_exclude_bench.json; tail -3 "$OUT"/r50_exclude_bench.err
python bench.py --gpus 1 --steps 10 --warmup 3 > "$OUT"/r50_bench.json 2> "$OUT"/r50_bench.err; echo "bench rc=$?"; tail -c 800 "$OUT"/r50_bench.json
python -m pytest tests -m gpu -q --ignore=tests/test_exclude_gpu.py > "$OUT"/r50_pytest_gpu.log 2>&1; echo "gpu suite rc=$?"; tail -5 "$OUT"/r50_pytest_gpu.log
