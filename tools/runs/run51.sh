# Label rank against the whole catalog (`label_ranks`, `rank_rows`, large ks): build, smoke, the new test files,
# tools/rank_bench.py at BASELINE config 5 (3 cases alternated in one process), the default bench line (its topk_ids
# checksum must stay 165473006011287), and the whole GPU suite.
set -u
OUT=${1:?usage: bash tools/runs/run51.sh OUTPUT_DIR}
mkdir -p "$OUT"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > "$OUT"/r51_gpu.txt 2>&1; cat "$OUT"/r51_gpu.txt
python -c "import __graft_entry__ as g; g.build()" > "$OUT"/r51_build.log 2>&1; echo "build rc=$?"
python -c "import __graft_entry__ as g; g.smoke()" > "$OUT"/r51_smoke.log 2>&1; echo "smoke rc=$?"
python -m pytest tests/test_label_rank_gpu.py tests/test_label_rank_host.py tests/test_nccl_label_rank_gpu.py -q -rxXfEs \
    --durations=10 > "$OUT"/r51_pytest_new.log 2>&1; echo "new tests rc=$?"
grep -E "FAILED|Error|SKIPPED|passed|failed" "$OUT"/r51_pytest_new.log | tail -20
python tools/rank_bench.py --iters 5 --warmup 2 > "$OUT"/r51_rank_bench.json 2> "$OUT"/r51_rank_bench.err; echo "rank bench rc=$?"
cat "$OUT"/r51_rank_bench.json; tail -3 "$OUT"/r51_rank_bench.err
python bench.py --gpus 1 --steps 10 --warmup 3 > "$OUT"/r51_bench.json 2> "$OUT"/r51_bench.err; echo "bench rc=$?"; tail -c 800 "$OUT"/r51_bench.json
python -m pytest tests -m gpu -q --ignore=tests/test_label_rank_gpu.py > "$OUT"/r51_pytest_gpu.log 2>&1; echo "gpu suite rc=$?"; tail -5 "$OUT"/r51_pytest_gpu.log
