# Label log-softmax over the whole catalog (`label_log_softmax`, `catalog_cross_entropy`): build, smoke, the new test
# files and the loss checks of tests/test_joint_eval.py, tools/lse_bench.py at BASELINE config 5 (5 cases alternated in
# one process), the default bench line (its topk_ids checksum must stay 165473006011287), and the whole GPU suite.
set -u
OUT=${1:?usage: bash tools/runs/run52.sh OUTPUT_DIR}
mkdir -p "$OUT"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > "$OUT"/r52_gpu.txt 2>&1; cat "$OUT"/r52_gpu.txt
python -c "import __graft_entry__ as g; g.build()" > "$OUT"/r52_build.log 2>&1; echo "build rc=$?"
python -c "import __graft_entry__ as g; g.smoke()" > "$OUT"/r52_smoke.log 2>&1; echo "smoke rc=$?"; tail -2 "$OUT"/r52_smoke.log
python -m pytest tests/test_label_log_softmax_gpu.py tests/test_label_log_softmax_host.py \
    tests/test_nccl_label_log_softmax_gpu.py tests/test_joint_eval.py -q -rxXfEs --durations=10 \
    > "$OUT"/r52_pytest_new.log 2>&1; echo "new tests rc=$?"
grep -E "FAILED|Error|SKIPPED|passed|failed" "$OUT"/r52_pytest_new.log | tail -30
python tools/lse_bench.py --iters 5 --warmup 2 > "$OUT"/r52_lse_bench.json 2> "$OUT"/r52_lse_bench.err; echo "lse bench rc=$?"
cat "$OUT"/r52_lse_bench.json; tail -3 "$OUT"/r52_lse_bench.err
python bench.py --gpus 1 --steps 10 --warmup 3 > "$OUT"/r52_bench.json 2> "$OUT"/r52_bench.err; echo "bench rc=$?"; tail -c 800 "$OUT"/r52_bench.json
python -m pytest tests -m gpu -q --ignore=tests/test_label_log_softmax_gpu.py > "$OUT"/r52_pytest_gpu.log 2>&1; echo "gpu suite rc=$?"
tail -5 "$OUT"/r52_pytest_gpu.log
