# sharded PCB / DARE merges: build, smoke, the new tests, the whole GPU suite, get_pcb_vectors of the parent library vs
# this one (K = 8 BLaIR-base, alternated in one process, checksums), and the pcb_sharded bench line on every GPU count
# the box has (G = 1, 2, 4, 8), next to the single-GPU get_pcb_vectors + merge.  `_cmp/lib_parent.so` is provided for
# this run only (a build of the parent commit: git stash; make -C mergerec_b200/csrc; cp the .so to _cmp/lib_parent.so).
set -u
OUT=${1:?usage: bash tools/runs/run48.sh OUTPUT_DIR}
mkdir -p "$OUT"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > "$OUT"/r48_gpu.txt 2>&1; cat "$OUT"/r48_gpu.txt
NG=$(nvidia-smi -L | wc -l)
python -c "import __graft_entry__ as g; g.build()" > "$OUT"/r48_build.log 2>&1; echo "build rc=$?"
python -c "import __graft_entry__ as g; g.smoke()" > "$OUT"/r48_smoke.log 2>&1; echo "smoke rc=$?"
python -m pytest tests/test_sharded_pcb_gpu.py -q -rs > "$OUT"/r48_pytest_new.log 2>&1; echo "new tests rc=$?"; tail -4 "$OUT"/r48_pytest_new.log
[ -f _cmp/lib_parent.so ] && { python tools/pcb_lib_compare.py _cmp/lib_parent.so > "$OUT"/r48_compare.json 2> "$OUT"/r48_compare.err; echo "compare rc=$?"; cat "$OUT"/r48_compare.json; }
for G in 1 2 4 8; do
  [ "$G" -gt "$NG" ] && break
  if [ "$G" -eq 1 ]; then
    python bench.py --gpus 1 --workload pcb_sharded --steps 10 --warmup 3 > "$OUT"/r48_bench_pcb_n1.json 2> "$OUT"/r48_bench_pcb_n1.err
  else
    python -m torch.distributed.run --nproc-per-node "$G" bench.py --workload pcb_sharded --gpus "$G" --steps 10 --warmup 3 \
      --no-cpu-baseline > "$OUT"/r48_bench_pcb_n$G.json 2> "$OUT"/r48_bench_pcb_n$G.err
  fi
  echo "bench G=$G rc=$?"; tail -c 600 "$OUT"/r48_bench_pcb_n$G.json
done
python -m pytest tests -m gpu -q --ignore=tests/test_sharded_pcb_gpu.py > "$OUT"/r48_pytest_gpu.log 2>&1; echo "gpu suite rc=$?"; tail -5 "$OUT"/r48_pytest_gpu.log
