# round-3 GPU job a: token-walk radix passes of the walker sort kernels.  Tests, the sort microbenchmark with the walk counters, and the
# bench alternating the token walk (default) with the old element walker (WM_SORT_TOKEN_MIN=0), three runs each, on one GPU.
# Usage: bash tools/gpu_jobs/r3a_token_walk.sh OUT_DIR (logs and JSON lines are written there)
OUT=${1:?usage: r3a_token_walk.sh OUT_DIR}
mkdir -p "$OUT"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee $OUT/r3a_gpu.txt
python -c "import __graft_entry__ as g; g.build()" > $OUT/r3a_build.log 2>&1 || { tail -20 $OUT/r3a_build.log; exit 1; }
timeout 1200 python -m pytest tests/test_sort_token_walk.py tests/test_gpu_stages.py tests/test_gpu_e2e.py -m gpu -q --timeout 900 \
	> $OUT/r3a_pytest.log 2>&1; rc=$?; tail -4 $OUT/r3a_pytest.log
[ $rc -eq 0 ] || exit 1
timeout 300 python -c "import __graft_entry__ as g; g.smoke(); print('smoke ok')" 2>&1 | tail -1
for args in "--n 30000 --arrays 100" "--n 150000 --arrays 16"; do
	for tm in 0 512 4096; do
		echo "== bench_sort $args WM_SORT_TOKEN_MIN=$tm"
		WM_SORT_TOKEN_MIN=$tm WM_SORT_DEBUG=1 timeout 600 python tools/bench_sort.py $args --check --repeat 1 2>&1 | grep -E "sort-debug|matches"
		WM_SORT_TOKEN_MIN=$tm timeout 600 python tools/bench_sort.py $args --repeat 7 | grep device
	done
done 2>&1 | tee $OUT/r3a_bench_sort.txt
for i in 1 2 3; do
	for arm in token walker; do
		tm=512; [ $arm = walker ] && tm=0
		WM_SORT_TOKEN_MIN=$tm WM_TIMING=1 WM_BENCH_NO_CPU=1 timeout 1200 python bench.py --gpus 1 --steps 20 --warmup 5 \
			> $OUT/r3a_bench_${arm}_$i.json 2> $OUT/r3a_bench_${arm}_$i.err
		python - $OUT/r3a_bench_${arm}_$i <<'PY'
import json, re, sys
d = json.load(open(sys.argv[1] + ".json"))
t = [l.strip() for l in open(sys.argv[1] + ".err") if re.search(r"seed\.(lookup_sort|c_concat_sort3)", l)]
print(f"{sys.argv[1]}: value {d['value']/1e6:.1f} e2e {d['e2e']['value']/1e6:.1f} Mbase/s parity {d.get('parity_checked')} "
      f"hbm {d['config']['hbm_used_gb']} GB | " + " | ".join(t))
PY
	done
done 2>&1 | tee $OUT/r3a_bench_summary.txt
# the default build as shipped, with the reference beside it: parity of the records
timeout 1800 python bench.py --gpus 1 --steps 20 --warmup 5 > $OUT/r3a_bench_parity.json 2> $OUT/r3a_bench_parity.err
python -c "import json; d = json.load(open('$OUT/r3a_bench_parity.json')); print('parity run: value', round(d['value'] / 1e6, 1), 'parity_checked', d['parity_checked'], 'hbm', d['config']['hbm_used_gb'])"
