#!/bin/bash
# First GPU call of a round: everything that has to be (re-)confirmed on a device, in one gpurun invocation.
#   /usr/local/graft/bin/gpurun --timeout 1800 -- 'bash tools/gpu_round_start.sh r2'   (about 20 minutes of box time)
# Writes into gpurun_out/ (merged back by gpurun); copy what should be judged into profiles/ afterwards.
# Order: tests first (the `reconstruct` kernels had their first device run pending at the end of round 1), then the
# bench lines WITHOUT a profiler, only then the ncu passes of the same commands.
tag=${1:-rN}
out=gpurun_out
mkdir -p $out
cd "${GRAFT_REPO_ROOT:-.}"
export PYTHONUNBUFFERED=1

echo "== M-step scatter microbenchmark (atomics vs the gather formulation)"
timeout 300 ./tools/ubench/mstep_scatter > $out/${tag}_ubench_mstep_scatter.txt 2>&1; echo "ubench rc=$?"; cat $out/${tag}_ubench_mstep_scatter.txt

echo "== pytest -m gpu"
timeout 900 python -m pytest tests -m gpu -x -q > $out/${tag}_pytest_gpu.log 2>&1; echo "pytest rc=$?"
tail -5 $out/${tag}_pytest_gpu.log

echo "== smoke"
timeout 300 python __graft_entry__.py --smoke > $out/${tag}_smoke.log 2>&1; echo "smoke rc=$?"; tail -2 $out/${tag}_smoke.log

echo "== bench (C2, model 4)"
timeout 900 python bench.py --steps 50 --warmup 5 > $out/${tag}_bench_c2.json 2> $out/${tag}_bench_c2.err; echo "bench rc=$?"
tail -c 600 $out/${tag}_bench_c2.json; echo

echo "== reconstruct bench (one sample, 96-sample cohort)"
timeout 900 python tools/bench_reconstruct.py > $out/${tag}_bench_reconstruct.json 2> $out/${tag}_bench_reconstruct.err
echo "bench_reconstruct rc=$?"; tail -c 1500 $out/${tag}_bench_reconstruct.json; echo; tail -3 $out/${tag}_bench_reconstruct.err

echo "== ncu launch lists (only after the commands above exited 0 without ncu)"
timeout 900 ncu --metrics gpu__time_duration.sum --clock-control none -c 400 --csv --log-file $out/${tag}_launches_c2.csv \
  python bench.py --steps 2 --warmup 1 --no-cpu > $out/${tag}_ncu_bench.log 2>&1; echo "ncu bench rc=$?"
timeout 900 ncu --metrics gpu__time_duration.sum --clock-control none -k regex:k_hmm -c 40 --csv \
  --log-file $out/${tag}_launches_reconstruct.csv python tools/bench_reconstruct.py --samples 16 --repeat 1 \
  > $out/${tag}_ncu_reconstruct.log 2>&1; echo "ncu reconstruct rc=$?"

echo "== ncu full capture: the HMM chain kernel of the cohort launch (launch index: emission, exp, chain per call)"
timeout 900 ncu --set full --clock-control none --import-source on -k regex:k_hmm_chain -s 2 -c 1 -o $out/${tag}_hmm_chain \
  python tools/bench_reconstruct.py --samples 16 --repeat 1 > $out/${tag}_ncu_full_reconstruct.log 2>&1; echo "ncu full rc=$?"
ncu -i $out/${tag}_hmm_chain.ncu-rep --page raw --csv > $out/${tag}_hmm_chain_raw.csv 2>/dev/null
python profiles/ncu_extract.py $out/${tag}_hmm_chain_raw.csv > $out/${tag}_hmm_chain_summary.txt 2>&1
tail -30 $out/${tag}_hmm_chain_summary.txt

echo "== compute-sanitizer (memcheck, then racecheck) on small runs: smoke() and the reconstruct golden cases"
timeout 900 compute-sanitizer --tool memcheck --error-exitcode 9 python __graft_entry__.py --smoke \
  > $out/${tag}_memcheck_smoke.log 2>&1; echo "memcheck smoke rc=$?"; tail -3 $out/${tag}_memcheck_smoke.log
timeout 900 compute-sanitizer --tool memcheck --error-exitcode 9 python -m pytest tests/test_zz_reconstruct_gpu.py -m gpu -q \
  -k "golden or other_haplotype" > $out/${tag}_memcheck_reconstruct.log 2>&1; echo "memcheck reconstruct rc=$?"
tail -3 $out/${tag}_memcheck_reconstruct.log
timeout 900 compute-sanitizer --tool racecheck --error-exitcode 9 python -m pytest tests/test_zz_reconstruct_gpu.py -m gpu -q \
  -k "golden" > $out/${tag}_racecheck_reconstruct.log 2>&1; echo "racecheck reconstruct rc=$?"
tail -3 $out/${tag}_racecheck_reconstruct.log

echo "== model 1"
timeout 900 python bench.py --model 1 --steps 20 --warmup 3 --no-cpu > $out/${tag}_bench_c2_model1.json 2> $out/${tag}_bench_c2_model1.err; echo "m1 rc=$?"
python - <<PY
import json
n = "${tag}_bench_c2_model1"
try:
    d = json.loads(open("$out/" + n + ".json").read().strip().splitlines()[-1])
    print(n, "ms_per_step", d["ms_per_step"], "row_pass_ms", d["roofline"]["per_kernel_ms"]["row_pass"])
except Exception as e:
    print(n, "unreadable:", e)
PY
