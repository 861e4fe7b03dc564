#!/bin/bash
# tools/gpu_round.sh <tag> [tests] [full] [sweep]: one GPU visit -- (tests) pytest -m gpu, the default bench line, the ncu launch list of
# two steady-state passes, (full) one ncu --set full capture of the same passes, (sweep) the four shapes of BASELINE configs[3].
tag=$1; shift
mkdir -p gpurun_out
for opt in "$@"; do eval "do_$opt=1"; done
if [ -n "$do_tests" ]; then
  ( time timeout 1500 python -m pytest tests -m gpu -x -q ) > gpurun_out/${tag}_pytest_gpu.log 2>&1; tail -4 gpurun_out/${tag}_pytest_gpu.log
fi
timeout 600 python bench.py --steps 2000 --warmup 200 ${BENCH_ARGS} 2> gpurun_out/${tag}_bench.err | tee gpurun_out/${tag}_bench.json | python -c "
import sys,json; d=json.loads(sys.stdin.read().strip().splitlines()[-1]); print('value %.4g  us/pass %.1f  frac %.3f  e2e %s  ended/pass %.0f' % (d['value'], d['roofline']['launch_us'], d['roofline']['frac'], d['e2e']['value'], d['config']['phase']['ended_envs_per_pass']))"
timeout 300 python bench.py --steps 20 --warmup 5 --no-cpu-baseline --no-e2e 2>/dev/null | tee gpurun_out/${tag}_bench_driver_args.json | python -c "
import sys,json; d=json.loads(sys.stdin.read().strip().splitlines()[-1]); print('driver-style 20 steps: value %.4g us/pass %.1f' % (d['value'], d['roofline']['launch_us']))"
DCM_PROFILE_AT=100 timeout 600 ncu --metrics gpu__time_duration.sum --clock-control none --profile-from-start off --csv --log-file gpurun_out/${tag}_launches.csv python bench.py --steps 200 --warmup 20 --no-e2e --no-cpu-baseline > /dev/null 2>&1
python - <<PY
import csv
rows=[r for r in csv.reader(open('gpurun_out/${tag}_launches.csv')) if len(r)>5 and r[0].isdigit()]
print([(r[4][:22], round(float(r[-1])/1000,1)) for r in rows])
PY
if [ -n "$do_full" ]; then
  DCM_PROFILE_AT=100 timeout 900 ncu --set full --clock-control none --import-source on --profile-from-start off -o gpurun_out/prof_${tag} -f python bench.py --steps 200 --warmup 20 --no-e2e --no-cpu-baseline > gpurun_out/${tag}_ncu_full.log 2>&1
  ls -la gpurun_out/prof_${tag}.ncu-rep
fi
if [ -n "$do_sweep" ]; then
  for shape in "10 20" "20 50" "30 100" "50 200"; do set -- $shape
    timeout 300 python bench.py --agents $1 --tasks $2 --steps 1000 --warmup 100 --no-e2e --no-cpu-baseline 2>/dev/null | tee -a gpurun_out/${tag}_shape_sweep.jsonl | python -c "
import sys,json; d=json.loads(sys.stdin.read().strip().splitlines()[-1]); print('$1A/$2T value %.4g us/pass %.1f frac %.3f' % (d['value'], d['roofline']['launch_us'], d['roofline']['frac']))"
  done
fi
if [ -n "$do_smoke" ]; then
  ( time python -c "import __graft_entry__ as g; g.smoke()" ) > gpurun_out/${tag}_smoke.log 2>&1; tail -4 gpurun_out/${tag}_smoke.log
fi
if [ -n "$do_refarm" ]; then
  timeout 600 python bench.py --impl reference 2>/dev/null
fi
if [ -n "$do_sanitize" ]; then bash tools/sanitize.sh $tag; fi
if [ -n "$do_greedy" ]; then
  timeout 300 python bench.py --policy greedy --steps 1000 --warmup 100 --no-cpu-baseline 2>/dev/null | tee gpurun_out/${tag}_bench_greedy.json | python -c "
import sys,json; d=json.loads(sys.stdin.read().strip().splitlines()[-1]); print('greedy: value %.4g us/pass %.1f frac %.3f e2e %.4g' % (d['value'], d['roofline']['launch_us'], d['roofline']['frac'], d['e2e']['value']))"
fi
if [ -n "$do_rollout" ]; then
  timeout 300 python bench.py --mode rollout --fused --iters 3 2>/dev/null | tee gpurun_out/${tag}_config5.jsonl | python -c "
import sys,json; d=json.loads(sys.stdin.read().strip().splitlines()[-1]); print('rollout --fused: value %.4g ms/iter %.1f' % (d['value'], d['ms_per_step']))"
fi
