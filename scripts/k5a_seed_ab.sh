# experiment: the seeded K5a trace against the parent build, alternating in one call (parent kernels built into
# deepemia_b200/libemia_parent.so from the parent commit with the NVCC_FLAGS of __graft_entry__.py; Python side identical)
set -u
O=${OUT:-${TMPDIR:-/tmp}/k5a_seed_ab}   # results (small files)
mkdir -p $O
D=$(mktemp -d)          # output dumps (large): compared here, not kept
trap 'rm -rf $D' EXIT
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > $O/gpu.csv
python -c "import __graft_entry__ as g; g.build(); g.smoke()" > $O/smoke.log 2>&1; echo "build+smoke: $?"
PARENT=$PWD/deepemia_b200/libemia_parent.so
NEW=$PWD/deepemia_b200/libemia.so
for r in 1 2 3; do for v in parent new; do
  lib=$PARENT; [ $v = new ] && lib=$NEW
  extra=""; [ $r = 1 ] && extra="--dump-outputs $D/dump_$v"
  EMIA_LIB_PATH=$lib timeout 900 python bench.py --gpus 1 --steps 20 --warmup 5 --no-cpu-baseline --no-flows --breakdown $extra \
    > $O/bench_${v}_$r.json 2> $O/bench_${v}_$r.err
  echo "bench $v $r: $? $(python -c "import json; d=json.loads(open('$O/bench_${v}_$r.json').read().strip().splitlines()[-1]); print(d['value'], d['ms_per_step'], d['gpu_launches'])")" \
    "k5_trace $(python -c "import json; print([json.loads(l)['stage_ms'].get('k5_trace') for l in open('$O/bench_${v}_$r.err') if l.startswith('{\"stage_ms')])")"
done; done
for f in $D/dump_parent/*; do cmp -s $f $D/dump_new/$(basename $f) && echo "same $(basename $f)" || echo "DIFF $(basename $f)"; done | sort | uniq -c | sort -rn | head -40
for r in 1 2 3; do for v in parent new; do
  lib=$PARENT; [ $v = new ] && lib=$NEW
  EMIA_LIB_PATH=$lib timeout 900 python bench.py --gpus 1 --steps 10 --warmup 3 --no-cpu-baseline --flows-only config2,config3a,config3b,config4 \
    > $O/flows_${v}_$r.json 2> $O/flows_${v}_$r.err
  echo "flows $v $r: $? $(python -c "import json; d=json.loads(open('$O/flows_${v}_$r.json').read().strip().splitlines()[-1]); print(*[(c, round(d[c]['ms_per_step'], 4)) for c in ('config2', 'config3a', 'config3b', 'config4')])")"
done; done
[ "${SKIP_SUITE:-0}" = 1 ] || { timeout 1500 python -m pytest -q -m gpu tests -p no:cacheprovider > $O/pytest_gpu.log 2>&1; echo "pytest gpu: $?"; tail -5 $O/pytest_gpu.log; }
timeout 300 python -m pytest -q -s tests/test_gpu_trace_seed.py -p no:cacheprovider > $O/pytest_seed.log 2>&1; echo "seed tests: $?"; grep -E "instances|masks|passed|failed" $O/pytest_seed.log
