B="python bench.py --steps 300 --warmup 10 --no-extra --no-cpu-baseline --e2e-sync"
run() { name=$1; shift; env "$@" $B $EXTRA 2>&1 | tail -1 | python -c "
import json,sys
d=json.loads(sys.stdin.read())
print('%s value %.1fM us/step %.1f parity %s' % ('$name', d['value']/1e6, d['ms_per_step']*1e3, d.get('parity_check',{}).get('ok')), d['step_us']['median'], d['step_us']['back_to_back_warm_l2'])
"; }
for F in "-Xptxas=-allow-expensive-optimizations=true" "-Xptxas=-O3 -extra-device-vectorization"; do
PAINTRL_NVCC_EXTRA="$F" python -m paintrl_b200.build --force 2>&1 | tail -1
EXTRA="--workload c2"; run "c2[$F]" A=1
EXTRA="--workload c5 --steps 60"; run "c5[$F]" A=1
done
