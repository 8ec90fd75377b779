B="python bench.py --steps 300 --warmup 10 --no-extra --no-cpu-baseline --no-parity --e2e-sync"
run() { name=$1; shift; env "$@" $B $EXTRA 2>&1 | tail -1 | python -c "
import json,sys
d=json.loads(sys.stdin.read())
print('%s value %.1fM us/step %.1f e2e %.1fM' % ('$name', d['value']/1e6, d['ms_per_step']*1e3, d['e2e']['value']/1e6), d['step_us'])
"; }
for F in 1 0; do
EXTRA="--workload c2"; run fused${F}_write PAINTRL_FUSED=$F
EXTRA="--workload c2 --no-flush"; run fused${F}_noflush PAINTRL_FUSED=$F
done
ncu --metrics gpu__time_duration.sum --clock-control none -s 10 -c 30 --csv --log-file gpurun_out/launches_fused.csv env PAINTRL_FUSED=1 python bench.py --steps 20 --warmup 5 --no-extra --no-cpu-baseline --no-parity --e2e-sync > /dev/null 2>&1
grep -E "step_fused|fill" gpurun_out/launches_fused.csv | head -12
