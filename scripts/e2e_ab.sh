# same-box A/B of the pipelined host entry: calls in flight, packer threads
run() { echo "$@ (host calls ${HC:-2})"; env "$@" timeout 300 python bench.py --steps 40 --warmup 3 --no-cpu-baseline --host-calls ${HC:-2} 2>/dev/null | tail -1 | python -c "
import json,sys; d=json.loads(sys.stdin.read()); print('   e2e', round(d['e2e']['value']), 'frames/s', round(d['e2e']['ms_per_step'],3), 'ms; one call at a time', round(d['e2e']['one_call_at_a_time']['value']))"; }
run CASA_X=0
HC=3 run CASA_HOST_DEPTH=3
HC=3 run CASA_HOST_DEPTH=3 CASA_HOST_THREADS=14
run CASA_HOST_THREADS=14
HC=4 run CASA_HOST_DEPTH=4
