#!/bin/bash
mkdir -p gpurun_out
for w in stream o12_decode train; do
  python bench.py --workload $w --no-cpu-baseline --steps 20 > gpurun_out/bench_$w.json 2> gpurun_out/bench_$w.err; echo "$w exit $?"
done
python - <<'PY'
import json
for w in ['stream','o12_decode','train']:
    try:
        j=json.loads(open(f'gpurun_out/bench_{w}.json').read().strip().split('\n')[-1])
        keys=['value','ms_per_step','per_chunk_ms','first_chunk_wall_ms_incl_d2h','exact_context_stream','tflops','clocks']
        print(w, {k:j[k] for k in keys if k in j})
    except Exception as e:
        print(w,'failed',e)
PY
