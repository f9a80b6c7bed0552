#!/bin/bash
# round 2, call F (1 GPU): determinism stress, full suite, bench after the compaction
mkdir -p gpurun_out; rm -f gpurun_out/parity_refbuild.jsonl
timeout 600 python tools/stress_determinism.py 120 1 0 0.0 > gpurun_out/f_stress_coord.log 2>&1; tail -4 gpurun_out/f_stress_coord.log
timeout 600 python tools/stress_determinism.py 60 1 1 0.1 > gpurun_out/f_stress_both.log 2>&1; tail -2 gpurun_out/f_stress_both.log
timeout 2400 python -m pytest tests -m gpu -q > gpurun_out/f_pytest.log 2>&1; echo "pytest rc=$?"; grep -E "passed|failed|FAILED|ERROR" gpurun_out/f_pytest.log | tail -12
timeout 600 python bench.py --steps 20 --warmup 5 > gpurun_out/f_bench_ours.json 2> gpurun_out/f_bench_ours.err; echo "bench ours rc=$?"; tail -3 gpurun_out/f_bench_ours.err
for cfg in C3 C4; do timeout 600 python bench.py --steps 10 --warmup 3 --config $cfg --no-cpu-baseline > gpurun_out/f_bench_ours_$cfg.json 2> gpurun_out/f_bench_ours_$cfg.err; echo "bench $cfg rc=$?"; done
python - <<'PY'
import json, glob
for f in sorted(glob.glob('gpurun_out/f_bench_*.json')):
    try:
        d = json.loads([l for l in open(f) if l.startswith('{')][-1])
        print(f, 'value %.1f' % d['value'], 'ms %.3f' % d['ms_per_step'], 'e2e %.1f (%.3f ms)' % (d['e2e']['value'], d['e2e']['ms_per_step']), {k: round(v,3) for k,v in (d.get('stage_ms') or {}).items()}, d.get('roofline_issue'), sep='\n   ')
    except Exception as e:
        print(f, 'ERR', e)
PY
