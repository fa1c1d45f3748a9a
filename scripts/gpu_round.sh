# usage: [SKIP_TESTS=1] [SKIP_BENCH=1] bash scripts/gpu_round.sh <tag> [ncu] [tune] [c5] [ncufull]   -- GPU tests + bench (+ optional ncu launch list, tuning sweep)
TAG=${1:-x}
mkdir -p gpurun_out
nvidia-smi -L | head -2; nproc
[ -z "$SKIP_TESTS" ] && timeout 1500 python -m pytest tests -m gpu -q --timeout 900 --durations=8 > gpurun_out/pytest_$TAG.log 2>&1; echo pytest rc=$?; tail -25 gpurun_out/pytest_$TAG.log
[ -z "$SKIP_BENCH" ] && timeout 600 python bench.py --steps 20 --warmup 5 > gpurun_out/bench_$TAG.json 2> gpurun_out/bench_$TAG.err; echo bench rc=$?
python - <<PY
import json
try:
    d=json.loads(open('gpurun_out/bench_$TAG.json').read().strip().splitlines()[-1])
    print('ms/frame', round(d['ms_per_step'],4), 'e2e ms', round(d['e2e']['ms_per_step'],4), 'e2e f32 ms', round(d['e2e_float_image']['ms_per_step'],4), 'G/s', round(d['value']/1e9,3))
    print({k:v['ms'] for k,v in d['stages'].items()}, d['sort_breakdown'])
    print('roofline', {k: d['roofline'].get(k) for k in ('achieved','frac','peak','E_examined_pairs','E_contrib')})
    print('roofline_sort', d['roofline_sort']['achieved'], d['roofline_sort']['frac'], 'clocks', d['clocks'])
    print('cpu', d.get('cpu_baseline',{}).get('ms_per_frame'), 'orbit', {k: d.get('orbit_n1',{}).get(k) for k in ('ms_per_step','frames_per_second','e2e_ms_per_step','consumed_frames_verified','flow_control_timeouts')})
except Exception as e:
    print('bench parse failed', e)
PY
tail -5 gpurun_out/bench_$TAG.err
for a in "$@"; do
if [ "$a" = "ncu" ]; then
ncu --metrics gpu__time_duration.sum --clock-control none -c 300 --csv --log-file gpurun_out/launches_$TAG.csv python bench.py --steps 2 --warmup 3 --no-cpu-baseline --no-orbit > gpurun_out/ncu_bench_$TAG.log 2>&1; echo ncu rc=$?
fi
if [ "$a" = "tune" ]; then
export LCGS_TUNING=1
for v in 2 3 4 5 6 7 8; do LCGS_SORT_VARIANT=$v timeout 120 python scripts/tune_frame.py C3 2>&1 | tail -1; done
for b in 32 64 256 1000000; do LCGS_EMIT_BIG=$b timeout 120 python scripts/tune_frame.py C3 2>&1 | tail -1; done
unset LCGS_TUNING
fi
if [ "$a" = "c5" ]; then
timeout 600 python bench.py --config C5 --shard rows --steps 10 --warmup 3 > gpurun_out/bench_c5_n1_$TAG.json 2> gpurun_out/bench_c5_n1_$TAG.err; echo bench_c5 rc=$?; tail -2 gpurun_out/bench_c5_n1_$TAG.err
python - <<PY
import json
try:
    d=json.loads(open('gpurun_out/bench_c5_n1_$TAG.json').read().strip().splitlines()[-1])
    print('C5 N=1 ms/frame', round(d['ms_per_step'],4), 'e2e', round(d['e2e']['ms_per_step'],4), d['tile_row_sharding']['per_rank_stage_ms'])
except Exception as e:
    print('parse failed', e)
PY
fi
if [ "$a" = "ncufull" ]; then
ncu --set full --clock-control none --import-source on -k "regex:blend2?_kernel|onesweep_pass|preprocess_fused|duplicate_keys_sorted|scan_compact|emit_big|tile_ranges|tile_order" -s 39 -c 13 -f -o gpurun_out/full_$TAG python bench.py --steps 2 --warmup 3 --no-cpu-baseline --no-orbit > gpurun_out/ncu_full_$TAG.log 2>&1; echo ncufull rc=$?
python scripts/ncu_export.py gpurun_out/full_$TAG.ncu-rep gpurun_out/full_$TAG.csv | tail -1
fi
done
