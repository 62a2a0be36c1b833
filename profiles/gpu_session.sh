#!/bin/bash
# One GPU session (TAG=r02 bash profiles/gpu_session.sh, about an hour): full GPU suite (parity table to profiles/parity_<TAG>.json or $PSL_PARITY_JSON), smoke,
# the bench lines of every config + the reference arm, the ncu launch list and a full ncu capture of the step kernels.  Everything
# that must come back goes to gpurun_out/ (the .ncu-rep with sources is ~25 MB, under the 64 MiB merge limit).
# A/B switches (environment): PSL_LIB=/path/to/other.so (another build of the same sources), PSL_GEO_MMA=0 (FFMA geometry kernels),
# PSL_H2=0 / PSL_H2_BWD=0 (3xTF32 colour kernels), PSL_FUSED_TAIL=0, PSL_HASH_APPEND=0, PSL_OVERLAP=0, PSL_TC=0, PSL_TC_BWD=0,
# PSL_CLOCKS_MS=<ms|0> (clock sampler period).  The 2-GPU lines: profiles/gpu_session_n2.sh under `gpurun --gpus 2`.
mkdir -p gpurun_out
T=${TAG:-f1}
export PSL_PARITY_JSON=${PSL_PARITY_JSON:-$PWD/profiles/parity_${T}.json}     # the session's parity table, beside parity_r02.json
( time timeout 1200 python -m pytest tests -m gpu -q --maxfail=8 -p no:cacheprovider -rxX ) > gpurun_out/${T}_tests.log 2>&1
echo "tests exit $?"; grep -E "^(FAILED|ERROR)|passed|failed" gpurun_out/${T}_tests.log | tail -8
( time timeout 300 python -c "import __graft_entry__ as g; g.smoke()" ) > gpurun_out/${T}_smoke.log 2>&1; echo "smoke exit $?"; tail -2 gpurun_out/${T}_smoke.log
( time timeout 500 python bench.py ) > gpurun_out/${T}_bench_c2.json 2> gpurun_out/${T}_bench_c2.err; echo "bench c2 exit $?"
for c in c1 c3 c4 rerender; do
  ( time timeout 500 python bench.py --config $c ) > gpurun_out/${T}_bench_$c.json 2> gpurun_out/${T}_bench_$c.err; echo "bench $c exit $?"
done
( time timeout 600 python bench.py --impl reference --steps 2 --warmup 1 ) > gpurun_out/${T}_bench_ref.json 2> gpurun_out/${T}_bench_ref.err; echo "bench ref exit $?"
timeout 400 ncu --profile-from-start off --metrics gpu__time_duration.sum --clock-control none --csv --log-file gpurun_out/${T}_launches.csv python profiles/prof_step.py 1 2 > gpurun_out/${T}_ncu_launches.log 2>&1
echo "ncu launches exit $?"
timeout 900 ncu --profile-from-start off --set full --clock-control none --import-source on -k regex:"k_color_fwd_h2|k_color_bwd_h2|k_wgrad_tc|k_geo_fwd_mma|k_geo_bwd_mma|k_knn|k_scatter_segments|k_render_tail_map" -f -o gpurun_out/${T}_full python profiles/prof_step.py 1 2 > gpurun_out/${T}_ncu_full.log 2>&1
echo "ncu full exit $?"
python - <<'PY'
import json, os
T = os.environ.get('TAG', 'f1')
for c in ('c2', 'c1', 'c3', 'c4', 'rerender', 'ref'):
    try:
        d = json.loads([l for l in open(f'gpurun_out/{T}_bench_{c}.json').read().splitlines() if l.startswith('{')][-1])
        print(c, round(d['ms_per_step'], 3), 'ms/step', 'value', round(d['value'] / 1e6, 3), 'e2e', round(d['e2e']['value'] / 1e6, 3), (d.get('roofline') or {}).get('kernel'),
              round((d.get('roofline') or {}).get('frac', 0), 4), (d.get('cpu_baseline') or {}).get('value'))
    except Exception as e:
        print(c, 'no line', e)
PY
