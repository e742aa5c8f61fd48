#!/bin/bash
# Head beside the forward recurrence (head_paced_kernel): early-dispatch trace, GPU suite, A/B timing of
# LFMQ_FWD_HEAD=0 / 1 (alternating), output comparison, and the cfg3 / predict workloads on the new build.
# Usage: tools/gpu_r03_head_beside_forward.sh OUTPUT_DIR   (run from the repository root; results go to OUTPUT_DIR/r03_*)
OUTDIR=${1:?usage: $0 OUTPUT_DIR}
mkdir -p "$OUTDIR"
O=$OUTDIR/r03
export R03_PREFIX=$O
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > ${O}_smi.txt 2>&1
cat ${O}_smi.txt

# 1. clock stamps of the paced head (CTA 0) during cfg2 train steps: forward counts already on its first tile when it
#    started, and per (t, tile) unit when h_t was there / when the unit was finished
LFMQ_TRACE_HEAD=1 timeout 300 python - > ${O}_trace.txt 2>&1 <<'PY'
import sys, numpy as np, torch
sys.path[:0] = ['.', 'oracle']
import bench
from lfm_quant_b200.engine import ForecasterEngine
w = bench.WORKLOADS['cfg2']
e = ForecasterEngine(max_batch=w['B'], seq_len=w['T'], n_inputs=w['F'], n_outputs=w['O'], num_hidden=w['H'],
                     num_layers=1, target_idx=bench.TARGET_IDX, precision='bf16', optimizer='Adadelta', seed=bench.SEED)
e.set_weights(bench.initial_weights(w))
x, y = (torch.from_numpy(a).cuda() for a in bench.synthetic(w['B'], np.random.default_rng(1), w))
for i in range(3):
    print('--- step', i, file=sys.stderr, flush=True)
    print(e.train_step(x, y, i, 0.6).cpu().numpy(), file=sys.stderr, flush=True)
PY
echo "trace rc $?"; grep -E "G=|unit +(0|1|2|3|10|11|30|31|46|47|60|61|80|81|94|95) " ${O}_trace.txt | tail -20

# 2. GPU suite (includes tests/test_gpu_head_beside_forward.py) and smoke
timeout 900 python -m pytest -q -m gpu tests > ${O}_pytest_gpu.log 2>&1
echo "pytest rc $?"; tail -5 ${O}_pytest_gpu.log
timeout 300 python __graft_entry__.py smoke > ${O}_smoke.log 2>&1
echo "smoke rc $?"; tail -3 ${O}_smoke.log

# 3. cfg2 timing, arms alternating
for r in 1 2 3; do
  for a in 0 1; do
    LFMQ_FWD_HEAD=$a timeout 300 python bench.py --no-cpu-baseline > ${O}_bench_head${a}_${r}.json 2> ${O}_bench_head${a}_${r}.err
  done
done

# 4. outputs: old once, new twice
LFMQ_FWD_HEAD=0 timeout 300 python bench.py --no-cpu-baseline --dump-outputs ${O}_dump_head0 > ${O}_dump_head0.json 2>&1
LFMQ_FWD_HEAD=1 timeout 300 python bench.py --no-cpu-baseline --dump-outputs ${O}_dump_head1a > ${O}_dump_head1a.json 2>&1
LFMQ_FWD_HEAD=1 timeout 300 python bench.py --no-cpu-baseline --dump-outputs ${O}_dump_head1b > ${O}_dump_head1b.json 2>&1

# 5. the other workloads on the new build
timeout 300 python bench.py --no-cpu-baseline --workload cfg3 > ${O}_bench_cfg3.json 2> ${O}_bench_cfg3.err
timeout 300 python bench.py --no-cpu-baseline --workload predict > ${O}_bench_predict.json 2> ${O}_bench_predict.err

python - <<'PY' | tee ${O}_summary.txt
import glob, json, os
import numpy as np
O = os.environ['R03_PREFIX']
def last(p):
    try:
        return json.loads(open(p).read().strip().splitlines()[-1])
    except Exception as e:
        return {'error': repr(e)}
for a in (0, 1):
    ms, fwd = [], []
    for r in (1, 2, 3):
        d = last('%s_bench_head%d_%d.json' % (O, a, r))
        if 'ms_per_step' not in d:
            print('head%d run %d' % (a, r), d); continue
        reg = d['roofline']['regions_ms_per_step']
        ms.append(d['ms_per_step']); fwd.append(reg['fwd'])
        print('LFMQ_FWD_HEAD=%d run %d: %.4f ms/step  regions %s  loss_check %s' % (
            a, r, d['ms_per_step'], {k: round(v, 4) for k, v in reg.items()}, d.get('loss_check', {}).get('ok')))
    if ms:
        print('LFMQ_FWD_HEAD=%d median %.4f ms (spread %.4f .. %.4f), fwd median %.4f ms' % (
            a, np.median(ms), min(ms), max(ms), np.median(fwd)))
def arrs(d):
    return {os.path.basename(f)[:-4]: np.load(f) for f in sorted(glob.glob(d + '/*.npy'))}
try:
    h0, h1a, h1b = (arrs('%s_dump_%s' % (O, n)) for n in ('head0', 'head1a', 'head1b'))
    for name in h0:
        a, b, c = (x[name].astype(np.float64) for x in (h0, h1a, h1b))
        print('%-28s old-new max|d| %.3e (rel %.3e)  new-new max|d| %.3e bit-identical %s' % (
            name, np.abs(a - b).max(), np.abs(a - b).max() / max(np.abs(a).max(), 1e-30), np.abs(b - c).max(),
            bool(np.array_equal(h1a[name], h1b[name]))))
except Exception as e:
    print('dump compare failed', repr(e))
for n in ('cfg3', 'predict'):
    d = last('%s_bench_%s.json' % (O, n))
    print(n, {k: d.get(k) for k in ('ms_per_step', 'value', 'metric', 'error') if k in d})
PY
