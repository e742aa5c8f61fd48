#!/usr/bin/env python
"""Headline benchmark: train-step sequences/sec of the recurrent forecaster (BASELINE.json).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl native|reference] [--precision bf16|fp32]
                    [--workload cfg2|cfg3|predict|batcher] [--dump-outputs DIR]

--dump-outputs DIR writes what the last timed step returned as DIR/<name>.npy (see dump_outputs).  The inputs depend only
on the arguments, so two builds run with the same arguments can be compared output for output -- with a tolerance: runs
of one build (cfg2, bf16, 20 steps, one B200 at its 1000 W power limit) wrote weights up to 4.4e-5 apart, not
bit-identical.

Default workload (what the driver runs) = BASELINE.json configs[1]: synthetic B=4096, T=48, F=32, O=16, 1-layer LSTM
H=256, one full Train._train_step_point (fwd, weighted-MSE loss, BPTT, clip, Adadelta, MaxNorm).  N>1 = configs[3]:
the company-batch axis sharded, 4096 windows per rank (weak scaling), ONE NCCL all-reduce of the flat gradient.
Other workloads (for profiles/, one GPU): cfg3 = configs[2] (2-layer H=512 + dropout 0.2), predict = configs[4]
(forward only, B=65536), batcher = the sliding-window gather kernel (HBM-bound, GB/s).
Prints ONE JSON line on rank 0 (contract in the task statement: value, e2e, roofline, cpu_baseline, clocks ...).

`--impl reference` times the reference's CPU path.  The reference is TensorFlow/Keras Python and TensorFlow is
not installable here (no wheel in /opt/wheelhouse, no network), so that arm runs the NumPy restatement of the
same step (oracle/, kind "port") on the host cores, on the FULL workload (4096 windows per step) -- labelled as such.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
for _p in (ROOT, os.path.join(ROOT, 'oracle')):
    if _p not in sys.path:
        sys.path.insert(0, _p)

TARGET_IDX = 3
SEED = 521                       # reference default, scripts/lfm_quant.py:72
METRIC = 'train-step sequences/sec at B=4096,T=48,H=256'

# name -> (B per GPU, T, F, O, H, L, dropout, mode, BASELINE configs index, metric)
WORKLOADS = {
    'cfg2': dict(B=4096, T=48, F=32, O=16, H=256, L=1, dropout=0.0, mode='train', cfg_index=1, metric=METRIC),
    'cfg3': dict(B=4096, T=48, F=32, O=16, H=512, L=2, dropout=0.2, mode='train', cfg_index=2,
                 metric='train-step sequences/sec at B=4096,T=48,H=512,L=2,dropout'),
    'predict': dict(B=65536, T=48, F=32, O=16, H=256, L=1, dropout=0.0, mode='predict', cfg_index=4,
                    metric='predict sequences/sec at B=65536,T=48,H=256'),
    'batcher': dict(B=4096, T=48, F=32, O=16, H=256, L=1, dropout=0.0, mode='batcher', cfg_index=1,
                    metric='sliding-window batcher GB/s at B=4096,T=48,F=32,O=16'),
}
# module-level dims of the default workload (imported by tests/test_gpu_baseline_shapes.py)
T, F, O, H, L = 48, 32, 16, 256, 1


def flops_per_seq(w):
    """SURVEY 8(d): algorithmic gate-GEMM FLOPs per window: fwd 2*T*(I+H)*4H per layer, weight gradient the same,
    data gradient 2*T*4H*H per layer (+ 2*T*4H*I for layers above the first)."""
    fwd = wg = dg = 0.0
    for l in range(w['L']):
        I = w['F'] if l == 0 else w['H']
        fwd += 2.0 * w['T'] * (I + w['H']) * 4 * w['H']
        wg += 2.0 * w['T'] * (I + w['H']) * 4 * w['H']
        dg += 2.0 * w['T'] * 4 * w['H'] * w['H'] + (2.0 * w['T'] * 4 * w['H'] * I if l > 0 else 0.0)
    return fwd, dg, wg


def hbm_bytes_per_seq(w, predict=False, fused_head=False):
    """Algorithmic HBM bytes per window of the three gate-GEMM kernels (DESIGN.md section 4; activations are bf16).
    Per time step and layer:
    forward   reads the layer input (2 I) and writes h (2 H), and in training the saved gates (8 H) + cell state (2 H);
    backward  reads the saved gates (8 H), the cell state once (2 H: c_t is kept for the next step as c_{t-1}) and
              dLoss/dh (2 H; with the head fused into the kernel the 64-byte dLoss/dpred row instead), writes dz (8 H);
    weight gradient reads [x | h] (2 (I + H)) and dz (8 H)."""
    T, H = w['T'], w['H']
    fwd = bwd = wg = 0.0
    for l in range(w['L']):
        I = w['F'] if l == 0 else H
        fwd += T * (2.0 * I + 2.0 * H + (0.0 if predict else 10.0 * H))
        bwd += T * (8.0 * H + 2.0 * H + (64.0 if fused_head else 2.0 * H) + 8.0 * H)
        wg += T * (2.0 * (I + H) + 8.0 * H)
    return fwd, bwd, wg


DUMP_BYTES = 64 * 10 ** 6        # --dump-outputs writes at most this many bytes of array data in all


def dump_outputs(d, arrays):
    """Writes {name: float32 / float64 array} as d/<name>.npy ('/' in a name becomes '.').  Smallest first, each array
    gets an equal share of the DUMP_BYTES still unused; one larger than its share keeps a fixed, seeded sample of its
    rows (leading axis, in order), so every run with the same arguments stores the same elements."""
    os.makedirs(d, exist_ok=True)
    left = DUMP_BYTES
    for i, name in enumerate(sorted(arrays, key=lambda n: arrays[n].nbytes)):
        a = np.asarray(arrays[name])
        assert a.dtype in (np.float32, np.float64), (name, a.dtype)
        share = left // (len(arrays) - i)
        if a.nbytes > share:
            keep = share // (a.nbytes // a.shape[0])
            a = a[np.sort(np.random.default_rng(SEED).choice(a.shape[0], keep, replace=False))]
        left -= a.nbytes
        np.save(os.path.join(d, name.replace('/', '.') + '.npy'), a)


def synthetic(batch, rng, w=None):
    w = w or WORKLOADS['cfg2']
    x = rng.standard_normal((batch, w['T'], w['F']), dtype=np.float32)
    y = rng.standard_normal((batch, w['T'], w['O']), dtype=np.float32)
    return x, y


def initial_weights(w=None):
    import lfm_oracle as orc
    w = w or WORKLOADS['cfg2']
    # W~U(-1,1) (init_scale=1.0, lfm_quant.py:54), U orthogonal, b=[0,1,0,0], gamma=1, beta=0, Glorot head
    return orc.init_params(w['L'], w['F'], w['O'], w['H'], init_scale=1.0, seed=SEED, dtype=np.float32)


def oracle_cfg(w):
    return dict(num_layers=w['L'], target_idx=TARGET_IDX, target_lambda=0.5, rnn_lambda=0.7, max_grad_norm=50.0,
                optimizer='Adadelta', max_norm=3.0, train=True, dropout=w['dropout'], recurrent_dropout=0.0, seed=SEED)


def cpu_port_seq_per_s(w, rows, steps, threads, warm=1):
    """Times oracle.train_step (fp32 NumPy; oracle.forward for the predict workload) on `rows` windows per step.  The
    BLAS thread count is scanned on a small sample (per-step matmuls this small do not scale to 128 threads) and the
    best one is kept; returns (windows/s, seconds/step, threads used)."""
    import lfm_oracle as orc
    from threadpoolctl import threadpool_limits
    rng = np.random.default_rng(SEED)
    cfg = oracle_cfg(w)

    def run(n_threads, n_rows, n_steps, warm):
        x, y = synthetic(n_rows, rng, w)
        with threadpool_limits(limits=n_threads):
            params = initial_weights(w)
            slots = orc.zero_slots('Adadelta', params)

            def one(it):
                nonlocal params
                if w['mode'] == 'predict':
                    orc.forward(params, x, num_layers=w['L'])
                else:
                    params, *_ = orc.train_step(params, slots, x, y, it, cfg, lr=0.6)
            for it in range(warm):
                one(it)
            t0 = time.perf_counter()
            for it in range(n_steps):
                one(warm + it)
            return (time.perf_counter() - t0) / n_steps

    cands = sorted({min(threads, c) for c in (4, 8, 16, 32, threads)})
    best = min(cands, key=lambda c: run(c, min(rows, 256), 1, 1))
    per_step = run(best, rows, steps, warm)
    return rows / per_step, per_step, best


class ClockSampler(object):
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""
    Q = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,'
         'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
         'clocks_event_reasons.sw_power_cap')

    def __init__(self, index=0):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.index), '--query-gpu=' + self.Q,
                                          '--format=csv,noheader,nounits', '-lms', '100'],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), [c.strip() for c in line.split(',')]))

    def stop(self, t0, t1):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        time.sleep(0.15)
        self.proc.terminate()
        rows = [r for (ts, r) in self.rows if t0 <= ts <= t1 + 0.2] or [r for (_, r) in self.rows[-3:]]
        sm, mx, pw, reasons = [], [], [], set()
        for r in rows:
            try:
                sm.append(float(r[0]))
                mx.append(float(r[1]))
                pw.append(float(r[2]))
            except Exception:
                continue
            for name, v in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), r[3:7]):
                if v.lower().startswith('active'):
                    reasons.add(name)
        return {'sm_mhz': float(np.median(sm)) if sm else None, 'sm_max_mhz': max(mx) if mx else None,
                'power_w_max': max(pw) if pw else None, 'reasons': sorted(reasons), 'samples': len(sm)}


def workload_text(w, B, world):
    if w['mode'] == 'predict':
        return ('BASELINE configs[4]: predict.py inference path, B=%d, T=%d, F=%d, O=%d, 1-layer LSTM H=%d; forward only'
                % (B, w['T'], w['F'], w['O'], w['H']))
    return ('BASELINE configs[%d]: B=%d per GPU (global %d), T=%d, F=%d, O=%d, %d-layer LSTM H=%d%s, Adadelta lr 0.6, '
            'clip 50, MaxNorm 3; full train step'
            % (w['cfg_index'] if world == 1 else 3, B, B * world, w['T'], w['F'], w['O'], w['L'], w['H'],
               ', dropout %.1f' % w['dropout'] if w['dropout'] > 0 else ''))


def run_reference(args, w, rank, world):
    """Reference arm: CPU path of the same step on the host cores, full workload per step, rank 0 only."""
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    rows = args.cpu_rows or (w['B'] if w['mode'] == 'train' else 4096)
    v, s_per_step, used = cpu_port_seq_per_s(w, rows, args.steps, cores, warm=args.warmup)   # W untimed steps, as asked
    full = rows == w['B']
    line = {
        'impl': 'reference', 'metric': w['metric'], 'value': v, 'unit': 'sequences/s', 'n_gpus': args.gpus,
        'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': s_per_step * 1e3, 'higher_is_better': True,
        'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': {'workload': workload_text(w, w['B'], 1) + (' -- all %d windows per step' % rows if full else
                                                              ' (bounded sample of %d windows per step)' % rows),
                   'same_config': bool(full)},
        'cpu_baseline': {'value': v, 'unit': 'sequences/s', 'cores': used, 'kind': 'port',
                         'sample': '%d of %d windows per step, %d steps after %d warm-up; NumPy fp32 restatement (oracle/) '
                                   '-- TensorFlow (the reference runtime) is not installable in this image; host has %d '
                                   'cores, `cores` = the BLAS thread count that was fastest and was used'
                                   % (rows, w['B'], args.steps, args.warmup, cores)},
        'e2e': {'value': v, 'unit': 'sequences/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
    }
    print(json.dumps(line), flush=True)


def load_peaks():
    pk = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.isfile(pk):
        p = json.load(open(pk))
        return dict(burst=p.get('bf16_tflops') or 1590.0, sustained=p.get('bf16_tflops_sustained') or 1400.0,
                    hbm=p.get('hbm_gbs') or 6650.0, src='MEASURED_PEAKS.json', sm_max=p.get('sm_max_mhz') or 1965.0,
                    sustained_mhz=(p.get('clocks_under_load') or {}).get('sm_mhz_median'))
    return dict(burst=1590.0, sustained=1400.0, hbm=6650.0, src='fallback (B200_PROFILING.md)', sm_max=1965.0,
                sustained_mhz=1300.0)


def pick_peak(peaks, clocks):
    """The sustained cuBLAS figure was measured at ~1365 MHz under the 1 kW power cap; a step that runs at the full
    clock with no power cap is compared with the burst figure (VERDICT r1 weak #4)."""
    sm = (clocks or {}).get('sm_mhz')
    capped = 'sw_power_cap' in ((clocks or {}).get('reasons') or [])
    if sm is not None and not capped and sm >= 0.9 * peaks['sm_max']:
        return peaks['burst'], 'burst (bf16_tflops): timed region ran at %.0f MHz with no power cap' % sm
    return peaks['sustained'], 'sustained (bf16_tflops_sustained): clocks %.0f MHz / power-capped' % (sm or 0)


def run_batcher(args, w, dev):
    """HBM-bound sliding-window gather (Dataset.get_batch, data_processing.py:307-368) over a resident fp64 table."""
    import torch
    from lfm_quant_b200.engine import gather_batch
    from lfm_quant_b200 import _native
    B, Tn, Fn, On = w['B'], w['T'], w['F'], w['O']
    stride, fn = 3, 3
    rng = np.random.default_rng(SEED)
    n_keys, n_months = 2000, 400                       # 800 K rows x 36 columns of fp64 = 230 MB: larger than L2
    n_cols = 3 + Fn + 1
    table = rng.standard_normal((n_keys * n_months, n_cols))
    table[:, -1] = np.exp(rng.normal(5, 2, size=table.shape[0]))
    n_rows = table.shape[0]
    span = (Tn - 1) * stride + 1
    ends = rng.integers(span + 1, n_rows - fn - 1, size=(8, B))
    idx = []
    for e in ends:
        inp = np.stack([e - span + 1, e, np.zeros_like(e)], axis=1).astype(np.int32)
        tar = np.stack([e - span + 1 + fn, e + fn, np.zeros_like(e)], axis=1).astype(np.int32)
        idx.append((torch.from_numpy(inp).to(dev), torch.from_numpy(tar).to(dev)))
    cu = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    kw = dict(seq_len=Tn, stride=stride, inp_cols=cu(np.arange(3, 3 + Fn, dtype=np.int32)),
              fin_cols=cu(np.arange(3, 3 + On, dtype=np.int32)), seq_norm_col=n_cols - 1,
              center=cu(rng.standard_normal(Fn)), scale=cu(np.abs(rng.standard_normal(Fn)) + 0.5),
              scale_flag=cu(np.ones(Fn, dtype=np.uint8)), aux_flag=cu(np.zeros(Fn, dtype=np.uint8)), log_squasher=True,
              aux_masking=False)
    tab = cu(table)
    for i in range(args.warmup):
        gather_batch(tab, *idx[i % 8], **kw)
    torch.cuda.synchronize()
    l0 = _native.load().lfmq_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(args.steps):
        out = gather_batch(tab, *idx[i % 8], **kw)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / args.steps
    launches = _native.load().lfmq_launch_count() - l0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {n: t.cpu().numpy() for n, t in zip(('x', 'y', 'seq_norm'), out)})
    written = B * Tn * (Fn + On) * 4 + B * 8
    read = B * Tn * (Fn + On) * 8 + B * 24
    peaks = load_peaks()
    gbs = (written + read) / (ms * 1e-3) / 1e9
    line = {'metric': w['metric'], 'value': gbs, 'unit': 'GB/s', 'n_gpus': 1, 'steps': args.steps, 'warmup': args.warmup,
            'ms_per_step': ms, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f64',
            'data': 'synthetic',
            'config': {'workload': 'Dataset.get_batch gather: B=%d windows, T=%d, F=%d, O=%d, stride %d, fp64 table of '
                                   '%d rows x %d columns (%.0f MB, resident)' % (B, Tn, Fn, On, stride, n_rows, n_cols,
                                                                                 table.nbytes / 1e6),
                       'l2': '8 rotating index sets over a table larger than L2'},
            'sequences_per_s': B / (ms * 1e-3), 'gpu_launches': int(launches),
            'roofline': {'bound': 'hbm', 'achieved': gbs, 'peak': peaks['hbm'], 'unit': 'GB/s', 'frac': gbs / peaks['hbm'],
                         'traffic': None, 'kernel': 'gather_batch_vec_kernel',
                         'algorithmic_bytes': {'written': written, 'read': read},
                         'peak_source': peaks['src'] + ' (hbm_gbs)'}}
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='native', choices=['native', 'reference'])
    ap.add_argument('--workload', default='cfg2', choices=sorted(WORKLOADS))
    ap.add_argument('--precision', default=os.environ.get('LFMQ_BENCH_PRECISION', 'bf16'),
                    choices=['bf16', 'fp32', 'bf16x3'])
    ap.add_argument('--batch', type=int, default=0, help='windows per GPU (default: the workload\'s)')
    ap.add_argument('--cpu-rows', type=int, default=0, help='windows per step of the CPU arm (default: all)')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-loss-check', action='store_true')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='write what the last timed step returned as DIR/<name>.npy')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl == 'reference':
        ap.error('--dump-outputs applies to --impl native (the reference arm draws its own inputs)')
    args.warmup = max(args.warmup, 3)
    w = dict(WORKLOADS[args.workload])
    if args.batch:
        w['B'] = args.batch

    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    if args.impl == 'reference':
        run_reference(args, w, rank, world)
        return

    import torch
    import torch.distributed as dist
    from lfm_quant_b200.engine import ForecasterEngine

    torch.cuda.set_device(local_rank)
    dev = torch.device('cuda', local_rank)
    if w['mode'] == 'batcher':
        if rank == 0:
            run_batcher(args, w, dev)
        return
    if world > 1:
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        dist.init_process_group('nccl', device_id=dev)
    B, Tn, Fn, On, Hn, Ln = w['B'], w['T'], w['F'], w['O'], w['H'], w['L']
    predict = w['mode'] == 'predict'

    def make_engine(precision):
        return ForecasterEngine(max_batch=B, seq_len=Tn, n_inputs=Fn, n_outputs=On, num_hidden=Hn, num_layers=Ln,
                                target_idx=TARGET_IDX, train=not predict, precision=precision, optimizer='Adadelta',
                                dropout=w['dropout'], target_lambda=0.5, rnn_lambda=0.7, max_grad_norm=50.0, max_norm=3.0,
                                seed=SEED, forward_only=predict)

    eng = make_engine(args.precision)
    eng.set_weights(initial_weights(w))
    lr = 0.6
    rng = np.random.default_rng(SEED + 1000 * rank)
    NB = 2 if predict else 4                            # rotating resident batches
    host = [synthetic(B, rng, w) for _ in range(NB)]
    pinned = [(torch.from_numpy(x).pin_memory(), torch.from_numpy(y).pin_memory()) for x, y in host]
    resident = [(px.to(dev), py.to(dev)) for px, py in pinned]
    denoms = None
    if world > 1:                                       # global loss denominators, once per batch (SURVEY 8e)
        denoms = []
        for _, y in resident:
            d = eng.mask_count(y)
            dist.all_reduce(d)
            denoms.append(d)

    preds_dev = torch.empty(B, Tn, On, dtype=torch.float32, device=dev) if predict else None
    preds_host = torch.empty(B, Tn, On, dtype=torch.float32).pin_memory() if predict else None

    def step_resident(i, e=None):
        e = e or eng
        x, y = resident[i % NB]
        if predict:
            return e.forward(x, out=preds_dev)
        if world > 1:
            return e.train_step_dp(x, y, i, lr, rank * B, denoms[i % NB])
        return e.train_step(x, y, i, lr)

    # e2e: the public host-batch API (lfm_quant_b200.engine.HostBatchPipeline): every step copies its own inputs
    # from pinned host memory (H2D on a copy stream, overlapped with the previous step's compute) and reads its
    # {loss, mse_0} back to the host.  predict: H2D of the windows, forward, D2H of all predictions, every call.
    from lfm_quant_b200.engine import HostBatchPipeline
    pipe = None
    if not predict:
        step_fn = (lambda x, y, i, lr_: eng.train_step_dp(x, y, i, lr_, rank * B, denoms[i % NB])) if world > 1 else None
        pipe = HostBatchPipeline(eng, B, step_fn=step_fn)

    def step_e2e(i):
        if predict:
            xd = pinned[i % NB][0].to(dev, non_blocking=True)
            eng.forward(xd, out=preds_dev)
            preds_host.copy_(preds_dev, non_blocking=True)
            return None
        return pipe.step(pinned[i % NB][0], pinned[i % NB][1], i, lr, next_batch=pinned[(i + 1) % NB])

    def sync():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, k, first):
        sync()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(k):
            last = fn(first + i)
        e1.record()
        sync()
        ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()), last

    it = 0
    for _ in range(args.warmup):
        step_resident(it)
        it += 1
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        time.sleep(0.3)
    eng.profile(True)
    l0 = eng.launch_count
    t0 = time.perf_counter()
    ms, last = timed(step_resident, args.steps, it)
    t1 = time.perf_counter()
    launches = eng.launch_count - l0
    regions = eng.profile_read()
    eng.profile(False)
    it += args.steps
    clocks = sampler.stop(t0, t1) if rank == 0 else None
    outputs = None
    if args.dump_outputs and rank == 0:
        # copied now: the e2e steps below overwrite preds_dev and move the weights on
        if predict:
            outputs = {'preds': last.cpu().numpy()}
        else:
            outputs = {'loss_mse': last.cpu().numpy()}
            outputs.update(('weights/' + spec[0], a) for spec, a in zip(eng.specs, eng.get_weights(trainable_only=False)))
    for _ in range(2):
        step_e2e(it)
        it += 1
    ms_e2e, _ = timed(step_e2e, args.steps, it)
    if pipe is not None:
        pipe.finish()
    it += args.steps
    final = None if predict else step_resident(it).float().cpu().numpy()
    n_steps_total = it + 1

    if rank == 0:
        value = world * B * args.steps / (ms * 1e-3)
        e2e = world * B * args.steps / (ms_e2e * 1e-3)
        peaks = load_peaks()
        peak_tf, peak_why = pick_peak(peaks, clocks)
        k = args.steps
        fwd_ms, bwd_ms, wg_ms, head_ms = (regions[n][0] / k for n in ('fwd', 'bwd', 'wgrad', 'head'))
        f_fwd, f_dg, f_wg = (f * B for f in flops_per_seq(w))

        def tf(flop, ms_):
            return flop / (ms_ * 1e-3) / 1e12 if ms_ > 0 else None

        def entry(flop, ms_):
            a = tf(flop, ms_)
            return {'ms': ms_, 'tflops': a, 'frac_of_burst': (a or 0) / peaks['burst'],
                    'frac_of_sustained': (a or 0) / peaks['sustained']}

        # Per-kernel gate-GEMM figures.  Algorithmic FLOPs per launch = per-window figure (SURVEY 8d) x the windows one
        # launch processes; durations = CUDA events recorded by the library around each kernel inside the timed region
        # (lfmq_profile_*), on the stream the kernels run on.
        names = {'fwd': 'forward recurrence', 'bwd': 'backward recurrence', 'wgrad': 'weight-gradient GEMM'}
        if args.precision == 'bf16' and Hn == 256 and Ln == 1 and w['dropout'] == 0:
            names = {'fwd': 'lstm_fwd_tc_kernel', 'bwd': 'lstm_bwd_tc_kernel', 'wgrad': 'wgrad_tc_kernel'}
        per = {names['fwd']: entry(f_fwd, fwd_ms)}
        if not predict:
            per[names['bwd']] = entry(f_dg, bwd_ms)
            per[names['wgrad']] = entry(f_wg, wg_ms)
        # the DOMINANT kernel = the gate-GEMM kernel with the longest duration; the headline roofline is its own
        dom = max(per, key=lambda n: per[n]['ms'])
        dom_flop = {names['fwd']: f_fwd, names['bwd']: f_dg, names['wgrad']: f_wg}[dom]
        achieved = per[dom]['tflops']
        gate_ms = fwd_ms + (0 if predict else bwd_ms + wg_ms)
        agg = tf(f_fwd + (0 if predict else f_dg + f_wg), gate_ms)
        # DRAM traffic (dram__bytes_read.sum + dram__bytes_write.sum per launch) comes ONLY from a committed
        # `ncu --set full` capture: profiles/r0N_ncu_traffic.json is written by tools/ncu_traffic.py from the .ncu-rep
        # and names the capture it was parsed from.  No file (or the kernel missing from it) -> null.
        traffic, traffic_src = None, None
        for tp in ('r02_ncu_traffic.json', 'r01_ncu_traffic.json'):
            tp = os.path.join(ROOT, 'profiles', tp)
            if args.workload == 'cfg2' and args.precision == 'bf16' and os.path.isfile(tp):
                tj = json.load(open(tp))
                if dom in tj.get('dram_bytes_per_launch', {}):
                    traffic = float(tj['dram_bytes_per_launch'][dom])
                    traffic_src = tj.get('source')
                    break
        # Which roof binds the dominant kernel: the one that needs the longer time for the kernel's algorithmic work
        # (FLOPs / measured bf16 peak  vs  HBM bytes / measured copy bandwidth).  `achieved / peak / frac` are quoted
        # against that roof; both are listed under `roofs`.
        by_fwd, by_bwd, by_wg = (b_ * B for b_ in hbm_bytes_per_seq(w, predict, fused_head=names['bwd'] == 'lstm_bwd_tc_kernel'))
        dom_bytes = {names['fwd']: by_fwd, names['bwd']: by_bwd, names['wgrad']: by_wg}[dom]
        dom_ms = per[dom]['ms']
        gbs = dom_bytes / (dom_ms * 1e-3) / 1e9 if dom_ms > 0 else None
        t_tensor_ms = dom_flop / (peak_tf * 1e12) * 1e3
        t_hbm_ms = dom_bytes / (peaks['hbm'] * 1e9) * 1e3
        roofs = {'tensor': {'achieved': achieved, 'peak': peak_tf, 'unit': 'TFLOP/s',
                            'frac': (achieved / peak_tf) if achieved else None, 'min_ms': t_tensor_ms,
                            'algorithmic_flop_per_launch': dom_flop},
                 'hbm': {'achieved': gbs, 'peak': peaks['hbm'], 'unit': 'GB/s',
                         'frac': (gbs / peaks['hbm']) if gbs else None, 'min_ms': t_hbm_ms,
                         'algorithmic_bytes_per_launch': dom_bytes}}
        bound = 'hbm' if t_hbm_ms > t_tensor_ms else 'tensor'
        roofline = {
            'bound': bound, 'kernel': dom, 'achieved': roofs[bound]['achieved'], 'peak': roofs[bound]['peak'],
            'unit': roofs[bound]['unit'], 'frac': roofs[bound]['frac'], 'ms': dom_ms,
            'roofs': roofs,
            'algorithmic_flop_per_launch': dom_flop, 'algorithmic_bytes_per_launch': dom_bytes,
            'traffic': traffic, 'traffic_source': traffic_src,
            'peak_source': '%s; %s' % (peaks['src'], peak_why),
            'peaks': {'bf16_tflops_burst': peaks['burst'], 'bf16_tflops_sustained': peaks['sustained'],
                      'hbm_gbs': peaks['hbm']},
            'per_kernel': per,
            'all_gate_gemms': {'ms': gate_ms, 'tflops': agg, 'frac_of_burst': (agg or 0) / peaks['burst'],
                               'frac_of_sustained': (agg or 0) / peaks['sustained']},
            'regions_ms_per_step': {n: v[0] / k for n, v in regions.items()},
        }
        if not predict and Hn == 256 and Ln == 1:
            # HBM-bound pieces, algorithmic bytes (SURVEY 8d): backward recurrence reads the saved gates + 2x cell state
            # + the dpred tile and writes dz (bf16); the head reads h + y and writes the dpred tiles
            bwd_bytes = B * Tn * (4 * Hn * 2 + 2 * Hn * 2 + 64) + B * Tn * 4 * Hn * 2
            head_bytes = B * Tn * (Hn * 2 + On * 4) + B * Tn * 64
            roofline['hbm_bound_pieces'] = {
                'backward recurrence': {'algorithmic_bytes': bwd_bytes,
                                        'gbs': bwd_bytes / (bwd_ms * 1e-3) / 1e9 if bwd_ms > 0 else None,
                                        'frac': bwd_bytes / (bwd_ms * 1e-3) / 1e9 / peaks['hbm'] if bwd_ms > 0 else None},
                'head (fused pointwise tail)': {'ms': head_ms, 'algorithmic_bytes': head_bytes,
                                                'gbs': head_bytes / (head_ms * 1e-3) / 1e9 if head_ms > 0 else None,
                                                'frac': head_bytes / (head_ms * 1e-3) / 1e9 / peaks['hbm'] if head_ms > 0 else None}}
        if predict:
            h2d, d2h = B * Tn * Fn * 4, B * Tn * On * 4
        else:
            h2d, d2h = B * Tn * (Fn + On) * 4, 8
        line = {
            'metric': w['metric'], 'value': value, 'unit': 'sequences/s', 'n_gpus': world, 'steps': args.steps,
            'warmup': args.warmup, 'ms_per_step': ms / args.steps, 'higher_is_better': True, 'scaling': 'weak',
            'vs_baseline': None, 'dtype': {'bf16': 'bf16', 'fp32': 'f32', 'bf16x3': 'bf16x3'}[args.precision],
            'data': 'synthetic',
            'config': {'workload': workload_text(w, B, world),
                       'parallelism': 'dp%d' % world,
                       'l2': 'per-step working set (saved activations, >0.5 GB) exceeds the 126 MB L2; %d rotating '
                             'input batches' % NB,
                       'precision': args.precision},
            'e2e': {'value': e2e, 'unit': 'sequences/s', 'ms_per_step': ms_e2e / args.steps,
                    'h2d_bytes_per_step': int(world * h2d), 'd2h_bytes_per_step': int(d2h * world),
                    'h2d_bytes_per_step_per_gpu': int(h2d)},
            'gpu_launches': int(launches),
            'roofline': roofline,
            'clocks': clocks,
        }
        if final is not None:
            line['final_loss_mse'] = [float(final[0]), float(final[1])]
        if final is not None and not args.no_loss_check and world == 1 and args.precision != 'fp32' and w['dropout'] == 0:
            # replay the very same step sequence on the fp32 parity path (1e-4 vs the oracle) and hold the tensor-core
            # path's final {loss, mse_0} to the bound of tests/test_gpu_baseline_shapes.py (TRAJ_BOUND = 2e-3)
            e32 = make_engine('fp32')
            e32.set_weights(initial_weights(w))
            out = None
            for i in range(n_steps_total):
                out = step_resident(i, e32)
            f32 = out.float().cpu().numpy()
            e32.close()
            rel = float(np.max(np.abs(final[:2] - f32[:2]) / np.abs(f32[:2])))
            line['loss_check'] = {'fp32_final_loss_mse': [float(f32[0]), float(f32[1])], 'steps_replayed': n_steps_total,
                                  'max_rel_diff': rel, 'bound': 2e-3, 'ok': bool(rel < 2e-3)}
        if not args.no_cpu_baseline:
            cores = os.cpu_count() or 1
            rows = args.cpu_rows or min(B, 4096)
            v, s_step, used = cpu_port_seq_per_s(w, rows, 2, cores)
            line['cpu_baseline'] = {'value': v, 'unit': 'sequences/s', 'cores': used, 'kind': 'port',
                                    'sample': '%d of %d windows per step, 2 steps after 1 warm-up (%.1f s); NumPy fp32 '
                                              'restatement of the reference step (TensorFlow unavailable); host has %d '
                                              'cores, `cores` = BLAS threads used' % (rows, B, 3 * s_step, cores)}
        if outputs is not None:
            dump_outputs(args.dump_outputs, outputs)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
