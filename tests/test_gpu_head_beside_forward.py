"""GPU tests of the training head that runs beside the forward recurrence (head_paced_kernel in csrc/lstm_tc.cu).

LFMQ_FWD_HEAD=0 selects the head after the recurrence (head_tc_kernel + head_reduce_kernel + head_fold_kernel).  The
switch is read when a handle is created, so every test builds one engine of each kind in this process and compares
them.  Both heads compute the same bf16 dLoss/dpred tiles; only the fp32 order in which the per-CTA partials of the
loss and of h^T dpred are summed differs.
"""
import numpy as np
import pytest
import torch

import bench
from util import make_engine, make_problem, rel_err

pytestmark = pytest.mark.gpu

F, O, H, L = 32, 16, 256, 1
AGREE = 1e-5


def _cuda(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _engine(monkeypatch, paced, B, T, **kw):
    monkeypatch.setenv('LFMQ_FWD_HEAD', '1' if paced else '0')
    return make_engine(B, T, F, O, H, L, target_idx=3, precision='bf16', **kw)


@pytest.mark.parametrize('B,removed', [(4096, 2), (300, 2), (4500, 0)])
def test_paced_head_launches(monkeypatch, B, removed):
    """The paced path drops head_reduce_kernel and head_fold_kernel; B=4500 needs a second tile iteration of the
    recurrence and keeps the head after it."""
    T = 6
    params, x, y = make_problem(B, T, F, O, H, L, seed=41)
    xc, yc = _cuda(x), _cuda(y)
    per_step = {}
    for paced in (False, True):
        eng = _engine(monkeypatch, paced, B, T)
        eng.set_weights(params)
        eng.train_step(xc, yc, 0, 0.1)          # first step: weight packing, streams, tensor maps
        torch.cuda.synchronize()
        n0 = eng.launch_count
        eng.train_step(xc, yc, 1, 0.1)
        torch.cuda.synchronize()
        per_step[paced] = eng.launch_count - n0
        eng.close()
    assert per_step[False] - per_step[True] == removed, per_step


@pytest.mark.parametrize('B', [4096, 300])
def test_paced_head_gradients_match(monkeypatch, B):
    T = 48
    params, x, y = make_problem(B, T, F, O, H, L, seed=42, init_scale=1.0)
    xc, yc = _cuda(x), _cuda(y)
    out = {}
    for paced in (False, True):
        eng = _engine(monkeypatch, paced, B, T)
        eng.set_weights(params)
        eng.backward(xc, yc)
        out[paced] = (eng.grads_list(), eng.grads[eng.n_trainable:eng.n_trainable + 2].cpu().numpy(),
                      [s[0] for s in eng.trainable_specs])
        eng.close()
    assert rel_err(out[True][1], out[False][1]) <= AGREE, (out[True][1], out[False][1])
    for name, g, r in zip(out[False][2], out[True][0], out[False][0]):
        assert np.isfinite(g).all(), name
        assert rel_err(g, r) <= AGREE, (name, rel_err(g, r))


def test_paced_head_trajectory_matches():
    """10 optimizer steps of the benchmark's workload (weights, batches, optimizer) agree in {loss, mse_0}."""
    w = bench.WORKLOADS['cfg2']
    B, T = w['B'], w['T']
    rng = np.random.default_rng(bench.SEED)
    batches = [tuple(_cuda(a) for a in bench.synthetic(B, rng, w)) for _ in range(4)]
    traj = {}
    mp = pytest.MonkeyPatch()
    try:
        for paced in (False, True):
            mp.setenv('LFMQ_FWD_HEAD', '1' if paced else '0')
            eng = make_engine(B, T, w['F'], w['O'], w['H'], w['L'], target_idx=bench.TARGET_IDX, precision='bf16',
                              optimizer='Adadelta', dropout=w['dropout'], target_lambda=0.5, rnn_lambda=0.7,
                              max_grad_norm=50.0, max_norm=3.0, seed=bench.SEED)
            eng.set_weights(bench.initial_weights(w))
            traj[paced] = np.array([eng.train_step(*batches[i % 4], i, 0.6).cpu().numpy() for i in range(10)])
            eng.close()
    finally:
        mp.undo()
    assert np.isfinite(traj[True]).all()
    for i in range(10):
        assert rel_err(traj[True][i], traj[False][i]) <= AGREE, (i, traj[True][i], traj[False][i])
