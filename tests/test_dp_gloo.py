"""N>1 path on CPU: world_size-2 gloo processes run the data-parallel step plumbing (lfm_quant_b200/dp.py) on
oracle gradients of their row shards and must reproduce the single-process gradient, loss and update."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import lfm_oracle as orc
from lfm_quant_b200 import dp
from util import make_problem

CFG = dict(num_layers=1, target_idx=1, target_lambda=0.5, rnn_lambda=0.7, max_grad_norm=0.5, optimizer='Adadelta',
           max_norm=3.0, train=True)
SHAPE = dict(B=10, T=5, F=6, O=3, H=8, L=1)


def _flat(grads, loss, mse):
    return torch.from_numpy(np.concatenate([g.ravel() for g in grads] + [np.array([loss, mse, 0.0, 0.0])]))


def _worker(rank, world, port, out_dir):
    os.environ['MASTER_ADDR'] = '127.0.0.1'
    os.environ['MASTER_PORT'] = str(port)
    dist.init_process_group('gloo', rank=rank, world_size=world)
    params, x, y = make_problem(SHAPE['B'], SHAPE['T'], SHAPE['F'], SHAPE['O'], SHAPE['H'], SHAPE['L'], seed=31)
    row0, n = dp.shard_rows(SHAPE['B'], rank, world)
    xs, ys = x[row0:row0 + n].astype(np.float64), y[row0:row0 + n].astype(np.float64)
    mask_local = float((~np.all(ys == 0.0, axis=-1)).sum())
    denom = dp.global_denominators(torch.tensor([float(n), mask_local], dtype=torch.float64), dist)
    preds, fc = orc.forward(params, xs, num_layers=1)
    loss, mse, dpred, _ = orc.loss_point_estimate(ys, preds, target_idx=1, target_lambda=0.5, rnn_lambda=0.7,
                                                  batch_global=denom[0].item(), mask_count_global=denom[1].item())
    grads = orc.backward(dpred, fc, num_layers=1)
    n_tr = sum(g.size for g in grads)
    flat = dp.allreduce_flat_gradient(_flat(grads, loss, mse), n_tr, dist)
    # replicated tail of the step: clip on the REDUCED gradient, optimizer, MaxNorm
    gl, off = [], 0
    for g in grads:
        gl.append(flat[off:off + g.size].numpy().reshape(g.shape).copy())
        off += g.size
    clipped, gn = orc.clip_by_global_norm(gl, CFG['max_grad_norm'])
    new = orc.optimizer_update('Adadelta', params, clipped, orc.zero_slots('Adadelta', params), 0.6, 0)
    new[0] = orc.max_norm_constraint(new[0], CFG['max_norm'])
    np.savez(os.path.join(out_dir, 'rank%d.npz' % rank), flat=flat.numpy(), denom=denom.numpy(), gn=gn,
             **{'w%d' % i: w for i, w in enumerate(new)})
    dist.destroy_process_group()


def _free_port():
    s = socket.socket()
    s.bind(('127.0.0.1', 0))
    p = s.getsockname()[1]
    s.close()
    return p


@pytest.mark.timeout(120)
def test_two_rank_step_equals_single_process(tmp_path):
    world = 2
    mp.spawn(_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    params, x, y = make_problem(SHAPE['B'], SHAPE['T'], SHAPE['F'], SHAPE['O'], SHAPE['H'], SHAPE['L'], seed=31)
    new, mse, loss, raw, gn = orc.train_step([p.copy() for p in params], orc.zero_slots('Adadelta', params),
                                             x.astype(np.float64), y.astype(np.float64), 0, CFG, lr=0.6)
    ref_flat = np.concatenate([g.ravel() for g in raw] + [np.array([loss, mse])])
    r0 = np.load(tmp_path / 'rank0.npz')
    r1 = np.load(tmp_path / 'rank1.npz')
    n = ref_flat.size
    np.testing.assert_allclose(r0['flat'][:n], ref_flat, rtol=1e-10, atol=1e-12)
    np.testing.assert_array_equal(r0['flat'][:n], r1['flat'][:n])           # replicas agree bit for bit
    assert r0['denom'][0] == SHAPE['B'] and r0['denom'][1] == (~np.all(y == 0, axis=-1)).sum()
    assert float(r0['gn']) == pytest.approx(float(gn), rel=1e-10)
    for i, w in enumerate(new):
        np.testing.assert_allclose(r0['w%d' % i], w, rtol=1e-9, atol=1e-12)
        np.testing.assert_array_equal(r0['w%d' % i], r1['w%d' % i])


def test_shard_rows_partition():
    for B in (7, 8, 4096, 32768):
        for world in (1, 2, 3, 8):
            spans = [dp.shard_rows(B, r, world) for r in range(world)]
            assert spans[0][0] == 0 and sum(n for _, n in spans) == B
            for (a, n), (b, _) in zip(spans, spans[1:]):
                assert a + n == b


def _cli_worker(rank, world, port, out_dir):
    """What scripts/train.py does under torchrun: dp.init_from_env() from the launcher's environment, then each rank
    takes its rows of every global batch of window indices."""
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world),
                      LOCAL_RANK=str(rank))
    r, w = dp.init_from_env()
    assert (r, w) == (rank, world) and dist.is_initialized()
    rows = []
    for n in (7, 2, 1):                                     # the last global batches of an epoch are ragged
        inp = np.arange(3 * n, dtype=np.int32).reshape(n, 3)
        tar = inp + 100
        meta = np.array([[b'd%d' % i, b'k', b'k'] for i in range(n)], dtype=object)
        a, b, m, row0 = dp.shard_batch_indices(inp, tar, meta, r, w)
        assert len(a) == len(b) == len(m)
        assert (b == a + 100).all()
        rows.append((n, row0, a[:, 0].tolist()))
    np.save(os.path.join(out_dir, 'cli%d.npy' % rank), np.array(rows, dtype=object), allow_pickle=True)
    dist.destroy_process_group()


def test_cli_sharding_covers_every_global_batch_exactly_once(tmp_path, monkeypatch):
    world = 2
    # the ranks take init_from_env's gloo branch on every machine: with CUDA visible it would give each rank a GPU of
    # its own (NCCL), which a machine with fewer GPUs than ranks does not have
    monkeypatch.setenv('CUDA_VISIBLE_DEVICES', '')
    mp.spawn(_cli_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    per_rank = [np.load(str(tmp_path / ('cli%d.npy' % r)), allow_pickle=True) for r in range(world)]
    for bi, n in enumerate((7, 2, 1)):
        got, expect_row0 = [], 0
        for r in range(world):
            nn, row0, firsts = per_rank[r][bi]
            assert nn == n and row0 == expect_row0
            expect_row0 += len(firsts)
            got += firsts
        assert got == [3 * i for i in range(n)]
