"""world_size-2 and 3 gloo runs of sharded.query_expansion_sharded and engine.test(aqe=True) on CPU.

numpy stand-ins for the two per-rank calls (the cosine lists of some rows of the joint set against all of it, and the
weighted mix) drive the same plumbing as the CUDA path: the query broadcast, the shard layout, the per-iteration
all-gather of the gallery rows and the global row bookkeeping.  Every rank must return the single-process result bit
for bit, with uneven and empty shards."""
import os

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from agrl.pytorch_b200 import engine, sharded
from oracle import distance as odist
from oracle import qe as oqe
from oracle import rank as orank
from test_engine_gloo import _shard
from test_engine_host import TinyModel, loaders
from test_rank_lists_gloo import ListOps
from test_sharded_gloo import _free_port


class QeOps(ListOps):
    """ListOps plus the query-expansion stand-ins (fp64 cosine rounded to fp32, stable lists, fp32 mix in list order)"""

    def qe_lists(self, x, ranges, k, fused=None):
        xd = x.numpy().astype(np.float64)
        n = xd / np.maximum(np.linalg.norm(xd, axis=1, keepdims=True), 1e-12)
        rows = np.concatenate([np.arange(r0, r1) for r0, r1 in ranges] + [np.zeros(0, np.int64)])
        d = np.stack([(1.0 - n @ n[r]).astype(np.float32) for r in rows]) if len(rows) else \
            np.zeros((0, len(xd)), np.float32)
        idx = np.argsort(d, axis=1, kind='stable')[:, :k]
        return torch.from_numpy(idx), torch.from_numpy(np.take_along_axis(d, idx, 1))

    def qe_mix(self, idx, d, x, alpha):
        idx, d, x = idx.numpy(), d.numpy(), x.numpy()
        k = idx.shape[1]
        w = np.power(np.float32(1.0) - d, np.float32(alpha))
        out = np.zeros((len(idx), x.shape[1]), np.float32)
        for j in range(k):
            out = out + w[:, j:j + 1] * x[idx[:, j]]
        return torch.from_numpy(out / np.float32(k))


def _worker(rank, world, port, case, out_dir):
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port))
    dist.init_process_group('gloo', rank=rank, world_size=world)
    try:
        qf, gf, k, times, alpha, bounds = case
        lo, hi = bounds[rank]
        qf_r = qf.clone() if rank == 0 else torch.zeros_like(qf)          # broadcast must repair this
        q, g = sharded.query_expansion_sharded(qf_r, gf[lo:hi], k, times, alpha, ops=QeOps())
        counts = [b - a for a, b in bounds]
        q2, g2 = sharded.query_expansion_sharded(qf, gf[lo:hi], k, times, alpha, ops=QeOps(), gallery_counts=counts,
                                                 broadcast_queries=False)
        np.savez(os.path.join(out_dir, 'r%d.npz' % rank), q=q.numpy(), g=g.numpy(), q2=q2.numpy(), g2=g2.numpy())
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize('world,shape,k,times,alpha,layout', [(2, (10, 40, 16), 5, 1, 3.0, 'even'),
                                                              (2, (9, 31, 8), 4, 3, 0.0, 'even'),
                                                              (3, (12, 48, 16), 5, 2, 0.5, 'skewed'),
                                                              (3, (7, 23, 9), 3, 3, 1.0, 'even')])
def test_sharded_expansion_matches_single_process(tmp_path, world, shape, k, times, alpha, layout):
    nq, ng, dim = shape
    qf, gf = oqe.grouped_features(nq, ng, dim, k, seed=nq + k, spread=0.3)
    bounds = [(0, 0), (0, ng - 7), (ng - 7, ng)] if layout == 'skewed' else sharded.shard_bounds(ng, world)
    mp.spawn(_worker, args=(world, _free_port(), (qf, gf, k, times, alpha, bounds), str(tmp_path)), nprocs=world,
             join=True)
    rq, rg = sharded.query_expansion_sharded(qf, gf, k, times, alpha, ops=QeOps())
    oq, og, _, _, margins = oqe.aqe(qf, gf, k, times, alpha)
    assert min(m.min() for m in margins) > 1e-4
    assert np.allclose(rq.numpy(), oq, atol=1e-5) and np.allclose(rg.numpy(), og, atol=1e-5)
    for r, (lo, hi) in enumerate(bounds):
        z = np.load(os.path.join(str(tmp_path), 'r%d.npz' % r))
        for q, g in (('q', 'g'), ('q2', 'g2')):
            assert np.array_equal(z[q], rq.numpy()), (r, q)
            assert z[g].shape == (hi - lo, dim) and np.array_equal(z[g], rg.numpy()[lo:hi]), (r, g)


def _engine_worker(rank, world, port, bounds, out_dir):
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port))
    dist.init_process_group('gloo', rank=rank, world_size=world)
    try:
        ql, gl, _ = loaders(nq=12, ng=41, seed=3)
        lo, hi = bounds[rank]
        r1, mAP = engine.test(TinyModel(), ql, _shard(gl, lo, hi), 'avg', True, max_rank=20, verbose=(rank == 0),
                              sharded_ops=QeOps(), aqe=True, qe_k=4, qe_times=2, qe_alpha=3.0)
        np.savez(os.path.join(out_dir, 'r%d.npz' % rank), r1=r1, mAP=mAP)
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize('world', [2, 3])
def test_engine_aqe_gallery_sharded_matches_single_process(tmp_path, world):
    bounds = sharded.shard_bounds(41, world)
    mp.spawn(_engine_worker, args=(world, _free_port(), bounds, str(tmp_path)), nprocs=world, join=True)
    ql, gl, (qp, qc, gp, gc) = loaders(nq=12, ng=41, seed=3)
    model = TinyModel()
    with torch.no_grad():
        qf = torch.cat([model(i, a) for i, _, _, a in ql])
        gf = torch.cat([model(i, a) for i, _, _, a in gl])
    qf, gf = sharded.query_expansion_sharded(qf, gf, 4, 2, 3.0, ops=QeOps())
    d = np.concatenate([odist.distance_matrix(qf, gf[lo:hi], 'euclidean').numpy() for lo, hi in bounds], axis=1)
    cmc, mAP = orank.mars_port(d, qp, gp, qc, gc, 20)
    for r in range(world):
        z = np.load(os.path.join(str(tmp_path), 'r%d.npz' % r))
        assert float(z['r1']) == cmc[0] and float(z['mAP']) == mAP


def test_argument_errors():
    qf, gf = oqe.grouped_features(4, 16, 8, 4, seed=1)
    for kw in (dict(qe_k=0), dict(qe_k=21), dict(qe_k=sharded.MAX_LIST_DEPTH + 1), dict(qe_times=0),
               dict(alpha=float('nan')), dict(alpha=float('inf'))):
        with pytest.raises(ValueError):
            sharded.query_expansion_sharded(qf, gf, **dict(dict(qe_k=4, qe_times=1, alpha=3.0), **kw), ops=QeOps())
    q, g = sharded.query_expansion_sharded(qf, gf, 20, 1, 0.0, ops=QeOps())       # qe_k == N, alpha 0: the plain mean
    mean = torch.cat([qf, gf]).mean(0).numpy()
    assert np.allclose(np.concatenate([q.numpy(), g.numpy()]), mean[None], atol=1e-6)
    with pytest.raises(AssertionError):
        sharded.query_expansion_sharded(qf, gf[:, :7], ops=QeOps())


def test_qe_symbol_is_exported_and_documented():
    from agrl.pytorch_b200 import _lib, metrics
    from test_abi import declared_symbols
    assert 'agrl_qe_mix_dev' in declared_symbols() and 'agrl_qe_mix_dev' in _lib.exported_names()
    assert hasattr(_lib.load(), 'agrl_qe_mix_dev')
    assert 'query_expansion' in metrics.__all__
    header = open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'include',
                               'agrl_b200.h')).read()
    doc = header[header.index('alpha query expansion'):header.index('agrl_qe_mix_dev(')]
    for must in ('powf(1 - dist[r, j], alpha)', '/ k', 'list order', 'must not', 'AGRL_E_INVALID', 'non-finite alpha'):
        assert must in doc, must
