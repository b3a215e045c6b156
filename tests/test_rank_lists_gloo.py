"""world_size-2 and 3 gloo runs of sharded.rank_lists_sharded on CPU, and the ABI of the ranked lists.

CPU stand-ins (written against the key contract of csrc/rank.cu: order-preserving distance bits << 32 | global gallery
index, all-ones = empty) drive the same plumbing as the CUDA kernels: the junk-depth all-reduce, the key all-gather, the
gallery-label all-gather and the per-list junk drop + rank merge.  Every rank's lists must equal the stable argsort of
the whole matrix, with and without the same-pid-same-camera columns."""
import os
import re

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from agrl.pytorch_b200 import sharded
from agrl.pytorch_b200 import synthetic as synth
from oracle import distance as odist
from test_sharded_gloo import KEY_MAX, CpuOps, _free_port, mono_keys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def decode(keys):
    """numpy twin of mono_key_value() in csrc/common.cuh: (index, distance) of uint64 keys, (-1, +inf) for empty ones"""
    idx = (keys & np.uint64(0xFFFFFFFF)).astype(np.int64)
    m = (keys >> np.uint64(32)).astype(np.uint32)
    bits = np.where(m & np.uint32(0x80000000), m & np.uint32(0x7FFFFFFF), ~m).astype(np.uint32)
    empty = keys == KEY_MAX
    return np.where(empty, -1, idx), np.where(empty, np.float32(np.inf), bits.view(np.float32))


class ListOps(CpuOps):
    """CpuOps plus the ranked-list stand-ins"""

    def keys(self, d, depth, offset):
        qp, gp = sharded._unlabelled(d.shape[0], d.shape[1], d.device)
        return self.partial(d, qp, gp, qp, gp, depth, offset)[0]

    def junk_depth(self, qp, gp, qc, gc):
        qp, gp, qc, gc = qp.numpy(), gp.numpy(), qc.numpy(), gc.numpy()
        j = max([int(np.sum((gp == p) & (gc == c))) for p, c in zip(qp, qc)] + [0])
        return torch.tensor([j], dtype=torch.int32), torch.zeros(1, dtype=torch.int32)

    def lists(self, keys_all, k, qp=None, gp=None, qc=None, gc=None, exclude_junk=False):
        keys = keys_all.numpy().view(np.uint64)
        parts, nq, depth = keys.shape
        out = np.full((nq, k), KEY_MAX, np.uint64)
        for q in range(nq):
            kept = []
            for p in range(parts):
                lst = keys[p, q]
                lst = lst[lst != KEY_MAX]
                if exclude_junk:
                    g = (lst & np.uint64(0xFFFFFFFF)).astype(np.int64)
                    lst = lst[~((gp.numpy()[g] == int(qp[q])) & (gc.numpy()[g] == int(qc[q])))]
                kept.append(lst[:k])            # only the first k kept keys of a list can reach the head
            head = np.sort(np.concatenate(kept))[:k]
            out[q, :len(head)] = head
        idx, dist_ = decode(out)
        return torch.from_numpy(idx), torch.from_numpy(dist_)


def reference_lists(d, k, labels=None):
    """np.argsort(kind='stable') of each row, without the query's same-pid-same-camera columns when labels are given"""
    nq, ng = d.shape
    idx = np.full((nq, k), -1, np.int64)
    val = np.full((nq, k), np.inf, np.float32)
    for q in range(nq):
        cols = np.arange(ng)
        if labels is not None:
            qp, qc, gp, gc = labels
            cols = cols[~((gp == qp[q]) & (gc == qc[q]))]
        order = cols[np.argsort(d[q, cols], kind='stable')][:k]
        idx[q, :len(order)] = order
        val[q, :len(order)] = d[q, order] + np.float32(0.0)
    return idx, val


def _worker(rank, world, port, case, out_dir):
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port))
    dist.init_process_group('gloo', rank=rank, world_size=world)
    try:
        qp, qc, gp, gc, qf, gf, metric, k, bounds = case
        lo, hi = bounds[rank]
        qf_r = qf.clone() if rank == 0 else torch.zeros_like(qf)          # broadcast must repair this
        qp_r = qp if rank == 0 else np.zeros_like(qp)
        qc_r = qc if rank == 0 else np.zeros_like(qc)
        res = {}
        for junk in (False, True):
            i, v = sharded.rank_lists_sharded(qf_r.clone(), gf[lo:hi], k, qp_r, gp[lo:hi], qc_r, gc[lo:hi], metric=metric,
                                              exclude_junk=junk, ops=ListOps())
            res['i%d' % junk], res['v%d' % junk] = i.numpy(), v.numpy()
        counts = [b - a for a, b in bounds]
        i, v = sharded.rank_lists_sharded(qf_r.clone(), gf[lo:hi], k, metric=metric, ops=ListOps(), gallery_counts=counts)
        res['i_nolabels'], res['v_nolabels'] = i.numpy(), v.numpy()
        np.savez(os.path.join(out_dir, 'r%d.npz' % rank), **res)
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize('world,shape,metric,k,layout', [(2, (30, 300, 10, 3), 'euclidean', 20, 'even'),
                                                         (2, (12, 9, 3, 2), 'cosine', 15, 'even'),
                                                         (3, (16, 200, 6, 4), 'euclidean', 25, 'skewed'),
                                                         (3, (20, 150, 5, 2), 'cosine', 7, 'even')])
def test_sharded_lists_match_the_stable_argsort(tmp_path, world, shape, metric, k, layout):
    qp, qc, gp, gc = synth.eval_labels(shape, seed=world + k)
    qf, gf = synth.eval_features(qp, gp, 16, seed=world + k, clustered=True)
    gf[1::2] = gf[0:-1:2][:len(gf[1::2])]                 # duplicated rows: ties across shard boundaries
    ng = len(gp)
    if layout == 'skewed':                                # an empty shard, and one holding every item of query 0's id
        gp = gp.copy()
        gp[gp == qp[0]] = qp[0] + 1000
        gp[-12:], gc[-12:] = qp[0], qc[0]                 # 12 junk items of query 0 in the last shard
        bounds = [(0, 0), (0, ng - 12), (ng - 12, ng)]
    else:
        bounds = sharded.shard_bounds(ng, world)
    mp.spawn(_worker, args=(world, _free_port(), (qp, qc, gp, gc, qf, gf, metric, k, bounds), str(tmp_path)),
             nprocs=world, join=True)
    d = odist.distance_matrix(qf, gf, metric).numpy()
    plain = reference_lists(d, k)
    junk = reference_lists(d, k, (qp, qc, gp, gc))
    assert not np.array_equal(plain[0], junk[0])
    for r in range(world):
        got = np.load(os.path.join(str(tmp_path), 'r%d.npz' % r))
        for key, (ri, rv) in (('0', plain), ('1', junk), ('_nolabels', plain)):
            assert np.array_equal(got['i' + key], ri), (r, key)
            assert np.array_equal(got['v' + key].view(np.int32), rv.view(np.int32)), (r, key)


def test_single_process_lists_and_padding():
    qp, qc, gp, gc = synth.eval_labels((10, 40, 4, 2), seed=3)
    qf, gf = synth.eval_features(qp, gp, 8, seed=3, clustered=True)
    d = odist.distance_matrix(qf, gf, 'euclidean').numpy()
    for k in (1, 39, 40, 41, 60):
        i, v = sharded.rank_lists_sharded(qf, gf, k, qp, gp, qc, gc, exclude_junk=True, ops=ListOps())
        ri, rv = reference_lists(d, k, (qp, qc, gp, gc))
        assert np.array_equal(i.numpy(), ri) and np.array_equal(v.numpy().view(np.int32), rv.view(np.int32))
        assert (i.numpy()[:, 40:] == -1).all()


def test_depth_limit_and_argument_errors():
    qp, qc, gp, gc = synth.eval_labels((4, 30, 3, 2), seed=5)
    qf, gf = synth.eval_features(qp, gp, 8, seed=5)
    with pytest.raises(ValueError, match='8192'):
        sharded.rank_lists_sharded(qf, gf, 8193, ops=ListOps())
    gp = gp.copy()
    gp[:], gc[:] = qp[0], qc[0]                            # 30 junk items: k + J = 8192 + 30
    with pytest.raises(ValueError, match='8192'):
        sharded.rank_lists_sharded(qf, gf, 8170, qp, gp, qc, gc, exclude_junk=True, ops=ListOps())
    with pytest.raises(ValueError, match='exclude_junk'):
        sharded.rank_lists_sharded(qf, gf, 5, exclude_junk=True, ops=ListOps())
    with pytest.raises(ValueError):
        sharded.rank_lists_sharded(qf, gf, 0, ops=ListOps())


def test_decode_inverts_the_key_map():
    x = np.array([0.0, -0.0, 1.5, -1.5, np.inf, -np.inf, 1e-45, -1e-45, 3.4e38, -3.4e38, np.nan], np.float32)
    keys = (mono_keys(x) << np.uint64(32)) | np.arange(len(x), dtype=np.uint64)
    idx, val = decode(keys)
    assert np.array_equal(idx, np.arange(len(x)))
    fin = ~np.isnan(x)
    assert np.array_equal(val[fin].view(np.uint32), (x[fin] + np.float32(0)).view(np.uint32))    # -0 -> +0
    assert val[-1].view(np.uint32) == 0x7FFFFFFF
    ranked = (keys[np.argsort(x, kind='stable')] >> np.uint64(32)).astype(np.int64)
    assert np.all(np.diff(ranked) >= 0)


def test_lists_symbols_are_exported_and_documented():
    from agrl.pytorch_b200 import _lib
    from test_abi import declared_symbols
    names = declared_symbols()
    for sym in ('agrl_rank_lists_dev', 'agrl_rank_junk_depth_dev'):
        assert sym in names and sym in _lib.exported_names()
        assert hasattr(_lib.load(), sym)
    header = open(os.path.join(ROOT, 'include', 'agrl_b200.h')).read()
    doc = header[header.index('Ranked lists'):header.index('agrl_rank_junk_depth_dev(')]
    for must in ('index -1', '+inf', 'exclude_junk', 'k + J', 'parts * depth <= 16384', 'AGRL_ST_LABEL_RANGE'):
        assert must in doc, must
    assert re.search(r'agrl_rank_lists_dev\(', header)
