"""Gallery-sharded k-reciprocal re-ranking (sharded.re_ranking_sharded, evaluate_mars_sharded(re_rank=True)) under gloo
on CPU, world sizes 2 and 3.

The three per-rank phases are CPU stand-ins built from oracle/rerank.py's per-row pieces on the rank's own rows, with the same
exchange contract as csrc/rerank.cu (rank rows (n_loc, K) padded with -1, k-reciprocal rows (n_loc, cap) + counts).
Features lie on a coarse integer grid, so every fp32 distance is exact and splitting the gallery cannot move a bit:
the concatenated blocks and the re-ranked CMC/mAP must equal the oracle on the whole gallery.  This checks the
padding, the global-index bookkeeping and the all-gathers of sharded.py."""
import os

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from agrl.pytorch_b200 import sharded
from agrl.pytorch_b200 import synthetic as synth
from oracle import rank as orank
from oracle import rerank as orr
from test_sharded_gloo import CpuOps, _free_port


class CpuRerankOps(CpuOps):
    """CpuOps (distance, partial, merge) plus stand-ins for the three re-ranking phases."""

    def rerank_rows(self, qg, qq, gg_slabs, offset, n_own, max_own, k1, k2):
        qg, qq = qg.numpy(), qq.numpy()
        nq, ng = qg.shape
        N = nq + ng
        cols = [np.concatenate([qq[:, c], qg[c, :]]) for c in range(nq)]                 # orig[:, c], query columns
        for s0, slab in gg_slabs:
            slab = slab.numpy()
            cols += [np.concatenate([qg[:, offset + s0 + t], slab[:, t]]) for t in range(slab.shape[1])]
        assert len(cols) == nq + n_own
        D = np.stack([orr.d_row(c) for c in cols])                                         # own rows of D
        K, _ = sharded.rerank_row_dims(k1, k2)
        rank = np.full((nq + n_own, K), -1, np.int32)
        top = orr.initial_rank(D, K)
        rank[:, :top.shape[1]] = top
        st = dict(D=D, nq=nq, N=N, offset=offset, n_own=n_own, k1=k1, k2=k2)
        return st, torch.from_numpy(rank)

    def _glob(self, st, l):
        return l if l < st['nq'] else l + st['offset']

    @staticmethod
    def _trim(rank_all, N):
        return rank_all.numpy()[:, :min(rank_all.shape[1], N)]

    def rerank_expand(self, st, rank_all):
        rank = self._trim(rank_all, st['N'])
        k1, D = st['k1'], st['D']
        _, cap = sharded.rerank_row_dims(k1, st['k2'])
        rows = D.shape[0]
        idx, val, cnt = np.zeros((rows, cap), np.int32), np.zeros((rows, cap), np.float32), np.zeros(rows, np.int32)
        for l in range(rows):
            ix = orr.expansion_row(rank, self._glob(st, l), k1)
            idx[l, :len(ix)], val[l, :len(ix)], cnt[l] = ix, orr.expansion_weights(D[l], ix), len(ix)
        return torch.from_numpy(idx), torch.from_numpy(val), torch.from_numpy(cnt)

    def rerank_finish(self, st, rank_all, idx_all, val_all, cnt_all, lambda_value):
        N, nq, n_own, k2, D = st['N'], st['nq'], st['n_own'], st['k2'], st['D']
        rank = self._trim(rank_all, N)
        idx_all, val_all, cnt_all = idx_all.numpy(), val_all.numpy(), cnt_all.numpy()
        V = [(idx_all[r, :cnt_all[r]], val_all[r, :cnt_all[r]]) for r in range(N)]
        rows = []
        for l in range(nq + n_own):
            g = self._glob(st, l)
            if k2 == 1:
                rows.append(V[g])
                continue
            rows.append(orr.qe_row([V[n] for n in rank[g, :k2]]))
        inv = {}                                                                           # over the own gallery rows
        for j in range(n_own):
            for c, v in zip(*rows[nq + j]):
                inv.setdefault(int(c), []).append((j, v))
        out = np.zeros((nq, n_own), np.float32)
        for i in range(nq):
            t = np.zeros(n_own, np.float32)
            for c, vi in zip(*rows[i]):
                if int(c) in inv:
                    js = np.array([j for j, _ in inv[int(c)]])
                    vs = np.array([v for _, v in inv[int(c)]], np.float32)
                    t[js] = t[js] + np.minimum(vi, vs)
            jac = 1 - t / (2. - t)
            lo = nq + st['offset']
            out[i] = jac * (1 - lambda_value) + D[i, lo:lo + n_own] * lambda_value
        return torch.from_numpy(out)


def grid_case(nq, ng, d, seed, dup=False):
    qp, qc, gp, gc = synth.eval_labels((nq, ng, max(4, nq // 3), 3), seed=seed)
    qf, gf = synth.eval_features(qp, gp, d, seed=seed, clustered=True)
    qf, gf = torch.round(2 * qf), torch.round(2 * gf)              # integers: every fp32 distance is exact
    if dup:                                                        # ties across shard boundaries
        gf[1::2] = gf[0:-1:2][:len(gf[1::2])]
        gf[-3:] = qf[:3]
    return qp, qc, gp, gc, qf.contiguous(), gf.contiguous()


def _worker(rank, world, port, case, out_dir):
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port))
    dist.init_process_group('gloo', rank=rank, world_size=world)
    try:
        qp, qc, gp, gc, qf, gf, k1, k2, bounds = case
        lo, hi = bounds[rank]
        qf_r = qf.clone() if rank == 0 else torch.zeros_like(qf)           # the broadcast must repair this
        block = sharded.re_ranking_sharded(qf_r, gf[lo:hi], k1=k1, k2=k2, ops=CpuRerankOps())
        qp_r = qp if rank == 0 else np.zeros_like(qp)
        qc_r = qc if rank == 0 else np.zeros_like(qc)
        cmc, mAP = sharded.evaluate_mars_sharded(qf_r, gf[lo:hi], qp_r, gp[lo:hi], qc_r, gc[lo:hi], max_rank=10,
                                                 ops=CpuRerankOps(), re_rank=True, k1=k1, k2=k2,
                                                 gallery_counts=[b - a for a, b in bounds])
        np.savez(os.path.join(out_dir, 'r%d.npz' % rank), block=block.numpy(), cmc=cmc, mAP=mAP)
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize('world,nq,ng,k1,k2,dup,uneven', [(2, 12, 61, 20, 6, False, False),
                                                          (3, 9, 40, 5, 1, True, False),
                                                          (3, 10, 47, 4, 3, True, True)])
def test_sharded_rerank_matches_unsharded_oracle(tmp_path, world, nq, ng, k1, k2, dup, uneven):
    qp, qc, gp, gc, qf, gf = grid_case(nq, ng, 16, seed=world + ng, dup=dup)
    bounds = sharded.shard_bounds(ng, world)
    if uneven:                                           # one short shard, one long, and an empty middle one
        bounds = [(0, 5), (5, 5), (5, ng)]
    mp.spawn(_worker, args=(world, _free_port(), (qp, qc, gp, gc, qf, gf, k1, k2, bounds), str(tmp_path)),
             nprocs=world, join=True)
    from oracle import distance as odist
    qg, qq, gg = (odist.distance_matrix(a, b).numpy() for a, b in ((qf, gf), (qf, qf), (gf, gf)))
    want = orr.re_ranking(qg, qq, gg, k1=k1, k2=k2)
    cmc, mAP = orank.mars_port(want, qp, gp, qc, gc, 10)
    got = [np.load(os.path.join(str(tmp_path), 'r%d.npz' % r)) for r in range(world)]
    full = np.concatenate([g['block'] for g in got], axis=1)
    assert full.shape == want.shape
    assert np.array_equal(full.view(np.uint32), want.view(np.uint32))
    for r, g in enumerate(got):
        assert np.array_equal(g['cmc'], cmc), r
        assert float(g['mAP']) == float(mAP), r


def test_single_process_rerank_without_init():
    qp, qc, gp, gc, qf, gf = grid_case(8, 30, 8, seed=5)
    block = sharded.re_ranking_sharded(qf, gf, k1=6, k2=2, ops=CpuRerankOps())
    from oracle import distance as odist
    qg, qq, gg = (odist.distance_matrix(a, b).numpy() for a, b in ((qf, gf), (qf, qf), (gf, gf)))
    assert np.array_equal(block.numpy(), orr.re_ranking(qg, qq, gg, k1=6, k2=2))


def test_unknown_metric_is_rejected_before_any_work():
    qf = torch.zeros(3, 4)
    with pytest.raises(ValueError):
        sharded.re_ranking_sharded(qf, qf, metric='manhattan', ops=CpuRerankOps())


def test_row_dims_match_the_header():
    assert sharded.rerank_row_dims(20, 6) == (21, 256)          # 21 * 12 = 252
    assert sharded.rerank_row_dims(30, 8) == (31, 1024)         # 31 * 17 = 527
    assert sharded.rerank_row_dims(1, 6) == (6, 4)              # 2 * 2 = 4 (round(0.5) = 0)
    assert sharded.rerank_row_dims(3, 1) == (4, 16)             # 4 * 4 = 16 (round(1.5) = 2)


def test_shard_workspace_query_needs_no_device():
    from agrl.pytorch_b200 import _lib
    lib = _lib.load()
    # the D rows dominate: (num_q + n_own) x N fp32, 64-bit positions beyond 2^31 elements
    nq, ng, n_own = 2000, 160000, 20000
    b = lib.agrl_rerank_shard_workspace_bytes(nq, ng, n_own, 20, 6)
    assert b >= 4 * (nq + n_own) * (nq + ng) > 4 * 2 ** 31
    assert b < 4 * (nq + n_own) * (nq + ng) + (1 << 30)
    assert lib.agrl_rerank_shard_workspace_bytes(1980, 9330, 0, 20, 6) > 4 * 1980 * 11310     # an empty shard
    assert lib.agrl_rerank_shard_workspace_bytes(1980, 9330, 50001, 20, 6) == 0                # n_own > 50000
    assert lib.agrl_rerank_shard_workspace_bytes(1980, 60000, 50000, 20, 6) > 0
    assert lib.agrl_rerank_shard_workspace_bytes(1980, 9330, 1000, 64, 6) == 0                 # k1 > 30
    assert lib.agrl_rerank_shard_workspace_bytes(1980, 9330, 1000, 20, 9) == 0                 # k2 > 8
    assert lib.agrl_rerank_shard_workspace_bytes(1980, 9330, 9331, 20, 6) == 0                 # more than the gallery
    assert lib.agrl_rerank_shard_workspace_bytes(0, 9330, 100, 20, 6) == 0
    assert lib.agrl_rerank_shard_workspace_bytes(1000, 16000000, 100, 20, 6) == 0              # N beyond the limit
    # the single-device query is unchanged by the sharded form
    assert lib.agrl_rerank_workspace_bytes(1980, 9330, 20, 6) > 4 * 11310 * 11310
    assert lib.agrl_rerank_workspace_bytes(1980, 46000, 20, 6) == 0
