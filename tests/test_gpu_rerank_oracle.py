"""Stage-wise parity of the k-reciprocal re-ranking (csrc/rerank.cu) with the oracle (oracle/rerank.py).

The GPU runs through the sharded phases (sharded.CudaOps: rerank_rows -> rerank_expand -> rerank_finish), which expose
the intermediate tables, and every final block is also required to be bit-identical to re_ranking_dev, so each check
here holds for the single-device path too.  Bars:
- rank table: int32-equal to the oracle's, including the -1 padding when N < K;
- k-reciprocal rows: counts and index sets equal, weights within WEIGHT_ULP ulp (expf against numpy's float32 exp is
  the only intended difference), NaN positions equal;
- final matrix: NaN positions equal; lambda = 1 returns D[:nq, nq:] bit for bit wherever the Jaccard term is not NaN
  (jac * 0 + D * 1 == D), which checks the normalisation exactly; otherwise within FINAL_TOL of the oracle.
Past the size the dense oracle can reach, the oracle's per-row pieces check a sample of rows: rank rows and weights
from the oracle's own D rows, expansion sets from the GPU's rank table, and whole final rows of sampled queries from the
GPU's k-reciprocal rows (stage-wise inputs, so those must agree bit for bit)."""
import time

import numpy as np
import pytest
import torch

from agrl.pytorch_b200 import _lib, metrics, sharded
from agrl.pytorch_b200.utils.re_ranking import re_ranking_dev
from oracle import rerank as orr
from oracle import synth
from test_gpu_rerank_sharded import bits_equal, run_phases
from test_oracle_rerank import GRID, grid_features, matrices, special_matrices, tie_features

pytestmark = pytest.mark.gpu

# A weight is exp(-d) over the sum of its row's exp(-d), so an exp that differs by a ulp or two moves the weight by
# more: its own term and the sum both shift, and the quotient can land in a lower binade than the term.  On one B200
# (1000 W power limit) the largest error measured here is 6 ulp (MARS size, cosine; 5 ulp for k1 = 29 / 30); on the
# CPU, numpy's float32 exp against the correctly rounded exp (at most 2 ulp apart) already moves normalised weights by
# up to 6 ulp.
WEIGHT_ULP = 8
FINAL_TOL = 1e-6
LAMS = (0.0, 0.3, 1.0)


def ulps(got, want):
    """|got - want| in units of the float32 spacing at want, for finite want"""
    return np.abs(got.astype(np.float64) - want.astype(np.float64)) / np.spacing(np.abs(want)).astype(np.float64)


def same_nan(a, b):
    return np.array_equal(np.isnan(a), np.isnan(b))


def bits_or_both_nan(a, b):
    nan = np.isnan(a)
    return np.array_equal(nan, np.isnan(b)) and np.array_equal(a[~nan].view(np.uint32), b[~nan].view(np.uint32))


def gpu_run(qg, qq, gg, k1, k2, lams=LAMS, bounds=None):
    """numpy (q_g, q_q, g_g) through the GPU phases; each final block is checked against re_ranking_dev bit for bit.
    Returns ([final block per lambda], rank table, (idx, val, cnt)) as numpy arrays."""
    qg_d, qq_d, gg_d = (torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in (qg, qq, gg))
    ng = qg.shape[1]
    outs, rank, v = run_phases(lambda: (qg_d, qq_d), lambda c0, c1: gg_d[:, c0:c1], bounds or [(0, ng)], k1, k2,
                               lams)
    for lam, out in zip(lams, outs):
        assert bits_equal(out, re_ranking_dev(qg_d, qq_d, gg_d, k1=k1, k2=k2, lambda_value=lam)), lam
    return [o.cpu().numpy() for o in outs], rank.cpu().numpy(), tuple(t.cpu().numpy() for t in v)


def check_rows(rank, v, want_rank, D_rows, rows):
    """rank rows and k-reciprocal rows of the given global rows against the oracle.  D_rows / rows: {r: D row},
    {r: (idx, weights)}.  Returns the largest weight error in ulps."""
    idx, val, cnt = v
    worst = 0.0
    for r, d in D_rows.items():
        assert np.array_equal(rank[r], want_rank[r]), r
        ix, w = rows[r]
        assert cnt[r] == len(ix) and np.array_equal(idx[r, :cnt[r]], ix), r
        got = val[r, :cnt[r]]
        assert same_nan(got, w), r
        fin = ~np.isnan(w)
        if fin.any():
            worst = max(worst, float(ulps(got[fin], w[fin]).max()))
    assert worst <= WEIGHT_ULP, worst
    return worst


def oracle_final(D, rank, rows, nq, k2, lam):
    N = D.shape[0]
    qe = orr.query_expansion(rows, rank, k2, N) if k2 != 1 else rows
    inv = orr.inverted_index(qe[nq:])
    jac = np.stack([orr.jaccard_row(qe[i], inv, N - nq) for i in range(nq)])
    return orr.blend(jac, D[:nq, nq:], lam)


def check_dense(qg, qq, gg, k1, k2, lams=LAMS, bounds=None, label=''):
    """every rank row, k-reciprocal row and final entry against the dense oracle"""
    t0 = time.time()
    outs, rank, v = gpu_run(qg, qq, gg, k1, k2, lams, bounds)
    t1 = time.time()
    nq, N = qg.shape[0], qg.shape[0] + qg.shape[1]
    K = max(k1 + 1, k2)
    with np.errstate(all='ignore'):
        D = orr.normalised_dist(qg, qq, gg)
        want_rank = np.full((N, K), -1, np.int32)
        top = orr.initial_rank(D, K)
        want_rank[:, :top.shape[1]] = top
        rows = orr.sparse_weights(D, top, k1)
        worst = check_rows(rank, v, want_rank, dict(enumerate(D)), dict(enumerate(rows)))
        err = 0.0
        for lam, out in zip(lams, outs):
            want = oracle_final(D, top, rows, nq, k2, lam)
            assert same_nan(out, want), lam
            fin = ~np.isnan(want)
            if lam == 1.0:                                # D itself wherever the Jaccard term is not NaN
                assert np.array_equal(out[fin].view(np.uint32), D[:nq, nq:][fin].view(np.uint32))
            if fin.any():
                e = float(np.abs(out[fin] - want[fin]).max())
                assert e <= FINAL_TOL, (lam, e)
                err = max(err, e)
    print('%s k1=%d k2=%d: max weight error %.2f ulp, max final error %.3g; GPU %.1f s, oracle %.1f s'
          % (label, k1, k2, worst, err, t1 - t0, time.time() - t1))
    return rank, v, D


def gpu_matrices(qf, gf, metric):
    cdm = metrics.compute_distance_matrix
    return tuple(cdm(a.cuda(), b.cuda(), metric).cpu().numpy() for a, b in ((qf, gf), (qf, qf), (gf, gf)))


def clustered(nq, ng, d, seed):
    qp, _, gp, _ = synth.eval_labels((nq, ng, max(4, min(625, nq // 3)), 6), seed=seed)
    return synth.eval_features(qp, gp, d, seed=seed + 1, clustered=True)


# ---- parameter grid: every k1, k2 and lambda value, both metrics --------------------------------------------------------
@pytest.mark.parametrize('k1,k2,metric', [(k1, k2, metric) for k1, k2, _, metric in GRID])
def test_parameter_grid(k1, k2, metric):
    """k1 in {1, 2, 5, 7, 9, 11, 20, 29, 30} (30: 31 forward neighbours fill the warp, cap = 1024; odd k1 exercise the
    round-half-even half), k2 in {1, 2, 6, 8} (8: 8192 sort keys; k1 = 1, k2 = 8: rank rows wider than k1 + 1); every
    case runs lambda = 0, 0.3 and 1 on the same phase A / B state"""
    qf, gf = clustered(300, 3000, 256, seed=k1 * 16 + k2)
    check_dense(*gpu_matrices(qf, gf, metric), k1, k2, label='grid %s' % metric)


# ---- ties ------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('k1,k2', [(20, 6), (7, 8), (30, 2)])
def test_ties(k1, k2):
    """integer-grid features: duplicated gallery rows (pairs 2t, 2t + 1), two of them split by the shard boundaries at
    499 and 1001, queries copied into the gallery and a row with k1 + 1 exact duplicates at lower indices, whose
    k-reciprocal set is empty"""
    qf, gf, empty_row = tie_features(200, 1500, 16, seed=k1, k1=k1)
    bounds = [(0, 499), (499, 1001), (1001, 1500)]
    assert torch.equal(gf[498], gf[499]) and torch.equal(gf[1000], gf[1001])
    _, (_, _, cnt), _ = check_dense(*gpu_matrices(qf, gf, 'euclidean'), k1, k2, bounds=bounds, label='ties')
    assert cnt[empty_row] == 0 and cnt[empty_row - 1] > 0


def test_quantised_distances():
    check_dense(*special_matrices('quantised'), 20, 6, bounds=sharded.shard_bounds(150, 2), label='quantised')


# ---- degenerate inputs -------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('nq,ng,k1,k2', [(1, 150, 20, 6), (40, 1, 20, 6), (3, 10, 20, 6), (5, 16, 20, 6), (2, 5, 1, 8)])
def test_degenerate_shapes(nq, ng, k1, k2):
    """one query, one gallery row, N < K (rank rows padded with -1), N == K"""
    check_dense(*matrices(*grid_features(nq, ng, 16, seed=nq + ng)), k1, k2, label='%dx%d' % (nq, ng))


def test_all_zero_distances():
    """every column maximum is 0: D = 0 / 0 is NaN everywhere, on both sides"""
    rank, _, _ = check_dense(*special_matrices('zeros'), 20, 6, label='zeros')
    assert np.array_equal(rank, np.tile(np.arange(21, dtype=np.int32), (100, 1)))      # NaN ties, by index


def test_inf_entries():
    check_dense(*special_matrices('inf'), 20, 6, label='inf')


@pytest.mark.parametrize('shards', [1, 2, 3])
def test_one_nan_entry(shards):
    """np.max propagates NaN, so the D rows of the columns holding the NaN are NaN throughout, in the rank table
    (NaN ties, by index), in the weights, and through np.minimum in the Jaccard sums"""
    qg, qq, gg = special_matrices('nan')
    _, _, D = check_dense(qg, qq, gg, 20, 6, bounds=sharded.shard_bounds(150, shards), label='nan/%d' % shards)
    assert list(np.flatnonzero(np.isnan(D).all(axis=1))) == [3, 30 + 17, 30 + 101]


# ---- MARS size, dense oracle ----------------------------------------------------------------------------------------
@pytest.mark.parametrize('metric', ['euclidean', 'cosine'])
def test_mars_size(metric):
    qf, gf = clustered(1980, 9330, 2048, seed=31)
    check_dense(*gpu_matrices(qf, gf, metric), 20, 6, lams=(0.3, 1.0), label='MARS %s' % metric)


# ---- past the dense oracle: sampled rows -------------------------------------------------------------------------------
def check_sampled(nq, ng, shards, seed, n_spread=60, n_queries=30):
    """2048-d clustered features, euclidean, k1 = 20, k2 = 6, lambda = 0.3 and 1 on the same phase A / B state.
    Sampled rows: the first and last query, the first and last gallery row, the rows on each side of every shard
    boundary, n_spread rows spread over all N rows and n_queries spread over the queries.  For them: rank rows exact
    and weights within WEIGHT_ULP against the oracle's own D rows (columns of the block matrix from
    compute_distance_matrix with the operand roles of the GPU path).  Expansion index sets: every row, from the GPU's
    rank table.  Final rows of the sampled queries: all ng entries, from the GPU's k-reciprocal rows, bit for bit; at
    lambda = 1 equal to D."""
    k1, k2, lam = 20, 6, 0.3
    cdm = metrics.compute_distance_matrix
    qf, gf = (t.cuda() for t in clustered(nq, ng, 2048, seed))
    N, K = nq + ng, k1 + 1
    bounds = sharded.shard_bounds(ng, shards)
    t0 = time.time()
    host = {}

    def q_dists():
        qg_d, qq_d = cdm(qf, gf), cdm(qf, qf)
        host.update(qg=qg_d.cpu().numpy(), qq=qq_d.cpu().numpy())
        return qg_d, qq_d

    outs, rank, v = run_phases(q_dists, lambda c0, c1: cdm(gf, gf[c0:c1]), bounds, k1, k2, [lam, 1.0])
    out, out1 = (o.cpu().numpy() for o in outs)
    del outs
    rank = rank.cpu().numpy()
    idx, val, cnt = (t.cpu().numpy() for t in v)
    del v
    torch.cuda.empty_cache()
    t1 = time.time()

    edges = {0, nq - 1, nq, N - 1}
    for lo, hi in bounds:
        edges |= {nq + lo - 1, nq + lo, nq + hi - 1, nq + hi}
    spread = set(np.linspace(0, N - 1, n_spread).astype(int).tolist())
    spread |= set(np.linspace(0, nq - 1, n_queries).astype(int).tolist())
    rows = sorted(r for r in edges | spread if 0 <= r < N)
    queries = [r for r in rows if r < nq]

    def column(r):
        gg_col = cdm(gf, gf[r - nq:r - nq + 1]).cpu().numpy()[:, 0] if r >= nq else None
        return orr.orig_column(host['qg'], host['qq'], r, gg_col)

    D_rows = {r: orr.d_row(column(r)) for r in rows}
    want_rank = {r: orr.rank_row(d, K) for r, d in D_rows.items()}
    exp_rows = {r: orr.expansion_row(rank, r, k1) for r in rows}
    worst = check_rows(rank, (idx, val, cnt), want_rank, D_rows,
                       {r: (ix, orr.expansion_weights(D_rows[r], ix)) for r, ix in exp_rows.items()})
    t2 = time.time()
    for r in range(N):
        ix = orr.expansion_row(rank, r, k1)
        assert cnt[r] == len(ix) and np.array_equal(idx[r, :cnt[r]], ix), r
    t3 = time.time()

    V = [(idx[r, :cnt[r]], val[r, :cnt[r]]) for r in range(N)]
    qe_gal = [orr.qe_row([V[n] for n in rank[nq + j, :k2]]) for j in range(ng)]
    inv = orr.inverted_index(qe_gal)
    for i in queries:
        jac = orr.jaccard_row(orr.qe_row([V[n] for n in rank[i, :k2]]), inv, ng)
        want = orr.blend(jac, D_rows[i][nq:], lam)
        assert bits_or_both_nan(out[i], want), i
        assert bits_or_both_nan(out1[i], D_rows[i][nq:]), i
    t4 = time.time()
    print('%d x %d, %d shards: %d sampled rows, %d expansion rows, %d whole final rows; max weight error %.2f ulp; '
          'GPU phases %.1f s, sampled rows %.1f s, expansion sets %.1f s, final rows %.1f s'
          % (nq, ng, shards, len(rows), N, len(queries), worst, t1 - t0, t2 - t1, t3 - t2, t4 - t3))


def test_near_the_single_device_ceiling():
    """4000 x 40000 (N = 44000), world 1 as a single shard"""
    check_sampled(4000, 40000, 1, seed=41)


def test_past_the_single_device_limit():
    """2000 x 160000 (N = 162000) in 4 shards: the D rows of a shard pass 2^31 elements, so sampled gallery rows at the
    end of a shard read D at 64-bit positions (rank rows, weights)"""
    assert _lib.load().agrl_rerank_workspace_bytes(2000, 160000, 20, 6) == 0
    check_sampled(2000, 160000, 4, seed=43)
