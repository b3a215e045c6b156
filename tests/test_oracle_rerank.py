"""Pin oracle/rerank.py to the reference's own re_ranking() (utils/re_ranking.py:30-94): tests/golden/rerank_*.npz
hold the three distance matrices (from the reference's compute_distance_matrix) and the re-ranked distances.  Then
pin the oracle's per-row pieces, bit for bit, to the dense statement of every stage, on the goldens and over the
k1 / k2 / lambda grid, ties, special values and degenerate shapes that tests/test_gpu_rerank_oracle.py runs."""
import os

import numpy as np
import pytest
import torch

from conftest import GOLDEN, golden_files
from oracle import distance as odist
from oracle import rerank as orr
from oracle import synth


@pytest.mark.parametrize('fname', golden_files('rerank_'))
def test_rerank_oracle_matches_reference_golden(fname):
    g = np.load(os.path.join(GOLDEN, fname))
    out = orr.re_ranking(g['q_g'], g['q_q'], g['g_g'], k1=int(g['k1']), k2=int(g['k2']), lambda_value=float(g['lam']))
    assert out.shape == g['out'].shape and out.dtype == np.float32
    assert np.array_equal(out, g['out']), (fname, float(np.abs(out - g['out']).max()))


def test_normalised_distance_definition():
    rng = np.random.RandomState(0)
    qg, qq, gg = rng.rand(3, 5).astype(np.float32), rng.rand(3, 3).astype(np.float32), rng.rand(5, 5).astype(np.float32)
    D = orr.normalised_dist(qg, qq, gg)
    orig = np.block([[qq, qg], [qg.T, gg]]).astype(np.float32) ** 2
    assert D.shape == (8, 8) and D.dtype == np.float32
    for i in range(8):
        assert np.array_equal(D[i], orig[:, i] / orig[:, i].max())


# ---- the row-local oracle against the dense statement ------------------------------------------------------------------
# The dense forms below are the reference's own (re_ranking.py:34-90): a full stable argsort, the (k2, N) dense mean and
# the dense V with its np.where inverted index.  Every per-row piece of oracle/rerank.py must reproduce them bit for bit.
def dense_rank(D, K):
    return np.argsort(D, axis=1, kind='stable')[:, :K].astype(np.int32)


def dense_qe(rows, rank, k2, N):
    out = []
    for i in range(N):
        dense = np.zeros((k2, N), np.float32)
        for r, n in enumerate(rank[i, :k2]):
            dense[r, rows[n][0]] = rows[n][1]
        acc = np.mean(dense[:len(rank[i, :k2])], axis=0)
        idx = np.where(acc != 0)[0]
        out.append((idx, acc[idx]))
    return out


def dense_final(rows, D, nq, lam):
    N = D.shape[0]
    V = np.zeros((N, N), np.float32)
    for i, (idx, w) in enumerate(rows):
        V[i, idx] = w
    inv = [np.where(V[:, c] != 0)[0] for c in range(N)]
    jac = np.zeros((nq, N), np.float32)
    for i in range(nq):
        t = np.zeros((1, N), np.float32)
        for c in rows[i][0]:
            t[0, inv[c]] = t[0, inv[c]] + np.minimum(V[i, c], V[inv[c], c])
        jac[i] = 1 - t / (2. - t)
    return (jac * (1 - lam) + D[:nq] * lam)[:, nq:]


def grid_features(nq, ng, d, seed):
    """clustered features on an integer grid: every fp32 squared-euclidean distance is exact, and ties are real"""
    qp, _, gp, _ = synth.eval_labels((nq, ng, max(4, nq // 3), 3), seed=seed)
    qf, gf = synth.eval_features(qp, gp, d, seed=seed, clustered=True)
    return torch.round(2 * qf).contiguous(), torch.round(2 * gf).contiguous()


def tie_features(nq, ng, d, seed, k1):
    """grid features with ties: duplicated gallery rows (pairs 2t, 2t + 1), the queries copied into the gallery's end,
    and k1 + 2 copies of one row from gallery index 40 on.  The last copy (gallery 41 + k1) has k1 + 1 exact duplicates
    at lower indices, so it is not among its own first k1 + 1 neighbours and its k-reciprocal set is empty."""
    qf, gf = grid_features(nq, ng, d, seed)
    gf[1::2] = gf[0:-1:2][:len(gf[1::2])]
    gf[-nq:] = qf
    gf[40:42 + k1] = gf[40] + 50                       # far from everything else
    return qf, gf.contiguous(), nq + 41 + k1


def matrices(qf, gf, metric='euclidean'):
    """(q_g, q_q, g_g) float32 numpy, the operand roles of the library's call sequence"""
    return tuple(odist.distance_matrix(a, b, metric).numpy() for a, b in ((qf, gf), (qf, qf), (gf, gf)))


def special_matrices(kind, seed=0):
    """numpy distance matrices for the edge cases: 'nan' (one NaN in q_g, one in g_g), 'inf' (+inf in q_g and g_g),
    'zeros' (all zero: every column maximum is 0, so D is 0 / 0 = NaN everywhere), 'quantised' (few distinct values).
    A NaN at q_g[a, b] sits in columns a and nq + b of the block matrix, one at g_g[a, b] in column nq + b only."""
    if kind == 'zeros':
        return np.zeros((20, 80), np.float32), np.zeros((20, 20), np.float32), np.zeros((80, 80), np.float32)
    if kind == 'quantised':
        qg = synth.quantised_distmat(30, 150, seed=seed, levels=16)
        qq = synth.quantised_distmat(30, 30, seed=seed + 1, levels=16)
        gg = synth.quantised_distmat(150, 150, seed=seed + 2, levels=16)
        np.fill_diagonal(qq, 0)
        np.fill_diagonal(gg, 0)
        return qg, qq, np.minimum(gg, gg.T)
    qg, qq, gg = matrices(*grid_features(30, 150, 16, seed))
    bad = np.float32('nan') if kind == 'nan' else np.float32('inf')
    qg[3, 17] = bad
    gg[60, 101] = bad
    return qg, qq, gg


def stagewise_oracle(qg, qq, gg, k1, k2, lam):
    """every stage from its own dense inputs: D, rank table, expansion rows, query-expanded rows, final block"""
    nq, N = qg.shape[0], qg.shape[0] + qg.shape[1]
    D = orr.normalised_dist(qg, qq, gg)
    rank = dense_rank(D, max(k1 + 1, k2))
    rows = orr.sparse_weights(D, rank, k1)
    qe = dense_qe(rows, rank, k2, N) if k2 != 1 else rows
    return D, rank, rows, qe, dense_final(qe, D, nq, lam)


def same(a, b):
    return a.shape == b.shape and np.array_equal(a, b, equal_nan=True)


def check_row_local(qg, qq, gg, k1, k2, lam):
    with np.errstate(all='ignore'):
        nq, N = qg.shape[0], qg.shape[0] + qg.shape[1]
        K = max(k1 + 1, k2)
        D, rank, rows, qe, final = stagewise_oracle(qg, qq, gg, k1, k2, lam)
        padded = np.full((N, K), -1, np.int32)                                     # the library's table when N < K
        padded[:, :rank.shape[1]] = rank
        for r in range(N):
            assert same(orr.d_row(orr.orig_column(qg, qq, r, gg[:, r - nq] if r >= nq else None)), D[r]), r
            assert same(orr.rank_row(D[r], K), rank[r]), r
            idx = orr.expansion_row(padded, r, k1)
            assert same(idx, rows[r][0]), r
            assert same(orr.expansion_weights(D[r], idx), rows[r][1]), r
            if k2 != 1:
                got = orr.qe_row([rows[n] for n in rank[r, :k2]])
                assert same(got[0], qe[r][0]) and same(got[1], qe[r][1]), r
        want = np.array([[orr.final_entry(qe[i], qe[nq + j], D[i, nq + j], lam) for j in range(N - nq)]
                         for i in range(nq)], np.float32).reshape(final.shape)
        assert same(want, final)
        assert same(orr.re_ranking(qg, qq, gg, k1=k1, k2=k2, lambda_value=lam), final)
    return D, rank, rows


@pytest.mark.parametrize('fname', golden_files('rerank_'))
def test_row_local_oracle_on_the_goldens(fname):
    g = np.load(os.path.join(GOLDEN, fname))
    check_row_local(g['q_g'], g['q_q'], g['g_g'], int(g['k1']), int(g['k2']), float(g['lam']))


# every k1 (odd ones give half = round-half-even(k1 / 2) + 1: 1 -> 1, 5 -> 3, 7 -> 5, 9 -> 5, 11 -> 7, 29 -> 15), k2
# (8 > k1 + 1 for k1 = 1 widens the rank rows past k1 + 1) and lambda of the GPU grid, both metrics
GRID = [(1, 8, 0.3, 'euclidean'), (1, 2, 1.0, 'cosine'), (2, 2, 0.0, 'euclidean'), (5, 6, 1.0, 'euclidean'),
        (7, 1, 0.3, 'cosine'), (9, 8, 0.3, 'euclidean'), (11, 6, 0.0, 'cosine'), (20, 6, 0.3, 'euclidean'),
        (29, 2, 1.0, 'euclidean'), (30, 8, 0.3, 'euclidean'), (30, 1, 0.0, 'cosine')]


@pytest.mark.parametrize('k1,k2,lam,metric', GRID)
def test_row_local_oracle_parameter_grid(k1, k2, lam, metric):
    check_row_local(*matrices(*grid_features(40, 200, 16, seed=k1 + 10 * k2), metric), k1, k2, lam)


@pytest.mark.parametrize('k1,k2', [(20, 6), (7, 8), (30, 2)])
def test_row_local_oracle_ties(k1, k2):
    qf, gf, empty_row = tie_features(30, 160, 16, seed=k1, k1=k1)
    _, _, rows = check_row_local(*matrices(qf, gf), k1, k2, 0.3)
    assert len(rows[empty_row][0]) == 0 and len(rows[empty_row - 1][0]) > 0


@pytest.mark.parametrize('kind', ['nan', 'inf', 'zeros', 'quantised'])
def test_row_local_oracle_special_values(kind):
    qg, qq, gg = special_matrices(kind)
    D, _, _ = check_row_local(qg, qq, gg, 20, 6, 0.3)
    nan_rows = np.isnan(D).all(axis=1)
    if kind == 'nan':                                  # np.max propagates NaN: the rows of both columns are all NaN
        assert list(np.flatnonzero(nan_rows)) == [3, 30 + 17, 30 + 101]
    if kind == 'zeros':
        assert nan_rows.all()
    if kind == 'inf':
        assert not nan_rows.any() and list(zip(*np.nonzero(np.isnan(D)))) == [(3, 47), (47, 3), (131, 90)]   # inf / inf


@pytest.mark.parametrize('nq,ng,k1,k2', [(3, 10, 20, 6), (5, 16, 20, 6), (1, 150, 20, 6), (40, 1, 20, 6), (2, 5, 1, 8)])
def test_row_local_oracle_degenerate_shapes(nq, ng, k1, k2):
    """N < K (3 x 10, k1 = 20), N == K (5 x 16), one query, one gallery row"""
    check_row_local(*matrices(*grid_features(nq, ng, 16, seed=nq + ng)), k1, k2, 0.3)


def test_rank_row_is_a_stable_argsort():
    rng = np.random.RandomState(3)
    for n in (1, 7, 31, 32, 500, 5000):
        for d in (rng.rand(n), np.round(4 * rng.rand(n)), np.zeros(n), -np.zeros(n)):
            d = d.astype(np.float32)
            d[rng.rand(n) < 0.05] = np.nan
            d[rng.rand(n) < 0.05] = np.inf
            for K in (1, 2, 21, 31, n, n + 3):
                assert np.array_equal(orr.rank_row(d, K), np.argsort(d, kind='stable')[:K]), (n, K)
