"""k-reciprocal re-ranking oracle -- TEST INFRASTRUCTURE ONLY (see oracle/__init__.py).

Restatement of the reference's torchreid/utils/re_ranking.py:30-94 (Zhong et al., CVPR 2017), the optional step
between the distance matrix and the ranking in test() (train_vidreid_xent_htri.py:523-527).  Same numpy float32
arithmetic in the same order, organised by stage with sparse rows instead of the dense N x N work matrices; ties in
the initial ranking are broken by index (numpy.argsort(kind='stable'); the reference's default quicksort leaves them
undefined, so the golden vectors are produced with argsort forced stable).  Pinned by tests/test_oracle_rerank.py
against tests/golden/rerank_*.npz, outputs of the reference's own re_ranking().

Every stage is also stated per row (``d_row``, ``rank_row``, ``expansion_row``, ``expansion_weights``, ``qe_row``,
``final_entry``): each computes one row or one entry from its own inputs, bit for bit what the dense form computes
there, so that problems too large for N x N matrices can be checked on a sample of rows.  ``re_ranking`` runs on
these pieces, except for the normalisation, which stays vectorised over the block matrix, and the Jaccard sums, which
run per query row over an inverted index (``inverted_index``, ``jaccard_row``) rather than entry by entry.
"""
import numpy as np


# ---- per-row pieces ------------------------------------------------------------------------------------------------
def orig_column(q_g, q_q, r, gg_col=None):
    """column r of the block matrix [[q_q, q_g], [q_g^T, g_g]] (N float32).  A query column needs only q_q and q_g; a
    gallery column r = nq + j also takes gg_col = g_g[:, j], so that g_g need not exist as a whole."""
    nq = q_g.shape[0]
    if r < nq:
        return np.concatenate([q_q[:, r], q_g[r, :]]).astype(np.float32)
    return np.concatenate([q_g[:, r - nq], gg_col]).astype(np.float32)


def d_row(col):
    """row r of D from column r of the block matrix (re_ranking.py:34-40): col^2 / max(col^2) in float32.  np.max
    propagates NaN, so a NaN anywhere in the column makes the whole row NaN."""
    sq = np.power(np.asarray(col, np.float32), 2).astype(np.float32)
    return 1. * sq / np.max(sq)


def rank_row(d, K):
    """first min(K, len(d)) entries of np.argsort(d, kind='stable'), without sorting the whole row: every value <= the
    K-th smallest is a candidate (so ties at the cut stay complete), and the candidates, in index order, are sorted
    stably by value.  NaN sorts last, as in np.argsort; a NaN K-th value falls back to the full sort."""
    d = np.asarray(d)
    n = d.shape[0]
    if K >= n:
        return np.argsort(d, kind='stable').astype(np.int32)
    kth = np.partition(d, K - 1)[K - 1]
    if np.isnan(kth):
        return np.argsort(d, kind='stable')[:K].astype(np.int32)
    cand = np.flatnonzero(d <= kth)
    return cand[np.argsort(d[cand], kind='stable')[:K]].astype(np.int32)


def reciprocal_row(rank, i, k):
    """re_ranking.py:50-53 (and :57-60 for the candidates): neighbours f of i within the first k with i in f's first k."""
    fwd = rank[i, :k]
    back = rank[fwd, :k]
    return fwd[np.where(back == i)[0]]


def expansion_row(rank, r, k1):
    """re_ranking.py:48-65: the sorted index set of row r -- its k-reciprocal set, grown by every candidate's
    half-size set that overlaps it by more than 2/3.  ``rank`` is any (N, >= k1 + 1) table of first columns; a table
    wider than N (padded with -1) is cut to N."""
    rank = rank[:, :min(rank.shape[1], rank.shape[0])]
    half = int(np.around(k1 / 2.)) + 1
    recip = reciprocal_row(rank, r, k1 + 1)
    expansion = recip
    for cand in recip:
        cr = reciprocal_row(rank, cand, half)
        if len(np.intersect1d(cr, recip)) > 2. / 3 * len(cr):
            expansion = np.append(expansion, cr)
    return np.unique(expansion)


def expansion_weights(d, idx):
    """re_ranking.py:66-67: exp(-D[r, idx]) normalised to sum 1 (numpy's pairwise float32 sum), from the D row"""
    w = np.exp(-d[idx])
    return (1. * w / np.sum(w)).astype(np.float32)


def qe_row(nb_rows, m=None):
    """re_ranking.py:69-74: the mean of the sparse V rows [(idx, w)] of a row's first k2 neighbours, given in rank
    order, as np.mean(dense, axis=0) computes it: rows added in order in float32 (an absent row adds an exact zero),
    then divided by the number of rows ``m`` (default len(nb_rows)).  Returns (idx, value) of the non-zero columns."""
    m = len(nb_rows) if m is None else m
    cols = np.unique(np.concatenate([np.asarray(ix, np.int64) for ix, _ in nb_rows])) if nb_rows else np.zeros(0, np.int64)
    acc = np.zeros(len(cols), np.float32)
    for ix, w in nb_rows:
        present = np.zeros(len(cols), np.float32)
        present[np.searchsorted(cols, ix)] = w
        acc = acc + present
    acc = acc / np.float32(m)
    keep = np.where(acc != 0)[0]
    return cols[keep], acc[keep]


def final_entry(vi, vj, d_ij, lambda_value):
    """re_ranking.py:76-90, one entry: the Jaccard term of the sparse rows vi = (idx, val) and vj = (idx, val)
    (jaccard_row over an inverted index of the single row vj), blended with D[i, j] (``d_ij``)."""
    jac = jaccard_row(vi, inverted_index([vj]), 1)
    return blend(jac, np.asarray([d_ij], np.float32), lambda_value)[0]


def blend(jac, d, lambda_value):
    """re_ranking.py:90: jac (1 - lambda) + D lambda in float32"""
    return jac * (1 - lambda_value) + d * lambda_value


def inverted_index(rows):
    """re_ranking.py:76-78 over the sparse rows [(idx, val)]: for every column c, the rows j with V[j, c] != 0
    (ascending) and their values.  Returns (bounds, row, val): column c holds entries bounds[c]:bounds[c + 1]."""
    n = int(max((int(ix.max()) + 1 for ix, _ in rows if len(ix)), default=0))
    r_of = np.repeat(np.arange(len(rows)), [len(ix) for ix, _ in rows])
    c_of = np.concatenate([np.asarray(ix, np.int64) for ix, _ in rows] + [np.zeros(0, np.int64)])
    v_of = np.concatenate([np.asarray(w, np.float32) for _, w in rows] + [np.zeros(0, np.float32)])
    nz = v_of != 0
    r_of, c_of, v_of = r_of[nz], c_of[nz], v_of[nz]
    order = np.argsort(c_of, kind='stable')
    return np.searchsorted(c_of[order], np.arange(n + 1)), r_of[order], v_of[order]


def jaccard_row(vi, inv, n):
    """re_ranking.py:80-88, one query: t[j] = sum over the query's columns c, ascending, of min(V[i, c], V[j, c]) for
    the n rows of the inverted index ``inv``, added in float32; returns 1 - t / (2 - t)"""
    bounds, r_of, v_of = inv
    t = np.zeros((1, n), np.float32)
    for c, vic in zip(*vi):
        if c + 1 >= len(bounds) or vic == 0:
            continue
        lo, hi = bounds[c], bounds[c + 1]
        t[0, r_of[lo:hi]] = t[0, r_of[lo:hi]] + np.minimum(vic, v_of[lo:hi])
    return (1 - t / (2. - t))[0]


# ---- the dense stages -----------------------------------------------------------------------------------------------
def normalised_dist(q_g, q_q, g_g):
    """re_ranking.py:34-40: D[i, j] = orig[j, i]^2 / max_k orig[k, i]^2 (float32), orig the (N, N) block matrix."""
    orig = np.concatenate([np.concatenate([q_q, q_g], axis=1), np.concatenate([q_g.T, g_g], axis=1)], axis=0)
    orig = np.power(orig, 2).astype(np.float32)
    return np.transpose(1. * orig / np.max(orig, axis=0))


def initial_rank(D, k):
    """first k columns of argsort(D) with ties by index (re_ranking.py:42)"""
    return np.stack([rank_row(d, k) for d in D]) if len(D) else np.zeros((0, min(k, D.shape[1])), np.int32)


def sparse_weights(D, rank, k1):
    """re_ranking.py:48-67: per row the sorted expansion set and exp(-D) weights normalised to sum 1 (float32)."""
    rows = []
    for i in range(D.shape[0]):
        idx = expansion_row(rank, i, k1)
        rows.append((idx, expansion_weights(D[i], idx)))
    return rows


def query_expansion(rows, rank, k2, N):
    """re_ranking.py:69-74: V_qe[i] = mean of the V rows of i's first k2 neighbours (float32, rows added in rank order)."""
    return [qe_row([rows[n] for n in rank[i, :k2]]) for i in range(N)]


def re_ranking(q_g_dist, q_q_dist, g_g_dist, k1=20, k2=6, lambda_value=0.3):
    q_g, q_q, g_g = (np.asarray(a) for a in (q_g_dist, q_q_dist, g_g_dist))
    nq, N = q_g.shape[0], q_g.shape[0] + q_g.shape[1]
    D = normalised_dist(q_g, q_q, g_g)
    rank = initial_rank(D, max(k1 + 1, k2))
    rows = sparse_weights(D, rank, k1)
    if k2 != 1:
        rows = query_expansion(rows, rank, k2, N)
    inv = inverted_index(rows)
    jac = np.stack([jaccard_row(rows[i], inv, N) for i in range(nq)]) if nq else np.zeros((0, N), np.float32)
    return blend(jac, D[:nq], lambda_value)[:, nq:]
