"""The ranking kernels (csrc/rank.cu) against the C oracle at every size where they change code path.

rank_market_kernel picks one of three paths per query from m, the number of gallery items of the query's
identity (positives plus same-camera junk), and from the row's length:
    fast      m <= 62 and no thread bins more than 65535 elements (u16 private histograms, warp sort of 64 keys)
    shared    m <= kListCap = 2048 otherwise (bitonic sort of n2 keys, u32 shared histogram)
    overflow  m > 2048 (rank_market_overflow_kernel, 8 CTAs looping over a query list)
The MARS evaluator keeps a streaming top-K (select_topk) whose buffer and sort trigger depend on K, and whose
first tile is short when K <= 128; its mAP is numpy's pairwise sum, replayed as a tree in rank_mars_finish_kernel.
The sharded forms size their lists by powers of two of parts * K (MARS merge) and parts * cap (market1501).

Every result is compared bit for bit with oracle/rank.py (rank_oracle.c): per-query AP, CMC, mAP, num_valid.
The label / distance constructor and its checks need no GPU; everything else is marked gpu.
"""
import numpy as np
import pytest
import torch

from oracle import rank as orank

gpu = pytest.mark.gpu

LIST_CAP = 2048                  # kListCap
FAST_MAX_M = 62                  # kFastBins - 2
RANK_THREADS = 256               # kRankThreads
U16_MAX = 65535

NAN_NEG = np.array([0xFFC00000], np.uint32).view(np.float32)[0]      # a NaN with the sign bit set
SPECIALS = np.array([np.nan, NAN_NEG, np.inf, -np.inf, -0.0, 0.0], np.float32)
PLACEMENTS = ('near', 'far', 'interleaved', 'tied')


def _bits32(x):
    return np.asarray(x, np.float32).view(np.uint32)


def _bits64(x):
    return np.asarray(x, np.float64).view(np.uint64)


# ------------------------------------------------------------------------------------------------
# label / distance constructor
# ------------------------------------------------------------------------------------------------
def make_case(specs, n_neg, seed, ng_mod4=None):
    """Labels and a float32 distance matrix from per-query specs (npos, njunk, placement).

    Query q has its own identity 1 + q and camera q % 6.  The gallery holds, for query q, npos positives (same
    identity, another camera) and njunk junk items (same identity, same camera), plus n_neg items of no query's
    identity: half distractors (pid -1), half filler identities.  (0, 0) is an identity absent from the gallery,
    (0, njunk) a junk-only identity.  The gallery is shuffled.  ng_mod4 pads the filler so that ng % 4 is that value.

    placement decides row q's distances: 'near' (same-pid items nearer than every other item), 'far' (farther),
    'interleaved' (one distribution for all) or 'tied' (four distance levels for all, so gallery index decides).
    Returns (q_pids, q_camids, g_pids, g_camids, distmat).
    """
    rng = np.random.RandomState(seed)
    if ng_mod4 is not None:
        n_neg += (ng_mod4 - (sum(p + j for p, j, _ in specs) + n_neg)) % 4
    nq = len(specs)
    qp = np.arange(1, nq + 1, dtype=np.int64)
    qc = np.arange(nq, dtype=np.int64) % 6
    gp, gc = [], []
    for q, (npos, njunk, _) in enumerate(specs):
        gp += [qp[q]] * (npos + njunk)
        gc += [(qc[q] + 1 + k % 5) % 6 for k in range(npos)] + [qc[q]] * njunk
    n_dis = n_neg // 2
    gp += [-1] * n_dis + list(10 ** 6 + rng.randint(0, 97, n_neg - n_dis))
    gc += list(rng.randint(0, 6, n_neg))
    perm = rng.permutation(len(gp))
    gp = np.asarray(gp, np.int64)[perm]
    gc = np.asarray(gc, np.int64)[perm]
    ng = len(gp)
    d = np.empty((nq, ng), np.float32)
    for q, (_, _, placement) in enumerate(specs):
        same = gp == qp[q]
        if placement == 'tied':
            d[q] = rng.randint(0, 4, ng) * 0.25
        elif placement == 'interleaved':
            d[q] = rng.rand(ng)
        elif placement == 'near':
            d[q] = 1 + rng.rand(ng)
            d[q, same] = rng.rand(int(same.sum()))
        elif placement == 'far':
            d[q] = rng.rand(ng)
            d[q, same] = 1 + rng.rand(int(same.sum()))
        else:
            raise ValueError(placement)
    return qp, qc, gp, gc, d


def inject_specials(qp, gp, d, seed, frac=0.03):
    """NaN (both signs), +-inf and -0.0 / +0.0: in about frac of every row and in a third of the same-pid items."""
    rng = np.random.RandomState(seed)
    d = d.copy()
    for q in range(d.shape[0]):
        hit = rng.rand(d.shape[1]) < frac
        same = np.flatnonzero(gp == qp[q])
        hit[same[rng.rand(len(same)) < 1 / 3]] = True
        d[q, hit] = SPECIALS[rng.randint(0, len(SPECIALS), int(hit.sum()))]
    return d


def same_pid_counts(qp, qc, gp, gc):
    """(m, npos, njunk) per query, counted from the labels."""
    same = gp[None, :] == qp[:, None]
    junk = same & (gc[None, :] == qc[:, None])
    return same.sum(1), (same & ~junk).sum(1), junk.sum(1)


def row_head(offset_floats):
    """Elements before the first 16-byte boundary of a row starting offset_floats floats past an aligned base."""
    return (4 - offset_floats % 4) % 4


def max_per_thread(ng, head):
    """Most elements one thread bins in rank_market_kernel's pass over a row (for_each_in_row): thread 0 takes
    the head element, ceil(nvec / 256) float4 vectors and a tail element."""
    head = min(head, ng)
    nvec = (ng - head) // 4
    return (head > 0) + 4 * -(-nvec // RANK_THREADS) + ((ng - head) % 4 > 0)


def market_path(m, ng, head):
    if m > LIST_CAP:
        return 'overflow'
    if m <= FAST_MAX_M and max_per_thread(ng, head) <= U16_MAX:
        return 'fast'
    return 'shared'


# the m of every path boundary, plus enough overflow queries (> 8) that the overflow CTAs loop
BOUNDARY_M = [1, 2, 31, 32, 33, 61, 62, 63, 64, 65, 127, 128, 129, 1023, 1024, 1025, 2047, 2048, 2049,
              4095, 4096, 4097]
EXTRA_OVERFLOW_M = [2050, 2051, 2200, 2500, 3000, 3333, 4098]


def boundary_specs(placement):
    specs = [(m - m // 3, m // 3, placement) for m in BOUNDARY_M + EXTRA_OVERFLOW_M]
    # identity absent from the gallery, junk-only identities (one of them past the fast path's size)
    return specs + [(0, 0, placement), (0, 3, placement), (0, 100, placement)]


def boundary_case(variant, seed=0):
    placement = variant if variant in PLACEMENTS else 'interleaved'
    specs = boundary_specs(placement)
    qp, qc, gp, gc, d = make_case(specs, 6000, seed, ng_mod4=3)          # ng % 4 == 3: host rows misaligned too
    if variant == 'specials':
        d = inject_specials(qp, gp, d, seed + 1)
    max_rank = d.shape[1] if variant == 'short_kept' else 50
    return specs, (qp, qc, gp, gc, d), max_rank


# ---- checks of the construction itself (no GPU): a boundary test must sit on the side it names ----
@pytest.mark.parametrize('placement', PLACEMENTS)
def test_constructor_gives_requested_counts(placement):
    specs, (qp, qc, gp, gc, d), _ = boundary_case(placement)
    m, npos, njunk = same_pid_counts(qp, qc, gp, gc)
    assert list(npos) == [s[0] for s in specs]
    assert list(njunk) == [s[1] for s in specs]
    assert list(m[:len(BOUNDARY_M)]) == BOUNDARY_M
    assert d.dtype == np.float32 and d.shape == (len(specs), len(gp)) and len(gp) % 4 == 3
    assert (gp == -1).sum() > 0                                            # distractors
    valid = npos > 0
    paths = [market_path(int(x), len(gp), 0) for x in m[valid]]
    assert paths.count('overflow') > 8
    assert {int(x) for x, p in zip(m[valid], paths) if p == 'fast'} == {x for x in BOUNDARY_M if x <= 62}
    assert {int(x) for x, p in zip(m[valid], paths) if p == 'shared'} == {x for x in BOUNDARY_M if 62 < x <= 2048}
    for q, (_, _, pl) in enumerate(specs):
        same = gp == qp[q]
        if not same.any() or same.all():
            continue
        a, b = d[q, same], d[q, ~same]
        if pl == 'near':
            assert a.max() < b.min()
        elif pl == 'far':
            assert a.min() > b.max()
        elif pl == 'tied':
            assert len(np.unique(d[q])) <= 4


def test_constructor_specials_and_short_kept():
    specs, (qp, qc, gp, gc, d), max_rank = boundary_case('specials')
    bits = d.view(np.uint32)
    for v in SPECIALS.view(np.uint32):
        assert (bits == v).sum() > 0, hex(v)
    for q in range(len(specs)):
        same = gp == qp[q]
        if same.sum() >= 30:
            assert not np.isfinite(d[q, same]).all()
    _, _, max_rank = boundary_case('short_kept')
    m, npos, njunk = same_pid_counts(qp, qc, gp, gc)
    kept = len(gp) - njunk
    short = (npos > 0) & (kept < min(max_rank, len(gp)))
    # the stale-cmc replay (flag bit 0) is reached by queries on each of the three paths
    assert {market_path(int(x), len(gp), 0) for x in m[short]} == {'fast', 'shared', 'overflow'}


def test_u16_window_arithmetic():
    """The rows whose thread 0 bins 65536 elements although ng <= 65535 * 256 (the former fast-path guard)."""
    limit = U16_MAX * RANK_THREADS
    assert limit == 16776960
    for head in range(4):
        window = [ng for ng in range(16776100, limit + 1) if max_per_thread(ng, head) > U16_MAX]
        assert window == list(range(16776196 + head, limit + 1)), head
    assert max_per_thread(16776195, 0) == 65533 and max_per_thread(16776196, 0) == 65536
    assert max_per_thread(16776960, 0) == 65536 and max_per_thread(16776961, 0) == 65537


# ------------------------------------------------------------------------------------------------
# market1501 (rank_market_kernel, _overflow, _finish)
# ------------------------------------------------------------------------------------------------
@pytest.fixture(scope='module')
def evaluate_cy():
    from agrl.pytorch_b200.metrics.rank_cylib.rank_cy import evaluate_cy as f
    return f


def strided(d, ld):
    """d on the device as a view with row stride ld > ng, so rows start off 16-byte boundaries."""
    buf = torch.full((d.shape[0], ld), float('nan'), device='cuda')
    buf[:, :d.shape[1]] = torch.from_numpy(d).cuda()
    return buf[:, :d.shape[1]]


def odd_ld(ng):
    """row stride > ng with ld % 4 == 1: consecutive rows start at all four offsets within 16 bytes"""
    return ng + ((1 - ng) % 4 or 4)


def market_inputs(d):
    yield 'host', d
    yield 'device', torch.from_numpy(d).cuda()
    yield 'device-ld', strided(d, odd_ld(d.shape[1]))


def check_market(evaluate_cy, labels_d, max_rank, ref=None):
    qp, qc, gp, gc, d = labels_d
    if ref is None:
        ref = orank.market1501_port(d, qp, gp, qc, gc, max_rank, return_ap=True)
    ref_cmc, ref_map, ref_ap, ref_nv = ref
    for name, dist in market_inputs(d):
        cmc, mAP, ap, nv = evaluate_cy(dist, qp, gp, qc, gc, max_rank, return_all_ap=True)
        bad = np.flatnonzero(_bits32(ap) != _bits32(ref_ap))
        assert bad.size == 0, (name, 'AP differs for queries', bad.tolist(), ap[bad].tolist(), ref_ap[bad].tolist())
        assert nv == ref_nv, name
        assert cmc.shape == ref_cmc.shape, name
        assert np.array_equal(_bits32(cmc), _bits32(ref_cmc)), (name, np.flatnonzero(_bits32(cmc) != _bits32(ref_cmc))[:10])
        assert mAP == ref_map, name
    return ref


@gpu
@pytest.mark.parametrize('variant', PLACEMENTS + ('specials', 'short_kept'))
def test_market1501_path_boundaries(evaluate_cy, variant):
    """m on both sides of 62 / 63 (fast | shared), of each power of two of the shared sort and of 2048 / 2049
    (shared | overflow) in one launch; 11 overflow queries; absent and junk-only identities."""
    specs, case, max_rank = boundary_case(variant, seed=PLACEMENTS.index(variant) if variant in PLACEMENTS else 7)
    check_market(evaluate_cy, case, max_rank)


@gpu
@pytest.mark.parametrize('m', [2047, 2048, 2049])
def test_market1501_list_cap_alone(evaluate_cy, m):
    """one query whose identity has m gallery items, the rest of the gallery nearer and farther"""
    specs = [(m - 100, 100, 'interleaved'), (5, 1, 'near')]
    qp, qc, gp, gc, d = make_case(specs, 3000, seed=m)
    check_market(evaluate_cy, (qp, qc, gp, gc, d), 50)


U16_NG = [16776195, 16776196, 16776960, 16776961]


POS = 1000          # in vector (1000 - head) // 4: 250 for head 0, 249 for heads 1-3; never thread 0's


def u16_case(ng, seed=0):
    """Rows 0-3: the worst case for one thread's counter -- the query's only positive is the farthest gallery
    item, so every other element lands in the first histogram bin (row 0 random below it, rows 1-3 constant, so
    index order decides).  The positive sits at index POS, which a thread other than 0 visits, so thread 0 bins
    all of its elements.  Row 4: random distances, 60 items of its identity scattered over the row, about a
    third of them junk."""
    rng = np.random.RandomState(seed)
    gp = np.full(ng, 2, np.int64)
    gc = np.ones(ng, np.int64)
    gp[POS] = 1
    idx = rng.choice(ng - POS - 1, 60, replace=False) + POS + 1
    gp[idx] = 3
    gc[idx] = rng.randint(0, 3, 60)
    qp = np.array([1, 1, 1, 1, 3], np.int64)
    qc = np.zeros(5, np.int64)
    d = np.empty((5, ng), np.float32)
    d[0] = rng.rand(ng)
    d[1:4] = 0.25
    d[:4, POS] = 2.0
    d[4] = rng.rand(ng)
    return qp, qc, gp, gc, d


@gpu
@pytest.mark.parametrize('ng', U16_NG)
def test_market1501_u16_counter_limit(evaluate_cy, ng):
    """Gallery sizes at the edge of the fast path's u16 per-thread counters.  On the host matrix rows start at
    offsets q * ng; on the strided device view at q * ld with ld % 4 == 1, so rows 0-3 take all four heads."""
    case = u16_case(ng)
    qp, qc, gp, gc, d = case
    for q in range(4):
        print('ng %d row %d: host thread-0 count %d, strided thread-0 count %d'
              % (ng, q, max_per_thread(ng, row_head(q * ng)), max_per_thread(ng, row_head(q * odd_ld(ng)))))
    ref = orank.market1501_port(d, qp, gp, qc, gc, 50, return_ap=True)
    # closed form of the worst case: one positive at kept rank ng - 1, AP = 1 / (kept rank + 1)
    assert np.array_equal(_bits32(ref[2][:4]), _bits32(np.full(4, 1.0 / ng, np.float32)))
    check_market(evaluate_cy, case, 50, ref=ref)


# ------------------------------------------------------------------------------------------------
# MARS (rank_mars_kernel<false> + select_topk, rank_mars_finish_kernel)
# ------------------------------------------------------------------------------------------------
@pytest.fixture(scope='module')
def evaluate_mars():
    from agrl.pytorch_b200.metrics.rank import evaluate_mars as f
    return f


MARS_ROWS = ('random', 'descending', 'ascending', 'constant', 'tie_at_k', 'special_beyond_k', 'signed_zeros',
             'distractors_first')


def mars_labels(nq, ng, seed):
    """pids drawn with about 20 items each, 10 % distractors; every query has a good item (another camera)."""
    rng = np.random.RandomState(seed)
    gp = rng.randint(0, max(2, ng // 20), ng).astype(np.int64)
    gc = rng.randint(0, 6, ng).astype(np.int64)
    gp[rng.rand(ng) < 0.1] = -1
    if (gp != -1).sum() == 0:
        gp[0] = 0
    anchors = rng.choice(np.flatnonzero(gp != -1), nq)
    qp = gp[anchors].copy()
    qc = (gc[anchors] + 1 + rng.randint(0, 5, nq)) % 6
    return qp, qc.astype(np.int64), gp, gc


def mars_row(kind, ng, K, gp, rng):
    if kind == 'descending':                  # every element beats the running threshold
        return -np.arange(ng, dtype=np.float32)
    if kind == 'ascending':
        return np.arange(ng, dtype=np.float32)
    if kind == 'constant':                    # index order decides
        return np.full(ng, 0.5, np.float32)
    if kind == 'signed_zeros':
        return np.where(rng.rand(ng) < 0.5, np.float32(-0.0), np.float32(0.0)).astype(np.float32)
    r = rng.rand(ng).astype(np.float32)
    order = np.argsort(r, kind='stable')
    if kind == 'tie_at_k' and ng > K:         # the K-th, (K+1)-th and (K+2)-th distances equal
        r[order[K:K + 2]] = r[order[K - 1]]
    elif kind == 'special_beyond_k':
        beyond = order[K:]
        r[beyond] = SPECIALS[:4][rng.randint(0, 4, len(beyond))]
    elif kind == 'distractors_first':
        dis = np.flatnonzero(gp == -1)
        r[dis[:K]] = -1.0 - rng.rand(min(K, len(dis))).astype(np.float32)
    return r


def mars_case(K, ng, seed):
    rng = np.random.RandomState(seed)
    qp, qc, gp, gc = mars_labels(len(MARS_ROWS), ng, seed)
    d = np.stack([mars_row(kind, ng, K, gp, rng) for kind in MARS_ROWS]).astype(np.float32)
    return qp, qc, gp, gc, d


def mars_inputs(d):
    yield 'host', d
    yield 'device', torch.from_numpy(d).cuda()
    yield 'device-ld', strided(d, d.shape[1] + 3)


def check_mars(evaluate_mars, case, K):
    qp, qc, gp, gc, d = case
    ref_cmc, ref_map, ref_ap = orank.mars_port(d, qp, gp, qc, gc, K, return_ap=True)
    for name, dist in mars_inputs(d):
        cmc, mAP, ap = evaluate_mars(dist, qp, gp, qc, gc, K, return_all_ap=True)
        bad = np.flatnonzero(_bits64(ap) != _bits64(ref_ap))
        assert bad.size == 0, (name, 'AP differs for rows', [MARS_ROWS[i] if len(ap) == len(MARS_ROWS) else i for i in bad])
        assert np.array_equal(_bits64(cmc), _bits64(ref_cmc)), name
        assert _bits64(mAP) == _bits64(ref_map), name
    return ref_ap


def _buf_len(K):
    L = 2048
    while L < 2 * K:
        L *= 2
    return L


MARS_K = [1, 2, 127, 128, 129, 256, 257, 1024, 4096, 8192]
MARS_CASES = [(K, ng) for K in MARS_K for ng in sorted({1023, 1024, 1025, 3 * _buf_len(K) + 5}) if ng >= K]


@gpu
@pytest.mark.parametrize('K,ng', MARS_CASES)
def test_mars_topk_boundaries(evaluate_mars, K, ng):
    check_mars(evaluate_mars, mars_case(K, ng, seed=K * 7 + ng), K)


@gpu
@pytest.mark.parametrize('K', [1, 2, 129, 1024, 8192])
def test_mars_num_g_equals_max_rank(evaluate_mars, K):
    check_mars(evaluate_mars, mars_case(K, K, seed=K), K)


@gpu
def test_mars_errors(evaluate_mars):
    qp, qc, gp, gc, d = mars_case(16, 100, seed=3)
    for name, dist in mars_inputs(d):
        with pytest.raises(ValueError):
            evaluate_mars(dist, qp, gp, qc, gc, 101)
    with pytest.raises(ValueError):
        orank.mars_port(d, qp, gp, qc, gc, 101)
    # query 0's identity has no item seen by another camera; its nearest item is a plain negative
    gp2 = gp.copy()
    gp2[gp2 == qp[0]] = -1
    gc2 = gc.copy()
    gp2[:3], gc2[:3] = qp[0], qc[0]
    gp2[3] = qp[0] + 1000
    d2 = d.copy()
    d2[0, 3] = -10.0
    with pytest.raises(ZeroDivisionError):
        orank.mars_port(d2, qp, gp2, qc, gc2, 16)
    for name, dist in mars_inputs(d2):
        with pytest.raises(ZeroDivisionError):
            evaluate_mars(dist, qp, gp2, qc, gc2, 16)


# 262 144 / 262 145: 2048 / 2049 leaves of the pairwise sum, either side of the leaf table of rank_mars_finish_kernel
# (kMaxLeaves); above it the leaves are summed during the tree walk
MAP_NQ = [1, 7, 8, 9, 127, 128, 129, 136, 1024, 8191, 8192, 8193, 100003, 262144, 262145]


@gpu
@pytest.mark.parametrize('nq', MAP_NQ)
def test_map_sum_order(evaluate_mars, evaluate_cy, nq):
    """MARS: mAP is np.mean of the GPU's own AP vector (numpy's pairwise sum: leaves of <= 128, splits at
    multiples of 8), besides equal to the oracle.  market1501: the sequential fp32 sum, against the oracle."""
    rng = np.random.RandomState(nq)
    ng, K = 40, 10
    gp = np.arange(ng, dtype=np.int64) % 12
    gc = rng.randint(1, 6, ng).astype(np.int64)
    qp = rng.randint(0, 12, nq).astype(np.int64)
    qc = np.zeros(nq, np.int64)
    d = (rng.rand(nq, ng) * rng.choice([1e-3, 1.0, 1e3], (nq, 1))).astype(np.float32)
    ref_cmc, ref_map, ref_ap = orank.mars_port(d, qp, gp, qc, gc, K, return_ap=True)
    for dist in (d, torch.from_numpy(d).cuda()):
        cmc, mAP, ap = evaluate_mars(dist, qp, gp, qc, gc, K, return_all_ap=True)
        assert len(np.unique(ap)) > min(nq, 8) // 2
        assert _bits64(mAP) == _bits64(np.mean(ap)), (mAP, np.mean(ap))
        assert np.array_equal(_bits64(ap), _bits64(ref_ap))
        assert _bits64(mAP) == _bits64(ref_map) and np.array_equal(_bits64(cmc), _bits64(ref_cmc))
    qp_m = qp.copy()
    qp_m[1::5] = 99                         # absent identities: num_valid < nq
    check_market(evaluate_cy, (qp_m, qc, gp, gc, d), 50)


# ------------------------------------------------------------------------------------------------
# sharded kernels, single process: shards are column slices of one matrix
# ------------------------------------------------------------------------------------------------
@pytest.fixture(scope='module')
def ops():
    from agrl.pytorch_b200 import sharded
    return sharded.CudaOps()


def clustered_labels(nq, ng, seed):
    """gallery ordered by pid (contiguous blocks), so most shards hold no item of most identities"""
    rng = np.random.RandomState(seed)
    gp = np.sort(rng.randint(0, max(2, ng // 30), ng)).astype(np.int64)
    gc = rng.randint(0, 6, ng).astype(np.int64)
    gp[rng.rand(ng) < 0.05] = -1
    anchors = rng.choice(np.flatnonzero(gp != -1), nq)
    qp = gp[anchors].copy()
    qc = ((gc[anchors] + 1 + rng.randint(0, 5, nq)) % 6).astype(np.int64)
    return qp, qc, gp, gc


def skewed_bounds(ng, parts):
    """parts contiguous shard ranges: a zero-width one first (stood in for by an all-pad list, see mars_sharded),
    then a 7-item one, then the rest near-equal"""
    from agrl.pytorch_b200 import sharded
    if parts == 1:
        return [(0, ng)]
    if parts == 2:
        return [(0, 0), (0, ng)]
    rest = sharded.shard_bounds(ng - 7, parts - 2)
    return [(0, 0), (0, 7)] + [(lo + 7, hi + 7) for lo, hi in rest]


def mars_sharded(ops, d, labels, bounds, K, permute):
    qp, qc, gp, gc = labels
    dev = torch.device('cuda')
    dd = torch.from_numpy(d).to(dev)
    tq, tqc = torch.as_tensor(qp).to(dev), torch.as_tensor(qc).to(dev)
    nq = len(qp)
    keys, cls, ngood, st = [], [], 0, torch.zeros(1, dtype=torch.int32, device=dev)
    for lo, hi in bounds:
        if hi == lo:
            # the partial kernel refuses a zero-width shard (test_mars_partial_refuses_empty_shard); what reaches
            # the merge for a shard without candidates is an all-pad list with no good image
            k = torch.full((nq, K), -1, dtype=torch.int64, device=dev)
            c = torch.zeros(nq, K, dtype=torch.uint8, device=dev)
            n = torch.zeros(nq, dtype=torch.int32, device=dev)
        else:
            k, c, n, st = ops.partial(dd[:, lo:hi], tq, torch.as_tensor(gp[lo:hi]).to(dev), tqc,
                                      torch.as_tensor(gc[lo:hi]).to(dev), K, lo)
        keys.append(k); cls.append(c); ngood = ngood + n
    keys, cls = torch.stack(keys), torch.stack(cls)
    if permute:                # lists not ascending: the merge must notice and sort
        perm = torch.randperm(K, generator=torch.Generator().manual_seed(K)).to(dev)
        keys, cls = keys[:, :, perm].contiguous(), cls[:, :, perm].contiguous()
    return ops.merge(keys, cls, ngood, K, st)


# (parts, K): parts * K below, at and above a power of two; up to the merge's limit of 16384
MERGE_CASES = [(3, 85), (4, 64), (1, 257), (2, 129), (2, 512), (5, 205), (3, 341), (8, 1023), (2, 4096),
               (3, 2731), (4, 4096), (3, 5461)]


@gpu
@pytest.mark.parametrize('layout', ['even', 'skewed'])
@pytest.mark.parametrize('parts,K', MERGE_CASES)
def test_mars_partial_merge_sizes(ops, parts, K, layout):
    from agrl.pytorch_b200 import sharded
    ng = max(3 * K, 2000) + 11
    nq = 24
    labels = clustered_labels(nq, ng, seed=parts * 100 + K)
    rng = np.random.RandomState(K)
    d = (rng.randint(0, 256, (nq, ng)) / 256.0).astype(np.float32)     # ties across shard boundaries
    d[1] = 0.5
    d[2] = -np.arange(ng, dtype=np.float32)
    qp, qc, gp, gc = labels
    ref_cmc, ref_map = orank.mars_port(d, qp, gp, qc, gc, K)
    bounds = sharded.shard_bounds(ng, parts) if layout == 'even' else skewed_bounds(ng, parts)
    assert len(bounds) == parts
    for permute in (False, True):
        cmc, mAP = mars_sharded(ops, d, labels, bounds, K, permute)
        assert np.array_equal(_bits64(cmc), _bits64(ref_cmc)), permute
        assert _bits64(mAP) == _bits64(ref_map), permute


@gpu
def test_mars_partial_refuses_empty_shard(ops):
    """a shard with no gallery row is refused before any launch (num_g < 1), never ranked"""
    qp, qc, gp, gc = clustered_labels(4, 100, seed=1)
    dev = torch.device('cuda')
    d = torch.zeros(4, 100, device=dev)
    with pytest.raises(ValueError):
        ops.partial(d[:, 0:0], torch.as_tensor(qp).to(dev), torch.as_tensor(gp[:0]).to(dev),
                    torch.as_tensor(qc).to(dev), torch.as_tensor(gc[:0]).to(dev), 8, 0)


def market_sharded_case(parts, cap, seed):
    """Identity A has exactly `cap` items in every shard but (for parts >= 3) the last, which holds none; other
    identities, distractors and filler fill each shard with 500 more items.  Distances take 64 levels."""
    rng = np.random.RandomState(seed)
    gp, gc, bounds = [], [], []
    for s in range(parts):
        n_a = 0 if (parts >= 3 and s == parts - 1) else cap
        other = np.where(rng.rand(500) < 0.2, -1, 100 + rng.randint(0, 6, 500))
        blk = np.concatenate([np.zeros(n_a, np.int64), other]).astype(np.int64)
        rng.shuffle(blk)
        bounds.append((len(gp), len(gp) + len(blk)))
        gp += list(blk)
        gc += list(rng.randint(0, 6, len(blk)))
    gp, gc = np.asarray(gp, np.int64), np.asarray(gc, np.int64)
    qp = np.array([0, 0, 0, 0, 0, 0, 100, 101, 102, 7777, 103], np.int64)
    qc = np.array([0, 1, 2, 3, 4, 5, 0, 1, 2, 0, 3], np.int64)
    gc[gp == 103] = 3                       # 103: junk-only for the query seen by camera 3
    d = (rng.randint(0, 64, (len(qp), len(gp))) / 64.0).astype(np.float32)
    return (qp, qc, gp, gc), d, bounds


def market_sharded(ops, d, labels, bounds, cap, K=50):
    qp, qc, gp, gc = labels
    dev = torch.device('cuda')
    dd = torch.from_numpy(d).to(dev)
    tq, tqc = torch.as_tensor(qp).to(dev), torch.as_tensor(qc).to(dev)
    lab = [(torch.as_tensor(gp[lo:hi]).to(dev), torch.as_tensor(gc[lo:hi]).to(dev)) for lo, hi in bounds]
    need = max(int(ops.market_count(tq, tg, tqc, tgc)[0].cpu()) for tg, tgc in lab)
    assert need <= cap
    keys, counts = [], 0
    for (lo, hi), (tg, tgc) in zip(bounds, lab):
        k, c, st = ops.market_gather(dd[:, lo:hi].contiguous(), tq, tg, tqc, tgc, lo, cap)
        keys.append(k); counts = counts + c
    keys_all = torch.stack(keys)
    cnt = 0
    for (lo, hi), (tg, tgc) in zip(bounds, lab):
        c, srt = ops.market_bin(dd[:, lo:hi].contiguous(), lo, keys_all)
        cnt = cnt + c
    return need, ops.market_finalize(cnt, srt, counts, len(gp), len(bounds), cap, K, st)


@gpu
@pytest.mark.parametrize('parts,cap', [(1, 8192), (2, 4096), (3, 2728), (4, 2048), (8, 1024)])
def test_market1501_sharded_list_limit(ops, parts, cap):
    """parts * cap up to 8192, the largest list the bin kernel admits; at (1, 8192), (2, 4096) ... every slot
    holds an item, so the sorted list has no pad at all"""
    labels, d, bounds = market_sharded_case(parts, cap, seed=parts)
    qp, qc, gp, gc = labels
    ref_cmc, ref_map = orank.market1501_port(d, qp, gp, qc, gc, 50)
    need, (cmc, mAP) = market_sharded(ops, d, labels, bounds, cap)
    assert need == cap
    assert np.array_equal(_bits32(cmc), _bits32(ref_cmc))
    assert mAP == ref_map


@gpu
@pytest.mark.parametrize('parts,cap', [(1, 8200), (2, 4100), (3, 2736)])
def test_market1501_sharded_list_over_limit_refused(ops, parts, cap):
    from agrl.pytorch_b200 import _lib
    labels, d, bounds = market_sharded_case(parts, 16, seed=parts)
    qp, qc, gp, gc = labels
    dev = torch.device('cuda')
    dd = torch.from_numpy(d).to(dev)
    tq, tqc = torch.as_tensor(qp).to(dev), torch.as_tensor(qc).to(dev)
    keys = []
    for lo, hi in bounds:
        k, c, st = ops.market_gather(dd[:, lo:hi].contiguous(), tq, torch.as_tensor(gp[lo:hi]).to(dev), tqc,
                                     torch.as_tensor(gc[lo:hi]).to(dev), lo, cap)
        keys.append(k)
    lo, hi = bounds[0]
    with pytest.raises(_lib.AgrlError):
        ops.market_bin(dd[:, lo:hi].contiguous(), lo, torch.stack(keys))
    assert ops.lib.agrl_rank_market1501_list_len(parts, cap) == 0
    assert ops.lib.agrl_rank_market1501_finalize_workspace_bytes(len(qp), parts, cap, 50) == 0
