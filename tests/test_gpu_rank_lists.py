"""Ranked lists on a B200 (metrics.rank_lists, metrics.retrieve, sharded.rank_lists_sharded; csrc/rank.cu
rank_lists_kernel and rank_junk_depth_kernel) against np.argsort(kind='stable') of the matrix the GPU's own
compute_distance_matrix produced -- the bits the fused epilogue sees too.  Distances are compared as int32 bit patterns
(-0 is ranked and returned as +0, every NaN as 0x7FFFFFFF), so NaN and signed zeros compare too."""
import numpy as np
import pytest
import torch

from oracle import rank as orank
from oracle import synth

pytestmark = pytest.mark.gpu

NAN_BITS = 0x7FFFFFFF


def canon_bits(v):
    """what the lists return for ranked values v: -0 -> +0, NaN -> 0x7FFFFFFF, as int32 bit patterns"""
    v = np.asarray(v, np.float32) + np.float32(0.0)
    b = v.view(np.int32).copy()
    b[np.isnan(v)] = NAN_BITS
    return b


def reference(d, k, labels=None):
    """(indices, distance bits) of the stable argsort of each row, junk columns deleted when labels are given"""
    nq, ng = d.shape
    idx = np.full((nq, k), -1, np.int64)
    bits = np.full((nq, k), np.float32(np.inf).view(np.int32), np.int32)
    for q in range(nq):
        cols = np.arange(ng)
        if labels is not None:
            qp, qc, gp, gc = labels
            cols = cols[~((gp == qp[q]) & (gc == qc[q]))]
        order = cols[np.argsort(d[q, cols], kind='stable')][:k]
        idx[q, :len(order)] = order
        bits[q, :len(order)] = canon_bits(d[q, order])
    return idx, bits


def check(got, ref, what=''):
    i, v = got
    assert i.is_cuda and v.is_cuda and i.dtype == torch.int64 and v.dtype == torch.float32
    ri, rb = ref
    i, b = i.cpu().numpy(), v.cpu().numpy().view(np.int32)
    bad = np.argwhere(i != ri)
    assert bad.size == 0, (what, 'index differs at', bad[:5].tolist())
    assert np.array_equal(b, rb), (what, 'distance bits differ at', np.argwhere(b != rb)[:5].tolist())


def strided(d, ld):
    buf = torch.full((d.shape[0], ld), float('nan'), device='cuda')
    buf[:, :d.shape[1]] = torch.from_numpy(d).cuda()
    return buf[:, :d.shape[1]]


def odd_ld(ng):
    """row stride with ld % 4 == 1: rows 0-3 start at all four offsets within 16 bytes"""
    return ng + ((1 - ng) % 4 or 4)


def _buf_len(K):
    L = 2048
    while L < 2 * K:
        L *= 2
    return L


LIST_K = [1, 2, 127, 128, 129, 256, 257, 1024, 4096, 8192]
LIST_CASES = [(k, ng) for k in LIST_K for ng in sorted({k - 1, k, k + 1, 1023, 1024, 1025, 3 * _buf_len(k) + 5}) if ng >= 1]


def boundary_matrix(nq, ng, seed):
    """quantised distances (ties everywhere) with special values sprinkled in"""
    rng = np.random.RandomState(seed)
    d = (rng.randint(-64, 256, (nq, ng)) / 64.0).astype(np.float32)
    sp = np.array([np.nan, -np.nan, np.inf, -np.inf, 0.0, -0.0], np.float32)
    m = rng.rand(nq, ng) < 0.02
    d[m] = sp[rng.randint(0, len(sp), int(m.sum()))]
    return d


@pytest.mark.parametrize('k,ng', LIST_CASES)
def test_matrix_route_depth_boundaries(k, ng):
    from agrl.pytorch_b200 import metrics
    d = boundary_matrix(6, ng, seed=k * 31 + ng)
    ref = reference(d, k)
    check(metrics.rank_lists(strided(d, odd_ld(ng)), k), ref, 'strided')
    if ng in (1023, 1025):
        check(metrics.rank_lists(d, k), ref, 'numpy')


def test_depth_over_8192_raises():
    from agrl.pytorch_b200 import metrics
    d = torch.zeros(2, 9000, device='cuda')
    with pytest.raises(ValueError, match='8192'):
        metrics.rank_lists(d, 8193)
    qp, gp = np.zeros(2, np.int64), np.zeros(9000, np.int64)
    qc, gc = np.zeros(2, np.int64), np.zeros(9000, np.int64)
    gc[:10] = 1
    with pytest.raises(ValueError, match='8192'):                     # k + J = 8000 + 8990
        metrics.rank_lists(d, 8000, qp, gp, qc, gc, exclude_junk=True)


def test_adversarial_rows():
    from agrl.pytorch_b200 import metrics
    ng = 1500
    rows = [np.full(ng, 1.0), np.full(ng, np.nan), np.full(ng, -np.nan), np.full(ng, -0.0),
            np.where(np.arange(ng) % 2, 0.0, -0.0), np.where(np.arange(ng) % 3 == 0, np.inf, -np.inf),
            np.where(np.arange(ng) % 5 == 0, np.nan, -np.nan)]
    rng = np.random.RandomState(1)
    mix = rng.choice(np.array([np.nan, -np.nan, np.inf, -np.inf, 0.0, -0.0, 1.0, -1.0, 1e-45, -3e38], np.float32), ng)
    rows += [mix, -np.arange(ng, dtype=np.float32), np.arange(ng, dtype=np.float32)[::-1].copy()]
    d = np.stack(rows).astype(np.float32)
    for k in (1, 7, 300, 1499, 1500, 1501, 3000):
        ref = reference(d, k)
        for ld in (ng, odd_ld(ng)):
            check(metrics.rank_lists(strided(d, ld), k), ref, (k, ld))
    got = metrics.rank_lists(d, 3000)
    assert (got[0][:, ng:] == -1).all() and torch.isinf(got[1][:, ng:]).all() and (got[1][:, ng:] > 0).all()


# ---- the fused route -------------------------------------------------------------------------------------------
def fused_vs_matrix(qf, gf, metric, split, ks, rows=None, labels=None):
    """retrieve (fused where it can) == rank_lists on the GPU's matrix; the matrix route == argsort on sampled rows"""
    from agrl.pytorch_b200 import metrics
    from agrl.pytorch_b200.metrics.distance import PreparedOperand
    gop = PreparedOperand(gf, metric, split)
    dm = metrics.compute_distance_matrix(qf, gf, metric, split=split)
    lab = labels or [None] * 4
    for k in ks:
        got = metrics.retrieve(qf, gop, k, q_pids=lab[0], g_pids=lab[1], q_camids=lab[2], g_camids=lab[3],
                               exclude_junk=labels is not None, fused=True)
        want = metrics.rank_lists(dm, k, *lab, exclude_junk=labels is not None)
        assert torch.equal(got[0], want[0]), (metric, split, k)
        assert torch.equal(got[1].view(torch.int32), want[1].view(torch.int32)), (metric, split, k)
        if rows is not None:
            r = torch.as_tensor(rows, device='cuda')
            dn = dm[r].cpu().numpy()
            lr = None if labels is None else (np.asarray(labels[0])[rows], np.asarray(labels[2])[rows],
                                              np.asarray(labels[1]), np.asarray(labels[3]))
            check((want[0][r], want[1][r]), reference(dn, k, lr), (metric, split, k))
    return dm


@pytest.mark.parametrize('split', [5, 3])
@pytest.mark.parametrize('metric', ['euclidean', 'cosine'])
def test_fused_route_mars_size(metric, split):
    qp, qc, gp, gc = synth.eval_labels('mars', seed=3)
    qf, gf = synth.eval_features(qp, gp, 4096, seed=3, clustered=True)
    qf, gf = qf.cuda(), gf.cuda()
    gf[100:200] = gf[300:400]                                          # exact duplicates
    fused_vs_matrix(qf, gf, metric, split, (1, 50, 255, 256, 257), rows=[0, 1, 977, 1979])


def test_fused_route_large_block():
    g = torch.Generator(device='cuda').manual_seed(4)
    qf = torch.randn(10000, 128, generator=g, device='cuda')
    gf = torch.randn(100000, 128, generator=g, device='cuda')
    gf[5000:5100] = gf[7000:7100]
    fused_vs_matrix(qf, gf, 'euclidean', 5, (50, 256), rows=[0, 4999, 9999])


def test_overflow_falls_back_to_the_same_lists():
    """gallery ordered by decreasing distance to query 0: the fused candidate list overflows, the blocks take over"""
    from agrl.pytorch_b200 import metrics, sharded
    from agrl.pytorch_b200.metrics.distance import PreparedOperand
    d, ng, nq = 64, 40000, 40
    g = torch.Generator(device='cuda').manual_seed(11)
    qf = torch.randn(nq, d, generator=g, device='cuda')
    u = torch.nn.functional.normalize(torch.randn(d, generator=g, device='cuda'), dim=0)
    gf = qf[0][None] + (ng - torch.arange(ng, device='cuda', dtype=torch.float32))[:, None] * 0.01 * u[None]
    ops = sharded.CudaOps()
    qop, gop = PreparedOperand(qf), PreparedOperand(gf)
    lab = [torch.zeros(nq, dtype=torch.int64, device='cuda'), torch.ones(ng, dtype=torch.int64, device='cuda')]
    st = ops.topk_fused(qop, gop, lab[0], lab[1], lab[0], lab[1], 50, 0, allow_fallback=False)[3]
    assert int(st.cpu()) & 8
    dm = metrics.compute_distance_matrix(qf, gf)
    for k in (50, 200, 256):
        got, want = metrics.retrieve(qf, gop, k), metrics.rank_lists(dm, k)
        assert torch.equal(got[0], want[0]) and torch.equal(got[1].view(torch.int32), want[1].view(torch.int32))
    check((want[0][:2], want[1][:2]), reference(dm[:2].cpu().numpy(), 256))


def test_retrieve_default_route_and_small_gallery():
    from agrl.pytorch_b200 import metrics
    g = torch.Generator(device='cuda').manual_seed(2)
    for ng in (1, 100, 40000):
        qf = torch.randn(50, 96, generator=g, device='cuda')
        gf = torch.randn(ng, 96, generator=g, device='cuda')
        dm = metrics.compute_distance_matrix(qf, gf, 'cosine')
        for k in (1, 64, 300):
            got, want = metrics.retrieve(qf, gf, k, metric='cosine'), metrics.rank_lists(dm, k)
            assert torch.equal(got[0], want[0]) and torch.equal(got[1].view(torch.int32), want[1].view(torch.int32))


# ---- junk exclusion --------------------------------------------------------------------------------------------
def junk_labels(nq, ng, seed, heavy=0, nid=60):
    """labels with distractors; query 0's identity gets `heavy` extra items under its own camera"""
    rng = np.random.RandomState(seed)
    gp = rng.randint(0, nid, ng).astype(np.int64)
    gc = rng.randint(0, 4, ng).astype(np.int64)
    gp[::9] = -1
    qp = rng.randint(0, nid, nq).astype(np.int64)
    qc = rng.randint(0, 4, nq).astype(np.int64)
    if heavy:
        where = rng.choice(ng, heavy, replace=False)
        gp[where], gc[where] = qp[0], qc[0]
    return qp, qc, gp, gc


@pytest.mark.parametrize('J', ['zero', 'one', 'large'])
def test_junk_exclusion_matrix_route(J):
    from agrl.pytorch_b200 import metrics, sharded
    nq, ng = 64, 5000
    qp, qc, gp, gc = junk_labels(nq, ng, seed=7, heavy=700 if J == 'large' else 0)
    if J == 'zero':
        gc = (gc % 2) + 10                             # no gallery item shares a query's camera
    elif J == 'one':
        gp = np.arange(ng, dtype=np.int64) + 1000      # unique gallery ids; queries 0-3 each own one same-camera item
        qp[:4], qc[:4] = gp[[5, 9, 11, 4000]], gc[[5, 9, 11, 4000]]
    rng = np.random.RandomState(8)
    d = (rng.randint(0, 512, (nq, ng)) / 64.0).astype(np.float32)
    d[0, np.flatnonzero((gp == qp[0]) & (gc == qc[0]))] = -1.0          # the junk ranks first
    dm = strided(d, odd_ld(ng))
    j, _ = sharded.CudaOps().junk_depth(*[torch.as_tensor(x).cuda() for x in (qp, gp, qc, gc)])
    want_j = max(int(np.sum((gp == p) & (gc == c))) for p, c in zip(qp, qc))
    assert int(j.cpu()) == want_j and want_j == {'zero': 0, 'one': 1}.get(J, want_j) and (J != 'large' or want_j >= 700)
    for k in (1, 20, 100, 1000):
        got = metrics.rank_lists(dm, k, qp, gp, qc, gc, exclude_junk=True)
        check(got, reference(d, k, (qp, qc, gp, gc)), (J, k))
        if k == 1000:
            listed = got[0].cpu().numpy()
            assert (listed >= 0).all()
            assert J == 'one' or (gp[listed] == -1).any()                 # distractors stay in the lists


def test_junk_depth_crosses_the_fused_limit():
    """k + J <= 256 stays fused, k + J > 256 takes the blocks: the same lists as the matrix route either way"""
    qp, qc, gp, gc = junk_labels(300, 40000, seed=9, heavy=100, nid=2000)
    g = torch.Generator(device='cuda').manual_seed(9)
    qf = torch.randn(300, 128, generator=g, device='cuda')
    gf = torch.randn(40000, 128, generator=g, device='cuda')
    own = np.flatnonzero((gp == qp[0]) & (gc == qc[0]))
    gf[torch.as_tensor(own, device='cuda')] = qf[0] + 0.01 * torch.randn(len(own), 128, generator=g, device='cuda')
    J = max(int(np.sum((gp == p) & (gc == c))) for p, c in zip(qp, qc))
    assert 100 <= J < 200
    ks = (1, 256 - J, 257 - J, 200)
    fused_vs_matrix(qf, gf, 'euclidean', 5, ks, rows=[0, 1, 299], labels=[qp, gp, qc, gc])


# ---- shards in one process ---------------------------------------------------------------------------------------
def shard_layouts(ng):
    from agrl.pytorch_b200 import sharded
    yield 'two', sharded.shard_bounds(ng, 2)
    yield 'three', sharded.shard_bounds(ng, 3)
    yield 'eight+empty', [(0, 0)] + sharded.shard_bounds(ng, 7)
    yield 'all-matches', [(0, 0), (0, ng - 100), (ng - 100, ng)]


def merged(ops, shard_keys, k, labels, exclude_junk):
    keys = torch.stack(shard_keys)
    return ops.lists(keys, k, *labels, exclude_junk=exclude_junk)


@pytest.mark.parametrize('source', ['plain', 'fused', 're_rank'])
def test_shards_merge_to_the_whole_gallery_lists(source):
    from agrl.pytorch_b200 import metrics, sharded
    from agrl.pytorch_b200.metrics.distance import PreparedOperand
    from agrl.pytorch_b200.utils.re_ranking import re_ranking_dev
    ops = sharded.CudaOps()
    nq, ng, dim = 120, (3000 if source == 're_rank' else 36000), 64
    qp, qc, gp, gc = junk_labels(nq, ng, seed=12, nid=1000)
    gp[gp == qp[1]] = -1
    gp[-100:], gc[-100:] = qp[1], qc[1]                            # the last shard: every item of query 1's identity
    g = torch.Generator(device='cuda').manual_seed(12)
    qf = torch.randint(-2, 3, (nq, dim), generator=g, device='cuda').float()     # quantised: many exact ties
    gf = torch.randint(-2, 3, (ng, dim), generator=g, device='cuda').float()
    gf[1::2] = gf[0:-1:2][:ng // 2]                                 # duplicates across shard boundaries
    dm = metrics.compute_distance_matrix(qf, gf)
    if source == 're_rank':
        dm = re_ranking_dev(dm, metrics.compute_distance_matrix(qf, qf), metrics.compute_distance_matrix(gf, gf))
    dev_lab = [torch.as_tensor(x).cuda() for x in (qp, gp, qc, gc)]
    for exclude_junk in (False, True):
        for k in (1, 50, 200):
            depth = sharded.list_depth(k, ops, dev_lab, exclude_junk)
            want = metrics.rank_lists(dm, k, qp, gp, qc, gc, exclude_junk=exclude_junk)
            for name, bounds in shard_layouts(ng):
                parts = []
                for lo, hi in bounds:
                    if hi == lo:
                        parts.append(torch.full((nq, depth), -1, dtype=torch.int64, device='cuda'))
                        continue
                    lab = [dev_lab[0], dev_lab[1][lo:hi], dev_lab[2], dev_lab[3][lo:hi]]
                    dj = sharded.list_depth(k, ops, lab, exclude_junk)
                    assert dj <= depth
                    if source == 'fused':
                        kk = ops.topk_keys(PreparedOperand(qf), PreparedOperand(gf[lo:hi]), depth, lo,
                                           fused=depth <= 256)
                    else:
                        kk = ops.keys(dm[:, lo:hi], depth, lo)
                    parts.append(kk)
                got = merged(ops, parts, k, dev_lab, exclude_junk)
                assert torch.equal(got[0], want[0]), (source, exclude_junk, k, name)
                assert torch.equal(got[1].view(torch.int32), want[1].view(torch.int32)), (source, exclude_junk, k, name)
            if k == 50:
                check(want, reference(dm.cpu().numpy(), k, (qp, qc, gp, gc) if exclude_junk else None), (source, k))
    if source == 're_rank':                                         # the sharded entry on one process
        got = sharded.rank_lists_sharded(qf, gf, 30, qp, gp, qc, gc, exclude_junk=True, re_rank=True)
        want = metrics.rank_lists(dm, 30, qp, gp, qc, gc, exclude_junk=True)
        assert torch.equal(got[0], want[0]) and torch.equal(got[1].view(torch.int32), want[1].view(torch.int32))
    else:
        for fused in (False, True):
            got = sharded.rank_lists_sharded(qf, gf, 30, qp, gp, qc, gc, exclude_junk=True, fused=fused)
            want = metrics.rank_lists(dm, 30, qp, gp, qc, gc, exclude_junk=True)
            assert torch.equal(got[0], want[0]) and torch.equal(got[1].view(torch.int32), want[1].view(torch.int32))


def test_lists_kernel_limits():
    from agrl.pytorch_b200 import _lib, sharded
    ops = sharded.CudaOps()
    keys = torch.full((3, 4, 5462), -1, dtype=torch.int64, device='cuda')      # 3 x 5462 > 16384
    with pytest.raises(_lib.AgrlError):
        ops.lists(keys, 10)
    with pytest.raises(ValueError):
        ops.lists(keys[:1, :, :5], 6)                                         # k > depth
    got = ops.lists(keys[:, :, :5461], 5461)                                  # 3 x 5461 <= 16384: all empty
    assert (got[0] == -1).all() and torch.isinf(got[1]).all()


# ---- the engine and the metrics --------------------------------------------------------------------------------
def test_engine_return_ranked():
    from agrl.pytorch_b200 import engine, metrics
    from test_gpu_engine import make_loaders, make_model
    model = make_model()
    ql, gl, labels = make_loaders()
    base = engine.test(model, ql, gl, 'avg', True, max_rank=20, verbose=False)
    d = engine.test(model, ql, gl, 'avg', True, return_distmat=True, max_rank=20, verbose=False)
    d2 = engine.test(model, ql, gl, 'avg', True, return_distmat=True, return_ranked=5, max_rank=20, verbose=False)
    assert isinstance(d2, np.ndarray) and np.array_equal(d, d2)
    r1, mAP, idx, dist_ = engine.test(model, ql, gl, 'avg', True, return_ranked=7, max_rank=20, verbose=False)
    assert len(base) == 2 and (r1, mAP) == base
    want = metrics.rank_lists(d, 7)
    assert torch.equal(idx, want[0]) and torch.equal(dist_.view(torch.int32), want[1].view(torch.int32))
    check((idx, dist_), reference(d, 7))


@pytest.mark.parametrize('shape', ['mars', (300, 2000, 40, 4)])
def test_lists_reproduce_the_mars_metric(shape):
    """the first max_rank columns, classified with the labels, give evaluate_rank(use_metric_mars=True) exactly"""
    from agrl.pytorch_b200 import metrics
    qp, qc, gp, gc = synth.eval_labels(shape, seed=5)
    qf, gf = synth.eval_features(qp, gp, 256, seed=5, clustered=True)
    dm = metrics.compute_distance_matrix(qf.cuda(), gf.cuda())
    R = 50
    cmc, mAP = metrics.evaluate_rank(dm, qp, gp, qc, gc, max_rank=R, use_metric_mars=True)
    idx = metrics.retrieve(qf.cuda(), gf.cuda(), R)[0].cpu().numpy()
    # a matrix that ranks exactly as the lists say over the first R places (the MARS metric reads no further)
    dl = np.full((len(qp), len(gp)), np.float32(R), np.float32)
    np.put_along_axis(dl, idx, np.arange(R, dtype=np.float32)[None], axis=1)
    rcmc, rmap = orank.mars_port(dl, qp, gp, qc, gc, R)
    assert np.array_equal(rcmc, cmc) and rmap == mAP
