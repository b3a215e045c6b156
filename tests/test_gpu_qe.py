"""Alpha query expansion on a B200 (csrc/qe.cu qe_mix_kernel, metrics.query_expansion, sharded.query_expansion_sharded,
engine.test(aqe=True)).

The mix kernel is checked against an fp64 restatement given the GPU's own lists, with sentinel guard bands around its
output; the composed call against the public calls it is made of, bit for bit; and the whole computation against the
fp64 oracle (oracle/qe.py) on features whose margin -- each row's k-th minus (k+1)-th similarity -- is asserted at every
iteration.  The lists are compared as sets: the margin decides a list's members, not their order, which changes only
the order of the fp32 sum."""
import os
import socket

import numpy as np
import pytest
import torch

from agrl.pytorch_b200 import _lib, metrics, sharded
from oracle import qe as oqe

pytestmark = pytest.mark.gpu

SENTINEL = 0x7FBADBAD                      # a NaN payload no computation produces
GUARD = 67


def lib():
    return _lib.require_device()


def stream():
    return torch.cuda.current_stream().cuda_stream


def padded(rows, cols, ld):
    """(buffer, view): a (rows, cols) view with row stride ld into a buffer with GUARD sentinel words on either side"""
    buf = torch.full((2 * GUARD + rows * ld,), SENTINEL, dtype=torch.int32, device='cuda').view(torch.float32)
    return buf, buf[GUARD:GUARD + rows * ld].view(rows, ld)[:, :cols]


def intact(buf, rows, cols, ld):
    """every word outside the (rows, cols) view is still the sentinel"""
    b = buf.view(torch.int32).cpu().numpy().copy()
    inner = b[GUARD:GUARD + rows * ld].reshape(rows, ld)
    inner[:, :cols] = SENTINEL
    return bool((b == SENTINEL).all())


def call_mix(idx, d, feats, alpha, out, rows=None, k=None):
    rows = idx.shape[0] if rows is None else rows
    k = idx.shape[1] if k is None else k
    return lib().agrl_qe_mix_dev(idx.data_ptr(), d.data_ptr(), idx.stride(0), rows, k, feats.data_ptr(),
                                 feats.stride(0), feats.shape[0], feats.shape[1], float(alpha), out.data_ptr(),
                                 out.stride(0), stream())


def mix_fp64(idx, d, feats, alpha):
    """out[r] = sum over the valid entries of powf(1 - d, alpha) * feats[idx] / k, in fp64 (1 - d rounded to fp32 as
    the kernel forms it), and the per-element scale sum |w| |x| / k the fp32 sum is judged against"""
    idx, d, x = idx.cpu().numpy(), d.cpu().numpy(), feats.cpu().numpy().astype(np.float64)
    rows, k = idx.shape
    out = np.zeros((rows, x.shape[1]))
    scale = np.zeros((rows, x.shape[1]))
    with np.errstate(invalid='ignore'):
        w = np.power((np.float32(1.0) - d).astype(np.float64), alpha)
    for r in range(rows):
        ok = (idx[r] >= 0) & (idx[r] < len(x))
        out[r] = w[r, ok] @ x[idx[r, ok]] / k
        scale[r] = np.abs(w[r, ok]) @ np.abs(x[idx[r, ok]]) / k
    return out, scale


def ld_of(dim, mod):
    """a row stride >= dim with ld % 4 == mod"""
    return dim + (mod - dim) % 4


DIMS = [1, 3, 4, 5, 63, 64, 65, 2048, 4096]


@pytest.mark.parametrize('k', [1, 2, 5, 31, 32, 33, 256, 257, 8192])
def test_mix_kernel_against_fp64(k):
    torch.manual_seed(k)
    ops = sharded.CudaOps()
    n = max(k + 64, 512)
    rows = 5 if k >= 256 else 37
    idx, d = ops.qe_lists(torch.randn(n, 32, device='cuda'), [(0, rows)], k)     # the GPU's own lists
    assert (idx[:, 0] == torch.arange(rows, device='cuda')).all()              # each row's list starts with itself
    idx, d = idx.clone(), d.clone()
    idx[1, k // 2] = -1                                                         # entries that contribute nothing
    if k > 1:
        idx[2, k - 1] = n
        idx[3, 0] = -(1 << 40)
    d[4, k // 3] = 1.5                                                          # similarity -0.5: NaN for alpha 0.5
    for mod in (0, 1):
        ldl = k + (3 if mod else 0)                                             # the lists at a row stride too
        lbuf_i = torch.full((rows, ldl), -7, dtype=torch.int64, device='cuda')
        lbuf_d = torch.full((rows, ldl), float('nan'), device='cuda')
        lbuf_i[:, :k], lbuf_d[:, :k] = idx, d
        li, ld_ = lbuf_i[:, :k], lbuf_d[:, :k]
        for dim in DIMS:
            ldf, ldo = ld_of(dim, mod), ld_of(dim, mod)
            feats = torch.empty(n, ldf, device='cuda')[:, :dim]
            feats.copy_(torch.randn(n, dim, device='cuda'))
            for alpha in (3.0, 0.5, 0.0):
                buf, out = padded(rows, dim, ldo)
                assert call_mix(li, ld_, feats, alpha, out) == 0
                torch.cuda.synchronize()
                assert intact(buf, rows, dim, ldo), (k, dim, mod, alpha)
                got = out.cpu().numpy()
                buf2, out2 = padded(rows, dim, ldo)
                assert call_mix(li, ld_, feats, alpha, out2) == 0
                assert np.array_equal(out2.cpu().numpy().view(np.int32), got.view(np.int32))    # repeatable
                ref, scale = mix_fp64(li, ld_, feats, alpha)
                assert np.array_equal(np.isnan(got), np.isnan(ref)), (k, dim, mod, alpha)
                assert np.isnan(got[4]).all() == (alpha == 0.5)
                fin = ~np.isnan(ref)
                tol = 1e-6 * max(1.0, np.sqrt(k)) * scale[fin] + 1e-30
                assert (np.abs(got[fin] - ref[fin]) <= tol).all(), (k, dim, mod, alpha)
            if dim % 4 == 0 and mod == 1:                           # the scalar path equals the 16-byte path
                f0 = torch.empty(n, dim, device='cuda')
                f0.copy_(feats)
                o0, o1 = torch.empty(rows, dim, device='cuda'), torch.empty(rows, dim, device='cuda')
                assert call_mix(idx, d, f0, 3.0, o0) == 0 and call_mix(li, ld_, feats, 3.0, o1) == 0
                assert torch.equal(o0.view(torch.int32), o1.view(torch.int32)), (k, dim)


def test_mix_limits():
    """AGRL_E_INVALID on one side of every limit, success on the other"""
    idx = torch.zeros(4, 8, dtype=torch.int64, device='cuda')
    d = torch.zeros(4, 8, device='cuda')
    x = torch.randn(10, 16, device='cuda')
    out = torch.empty(4, 16, device='cuda')
    L = lib()

    def mix(rows=4, k=8, ld_list=8, feats=x, ld_feat=16, num=10, dim=16, alpha=3.0, o=out, ld_out=16):
        rc = L.agrl_qe_mix_dev(idx.data_ptr(), d.data_ptr(), ld_list, rows, k, feats.data_ptr(), ld_feat, num, dim,
                               alpha, o.data_ptr(), ld_out, stream())
        torch.cuda.synchronize()
        return rc
    E = _lib.E_INVALID
    assert mix() == 0
    assert mix(rows=-1) == E and mix(rows=0) == 0
    assert mix(k=0) == E and mix(k=1) == 0
    assert mix(ld_list=7) == E and mix(k=7, ld_list=7) == 0
    assert mix(ld_feat=15) == E and mix(ld_feat=15, dim=15, ld_out=15) == 0
    assert mix(ld_out=15) == E
    assert mix(num=-1) == E and mix(num=0) == 0
    assert mix(dim=-1) == E and mix(dim=0) == 0
    for a in (float('nan'), float('inf'), float('-inf')):
        assert mix(alpha=a) == E
    assert mix(alpha=3.4e38) == 0 and mix(alpha=0.0) == 0
    assert mix(o=x, ld_out=16) == E                                             # out over feats
    assert mix(o=x[6:], ld_out=16) == E
    assert mix(o=x[6:], num=6) == 0                                             # just past the rows that are read
    assert torch.equal(mix_zero_rows(), torch.zeros(4, 16))


def mix_zero_rows():
    """num_feats == 0: every entry is out of range, every row is 0"""
    out = torch.full((4, 16), 5.0, device='cuda')
    idx = torch.zeros(4, 3, dtype=torch.int64, device='cuda')
    d = torch.zeros(4, 3, device='cuda')
    assert lib().agrl_qe_mix_dev(idx.data_ptr(), d.data_ptr(), 3, 4, 3, None, 16, 0, 16, 3.0, out.data_ptr(), 16,
                                 stream()) == 0
    return out.cpu()


def test_query_expansion_limits():
    qf, gf = torch.randn(3, 8, device='cuda'), torch.randn(5, 8, device='cuda')
    for kw in (dict(qe_k=0), dict(qe_k=9), dict(qe_k=8193), dict(qe_times=0), dict(alpha=float('nan')),
               dict(alpha=float('inf'))):
        with pytest.raises(ValueError):
            metrics.query_expansion(qf, gf, **kw)
    q, g = metrics.query_expansion(qf, gf, qe_k=8)                              # qe_k == N
    assert q.is_cuda and q.dtype == torch.float32 and q.shape == (3, 8) and g.shape == (5, 8)
    q, g = metrics.query_expansion(qf.cpu(), gf.cpu(), qe_k=1, alpha=0.0)       # alpha 0, k 1: each row itself
    assert torch.equal(q, qf) and torch.equal(g, gf)
    with pytest.raises(AssertionError):
        metrics.query_expansion(qf[0], gf)
    with pytest.raises(AssertionError):
        metrics.query_expansion(qf, gf[:, :7])
    big = torch.randn(8200, 8, device='cuda')
    metrics.query_expansion(big[:10], big[10:], qe_k=8192)                     # the deepest list
    with pytest.raises(ValueError):
        metrics.query_expansion(big[:10], big[10:], qe_k=8193)


def chain(qf, gf, k, times, alpha):
    """the public calls query_expansion is made of"""
    x = torch.cat([qf, gf])
    for _ in range(times):
        idx, d = metrics.rank_lists(metrics.compute_distance_matrix(x, x, 'cosine'), k)
        out = torch.empty_like(x)
        assert call_mix(idx, d, x, alpha, out) == 0
        x = out
    return x[:len(qf)], x[len(qf):]


def bits(t):
    return t.contiguous().view(torch.int32).cpu().numpy()


@pytest.mark.parametrize('shape,k,times,alpha', [((300, 2700, 512), 5, 2, 3.0), ((1980, 9330, 4096), 5, 1, 3.0),
                                                 ((40, 400, 65), 31, 3, 0.5), ((2000, 31000, 256), 5, 1, 3.0)])
def test_query_expansion_equals_the_chained_calls(shape, k, times, alpha):
    nq, ng, dim = shape
    torch.manual_seed(nq)
    qf, gf = torch.randn(nq, dim, device='cuda'), torch.randn(ng, dim, device='cuda')
    q, g = metrics.query_expansion(qf, gf, k, times, alpha)
    cq, cg = chain(qf, gf, k, times, alpha)
    assert np.array_equal(bits(q), bits(cq)) and np.array_equal(bits(g), bits(cg))
    if nq + ng >= sharded.FUSED_MIN_GALLERY:                                    # the fused route and distance blocks
        for fused in (True, False):
            fq, fg = metrics.query_expansion(qf, gf, k, times, alpha, fused=fused)
            assert np.array_equal(bits(fq), bits(q)) and np.array_equal(bits(fg), bits(g)), fused


def expand_stepwise(qf, gf, k, times, alpha):
    """query_expansion one iteration at a time, keeping each iteration's lists"""
    ops = sharded.CudaOps()
    x = torch.cat([qf, gf]).cuda()
    lists = []
    for _ in range(times):
        idx, d = ops.qe_lists(x, [(0, len(x))], k)
        lists.append(idx.cpu().numpy())
        x = ops.qe_mix(idx, d, x, alpha)
    return x, lists


@pytest.mark.parametrize('shape', [(1980, 9330, 4096), (10000, 100000, 2048)])
@pytest.mark.parametrize('times', [1, 3])
def test_against_the_oracle(shape, times):
    nq, ng, dim = shape
    k, alpha = 5, 3.0
    qf, gf = oqe.grouped_features(nq, ng, dim, k, seed=7)
    x, lists = expand_stepwise(qf, gf, k, times, alpha)
    q, g = metrics.query_expansion(qf, gf, k, times, alpha)
    assert np.array_equal(bits(x), bits(torch.cat([q, g])))
    oq, og, olists, _, margins = oqe.aqe(qf, gf, k, times, alpha, device='cuda')
    torch.cuda.empty_cache()
    for it in range(times):
        assert margins[it].min() > 1e-3, (it, margins[it].min())
        assert np.array_equal(np.sort(lists[it], 1), np.sort(olists[it], 1)), it
    ref = np.concatenate([oq, og])
    err = np.abs(x.cpu().numpy() - ref).max(1) / np.linalg.norm(ref, axis=1)
    assert err.max() < 1e-5, err.max()


def run_shards(qf, gf, bounds, k, times, alpha):
    """every shard of query_expansion_sharded in sequence, the all-gather written as a concatenation"""
    ops = sharded.CudaOps()
    nq = len(qf)
    gfs = [gf[lo:hi] for lo, hi in bounds]
    for _ in range(times):
        x = torch.cat([qf] + gfs)
        outs = []
        for lo, hi in bounds:
            idx, d = ops.qe_lists(x, [(0, nq), (nq + lo, nq + hi)], k)
            outs.append(ops.qe_mix(idx, d, x, alpha))
        for o in outs[1:]:
            assert torch.equal(o[:nq].view(torch.int32), outs[0][:nq].view(torch.int32))
        qf, gfs = outs[0][:nq], [o[nq:] for o in outs]
    return qf, torch.cat(gfs)


@pytest.mark.parametrize('shape,world,layout', [((1980, 9330, 2048), 2, 'even'), ((1980, 9330, 2048), 3, 'empty'),
                                                ((1980, 9330, 2048), 8, 'even'), ((3000, 37000, 256), 3, 'empty')])
def test_sharded_in_sequence_equals_one_device(shape, world, layout):
    nq, ng, dim = shape
    torch.manual_seed(world)
    qf, gf = torch.randn(nq, dim, device='cuda'), torch.randn(ng, dim, device='cuda')
    bounds = sharded.shard_bounds(ng, world)
    if layout == 'empty':
        bounds = [(0, 0)] + sharded.shard_bounds(ng, world - 1)
    q, g = metrics.query_expansion(qf, gf, 5, 2, 3.0)
    sq, sg = run_shards(qf, gf, bounds, 5, 2, 3.0)
    assert np.array_equal(bits(sq), bits(q)) and np.array_equal(bits(sg), bits(g))
    q1, g1 = sharded.query_expansion_sharded(qf, gf, 5, 2, 3.0)                 # no process group: one shard
    assert np.array_equal(bits(q1), bits(q)) and np.array_equal(bits(g1), bits(g))


def _nccl_worker(rank, world, port, qf, gf, out_dir):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dist.init_process_group('nccl', rank=rank, world_size=world)
    try:
        lo, hi = sharded.shard_bounds(len(gf), world)[rank]
        q, g = sharded.query_expansion_sharded(qf.cuda(), gf[lo:hi].cuda(), 5, 2, 3.0)
        np.savez(os.path.join(out_dir, 'r%d.npz' % rank), q=q.cpu().numpy(), g=g.cpu().numpy())
    finally:
        dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason='needs 2 GPUs')
def test_sharded_nccl(tmp_path):
    import torch.multiprocessing as mp
    world = torch.cuda.device_count()
    torch.manual_seed(3)
    qf, gf = torch.randn(500, 1024), torch.randn(4000, 1024)
    s = socket.socket()
    s.bind(('127.0.0.1', 0))
    port = s.getsockname()[1]
    s.close()
    mp.spawn(_nccl_worker, args=(world, port, qf, gf, str(tmp_path)), nprocs=world, join=True)
    q, g = metrics.query_expansion(qf.cuda(), gf.cuda(), 5, 2, 3.0)
    for r, (lo, hi) in enumerate(sharded.shard_bounds(len(gf), world)):
        z = np.load(os.path.join(str(tmp_path), 'r%d.npz' % r))
        assert np.array_equal(z['q'].view(np.int32), bits(q)) and np.array_equal(z['g'].view(np.int32), bits(g)[lo:hi])


@pytest.mark.parametrize('re_rank,ranked', [(False, None), (True, None), (False, 7), (True, 7)])
def test_engine_aqe_equals_the_steps_by_hand(re_rank, ranked):
    from agrl.pytorch_b200 import engine
    from agrl.pytorch_b200.utils.re_ranking import re_ranking_dev
    from test_gpu_engine import make_loaders, make_model
    model = make_model()
    ql, gl, (qp, qc, gp, gc) = make_loaders()
    kw = dict(re_rank=re_rank, max_rank=20, verbose=False, aqe=True, qe_k=4, qe_times=2, qe_alpha=2.0)
    res = engine.test(model, ql, gl, 'avg', True, return_ranked=ranked, **kw)
    dm = engine.test(model, ql, gl, 'avg', True, return_distmat=True, **kw)
    with torch.no_grad():
        qf = engine.extract_features(model, ql)[0]
        gf = engine.extract_features(model, gl)[0]
        assert torch.equal(engine.extract_features(model, gl)[0].view(torch.int32), gf.view(torch.int32))
    qf, gf = metrics.query_expansion(qf, gf, 4, 2, 2.0)
    cdm = metrics.compute_distance_matrix
    d = cdm(qf, gf)
    if re_rank:
        d = re_ranking_dev(d, cdm(qf, qf), cdm(gf, gf))
    cmc, mAP = metrics.evaluate_rank(d, qp, gp, qc, gc, max_rank=20, use_metric_mars=True)
    assert np.array_equal(dm.view(np.int32), bits(d))
    assert res[0] == cmc[0] and res[1] == mAP
    if ranked:
        i, v = metrics.rank_lists(d, ranked)
        assert torch.equal(res[2], i) and np.array_equal(bits(res[3]), bits(v))
    else:
        assert len(res) == 2
    r_args = engine.test(model, ql, gl, 'avg', True, max_rank=20, verbose=False,
                         args=type('A', (), dict(re_rank=re_rank, aqe=True, qe_k=4, qe_times=2, qe_alpha=2.0))())
    assert r_args[:2] == tuple(res[:2])
