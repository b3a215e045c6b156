"""Gallery-sharded k-reciprocal re-ranking on the GPU (agrl_rerank_shard_*, sharded.re_ranking_sharded).

The shards of one process run in sequence; the two exchanges are written out as concatenations (the query rows once,
then every shard's gallery rows in order), the way test_sharded_partial_and_merge_kernels treats the MARS merge.  The
bar is bit identity with re_ranking_dev on the whole problem, compared as int32 so that NaNs compare too.  It rests
on the premise, checked first, that a distance block computed on a slice of the operands equals the slice of the
whole matrix bit for bit."""
import os
import socket

import numpy as np
import pytest
import torch

from agrl.pytorch_b200 import _lib, metrics, sharded
from agrl.pytorch_b200.utils.re_ranking import re_ranking_dev
from oracle import synth

pytestmark = pytest.mark.gpu

MARS = (1980, 9330, 4096)


def features(nq, ng, d, seed, clustered=True):
    qp, qc, gp, gc = synth.eval_labels((nq, ng, max(4, min(625, nq // 3)), 6), seed=seed)
    qf, gf = synth.eval_features(qp, gp, d, seed=seed + 1, clustered=clustered)
    return (qp, qc, gp, gc), qf.cuda(), gf.cuda()


def single_device(qf, gf, metric='euclidean', k1=20, k2=6, lam=0.3):
    cdm = metrics.compute_distance_matrix
    return re_ranking_dev(cdm(qf, gf, metric), cdm(qf, qf, metric), cdm(gf, gf, metric), k1=k1, k2=k2, lambda_value=lam)


def run_shards(qf, gf, bounds, metric='euclidean', k1=20, k2=6, lam=0.3, slab_cols=None):
    """every shard's phases A, B, C in sequence, with the exchanges as concatenations; returns the blocks side by side"""
    ops = sharded.CudaOps()
    outs, _, _ = run_phases(lambda: (ops.distance(qf, gf, metric), ops.distance(qf, qf, metric)),
                            lambda c0, c1: ops.distance(gf, gf[c0:c1], metric), bounds, k1, k2, [lam], slab_cols,
                            ops)
    return outs[0]


def run_phases(q_dists, gg_cols, bounds, k1=20, k2=6, lams=(0.3,), slab_cols=None, ops=None):
    """phases A, B, C of every shard on the block matrix [[qq, qg], [qg^T, gg]]: q_dists() gives (qg, qq) and
    gg_cols(c0, c1) gives gg[:, c0:c1].  The references to qg and qq taken here are dropped after phase A, so the two
    matrices are freed then unless the caller keeps its own (run_shards keeps none).  Returns ([the blocks side by
    side, one matrix per lambda of ``lams``, all from the same phase A / B state], the exchanged rank table (N, K),
    the exchanged k-reciprocal rows [idx (N, cap), val (N, cap), cnt (N)])."""
    ops = ops or sharded.CudaOps()
    qg, qq = q_dists()
    nq, ng = qg.shape
    counts = [hi - lo for lo, hi in bounds]
    width = slab_cols or max(1, sharded.RERANK_SLAB_BYTES // (4 * ng))
    states, ranks = [], []
    for lo, hi in bounds:
        slabs = ((s0, gg_cols(lo + s0, min(hi, lo + s0 + width))) for s0 in range(0, hi - lo, width))
        st, rr = ops.rerank_rows(qg, qq, slabs, lo, hi - lo, max(counts), k1, k2)
        states.append(st)
        ranks.append(rr)
    del qq, qg
    for rr in ranks[1:]:
        assert torch.equal(rr[:nq], ranks[0][:nq])                 # query rows are the same on every shard
    rank_all = torch.cat([ranks[0][:nq]] + [rr[nq:] for rr in ranks])
    del ranks
    vs = [ops.rerank_expand(st, rank_all) for st in states]
    v_all = [torch.cat([vs[0][k][:nq]] + [v[k][nq:] for v in vs]) for k in range(3)]
    del vs
    outs = []
    for lam in lams:
        blocks = [ops.rerank_finish(st, rank_all, v_all[0], v_all[1], v_all[2], lam) for st in states]
        for blk, (lo, hi) in zip(blocks, bounds):
            assert tuple(blk.shape) == (nq, hi - lo)
        outs.append(torch.cat(blocks, dim=1))
        del blocks
    del states
    return outs, rank_all, v_all


def bits_equal(a, b):
    return a.shape == b.shape and torch.equal(a.contiguous().view(torch.int32), b.contiguous().view(torch.int32))


# ---- the premise -------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('metric', ['euclidean', 'cosine'])
@pytest.mark.parametrize('split', [_lib.SPLIT_FP16X2, _lib.SPLIT_BF16X3])
def test_distance_blocks_are_slices_of_the_whole_matrix(metric, split):
    _, qf, gf = features(*MARS, seed=11)
    cdm = metrics.compute_distance_matrix
    whole = cdm(gf, gf, metric, split=split)
    for lo, hi in sharded.shard_bounds(MARS[1], 8)[2:4] + [(3001, 3008), (9329, 9330)]:
        assert bits_equal(cdm(gf, gf[lo:hi], metric, split=split), whole[:, lo:hi]), (lo, hi)
        assert bits_equal(cdm(gf[lo:hi], gf, metric, split=split), whole[lo:hi]), (lo, hi)
    qg = cdm(qf, gf, metric, split=split)
    lo, hi = sharded.shard_bounds(MARS[1], 3)[1]
    assert bits_equal(cdm(qf, gf[lo:hi], metric, split=split), qg[:, lo:hi])
    assert bits_equal(cdm(qf[100:1000], gf, metric, split=split), qg[100:1000])


# ---- bit identity with the single-device path --------------------------------------------------------------------------
@pytest.fixture(scope='module')
def mars_case():
    return features(*MARS, seed=3)


@pytest.mark.parametrize('metric', ['euclidean', 'cosine'])
def test_mars_shape_bit_identical(mars_case, metric):
    _, qf, gf = mars_case
    want = single_device(qf, gf, metric)
    for world in (2, 3, 8):
        got = run_shards(qf, gf, sharded.shard_bounds(MARS[1], world), metric,
                         slab_cols=777 if world == 2 else None)        # several column slabs per shard
        assert bits_equal(got, want), (metric, world)


@pytest.mark.parametrize('k1', [1, 20, 30])
@pytest.mark.parametrize('k2', [1, 6])
def test_k1_k2_bit_identical(k1, k2):
    _, qf, gf = features(300, 2000, 256, seed=k1 + k2)
    want = single_device(qf, gf, k1=k1, k2=k2, lam=0.25)
    got = run_shards(qf, gf, sharded.shard_bounds(2000, 3), k1=k1, k2=k2, lam=0.25, slab_cols=301)
    assert bits_equal(got, want), (k1, k2)


@pytest.mark.parametrize('metric', ['euclidean', 'cosine'])
def test_tie_heavy_bit_identical(metric):
    _, qf, gf = features(200, 1500, 64, seed=21)
    gf[1::2] = gf[0:-1:2][:len(gf[1::2])]                              # duplicated gallery rows across shard boundaries
    gf[-200:] = qf                                                     # queries copied into the gallery
    gf[700:720] = gf[700]
    want = single_device(qf, gf, metric)
    for world in (2, 3):
        assert bits_equal(run_shards(qf, gf, sharded.shard_bounds(1500, world), metric), want), (metric, world)


def test_tiny_problem_bit_identical():
    _, qf, gf = features(3, 10, 16, seed=4)                            # N = 13 < k1 + 1
    want = single_device(qf, gf)
    for bounds in (sharded.shard_bounds(10, 2), [(0, 1), (1, 9), (9, 10)]):
        assert bits_equal(run_shards(qf, gf, bounds), want), bounds


def test_empty_shard_bit_identical():
    _, qf, gf = features(120, 1000, 128, seed=5)
    want = single_device(qf, gf, k2=3)
    got = run_shards(qf, gf, [(0, 0), (0, 500), (500, 500), (500, 1000)], k2=3)
    assert bits_equal(got, want)
    got = run_shards(qf, gf, [(0, 1000), (1000, 1000)], k2=1)
    assert bits_equal(got, single_device(qf, gf, k2=1))


def test_near_the_single_device_ceiling_bit_identical():
    _, qf, gf = features(4000, 40000, 2048, seed=6)
    want = single_device(qf, gf)
    got = run_shards(qf, gf, sharded.shard_bounds(40000, 4))
    assert bits_equal(got, want)


def test_beyond_one_device_4_and_8_shards_agree():
    """2000 x 160000: N = 162000 is past the single-device limit (46000); a shard's D rows exceed 2^31 elements"""
    lib = _lib.load()
    assert lib.agrl_rerank_workspace_bytes(2000, 160000, 20, 6) == 0
    _, qf, gf = features(2000, 160000, 2048, seed=7)
    got4 = run_shards(qf, gf, sharded.shard_bounds(160000, 4)).cpu()
    torch.cuda.empty_cache()
    got8 = run_shards(qf, gf, sharded.shard_bounds(160000, 8)).cpu()
    torch.cuda.empty_cache()
    assert got4.shape == (2000, 160000)
    assert bool(torch.isfinite(got4).all()) and float(got4.min()) >= 0.0
    assert bits_equal(got4, got8)


# ---- public entry points -----------------------------------------------------------------------------------------------
def test_evaluate_mars_sharded_re_rank_world_1(mars_case):
    (qp, qc, gp, gc), qf, gf = mars_case
    want = single_device(qf, gf)
    block = sharded.re_ranking_sharded(qf, gf)
    assert bits_equal(block, want)
    cmc, mAP = sharded.evaluate_mars_sharded(qf, gf, qp, gp, qc, gc, re_rank=True)
    rcmc, rmAP = metrics.evaluate_rank(want, qp, gp, qc, gc, use_metric_mars=True)
    assert np.array_equal(cmc, rcmc) and float(mAP) == float(rmAP)


def test_limits_and_errors():
    _, qf, gf = features(20, 300, 32, seed=8)
    with pytest.raises(_lib.AgrlError):
        sharded.re_ranking_sharded(qf, gf, k1=64)
    with pytest.raises(_lib.AgrlError):
        sharded.re_ranking_sharded(qf, gf, k2=9)
    with pytest.raises(ValueError):
        sharded.re_ranking_sharded(qf, gf, metric='hamming')
    big = torch.randn(50001, 32, device='cuda')
    with pytest.raises(_lib.AgrlError):                                # n_r > 50000: one rank's t_min no longer fits
        sharded.re_ranking_sharded(qf, big)
    lib = _lib.load()
    assert lib.agrl_rerank_shard_workspace_bytes(20, 50001, 50001, 20, 6) == 0
    assert lib.agrl_rerank_shard_workspace_bytes(20, 100000, 50000, 20, 6) > 0
    ws = torch.empty(16, dtype=torch.uint8, device='cuda')
    rank = torch.empty(20, 21, dtype=torch.int32, device='cuda')
    qq = torch.zeros(20, 20, device='cuda')
    qg = torch.zeros(20, 300, device='cuda')
    assert lib.agrl_rerank_shard_rows_dev(qg.data_ptr(), 300, qq.data_ptr(), 20, None, 0, 20, 300, 0, 0, 0, 20, 20, 6,
                                          rank.data_ptr(), ws.data_ptr(), 16, None) == _lib.E_WORKSPACE
    assert lib.agrl_rerank_shard_rows_dev(qg.data_ptr(), 300, qq.data_ptr(), 20, None, 0, 20, 300, 0, 10, 0, 25, 20, 6,
                                          rank.data_ptr(), ws.data_ptr(), 16, None) == _lib.E_INVALID   # no g_cols
    assert lib.agrl_rerank_shard_rows_dev(qg.data_ptr(), 300, qq.data_ptr(), 20, None, 0, 20, 300, 295, 10, 0, 20, 20, 6,
                                          rank.data_ptr(), ws.data_ptr(), 16, None) == _lib.E_INVALID   # past the gallery


# ---- NCCL, one process per GPU --------------------------------------------------------------------------------------
def _free_port():
    s = socket.socket()
    s.bind(('127.0.0.1', 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _nccl_worker(rank, world, port, qf, gf, out_dir):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dist.init_process_group('nccl', rank=rank, world_size=world, device_id=torch.device('cuda', rank))
    try:
        lo, hi = sharded.shard_bounds(gf.shape[0], world)[rank]
        q = qf.cuda() if rank == 0 else torch.zeros_like(qf, device='cuda')
        block = sharded.re_ranking_sharded(q, gf[lo:hi].cuda())
        np.save(os.path.join(out_dir, 'b%d.npy' % rank), block.cpu().numpy())
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize('world', [2, 4])
def test_nccl_blocks_equal_single_device(tmp_path, world):
    if torch.cuda.device_count() < world:
        pytest.skip('needs %d GPUs' % world)
    import torch.multiprocessing as mp
    _, qf, gf = features(500, 4000, 512, seed=9)
    want = single_device(qf, gf).cpu().numpy()
    mp.spawn(_nccl_worker, args=(world, _free_port(), qf.cpu(), gf.cpu(), str(tmp_path)), nprocs=world, join=True)
    got = np.concatenate([np.load(os.path.join(str(tmp_path), 'b%d.npy' % r)) for r in range(world)], axis=1)
    assert np.array_equal(got.view(np.int32), want.view(np.int32))
