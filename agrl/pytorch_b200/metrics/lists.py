"""Ranked lists: each query's first ``k`` gallery items with their distances, on the GPU.

Row i of the result is ``np.argsort(d[i], kind='stable')[:k]`` -- ascending distance, ties by the lower gallery index,
NaN last, -0 == +0 -- the order every evaluator of this package ranks in (include/agrl_b200.h, section 3).  The
distances are the ranked values decoded from the ranking keys, not recomputed: -0 comes back as +0 and every NaN as the
NaN 0x7FFFFFFF.  Where fewer than k items qualify the tail holds index -1 and distance +inf.

    rank_lists(distmat, k)            from a distance matrix (CUDA tensor with any row stride, or numpy)
    retrieve(qf, gallery, k)          from features, the matrix never written for large galleries
    sharded.rank_lists_sharded(...)   the gallery split over the GPUs of a process group

``exclude_junk=True`` (needs the four label vectors) drops the gallery items that share the query's pid and camera, the
junk of rank_cy.pyx:197 and rank.py:166-169; pid -1 distractors stay, they are results a viewer wants to see.
"""
import numpy as np
import torch

from .. import _lib
from .distance import PreparedOperand

_ops = None


def _cuda_ops():
    global _ops
    if _ops is None:
        from ..sharded import CudaOps
        _ops = CudaOps()
    return _ops


def _labels(q_pids, g_pids, q_camids, g_camids, dev):
    if q_pids is None:
        return None
    from ..sharded import _as_dev_i64
    return [_as_dev_i64(x, dev) for x in (q_pids, g_pids, q_camids, g_camids)]


def rank_lists(distmat, k, q_pids=None, g_pids=None, q_camids=None, g_camids=None, exclude_junk=False):
    """(indices, distances): (num_q, k) int64 and fp32 CUDA tensors, the first k items of every row of ``distmat``.

    ``distmat`` is a (num_q, num_g) fp32 CUDA tensor (any row stride) or a numpy array, which is copied to the current
    device.  Raises ValueError when k plus the junk depth (the most items of one query's pid and camera) exceeds 8192."""
    from .. import sharded
    ops = _cuda_ops()
    if not isinstance(distmat, torch.Tensor):
        distmat = torch.from_numpy(np.ascontiguousarray(distmat, dtype=np.float32)).cuda()
    assert distmat.dim() == 2 and distmat.dtype == torch.float32 and distmat.is_cuda
    if distmat.stride(1) != 1:
        distmat = distmat.contiguous()
    dev = distmat.device
    nq, ng = distmat.shape
    labels = _labels(q_pids, g_pids, q_camids, g_camids, dev)
    with torch.cuda.device(dev):
        depth = sharded.list_depth(k, ops, labels, exclude_junk)
        if ng == 0:
            keys = torch.full((nq, depth), -1, dtype=torch.int64, device=dev)
        else:
            keys = ops.keys(distmat, depth, 0)
        return ops.lists(keys.unsqueeze(0), int(k), *(labels or [None] * 4), exclude_junk=exclude_junk)


def retrieve(qf, gallery, k, metric='euclidean', q_pids=None, g_pids=None, q_camids=None, g_camids=None,
             exclude_junk=False, split=_lib.SPLIT_FP16X2, fused=None):
    """``rank_lists(compute_distance_matrix(qf, gallery, metric), k, ...)`` without the matrix.

    ``gallery`` is a (num_g, dim) CUDA feature tensor or a PreparedOperand (split once, reused for every query batch;
    its metric and split then apply).  Lists of k + J <= 256 keys come from the distance -> top-k fused into the GEMM
    epilogue, from sharded.FUSED_MIN_GALLERY gallery rows on (``fused`` overrides); deeper lists, smaller galleries and
    queries whose candidate list overflows the fused route go through distance blocks.  The lists are the same either
    way."""
    from .. import sharded
    ops = _cuda_ops()
    gop = gallery if isinstance(gallery, PreparedOperand) else PreparedOperand(gallery, metric, split)
    dev = gop.device
    qop = PreparedOperand(qf.to(dev), gop.metric, gop.split)
    labels = _labels(q_pids, g_pids, q_camids, g_camids, dev)
    with torch.cuda.device(dev):
        depth = sharded.list_depth(k, ops, labels, exclude_junk)
        if fused is None:
            fused = gop.rows >= sharded.FUSED_MIN_GALLERY
        if gop.rows == 0:
            keys = torch.full((qop.rows, depth), -1, dtype=torch.int64, device=dev)
        else:
            keys = ops.topk_keys(qop, gop, depth, 0, fused=fused and depth <= sharded.FUSED_MAX_DEPTH)
        return ops.lists(keys.unsqueeze(0), int(k), *(labels or [None] * 4), exclude_junk=exclude_junk)
