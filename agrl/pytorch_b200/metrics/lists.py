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
from .rank import _dev_labels


def _lists(ops, keys_of, nq, ng, dev, k, labels, exclude_junk):
    """The (indices, distances) lists of k from the keys ``keys_of(depth)`` of a non-empty gallery of ng rows."""
    from .. import sharded
    labels = None if labels[0] is None else [_dev_labels(x, dev) for x in labels]
    with torch.cuda.device(dev):
        depth = sharded.list_depth(k, ops, labels, exclude_junk)
        keys = keys_of(depth) if ng else torch.full((nq, depth), -1, dtype=torch.int64, device=dev)
        return ops.lists(keys.unsqueeze(0), int(k), *(labels or [None] * 4), exclude_junk=exclude_junk)


def rank_lists(distmat, k, q_pids=None, g_pids=None, q_camids=None, g_camids=None, exclude_junk=False):
    """(indices, distances): (num_q, k) int64 and fp32 CUDA tensors, the first k items of every row of ``distmat``.

    ``distmat`` is a (num_q, num_g) fp32 CUDA tensor (any row stride) or a numpy array, which is copied to the current
    device.  Raises ValueError when k plus the junk depth (the most items of one query's pid and camera) exceeds 8192."""
    from ..sharded import CudaOps
    ops = CudaOps()
    if not isinstance(distmat, torch.Tensor):
        distmat = torch.from_numpy(np.ascontiguousarray(distmat, dtype=np.float32)).cuda()
    assert distmat.dim() == 2 and distmat.dtype == torch.float32 and distmat.is_cuda
    if distmat.stride(1) != 1:
        distmat = distmat.contiguous()
    return _lists(ops, lambda depth: ops.keys(distmat, depth, 0), distmat.shape[0], distmat.shape[1], distmat.device, k,
                  (q_pids, g_pids, q_camids, g_camids), exclude_junk)


def retrieve(qf, gallery, k, metric='euclidean', q_pids=None, g_pids=None, q_camids=None, g_camids=None,
             exclude_junk=False, split=_lib.SPLIT_FP16X2, fused=None):
    """``rank_lists(compute_distance_matrix(qf, gallery, metric), k, ...)`` without the matrix.

    ``gallery`` is a (num_g, dim) CUDA feature tensor or a PreparedOperand (split once, reused for every query batch;
    its metric and split then apply).  Lists of k + J <= 256 keys come from the distance -> top-k fused into the GEMM
    epilogue, from sharded.FUSED_MIN_GALLERY gallery rows on (``fused`` overrides); deeper lists, smaller galleries and
    queries whose candidate list overflows the fused route go through distance blocks.  The lists are the same either
    way."""
    from .. import sharded
    ops = sharded.CudaOps()
    gop = gallery if isinstance(gallery, PreparedOperand) else PreparedOperand(gallery, metric, split)
    qop = PreparedOperand(qf.to(gop.device), gop.metric, gop.split)

    def keys_of(depth):
        use = sharded.fused_default(gop.rows, depth) if fused is None else fused and depth <= sharded.FUSED_MAX_DEPTH
        return ops.topk_keys(qop, gop, depth, 0, fused=use)
    return _lists(ops, keys_of, qop.rows, gop.rows, gop.device, k, (q_pids, g_pids, q_camids, g_camids), exclude_junk)
