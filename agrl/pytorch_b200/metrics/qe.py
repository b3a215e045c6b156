"""Alpha query expansion (FastReID fastreid/evaluation/query_expansion.py ``aqe``, TEST.AQE), on the GPU.

One iteration over the joint set X = [queries; gallery] replaces every row by the mean of its k nearest neighbours'
rows (itself included), each weighted by its cosine similarity to the power alpha:

    idx, d = rank_lists(compute_distance_matrix(X, X, 'cosine'), k)       # ties to the lower index
    X'[i] = sum_j powf(1 - d[i, j], alpha) * X[idx[i, j]] / k             # fp32, in list order

The expansion is transductive (queries and gallery are expanded together) and the similarity is always the cosine,
whatever metric ranks the expanded features afterwards.  The lists never write the N x N matrix: from
sharded.FUSED_MIN_GALLERY rows on they come from the distance -> top-k fused into the GEMM epilogue.
sharded.query_expansion_sharded is the same computation with the gallery split over the GPUs of a process group.
"""
import torch

from .. import _lib


def query_expansion(qf, gf, qe_k=5, qe_times=1, alpha=3.0, split=_lib.SPLIT_FP16X2, fused=None):
    """(qf', gf'): the query and gallery features after ``qe_times`` iterations of alpha query expansion over their
    ``qe_k`` nearest neighbours, as CUDA fp32 tensors (CPU inputs are moved to the current device).  FastReID's defaults:
    QE_TIME = 1, QE_K = 5, ALPHA = 3.0; ``alpha=0`` is plain mean query expansion.  ``split`` is the operand split of the
    cosine distances; ``fused`` overrides the choice of the fused distance -> top-k (the result is the same either way).

    Raises AssertionError for inputs that are not 2-D or differ in dim (as compute_distance_matrix), ValueError when
    qe_k < 1, qe_k > num_q + num_g, qe_k > sharded.MAX_LIST_DEPTH, qe_times < 1 or alpha is not finite."""
    from .. import sharded
    assert isinstance(qf, torch.Tensor) and isinstance(gf, torch.Tensor)
    assert qf.dim() == 2, 'Expected 2-D tensor, but got {}-D'.format(qf.dim())
    assert gf.dim() == 2, 'Expected 2-D tensor, but got {}-D'.format(gf.dim())
    assert qf.size(1) == gf.size(1)
    sharded.check_qe_args(qe_k, qe_times, alpha, qf.size(0) + gf.size(0))
    lib_ops = sharded.CudaOps(split)
    dev = qf.device if qf.is_cuda else torch.device('cuda', torch.cuda.current_device())
    x = torch.cat([qf.detach().to(device=dev, dtype=torch.float32), gf.detach().to(device=dev, dtype=torch.float32)])
    nq, n = qf.size(0), x.size(0)
    with torch.cuda.device(dev):
        for _ in range(qe_times):
            idx, d = lib_ops.qe_lists(x, [(0, n)], qe_k, fused)
            x = lib_ops.qe_mix(idx, d, x, alpha)
    return x[:nq], x[nq:]
