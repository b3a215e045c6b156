"""Mirror of torchreid/metrics/rank.py for the hot path: ``evaluate_rank`` with the reference's
signature (rank.py:215-216), dispatch (:232-238) and return types, computed on the GPU.

    use_metric_market1501 -> rank_cylib.rank_cy.evaluate_cy (fp32 semantics of the Cython evaluator)
    use_metric_mars       -> MARS metric of evaluate_mars / Compute_AP (rank.py:160-212), float64
    neither flag          -> None, like the reference (the function falls off its end)
    use_metric_cuhk03     -> NotImplementedError (random-sampling metric, out of scope)

``use_cython=False`` selects the reference's float64 numpy evaluator (rank.py:95-150); here it only changes the
RETURN TYPE of mAP to numpy.float64 as that function has -- the native evaluator is the only implementation
(there is no Python fallback to select), so the value is rank_cy's fp32-accumulated one (equal to ~1e-9).

Beyond the reference: ``distmat`` may also be a CUDA torch tensor, in which case nothing is copied
through the host (labels may then be numpy arrays or CUDA int64 tensors).
"""
import ctypes

import numpy as np

from .. import _lib
from .rank_cylib.rank_cy import evaluate_cy, _as, _is_cuda_tensor

IS_CYTHON_AVAI = True     # rank.py:11-19: the native evaluator is always present here


def evaluate_mars(distmat, q_pids, g_pids, q_camids, g_camids, max_rank, return_all_ap=False):
    """(numpy.float64[max_rank], numpy.float64) -- rank.py:160-177."""
    if _is_cuda_tensor(distmat):
        return _mars_device(distmat, q_pids, g_pids, q_camids, g_camids, max_rank, return_all_ap)
    lib = _lib.require_device()
    d = _as(distmat, np.float32)
    qp, gp = _as(q_pids, np.int64), _as(g_pids, np.int64)
    qc, gc = _as(q_camids, np.int64), _as(g_camids, np.int64)
    num_q, num_g = d.shape
    max_rank = int(max_rank)
    if num_g < max_rank:
        # rank.py:174 assigns a length-num_g row into a length-max_rank slot
        raise ValueError('could not broadcast input array from shape ({},) into shape ({},)'.format(num_g, max_rank))
    cmc = np.zeros(max_rank, np.float64)
    mAP = ctypes.c_double(0.0)
    all_ap = np.zeros(num_q, np.float64) if return_all_ap else None
    rc = lib.agrl_rank_mars_host(d.ctypes.data, qp.ctypes.data, gp.ctypes.data, qc.ctypes.data, gc.ctypes.data,
                                 num_q, num_g, max_rank, cmc.ctypes.data, ctypes.addressof(mAP),
                                 all_ap.ctypes.data if return_all_ap else None)
    _lib.check(rc)
    out = (cmc, np.float64(mAP.value))
    return out + (all_ap,) if return_all_ap else out


def evaluate_rank(distmat, q_pids, g_pids, q_camids, g_camids, max_rank=50, use_metric_cuhk03=False,
                  use_metric_market1501=False, use_metric_mars=False, use_cython=True):
    """Evaluate CMC and mAP (signature of rank.py:215-216)."""
    if use_metric_market1501 or use_metric_cuhk03:
        res = evaluate_cy(distmat, q_pids, g_pids, q_camids, g_camids, max_rank, use_metric_cuhk03)
        if not use_cython:
            # rank.py:236 -> eval_market1501 (:95-150) returns (np.float32[max_rank], np.float64); the VALUE here is still the
            # native evaluator's fp32-accumulated mAP (the float64 numpy path agrees with it to ~1e-9, SURVEY App. A)
            return res[0], np.float64(res[1])
        return res
    elif use_metric_mars:
        return evaluate_mars(distmat, q_pids, g_pids, q_camids, g_camids, max_rank)


# ------------------------------------------------------------------------------------------------
# device-resident inputs (no host round trip)
# ------------------------------------------------------------------------------------------------
def _dev_labels(x, device):
    import torch
    if isinstance(x, torch.Tensor):
        return x.to(device=device, dtype=torch.int64).contiguous()
    return torch.as_tensor(np.ascontiguousarray(np.asarray(x), dtype=np.int64)).to(device)


def _market1501_device(distmat, q_pids, g_pids, q_camids, g_camids, max_rank, return_all_ap=False):
    import torch
    lib = _lib.require_device()
    assert distmat.dim() == 2 and distmat.dtype == torch.float32
    dev = distmat.device
    num_q, num_g = distmat.shape
    max_rank = int(max_rank)
    if num_g < max_rank:
        print('Note: number of gallery samples is quite small, got {}'.format(num_g))
    if distmat.stride(1) != 1:
        distmat = distmat.contiguous()
    qp, gp, qc, gc = (_dev_labels(x, dev) for x in (q_pids, g_pids, q_camids, g_camids))
    rank_len = min(max_rank, num_g)
    cmc = torch.empty(rank_len, dtype=torch.float32, device=dev)
    scal = torch.zeros(4, dtype=torch.float32, device=dev)              # [mAP, status(u32), num_valid(i64)]
    all_ap = torch.empty(max(num_q, 1), dtype=torch.float32, device=dev)
    wsb = lib.agrl_rank_workspace_bytes(num_q, num_g, max_rank)
    ws = torch.empty(wsb, dtype=torch.uint8, device=dev)
    _lib.call(dev, lib.agrl_rank_market1501_dev,
              distmat.data_ptr(), distmat.stride(0), qp.data_ptr(), gp.data_ptr(), qc.data_ptr(), gc.data_ptr(),
              num_q, num_g, max_rank, cmc.data_ptr(), scal.data_ptr(), all_ap.data_ptr(),
              scal.data_ptr() + 8, scal.data_ptr() + 4, ws.data_ptr(), wsb)
    host = scal.cpu()                                                    # synchronises the stream
    status = int(host.view(torch.int32)[1])
    _raise_status(status)
    out = (cmc.cpu().numpy(), float(host[0]))
    if return_all_ap:
        return out + (all_ap[:num_q].cpu().numpy(), int(host.view(torch.int64)[1]))
    return out


def _mars_device(distmat, q_pids, g_pids, q_camids, g_camids, max_rank, return_all_ap=False):
    import torch
    lib = _lib.require_device()
    assert distmat.dim() == 2 and distmat.dtype == torch.float32
    dev = distmat.device
    num_q, num_g = distmat.shape
    max_rank = int(max_rank)
    if num_g < max_rank:
        raise ValueError('could not broadcast input array from shape ({},) into shape ({},)'.format(num_g, max_rank))
    if distmat.stride(1) != 1:
        distmat = distmat.contiguous()
    qp, gp, qc, gc = (_dev_labels(x, dev) for x in (q_pids, g_pids, q_camids, g_camids))
    out = torch.zeros(max_rank + 2, dtype=torch.float64, device=dev)       # [cmc.., mAP, status]
    all_ap = torch.empty(num_q, dtype=torch.float64, device=dev)
    wsb = lib.agrl_rank_workspace_bytes(num_q, num_g, max_rank)
    ws = torch.empty(wsb, dtype=torch.uint8, device=dev)
    _lib.call(dev, lib.agrl_rank_mars_dev,
              distmat.data_ptr(), distmat.stride(0), qp.data_ptr(), gp.data_ptr(), qc.data_ptr(), gc.data_ptr(),
              num_q, num_g, max_rank, out.data_ptr(), out.data_ptr() + 8 * max_rank, all_ap.data_ptr(),
              out.data_ptr() + 8 * (max_rank + 1), ws.data_ptr(), wsb)
    host = out.cpu()
    _raise_status(int(host.view(torch.int32)[2 * (max_rank + 1)]))
    res = (host[:max_rank].numpy().copy(), np.float64(host[max_rank]))
    return res + (all_ap.cpu().numpy(),) if return_all_ap else res


def _raise_status(status):
    if status & _lib.ST_LABEL_RANGE:
        _lib.check(_lib.E_LABEL_RANGE)
    if status & _lib.ST_NO_VALID_QUERY:
        _lib.check(_lib.E_NO_VALID_QUERY)
    if status & _lib.ST_ZERO_DIVISION:
        _lib.check(_lib.E_ZERO_DIVISION)
