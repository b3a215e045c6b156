"""k-reciprocal re-ranking on the GPU -- mirror of ``torchreid/utils/re_ranking.py`` (reference :30-94), the optional
step of test() between the distance matrix and the ranking (train_vidreid_xent_htri.py:523-527).

Same signature and return type: three distance matrices in (numpy arrays or torch tensors, as test() mixes them),
one float32 numpy array (num_query, num_gallery) out.  Ties in the initial ranking are broken by index
(numpy.argsort(kind='stable')); the reference's default argsort leaves them undefined.
"""
import numpy as np
import torch

from .. import _lib

__all__ = ['re_ranking', 're_ranking_dev']


def _to_device(a, dev):
    t = torch.as_tensor(a)
    t = t.to(device=dev, dtype=torch.float32)
    return t if t.stride(-1) == 1 else t.contiguous()


def re_ranking_dev(q_g_dist, q_q_dist, g_g_dist, k1=20, k2=6, lambda_value=0.3):
    """Device-resident variant: CUDA tensors in, CUDA tensor (num_query, num_gallery) out, asynchronous."""
    lib = _lib.require_device()
    dev = next((t.device for t in (q_g_dist, q_q_dist, g_g_dist) if isinstance(t, torch.Tensor) and t.is_cuda),
               torch.device('cuda', torch.cuda.current_device()))
    qg, qq, gg = (_to_device(a, dev) for a in (q_g_dist, q_q_dist, g_g_dist))
    nq, ng = qg.shape
    assert tuple(qq.shape) == (nq, nq) and tuple(gg.shape) == (ng, ng), 'expected (nq, ng), (nq, nq), (ng, ng)'
    wsb = lib.agrl_rerank_workspace_bytes(nq, ng, int(k1), int(k2))
    if wsb == 0:
        _lib.check(_lib.E_UNSUPPORTED)
    out = torch.empty(nq, ng, dtype=torch.float32, device=dev)
    ws = torch.empty(wsb, dtype=torch.uint8, device=dev)
    _lib.call(dev, lib.agrl_rerank_dev, qg.data_ptr(), qg.stride(0), qq.data_ptr(), qq.stride(0), gg.data_ptr(), gg.stride(0),
              nq, ng, int(k1), int(k2), float(lambda_value), out.data_ptr(), out.stride(0), ws.data_ptr(), wsb)
    return out


def re_ranking(q_g_dist, q_q_dist, g_g_dist, k1=20, k2=6, lambda_value=0.3):
    """Drop-in for the reference's re_ranking(): returns a numpy float32 array (num_query, num_gallery)."""
    return re_ranking_dev(q_g_dist, q_q_dist, g_g_dist, k1, k2, lambda_value).cpu().numpy()
