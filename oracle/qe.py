"""Alpha query expansion oracle -- TEST INFRASTRUCTURE ONLY (see oracle/__init__.py).

fp64 restatement of FastReID's ``aqe`` (fastreid/evaluation/query_expansion.py) with the tie order of this package.
One iteration over the joint set X = [queries; gallery] (N rows):
    s       = cosine similarity of the rows, x / max(||x||, 1e-12) as F.normalize
    idx[i]  = the first k of np.argsort(-s[i], kind='stable'): itself included, ties to the lower index
    X'[i]   = sum_j s[i, idx[i, j]] ** alpha * X[idx[i, j]] / k          (np.power: NaN for s < 0 and non-integer alpha)
repeated qe_times times.  Each iteration also reports every row's margin, s_k - s_(k+1) (its k-th and (k+1)-th
similarity; +inf when N == k): where it exceeds the error of an fp32 similarity, the list's members are decided.

Arithmetic is torch float64, on the CPU by default; ``device='cuda'`` runs the same fp64 products on a GPU for sets of
10^5 rows, where the CPU takes minutes per iteration.  The similarity rows are formed ``block`` at a time, so no
N x N matrix is held.
"""
import numpy as np
import torch


def _lists(n, k, device, block):
    """(idx (N, k) int64, sims (N, k) fp64, margins (N,) fp64) for the normalised rows n (fp64, on device)."""
    N = n.shape[0]
    kk = min(k + 1, N)
    idx = np.empty((N, k), np.int64)
    sims = np.empty((N, k), np.float64)
    margin = np.full(N, np.inf)
    for r0 in range(0, N, block):
        s = n[r0:r0 + block] @ n.t()
        top_v, top_i = torch.topk(s, kk, dim=1)
        s_cut = top_v[:, kk - 1:kk]
        count = (s >= s_cut).sum(dim=1).cpu().numpy()
        top_v, top_i = top_v.cpu().numpy(), top_i.cpu().numpy()
        for b in range(top_v.shape[0]):
            if count[b] == kk:                       # the candidates are exactly the first kk: order them stably
                o = np.lexsort((top_i[b], -top_v[b]))
                cols, vals = top_i[b][o], top_v[b][o]
            else:                                    # a tie at the (k+1)-th place: the whole row
                row = s[b].cpu().numpy()
                cols = np.argsort(-row, kind='stable')[:kk]
                vals = row[cols]
            idx[r0 + b], sims[r0 + b] = cols[:k], vals[:k]
            if kk > k:
                margin[r0 + b] = vals[k - 1] - vals[k]
    return idx, sims, margin


def aqe(qf, gf, qe_k=5, qe_times=1, alpha=3.0, device='cpu', block=2048):
    """(qf', gf', lists, sims, margins): the expanded features (fp64 numpy), and per iteration the ranked lists
    (N, qe_k), their similarities and the margins (N,)."""
    x = torch.cat([torch.as_tensor(qf), torch.as_tensor(gf)]).to(device=device, dtype=torch.float64)
    assert torch.isfinite(x).all(), 'the oracle ranks finite features only'
    nq = len(qf)
    lists, sims, margins = [], [], []
    for _ in range(qe_times):
        n = x / x.norm(dim=1, keepdim=True).clamp(min=1e-12)
        idx, s, m = _lists(n, qe_k, device, block)
        with np.errstate(invalid='ignore'):
            w = torch.from_numpy(np.power(s, alpha)).to(device)
        gi = torch.from_numpy(idx).to(device)
        x = sum(w[:, j:j + 1] * x[gi[:, j]] for j in range(qe_k)) / qe_k
        lists.append(idx)
        sims.append(s)
        margins.append(m)
    x = x.cpu().numpy()
    return x[:nq], x[nq:], lists, sims, margins


def grouped_features(nq, ng, dim, k, seed=0, spread=0.3):
    """(qf, gf) fp32: the N = nq + ng rows fall, in a random order, into groups of exactly k rows around a shared random
    direction (+ spread * noise), with row norms between 0.5 and 2.  Each row's k most similar rows are then its own
    group, separated from the rest by a wide margin that the expansion keeps (the caller asserts it).  N % k == 0."""
    N = nq + ng
    assert N % k == 0
    g = torch.Generator().manual_seed(seed)
    cent = torch.randn(N // k, dim, generator=g)
    group = torch.randperm(N, generator=g) // k
    x = cent[group] + spread * torch.randn(N, dim, generator=g)
    x = x / x.norm(dim=1, keepdim=True) * (0.5 + 1.5 * torch.rand(N, 1, generator=g))
    return x[:nq].contiguous(), x[nq:].contiguous()
