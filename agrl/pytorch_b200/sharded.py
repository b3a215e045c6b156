"""Gallery-sharded evaluation over the GPUs of one box (SURVEY.md section 8e).

The only part of AGRL's test-time path that needs communication: each rank owns a slice of the
gallery (its rows of the feature matrix are already there when the head ran sharded), computes its
block of the distance matrix and, per query, its best ``max_rank`` candidates + good-image count with
the kernels of libagrl_b200; one NCCL all-gather of the (key, class) lists and one all-reduce of the
counts later, every rank merges them into exactly the CMC/mAP the unsharded evaluator would return.
Messages are tiny (num_q x max_rank x 9 B per rank), so the merge is latency-bound and the flat
one-shot collectives of NVSwitch are the right shape.  The graph head needs no collective at all.

    cmc, mAP = evaluate_mars_sharded(qf, gf_local, q_pids, g_pids_local, q_camids, g_camids_local)

k-reciprocal re-ranking shards too (``re_ranking_sharded``, or ``re_rank=True`` above): every rank holds all
features after one all-gather, computes the D rows of its queries + gallery rows, and two all-gathers of sparse
tables (rank lists, k-reciprocal rows) later produces its (num_q x num_g_r) block of the re-ranked matrix.

``ops`` lets the tests drive the same plumbing with CPU stand-ins under gloo; the product default is
the CUDA implementation and there is no fallback.
"""
import math
from types import SimpleNamespace

import numpy as np
import torch
import torch.distributed as dist

from . import _lib
from .metrics.distance import PreparedOperand, _check_metric, _workspace, _METRICS, distance_prepared
from .metrics.rank import _dev_labels, _raise_status


def shard_bounds(n, world):
    """Contiguous, near-equal row ranges [(lo, hi)] of a length-n gallery for `world` ranks."""
    base, extra = divmod(n, world)
    out, lo = [], 0
    for r in range(world):
        hi = lo + base + (1 if r < extra else 0)
        out.append((lo, hi))
        lo = hi
    return out


def or_across_ranks(status, group=None):
    """Bitwise OR of every rank's status word (bit flags: LABEL_RANGE, ZERO_DIVISION, TOPK_OVERFLOW, ...), in place."""
    return status.copy_(_max_and_or(None, status, group)[1])


def _max_and_or(maxed, status, group):
    """(MAX over the ranks of the int32 tensor ``maxed``, bitwise OR over the ranks of the status words) in one
    all-reduce.  NCCL has no BOR reduction: each word is expanded into one 0/1 lane per bit, all-reduced with MAX and
    re-packed."""
    shifts = torch.arange(16, device=status.device, dtype=torch.int32)
    lanes = ((status.to(torch.int32).view(-1, 1) >> shifts) & 1).view(-1)
    n = 0 if maxed is None else maxed.numel()
    word = lanes if maxed is None else torch.cat([maxed.to(torch.int32).view(-1), lanes])
    dist.all_reduce(word, op=dist.ReduceOp.MAX, group=group)
    return word[:n], (word[n:].view(-1, 16) << shifts).sum(dim=1).to(status.dtype).view_as(status)


TOPK_BLOCK_BYTES = 1 << 31       # largest distance block (num_q rows x num_g fp32) of the unfused top-k routes


class CudaOps(object):
    """Per-rank compute on the rank's current CUDA device (libagrl_b200)."""

    def __init__(self, split=_lib.SPLIT_FP16X2):
        self.lib = _lib.require_device()
        self.split = split

    def distance(self, qf, gf, metric):
        from .metrics import compute_distance_matrix
        return compute_distance_matrix(qf, gf, metric, split=self.split)

    def partial(self, d, q_pids, g_pids, q_camids, g_camids, max_rank, offset):
        dev = d.device
        nq, ng = d.shape
        keys = torch.empty(nq, max_rank, dtype=torch.int64, device=dev)
        cls = torch.empty(nq, max_rank, dtype=torch.uint8, device=dev)
        ngood = torch.empty(nq, dtype=torch.int32, device=dev)
        status = torch.zeros(1, dtype=torch.int32, device=dev)
        wsb = self.lib.agrl_rank_workspace_bytes(nq, ng, max_rank)
        _lib.call(dev, self.lib.agrl_rank_mars_partial_dev,
                  d.data_ptr(), d.stride(0), q_pids.data_ptr(), g_pids.data_ptr(), q_camids.data_ptr(),
                  g_camids.data_ptr(), nq, ng, max_rank, offset, keys.data_ptr(), cls.data_ptr(), ngood.data_ptr(),
                  status.data_ptr(), _workspace(dev, wsb).data_ptr(), wsb)
        return keys, cls, ngood, status

    def _fused_keys(self, qop, gop, depth, offset):
        """(keys (num_q, depth) int64, status) of two PreparedOperand from the distance -> top-k fused into the GEMM
        epilogue (agrl_distance_topk_dev); the status has ST_TOPK_OVERFLOW when a query's candidate list overflowed."""
        assert (qop.metric, qop.split, qop.dim, qop.device) == (gop.metric, gop.split, gop.dim, gop.device)
        dev, nq = qop.device, qop.rows
        keys = torch.empty(nq, depth, dtype=torch.int64, device=dev)
        status = torch.zeros(1, dtype=torch.int32, device=dev)
        wsb = self.lib.agrl_distance_topk_workspace_bytes(nq)
        _lib.call(dev, self.lib.agrl_distance_topk_dev,
                  qop.buf.data_ptr(), nq, gop.buf.data_ptr(), gop.rows, qop.dim, _METRICS[qop.metric], qop.split, depth,
                  offset, keys.data_ptr(), status.data_ptr(), _workspace(dev, wsb).data_ptr(), wsb)
        return keys, status

    def topk_fused(self, qop, gop, q_pids, g_pids, q_camids, g_camids, max_rank, offset, allow_fallback=True):
        """Same outputs as ``partial`` from two PreparedOperand, with the distance -> top-k fused into the GEMM epilogue
        (agrl_distance_topk_dev + agrl_rank_mars_classify_dev): no (num_q x num_g) matrix is allocated.  When a query's
        candidate list overflows (a gallery ordered by distance to the query) the call falls back to distance blocks +
        ``partial`` -- the results are the same either way."""
        keys, status = self._fused_keys(qop, gop, max_rank, offset)
        dev, nq, ng = qop.device, qop.rows, gop.rows
        cls = torch.empty(nq, max_rank, dtype=torch.uint8, device=dev)
        ngood = torch.empty(nq, dtype=torch.int32, device=dev)
        wsb = self.lib.agrl_rank_mars_classify_workspace_bytes(nq, ng)
        _lib.call(dev, self.lib.agrl_rank_mars_classify_dev,
                  keys.data_ptr(), q_pids.data_ptr(), g_pids.data_ptr(), q_camids.data_ptr(), g_camids.data_ptr(),
                  nq, ng, max_rank, offset, cls.data_ptr(), ngood.data_ptr(), status.data_ptr(),
                  _workspace(dev, wsb).data_ptr(), wsb)
        if allow_fallback and int(status.cpu()) & _lib.ST_TOPK_OVERFLOW:
            return self.topk_unfused(qop, gop, q_pids, g_pids, q_camids, g_camids, max_rank, offset)
        return keys, cls, ngood, status

    def topk_unfused(self, qop, gop, q_pids, g_pids, q_camids, g_camids, max_rank, offset, block_bytes=TOPK_BLOCK_BYTES):
        """distance blocks (at most ``block_bytes`` each) written to HBM + the streaming top-k kernel"""
        dev, nq = qop.device, qop.rows
        keys = torch.empty(nq, max_rank, dtype=torch.int64, device=dev)
        cls = torch.empty(nq, max_rank, dtype=torch.uint8, device=dev)
        ngood = torch.empty(nq, dtype=torch.int32, device=dev)
        status = torch.zeros(1, dtype=torch.int32, device=dev)
        for q0, q1, dm in _distance_blocks(qop, gop, block_bytes):
            k, c, n, st = self.partial(dm, q_pids[q0:q1], g_pids, q_camids[q0:q1], g_camids, max_rank, offset)
            keys[q0:q1], cls[q0:q1], ngood[q0:q1] = k, c, n
            status |= st
        return keys, cls, ngood, status

    def merge(self, keys_all, cls_all, ngood, max_rank, status_parts):
        dev = keys_all.device
        parts, nq = keys_all.shape[0], keys_all.shape[1]
        out = torch.zeros(max_rank + 2, dtype=torch.float64, device=dev)      # [cmc.., mAP, status]
        wsb = self.lib.agrl_rank_workspace_bytes(nq, 0, max_rank)
        _lib.call(dev, self.lib.agrl_rank_mars_merge_dev,
                  keys_all.data_ptr(), cls_all.data_ptr(), ngood.data_ptr(), parts, nq, max_rank,
                  out.data_ptr(), out.data_ptr() + 8 * max_rank, None, out.data_ptr() + 8 * (max_rank + 1),
                  _workspace(dev, wsb).data_ptr(), wsb)
        host = out.cpu()
        _raise_status(int(host.view(torch.int32)[2 * (max_rank + 1)]) | int(status_parts.cpu()))
        return host[:max_rank].numpy().copy(), np.float64(host[max_rank])

    # ---- ranked lists (agrl_rank_lists_dev) ---------------------------------------------------------------------------
    def keys(self, d, depth, offset):
        """Each query's first ``depth`` keys of the distance block ``d`` (agrl_rank_mars_partial_dev)."""
        qp, lab = _unlabelled(d.shape[0], d.shape[1], d.device)
        return self.partial(d, qp, lab, qp, lab, depth, offset)[0]

    def topk_keys(self, qop, gop, depth, offset, fused=True):
        """``keys`` of the distance block of two PreparedOperand without materialising it: distance -> top-k fused into
        the GEMM epilogue (depth <= 256); when a query's candidate list overflows, or with ``fused=False``, distance blocks
        of at most TOPK_BLOCK_BYTES + ``keys``.  The keys are the same either way."""
        if fused:
            keys, status = self._fused_keys(qop, gop, depth, offset)
            if not int(status.cpu()) & _lib.ST_TOPK_OVERFLOW:
                return keys
        else:
            keys = torch.empty(qop.rows, depth, dtype=torch.int64, device=qop.device)
        for q0, q1, dm in _distance_blocks(qop, gop):
            keys[q0:q1] = self.keys(dm, depth, offset)
        return keys

    def junk_depth(self, q_pids, g_pids, q_camids, g_camids):
        """(J, status) as int32 tensors of one element: the most gallery items of this shard sharing a query's pid and
        camera, over the queries (agrl_rank_junk_depth_dev)."""
        dev = q_pids.device
        nq, ng = q_pids.numel(), g_pids.numel()
        out = torch.zeros(2, dtype=torch.int32, device=dev)                   # [J, status]
        wsb = self.lib.agrl_rank_mars_classify_workspace_bytes(nq, ng)
        _lib.call(dev, self.lib.agrl_rank_junk_depth_dev,
                  q_pids.data_ptr(), g_pids.data_ptr(), q_camids.data_ptr(), g_camids.data_ptr(), nq, ng, out.data_ptr(),
                  out.data_ptr() + 4, _workspace(dev, wsb).data_ptr(), wsb)
        return out[0:1], out[1:2]

    def lists(self, keys_all, k, q_pids=None, g_pids=None, q_camids=None, g_camids=None, exclude_junk=False):
        """(indices int64, distances fp32), (num_q, k) each, from the [part][query][depth] key lists (agrl_rank_lists_dev);
        with ``exclude_junk`` the gallery labels are indexed by global gallery index."""
        dev = keys_all.device
        keys_all = keys_all.contiguous()
        parts, nq, depth = keys_all.shape
        index = torch.empty(nq, k, dtype=torch.int64, device=dev)
        dist_ = torch.empty(nq, k, dtype=torch.float32, device=dev)
        status = torch.zeros(1, dtype=torch.int32, device=dev)
        ng = g_pids.numel() if exclude_junk else 0
        wsb = self.lib.agrl_rank_mars_classify_workspace_bytes(nq, ng) if exclude_junk else 0
        ws = _workspace(dev, max(wsb, 1))
        lab = [x.data_ptr() if exclude_junk else None for x in (q_pids, g_pids, q_camids, g_camids)]
        _lib.call(dev, self.lib.agrl_rank_lists_dev,
                  keys_all.data_ptr(), parts, nq, depth, k, lab[0], lab[1], lab[2], lab[3], ng, int(bool(exclude_junk)),
                  index.data_ptr(), dist_.data_ptr(), k, status.data_ptr(), ws.data_ptr(), wsb)
        _raise_status(int(status.cpu()))
        return index, dist_

    # ---- alpha query expansion (agrl_qe_mix_dev) ----------------------------------------------------------------------
    def qe_lists(self, x, ranges, k, fused=None):
        """(indices int64, cosine distances fp32), (rows, k) each: the ranked lists of the rows x[r0:r1] of every
        (r0, r1) in ``ranges``, in order, against all rows of x (each row's list includes itself).  x is split into
        cosine operand planes once; a range that is not the whole of x is a rows_view of those planes.  The distance ->
        top-k is fused into the GEMM epilogue as fused_default decides for the rows of x (``fused`` overrides); the
        lists are the same either way."""
        n, dev = x.shape[0], x.device
        if fused is None:
            fused = fused_default(n, k)
        op = PreparedOperand(x, 'cosine', self.split)
        keys = [self.topk_keys(op if (r0, r1) == (0, n) else op.rows_view(r0, r1), op, k, 0,
                               fused=fused and k <= FUSED_MAX_DEPTH) for r0, r1 in ranges if r1 > r0]
        if not keys:
            return torch.empty(0, k, dtype=torch.int64, device=dev), torch.empty(0, k, dtype=torch.float32, device=dev)
        return self.lists(torch.cat(keys).unsqueeze(0), k)

    def qe_mix(self, idx, d, x, alpha):
        """(rows, dim) fp32: row r = sum_j powf(1 - d[r, j], alpha) * x[idx[r, j]] / k, in list order
        (agrl_qe_mix_dev)."""
        assert idx.stride() == d.stride() and x.dtype == torch.float32 and x.stride(1) == 1
        rows, k = idx.shape
        dim = x.shape[1]
        out = torch.empty(rows, dim, dtype=torch.float32, device=x.device)
        _lib.call(x.device, self.lib.agrl_qe_mix_dev,
                  idx.data_ptr(), d.data_ptr(), idx.stride(0), rows, k, x.data_ptr(), x.stride(0), x.shape[0], dim,
                  float(alpha), out.data_ptr(), dim)
        return out


    # ---- market1501 metric -------------------------------------------------------------------------
    def market_count(self, q_pids, g_pids, q_camids, g_camids):
        dev = g_pids.device
        nq, ng = q_pids.numel(), g_pids.numel()
        out = torch.zeros(2, dtype=torch.int32, device=dev)                   # [max_count, status]
        wsb = self.lib.agrl_rank_workspace_bytes(nq, ng, 1)
        _lib.call(dev, self.lib.agrl_rank_market1501_count_dev,
                  q_pids.data_ptr(), g_pids.data_ptr(), q_camids.data_ptr(), g_camids.data_ptr(), nq, ng,
                  out.data_ptr(), out.data_ptr() + 4, _workspace(dev, wsb).data_ptr(), wsb)
        return out[0:1], out[1:2]

    def market_gather(self, d, q_pids, g_pids, q_camids, g_camids, offset, cap):
        dev = d.device
        nq, ng = d.shape
        keys = torch.empty(nq, cap, dtype=torch.int64, device=dev)
        counts = torch.empty(2, nq, dtype=torch.int32, device=dev)            # [npos, njunk]
        status = torch.zeros(1, dtype=torch.int32, device=dev)
        wsb = self.lib.agrl_rank_workspace_bytes(nq, ng, 1)
        _lib.call(dev, self.lib.agrl_rank_market1501_gather_dev,
                  d.data_ptr(), d.stride(0), q_pids.data_ptr(), g_pids.data_ptr(), q_camids.data_ptr(), g_camids.data_ptr(),
                  nq, ng, offset, cap, keys.data_ptr(), counts[0].data_ptr(), counts[1].data_ptr(), status.data_ptr(),
                  _workspace(dev, wsb).data_ptr(), wsb)
        return keys, counts, status

    def market_bin(self, d, offset, keys_all):
        dev = d.device
        nq, ng = d.shape
        parts, cap = keys_all.shape[0], keys_all.shape[2]
        n2 = self.lib.agrl_rank_market1501_list_len(parts, cap)
        if n2 == 0:
            _lib.check(_lib.E_UNSUPPORTED)
        cnt = torch.empty(nq, n2, dtype=torch.int32, device=dev)
        srt = torch.empty(nq, n2, dtype=torch.int64, device=dev)
        _lib.call(dev, self.lib.agrl_rank_market1501_bin_dev,
                  d.data_ptr(), d.stride(0), nq, ng, offset, keys_all.data_ptr(), parts, cap, cnt.data_ptr(), srt.data_ptr())
        return cnt, srt

    def market_finalize(self, cnt, srt, counts, ng_total, parts, cap, max_rank, status_parts):
        dev = cnt.device
        nq = cnt.shape[0]
        rank_len = min(max_rank, ng_total)
        cmc = torch.empty(rank_len, dtype=torch.float32, device=dev)
        scal = torch.zeros(4, dtype=torch.float32, device=dev)               # [mAP, status(u32), num_valid(i64)]
        wsb = self.lib.agrl_rank_market1501_finalize_workspace_bytes(nq, parts, cap, max_rank)
        _lib.call(dev, self.lib.agrl_rank_market1501_finalize_dev,
                  cnt.data_ptr(), srt.data_ptr(), counts[0].data_ptr(), counts[1].data_ptr(), nq, ng_total, parts, cap,
                  max_rank, cmc.data_ptr(), scal.data_ptr(), None, scal.data_ptr() + 8, scal.data_ptr() + 4,
                  _workspace(dev, wsb).data_ptr(), wsb)
        host = scal.cpu()
        _raise_status(int(host.view(torch.int32)[1]) | int(status_parts.cpu()))
        return cmc.cpu().numpy(), float(host[0])

    # ---- gallery-sharded k-reciprocal re-ranking (agrl_rerank_shard_*) ----------------------------------------------
    def rerank_rows(self, qg, qq, gg_slabs, offset, n_own, max_own, k1, k2):
        """Phase A.  ``gg_slabs`` yields (s0, g_g[:, offset + s0 : offset + s0 + w]) in order; each slab is released
        once consumed.  Returns (state for the next two phases, int32 rank rows (num_q + n_own, K))."""
        lib, dev = self.lib, qg.device
        nq, ng = qg.shape
        if lib.agrl_rerank_shard_workspace_bytes(nq, ng, max_own, k1, k2) == 0:      # the same verdict on every rank
            _lib.check(_lib.E_UNSUPPORTED)
        wsb = lib.agrl_rerank_shard_workspace_bytes(nq, ng, n_own, k1, k2)
        K, _ = rerank_row_dims(k1, k2)
        st = SimpleNamespace(ws=torch.empty(wsb, dtype=torch.uint8, device=dev), wsb=wsb, nq=nq, ng=ng, offset=offset,
                             n_own=n_own, k1=k1, k2=k2)
        rank_rows = torch.empty(nq + n_own, K, dtype=torch.int32, device=dev)

        def rows(slab, r0, r1):
            _lib.call(dev, lib.agrl_rerank_shard_rows_dev,
                      qg.data_ptr(), qg.stride(0), qq.data_ptr(), qq.stride(0), slab.data_ptr() if slab is not None else None,
                      slab.stride(0) if slab is not None else 0, nq, ng, offset, n_own, r0, r1, k1, k2, rank_rows.data_ptr(),
                      st.ws.data_ptr(), wsb)
        rows(None, 0, nq)
        for s0, slab in gg_slabs:
            rows(slab.contiguous(), nq + s0, nq + s0 + slab.shape[1])
        return st, rank_rows

    def rerank_expand(self, st, rank_all):
        """Phase B: this rank's k-reciprocal rows (idx int32, val fp32 (num_q + n_own, cap); cnt int32 (num_q + n_own))."""
        dev = rank_all.device
        _, cap = rerank_row_dims(st.k1, st.k2)
        rows = st.nq + st.n_own
        idx = torch.empty(rows, cap, dtype=torch.int32, device=dev)
        val = torch.empty(rows, cap, dtype=torch.float32, device=dev)
        cnt = torch.empty(rows, dtype=torch.int32, device=dev)
        _lib.call(dev, self.lib.agrl_rerank_shard_expand_dev,
                  rank_all.data_ptr(), st.nq, st.ng, st.offset, st.n_own, st.k1, st.k2, idx.data_ptr(), val.data_ptr(),
                  cnt.data_ptr(), st.ws.data_ptr(), st.wsb)
        return idx, val, cnt

    def rerank_finish(self, st, rank_all, idx_all, val_all, cnt_all, lambda_value):
        """Phase C: this rank's (num_q, n_own) block of the re-ranked distance matrix."""
        dev = rank_all.device
        out = torch.empty(st.nq, st.n_own, dtype=torch.float32, device=dev)
        _lib.call(dev, self.lib.agrl_rerank_shard_finish_dev,
                  rank_all.data_ptr(), idx_all.data_ptr(), val_all.data_ptr(), cnt_all.data_ptr(), st.nq, st.ng, st.offset,
                  st.n_own, st.k1, st.k2, float(lambda_value), out.data_ptr() if st.n_own else None, max(st.n_own, 1),
                  st.ws.data_ptr(), st.wsb)
        return out


def _distance_blocks(qop, gop, block_bytes=TOPK_BLOCK_BYTES):
    """(q0, q1, distance rows q0:q1 of two PreparedOperand) over the queries, in blocks of at most ``block_bytes`` that
    reuse one buffer: consume each block before taking the next."""
    assert (qop.metric, qop.split, qop.dim, qop.device) == (gop.metric, gop.split, gop.dim, gop.device)
    nq, ng = qop.rows, gop.rows
    rows = max(1, min(nq, block_bytes // max(4 * ng, 1)))
    dbuf = torch.empty(rows, ng, device=qop.device)
    for q0 in range(0, nq, rows):
        q1 = min(nq, q0 + rows)
        yield q0, q1, distance_prepared(qop.rows_view(q0, q1), gop, out=dbuf[:q1 - q0])


def rerank_row_dims(k1, k2):
    """(K, cap): widths of the rank-table rows and of the k-reciprocal rows exchanged by the sharded re-ranking
    (include/agrl_b200.h): K = max(k1 + 1, k2), cap = least power of two >= (k1 + 1)(round(k1 / 2) + 2)."""
    need = (k1 + 1) * (int(np.around(k1 / 2.)) + 2)
    cap = 2
    while cap < need:
        cap *= 2
    return max(k1 + 1, k2), cap


def _unlabelled(nq, ng, dev):
    """query / gallery labels for a ranking that needs none: no gallery item shares a query's pid"""
    return torch.zeros(nq, dtype=torch.int64, device=dev), torch.ones(ng, dtype=torch.int64, device=dev)


MAX_LIST_DEPTH = 8192            # k + J per query and shard (agrl_rank_mars_partial_dev / agrl_rank_lists_dev)
FUSED_MAX_DEPTH = 256            # deepest list the fused distance -> top-k keeps (agrl_distance_topk_dev)
FUSED_MIN_GALLERY = 32768        # gallery rows per shard from which the fused distance -> top-k is the default


def fused_default(gallery_rows, depth):
    """Whether lists of ``depth`` keys against ``gallery_rows`` rows come from the distance -> top-k fused into the
    GEMM epilogue unless the caller says otherwise: from FUSED_MIN_GALLERY rows on, up to FUSED_MAX_DEPTH keys."""
    return gallery_rows >= FUSED_MIN_GALLERY and depth <= FUSED_MAX_DEPTH


def list_depth(k, ops, labels, exclude_junk, group=None, world=1):
    """Keys every shard must keep per query for lists of length k: k, plus with ``exclude_junk`` the most junk items
    (same pid and camera) any query has in one shard, all-reduced (MAX) over the ranks with their status words.  Raises
    ValueError beyond MAX_LIST_DEPTH."""
    k = int(k)
    if k < 1:
        raise ValueError('k must be at least 1, got {}'.format(k))
    J = 0
    if exclude_junk:
        if labels is None:
            raise ValueError('exclude_junk needs q_pids, g_pids, q_camids and g_camids')
        j, status = ops.junk_depth(*labels)
        if world > 1:
            j, status = _max_and_or(j, status, group)
        host = torch.cat([j, status.to(j.dtype)]).cpu()
        _raise_status(int(host[1]))
        J = int(host[0])
    if k + J > MAX_LIST_DEPTH:
        raise ValueError('ranked lists reach {} keys per query (k = {} plus {} junk items of one identity and camera); '
                         'at most {} are supported'.format(k + J, k, J, MAX_LIST_DEPTH))
    return k + J


def rank_lists_sharded(qf, gf_local, k, q_pids=None, g_pids_local=None, q_camids=None, g_camids_local=None,
                       metric='euclidean', exclude_junk=False, group=None, broadcast_queries=True, ops=None,
                       gallery_counts=None, fused=None, re_rank=False, k1=20, k2=6, lambda_value=0.3):
    """Ranked lists of ``qf`` against the union of every rank's gallery shard: (indices int64, distances fp32) CUDA
    tensors of shape (num_q, k), the same on every rank, bit-identical to ``metrics.rank_lists`` on the whole distance
    matrix -- row i is np.argsort(d[i], kind='stable')[:k] with GLOBAL gallery indices, padded with (-1, +inf).
    Arguments as in evaluate_mars_sharded; labels are only needed for ``exclude_junk`` (skip the gallery items with the
    query's pid and camera; pid -1 distractors stay).  ``re_rank`` ranks the block of re_ranking_sharded instead.
    Exchanges: the query broadcast and shard layout of evaluate_mars_sharded, one all-reduce(max) of the junk depth J with
    ``exclude_junk`` (plus one all-gather of the gallery labels), and one all-gather of num_q x (k + J) keys.
    Raises ValueError when k + J exceeds MAX_LIST_DEPTH."""
    _check_metric(metric)
    dev = qf.device
    ops = ops or CudaOps()
    qf = qf.contiguous()
    labels = None
    if q_pids is not None:
        labels = [_dev_labels(x, dev) for x in (q_pids, g_pids_local, q_camids, g_camids_local)]
    world, rank, counts, offset, n_own = _shard_prologue(qf, gf_local, group, broadcast_queries, gallery_counts,
                                                         *(labels[0::2] if labels else ()))      # q_pids, q_camids
    nq = qf.shape[0]
    depth = list_depth(k, ops, labels, exclude_junk, group, world)
    if fused is None:
        fused = hasattr(ops, 'topk_keys') and fused_default(n_own, depth)
    if re_rank:
        d = re_ranking_sharded(qf, gf_local, metric, k1, k2, lambda_value, group=group, broadcast_queries=False, ops=ops,
                               gallery_counts=counts)
    if n_own == 0:                        # no candidates: an all-empty list
        keys = torch.full((nq, depth), -1, dtype=torch.int64, device=dev)
    elif re_rank:
        keys = ops.keys(d, depth, offset)
    elif fused:
        keys = ops.topk_keys(PreparedOperand(qf, metric, ops.split), PreparedOperand(gf_local, metric, ops.split), depth,
                             offset, fused=depth <= FUSED_MAX_DEPTH)
    else:
        keys = ops.keys(ops.distance(qf, gf_local, metric), depth, offset)
    keys_all = _gather_lists(keys, world, group)
    if world > 1 and exclude_junk:        # the junk test needs the labels of every listed item
        labels[1] = _gather_shard_rows(labels[1], 0, counts, rank, group)
        labels[3] = _gather_shard_rows(labels[3], 0, counts, rank, group)
    return ops.lists(keys_all, k, *(labels or [None] * 4), exclude_junk=exclude_junk)


def check_qe_args(qe_k, qe_times, alpha, n):
    """ValueError for alpha query expansion parameters it cannot honour on a joint set of n rows."""
    if qe_k < 1 or qe_k > MAX_LIST_DEPTH:
        raise ValueError('qe_k must be between 1 and {}, got {}'.format(MAX_LIST_DEPTH, qe_k))
    if qe_k > n:
        raise ValueError('qe_k = {} exceeds the {} query and gallery rows'.format(qe_k, n))
    if qe_times < 1:
        raise ValueError('qe_times must be at least 1, got {}'.format(qe_times))
    if not math.isfinite(alpha):
        raise ValueError('alpha must be finite, got {}'.format(alpha))


def query_expansion_sharded(qf, gf_local, qe_k=5, qe_times=1, alpha=3.0, group=None, broadcast_queries=True, ops=None,
                            gallery_counts=None):
    """Alpha query expansion (metrics.query_expansion) of ``qf`` and the union of every rank's gallery shard.

    Returns (qf', gf_local'): the expanded queries (the same on every rank) and this rank's expanded gallery rows,
    bit-identical to the matching rows of metrics.query_expansion on the whole sets.  Arguments as in
    evaluate_mars_sharded; shards may be empty.  Each iteration all-gathers the gallery rows; each rank then ranks its
    query and gallery rows against the whole joint set and mixes them.  Raises ValueError as check_qe_args."""
    ops = ops or CudaOps()
    assert qf.dim() == 2 and gf_local.dim() == 2 and qf.size(1) == gf_local.size(1)
    dev = qf.device
    qf = qf.detach().to(torch.float32).contiguous()
    gf = gf_local.detach().to(device=dev, dtype=torch.float32).contiguous()
    if broadcast_queries and _world_size(group) > 1:
        qf = qf.clone()                   # the broadcast writes into it
    _, rank, counts, offset, n_own = _shard_prologue(qf, gf, group, broadcast_queries, gallery_counts)
    nq = qf.shape[0]
    check_qe_args(qe_k, qe_times, alpha, nq + sum(counts))
    lo = nq + offset
    for _ in range(qe_times):
        x = torch.cat([qf, _gather_shard_rows(gf, 0, counts, rank, group)])
        idx, d = ops.qe_lists(x, [(0, nq), (lo, lo + n_own)], qe_k)
        mixed = ops.qe_mix(idx, d, x, alpha)
        qf, gf = mixed[:nq], mixed[nq:]
    return qf, gf


def _world_size(group):
    return dist.get_world_size(group) if dist.is_initialized() else 1


def _shard_prologue(qf, gf_local, group, broadcast_queries, gallery_counts, qp=None, qc=None):
    """(world, rank, counts, offset, n_own) of a sharded entry: rank 0's queries (and their labels qp, qc) broadcast
    into qf (qp, qc) with ``broadcast_queries``, then the rows of every rank's gallery shard (_shard_layout), the global
    index of this rank's first gallery row and its number of rows."""
    world = _world_size(group)
    if world > 1 and broadcast_queries:
        _broadcast_queries(qf, qp, qc, group)
    counts, rank = _shard_layout(gf_local.shape[0], qf.device, world, group, gallery_counts)
    return world, rank, counts, sum(counts[:rank]), counts[rank]


def _shard_layout(n_local_rows, dev, world, group, gallery_counts):
    """(rows of every shard, this rank): from ``gallery_counts`` when the caller knows them (no collective, no host
    sync), else one all-gather of the local row count."""
    if world == 1:
        return [int(n_local_rows)], 0
    rank = dist.get_rank(group)
    if gallery_counts is not None:
        counts = [int(c) for c in gallery_counts]
        assert len(counts) == world and counts[rank] == int(n_local_rows), 'gallery_counts must list every rank\'s shard rows'
        return counts, rank
    n_local = torch.tensor([n_local_rows], dtype=torch.int64, device=dev)
    counts = torch.empty(world, dtype=torch.int64, device=dev)
    dist.all_gather_into_tensor(counts, n_local, group=group)
    return counts.cpu().tolist(), rank


def _broadcast_queries(qf, qp, qc, group):
    """rank 0's query features and labels to every rank: two collectives (features; both label vectors packed)"""
    src = dist.get_global_rank(group, 0) if group is not None else 0
    dist.broadcast(qf, src=src, group=group)
    if qp is None:
        return
    lab = torch.stack([qp, qc])
    dist.broadcast(lab, src=src, group=group)
    qp.copy_(lab[0]); qc.copy_(lab[1])


def _gather_shard_rows(t, head, counts, rank, group):
    """t[:head] followed by every rank's rows t[head:] in rank order (one all-gather, padded to the largest shard)."""
    world = len(counts)
    if world == 1:
        return t
    most = max(counts)
    pad = t.new_zeros((most,) + tuple(t.shape[1:]))
    pad[:counts[rank]] = t[head:]
    buf = t.new_empty((world * most,) + tuple(t.shape[1:]))
    dist.all_gather_into_tensor(buf, pad, group=group)
    return torch.cat([t[:head]] + [buf[r * most:r * most + c] for r, c in enumerate(counts)])


def _gather_lists(t, world, group):
    """(world, num_q, depth) view of every rank's per-query lists t (num_q, depth), in rank order (one all-gather)."""
    if world == 1:
        return t.unsqueeze(0)
    out = t.new_empty((world * t.shape[0],) + tuple(t.shape[1:]))
    dist.all_gather_into_tensor(out, t.contiguous(), group=group)
    return out.view((world,) + tuple(t.shape))


RERANK_SLAB_BYTES = 1 << 31      # largest g_g column slab (num_g x columns fp32) alive at a time


def re_ranking_sharded(qf, gf_local, metric='euclidean', k1=20, k2=6, lambda_value=0.3, group=None,
                       broadcast_queries=True, ops=None, gallery_counts=None):
    """k-reciprocal re-ranking (utils/re_ranking.py:30-94) of ``qf`` against the union of every rank's gallery shard.

    Returns this rank's (num_q, num_g_r) block of the re-ranked distance matrix as a CUDA tensor: bit-identical to
    ``re_ranking_dev(qg, qq, gg)[:, off:off + num_g_r]`` with the three matrices from ``compute_distance_matrix`` on
    the whole sets and ``off`` the global index of this rank's first gallery row.  Arguments as in
    evaluate_mars_sharded.  Exchanges: the gallery features (all-gather), then the gallery rows of the rank table
    (num_g x K int32) and of the k-reciprocal rows (num_g x cap x 8 B + counts).  Per-rank limits: k1 <= 30, k2 <= 8,
    num_g_r <= 50000 (agrl_rerank_shard_workspace_bytes); the D rows take 4 (num_q + num_g_r)(num_q + num_g) bytes.
    """
    _check_metric(metric)
    ops = ops or CudaOps()
    qf, gf_own = qf.contiguous(), gf_local.contiguous()
    _, rank, counts, offset, n_own = _shard_prologue(qf, gf_own, group, broadcast_queries, gallery_counts)
    nq, ng = qf.shape[0], sum(counts)
    gf_all = _gather_shard_rows(gf_own, 0, counts, rank, group)
    # the operand roles of the single-device path: qq = d(q, q), qg = d(q, g), gg[:, own] = d(g, g_own)
    qq = ops.distance(qf, qf, metric)
    qg = ops.distance(qf, gf_all, metric)
    width = max(1, RERANK_SLAB_BYTES // (4 * ng))
    slabs = ((s0, ops.distance(gf_all, gf_own[s0:s0 + width], metric)) for s0 in range(0, n_own, width))
    st, rank_rows = ops.rerank_rows(qg, qq, slabs, offset, n_own, max(counts), k1, k2)
    del qq, qg, gf_all
    rank_all = _gather_shard_rows(rank_rows, nq, counts, rank, group)
    v_all = [_gather_shard_rows(t, nq, counts, rank, group) for t in ops.rerank_expand(st, rank_all)]
    return ops.rerank_finish(st, rank_all, v_all[0], v_all[1], v_all[2], lambda_value)


def evaluate_mars_sharded(qf, gf_local, q_pids, g_pids_local, q_camids, g_camids_local, metric='euclidean',
                          max_rank=50, group=None, broadcast_queries=True, ops=None, fused=None, gallery_counts=None,
                          re_rank=False, k1=20, k2=6, lambda_value=0.3):
    """MARS-metric CMC/mAP (rank.py:160-212) of ``qf`` against the union of every rank's gallery shard.

    qf (num_q, d) and the query labels must be the same on every rank (``broadcast_queries`` copies
    rank 0's); gf_local (num_g_r, d) and its labels are this rank's rows.  Gallery indices are global:
    shard r starts at sum(num_g_0..r-1), which is also how ties are broken (by global index).
    ``gallery_counts``: rows of every rank's shard when the caller knows them (skips one all-gather and its host sync).
    ``fused``: distance -> top-k in the GEMM epilogue, no (num_q x num_g_r) matrix (default: from FUSED_MIN_GALLERY
    gallery rows per shard on; same result either way).
    ``re_rank``: rank the k-reciprocal re-ranked distances (re_ranking_sharded with k1, k2, lambda_value) instead,
    through the per-shard top-k + merge (``fused`` does not apply): the CMC/mAP of re_ranking_dev followed by
    evaluate_rank(use_metric_mars=True) on one device.
    Returns (numpy.float64[max_rank], numpy.float64) on every rank.
    """
    dev = qf.device
    ops = ops or CudaOps()
    qp, qc = _dev_labels(q_pids, dev), _dev_labels(q_camids, dev)
    gp, gc = _dev_labels(g_pids_local, dev), _dev_labels(g_camids_local, dev)
    qf = qf.contiguous()
    world, _, counts, offset, n_own = _shard_prologue(qf, gf_local, group, broadcast_queries, gallery_counts, qp, qc)
    total = sum(counts)
    if total < max_rank:
        raise ValueError('could not broadcast input array from shape ({},) into shape ({},)'.format(total, max_rank))

    if fused is None:
        fused = hasattr(ops, 'topk_fused') and fused_default(n_own, max_rank)
    if re_rank:
        d = re_ranking_sharded(qf, gf_local, metric, k1, k2, lambda_value, group=group, broadcast_queries=False, ops=ops,
                               gallery_counts=counts)
        keys, cls, ngood, status = ops.partial(d, qp, gp, qc, gc, max_rank, offset)
    elif fused:
        keys, cls, ngood, status = ops.topk_fused(PreparedOperand(qf, metric, ops.split), PreparedOperand(gf_local, metric, ops.split),
                                                  qp, gp, qc, gc, max_rank, offset)
    else:
        d = ops.distance(qf, gf_local, metric)
        keys, cls, ngood, status = ops.partial(d, qp, gp, qc, gc, max_rank, offset)
    keys_all, cls_all = _gather_lists(keys, world, group), _gather_lists(cls, world, group)
    if world > 1:
        dist.all_reduce(ngood, op=dist.ReduceOp.SUM, group=group)
        or_across_ranks(status, group)
    return ops.merge(keys_all, cls_all, ngood, max_rank, status)


def evaluate_market1501_sharded(qf, gf_local, q_pids, g_pids_local, q_camids, g_camids_local, metric='euclidean',
                                max_rank=50, group=None, broadcast_queries=True, ops=None, gallery_counts=None):
    """market1501-metric CMC/mAP (rank_cy.pyx:154-241 semantics) of ``qf`` against the union of every
    rank's gallery shard: same arguments as evaluate_mars_sharded, returns (numpy.float32[rank_len], float)
    on every rank, bit-identical to the unsharded evaluator (ties by global gallery index).

    Exchanges: all-reduce(max) of one int, all-gather of the per-query same-pid key lists, all-reduce(sum)
    of their positive / junk counts, all-reduce(sum) of the per-list-item rank counts."""
    dev = qf.device
    ops = ops or CudaOps()
    qp, qc = _dev_labels(q_pids, dev), _dev_labels(q_camids, dev)
    gp, gc = _dev_labels(g_pids_local, dev), _dev_labels(g_camids_local, dev)
    qf = qf.contiguous()
    world, _, counts_g, offset, _ = _shard_prologue(qf, gf_local, group, broadcast_queries, gallery_counts, qp, qc)
    ng_total = sum(counts_g)
    if ng_total < max_rank:
        print('Note: number of gallery samples is quite small, got {}'.format(ng_total))     # rank_cy.pyx:160-162

    max_count, status = ops.market_count(qp, gp, qc, gc)
    if world > 1:
        dist.all_reduce(max_count, op=dist.ReduceOp.MAX, group=group)
    cap = max(8, (int(max_count.cpu()) + 7) // 8 * 8)

    d = ops.distance(qf, gf_local, metric)
    keys, counts, st2 = ops.market_gather(d, qp, gp, qc, gc, offset, cap)
    status = torch.bitwise_or(status, st2)
    keys_all = _gather_lists(keys, world, group)
    if world > 1:
        dist.all_reduce(counts, op=dist.ReduceOp.SUM, group=group)
        or_across_ranks(status, group)
    cnt, srt = ops.market_bin(d, offset, keys_all)
    if world > 1:
        dist.all_reduce(cnt, op=dist.ReduceOp.SUM, group=group)
    return ops.market_finalize(cnt, srt, counts, ng_total, world, cap, max_rank, status)
