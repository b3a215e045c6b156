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
from types import SimpleNamespace

import numpy as np
import torch
import torch.distributed as dist

from . import _lib


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
    """Bitwise OR of every rank's status word (bit flags: LABEL_RANGE, ZERO_DIVISION, TOPK_OVERFLOW, ...), in place.
    NCCL has no BOR reduction: the word is expanded into one 0/1 lane per bit, all-reduced with MAX and re-packed."""
    shifts = torch.arange(16, device=status.device, dtype=torch.int32)
    bits = (status.to(torch.int32).view(-1, 1) >> shifts) & 1
    dist.all_reduce(bits, op=dist.ReduceOp.MAX, group=group)
    status.copy_((bits << shifts).sum(dim=1).to(status.dtype).view_as(status))
    return status


class CudaOps(object):
    """Per-rank compute on the rank's current CUDA device (libagrl_b200)."""

    def __init__(self, split=_lib.SPLIT_FP16X2):
        self.lib = _lib.require_device()
        self.split = split
        self._ws = {}

    def _workspace(self, dev, nbytes):
        key = (dev, torch.cuda.current_stream(dev).cuda_stream)       # never shared between streams
        ws = self._ws.get(key)
        if ws is None or ws.numel() < nbytes:
            ws = self._ws[key] = torch.empty(nbytes, dtype=torch.uint8, device=dev)
        return ws

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
        ws = self._workspace(dev, wsb)
        with torch.cuda.device(dev):
            _lib.check(self.lib.agrl_rank_mars_partial_dev(
                d.data_ptr(), d.stride(0), q_pids.data_ptr(), g_pids.data_ptr(), q_camids.data_ptr(),
                g_camids.data_ptr(), nq, ng, max_rank, offset, keys.data_ptr(), cls.data_ptr(), ngood.data_ptr(),
                status.data_ptr(), ws.data_ptr(), wsb, torch.cuda.current_stream(dev).cuda_stream))
        return keys, cls, ngood, status

    def topk_fused(self, qop, gop, q_pids, g_pids, q_camids, g_camids, max_rank, offset, allow_fallback=True):
        """Same outputs as ``partial`` from two PreparedOperand, with the distance -> top-k fused into the GEMM epilogue
        (agrl_distance_topk_dev + agrl_rank_mars_classify_dev): no (num_q x num_g) matrix is allocated.  When a query's
        candidate list overflows (a gallery ordered by distance to the query) the call falls back to distance blocks +
        ``partial`` -- the results are the same either way."""
        from .metrics.distance import _METRICS
        assert (qop.metric, qop.split, qop.dim, qop.device) == (gop.metric, gop.split, gop.dim, gop.device)
        dev, nq, ng = qop.device, qop.rows, gop.rows
        keys = torch.empty(nq, max_rank, dtype=torch.int64, device=dev)
        cls = torch.empty(nq, max_rank, dtype=torch.uint8, device=dev)
        ngood = torch.empty(nq, dtype=torch.int32, device=dev)
        status = torch.zeros(1, dtype=torch.int32, device=dev)
        lib = self.lib
        wsb = max(lib.agrl_distance_topk_workspace_bytes(nq), lib.agrl_rank_mars_classify_workspace_bytes(nq, ng))
        ws = self._workspace(dev, wsb)
        with torch.cuda.device(dev):
            stream = torch.cuda.current_stream(dev).cuda_stream
            _lib.check(lib.agrl_distance_topk_dev(
                qop.buf.data_ptr(), nq, gop.buf.data_ptr(), ng, qop.dim, _METRICS[qop.metric], qop.split, max_rank, offset,
                keys.data_ptr(), status.data_ptr(), ws.data_ptr(), wsb, stream))
            _lib.check(lib.agrl_rank_mars_classify_dev(
                keys.data_ptr(), q_pids.data_ptr(), g_pids.data_ptr(), q_camids.data_ptr(), g_camids.data_ptr(),
                nq, ng, max_rank, offset, cls.data_ptr(), ngood.data_ptr(), status.data_ptr(), ws.data_ptr(), wsb, stream))
        if allow_fallback and int(status.cpu()) & _lib.ST_TOPK_OVERFLOW:
            return self.topk_unfused(qop, gop, q_pids, g_pids, q_camids, g_camids, max_rank, offset)
        return keys, cls, ngood, status

    def topk_unfused(self, qop, gop, q_pids, g_pids, q_camids, g_camids, max_rank, offset, block_bytes=1 << 31):
        """distance blocks (at most ``block_bytes`` each) written to HBM + the streaming top-k kernel"""
        from .metrics.distance import distance_prepared
        dev, nq, ng = qop.device, qop.rows, gop.rows
        rows = max(1, min(nq, block_bytes // max(4 * ng, 1)))
        keys = torch.empty(nq, max_rank, dtype=torch.int64, device=dev)
        cls = torch.empty(nq, max_rank, dtype=torch.uint8, device=dev)
        ngood = torch.empty(nq, dtype=torch.int32, device=dev)
        status = torch.zeros(1, dtype=torch.int32, device=dev)
        dbuf = torch.empty(rows, ng, device=dev)
        for q0 in range(0, nq, rows):
            q1 = min(nq, q0 + rows)
            dm = distance_prepared(qop.rows_view(q0, q1), gop, out=dbuf[:q1 - q0])
            k, c, n, st = self.partial(dm, q_pids[q0:q1], g_pids, q_camids[q0:q1], g_camids, max_rank, offset)
            keys[q0:q1], cls[q0:q1], ngood[q0:q1] = k, c, n
            status |= st
        return keys, cls, ngood, status

    def merge(self, keys_all, cls_all, ngood, max_rank, status_parts):
        dev = keys_all.device
        parts, nq = keys_all.shape[0], keys_all.shape[1]
        out = torch.zeros(max_rank + 2, dtype=torch.float64, device=dev)      # [cmc.., mAP, status]
        wsb = self.lib.agrl_rank_workspace_bytes(nq, 0, max_rank)
        ws = self._workspace(dev, wsb)
        with torch.cuda.device(dev):
            _lib.check(self.lib.agrl_rank_mars_merge_dev(
                keys_all.data_ptr(), cls_all.data_ptr(), ngood.data_ptr(), parts, nq, max_rank,
                out.data_ptr(), out.data_ptr() + 8 * max_rank, None, out.data_ptr() + 8 * (max_rank + 1),
                ws.data_ptr(), wsb, torch.cuda.current_stream(dev).cuda_stream))
            host = out.cpu()
            st_parts = int(status_parts.cpu())
        status = int(host.view(torch.int32)[2 * (max_rank + 1)]) | st_parts
        from .metrics.rank import _raise_status
        _raise_status(status)
        return host[:max_rank].numpy().copy(), np.float64(host[max_rank])


    # ---- market1501 metric -------------------------------------------------------------------------
    def market_count(self, q_pids, g_pids, q_camids, g_camids):
        dev = g_pids.device
        nq, ng = q_pids.numel(), g_pids.numel()
        out = torch.zeros(2, dtype=torch.int32, device=dev)                   # [max_count, status]
        wsb = self.lib.agrl_rank_workspace_bytes(nq, ng, 1)
        ws = self._workspace(dev, wsb)
        with torch.cuda.device(dev):
            _lib.check(self.lib.agrl_rank_market1501_count_dev(
                q_pids.data_ptr(), g_pids.data_ptr(), q_camids.data_ptr(), g_camids.data_ptr(), nq, ng,
                out.data_ptr(), out.data_ptr() + 4, ws.data_ptr(), wsb, torch.cuda.current_stream(dev).cuda_stream))
        return out[0:1], out[1:2]

    def market_gather(self, d, q_pids, g_pids, q_camids, g_camids, offset, cap):
        dev = d.device
        nq, ng = d.shape
        keys = torch.empty(nq, cap, dtype=torch.int64, device=dev)
        counts = torch.empty(2, nq, dtype=torch.int32, device=dev)            # [npos, njunk]
        status = torch.zeros(1, dtype=torch.int32, device=dev)
        wsb = self.lib.agrl_rank_workspace_bytes(nq, ng, 1)
        ws = self._workspace(dev, wsb)
        with torch.cuda.device(dev):
            _lib.check(self.lib.agrl_rank_market1501_gather_dev(
                d.data_ptr(), d.stride(0), q_pids.data_ptr(), g_pids.data_ptr(), q_camids.data_ptr(), g_camids.data_ptr(),
                nq, ng, offset, cap, keys.data_ptr(), counts[0].data_ptr(), counts[1].data_ptr(), status.data_ptr(),
                ws.data_ptr(), wsb, torch.cuda.current_stream(dev).cuda_stream))
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
        with torch.cuda.device(dev):
            _lib.check(self.lib.agrl_rank_market1501_bin_dev(
                d.data_ptr(), d.stride(0), nq, ng, offset, keys_all.data_ptr(), parts, cap, cnt.data_ptr(), srt.data_ptr(),
                torch.cuda.current_stream(dev).cuda_stream))
        return cnt, srt

    def market_finalize(self, cnt, srt, counts, ng_total, parts, cap, max_rank, status_parts):
        dev = cnt.device
        nq = cnt.shape[0]
        rank_len = min(max_rank, ng_total)
        cmc = torch.empty(rank_len, dtype=torch.float32, device=dev)
        scal = torch.zeros(4, dtype=torch.float32, device=dev)               # [mAP, status(u32), num_valid(i64)]
        wsb = self.lib.agrl_rank_market1501_finalize_workspace_bytes(nq, parts, cap, max_rank)
        ws = self._workspace(dev, wsb)
        with torch.cuda.device(dev):
            _lib.check(self.lib.agrl_rank_market1501_finalize_dev(
                cnt.data_ptr(), srt.data_ptr(), counts[0].data_ptr(), counts[1].data_ptr(), nq, ng_total, parts, cap, max_rank,
                cmc.data_ptr(), scal.data_ptr(), None, scal.data_ptr() + 8, scal.data_ptr() + 4, ws.data_ptr(), wsb,
                torch.cuda.current_stream(dev).cuda_stream))
            host = scal.cpu()
            st_parts = int(status_parts.cpu())
        from .metrics.rank import _raise_status
        _raise_status(int(host.view(torch.int32)[1]) | st_parts)
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
        with torch.cuda.device(dev):
            stream = torch.cuda.current_stream(dev).cuda_stream

            def rows(slab, r0, r1):
                _lib.check(lib.agrl_rerank_shard_rows_dev(
                    qg.data_ptr(), qg.stride(0), qq.data_ptr(), qq.stride(0), slab.data_ptr() if slab is not None else None,
                    slab.stride(0) if slab is not None else 0, nq, ng, offset, n_own, r0, r1, k1, k2, rank_rows.data_ptr(),
                    st.ws.data_ptr(), wsb, stream))
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
        with torch.cuda.device(dev):
            _lib.check(self.lib.agrl_rerank_shard_expand_dev(
                rank_all.data_ptr(), st.nq, st.ng, st.offset, st.n_own, st.k1, st.k2, idx.data_ptr(), val.data_ptr(),
                cnt.data_ptr(), st.ws.data_ptr(), st.wsb, torch.cuda.current_stream(dev).cuda_stream))
        return idx, val, cnt

    def rerank_finish(self, st, rank_all, idx_all, val_all, cnt_all, lambda_value):
        """Phase C: this rank's (num_q, n_own) block of the re-ranked distance matrix."""
        dev = rank_all.device
        out = torch.empty(st.nq, st.n_own, dtype=torch.float32, device=dev)
        with torch.cuda.device(dev):
            _lib.check(self.lib.agrl_rerank_shard_finish_dev(
                rank_all.data_ptr(), idx_all.data_ptr(), val_all.data_ptr(), cnt_all.data_ptr(), st.nq, st.ng, st.offset,
                st.n_own, st.k1, st.k2, float(lambda_value), out.data_ptr() if st.n_own else None, max(st.n_own, 1),
                st.ws.data_ptr(), st.wsb, torch.cuda.current_stream(dev).cuda_stream))
        return out


def rerank_row_dims(k1, k2):
    """(K, cap): widths of the rank-table rows and of the k-reciprocal rows exchanged by the sharded re-ranking
    (include/agrl_b200.h): K = max(k1 + 1, k2), cap = least power of two >= (k1 + 1)(round(k1 / 2) + 2)."""
    need = (k1 + 1) * (int(np.around(k1 / 2.)) + 2)
    cap = 2
    while cap < need:
        cap *= 2
    return max(k1 + 1, k2), cap


def _as_dev_i64(x, dev):
    if isinstance(x, torch.Tensor):
        return x.to(device=dev, dtype=torch.int64).contiguous()
    return torch.as_tensor(np.ascontiguousarray(np.asarray(x), dtype=np.int64)).to(dev)


FUSED_MIN_GALLERY = 32768        # gallery rows per shard from which the fused distance -> top-k is the default


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
    if metric not in ('euclidean', 'cosine'):
        raise ValueError('Unknown distance metric: {}. Please choose either "euclidean" or "cosine"'.format(metric))
    world = dist.get_world_size(group) if dist.is_initialized() else 1
    ops = ops or CudaOps()
    qf, gf_own = qf.contiguous(), gf_local.contiguous()
    if world > 1 and broadcast_queries:
        _broadcast_queries(qf, None, None, group)
    counts, rank = _shard_layout(gf_own.shape[0], qf.device, world, group, gallery_counts)
    nq, ng, n_own, offset = qf.shape[0], sum(counts), counts[rank], sum(counts[:rank])
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
    world = dist.get_world_size(group) if dist.is_initialized() else 1
    dev = qf.device
    ops = ops or CudaOps()
    qp, qc = _as_dev_i64(q_pids, dev), _as_dev_i64(q_camids, dev)
    gp, gc = _as_dev_i64(g_pids_local, dev), _as_dev_i64(g_camids_local, dev)
    qf = qf.contiguous()
    if world > 1 and broadcast_queries:
        _broadcast_queries(qf, qp, qc, group)
    # global index of this shard's first row
    counts, rank = _shard_layout(gf_local.shape[0], dev, world, group, gallery_counts)
    total = sum(counts)
    if total < max_rank:
        raise ValueError('could not broadcast input array from shape ({},) into shape ({},)'.format(total, max_rank))
    offset = sum(counts[:rank])

    if fused is None:
        fused = gf_local.shape[0] >= FUSED_MIN_GALLERY and hasattr(ops, 'topk_fused') and max_rank <= 256
    if re_rank:
        d = re_ranking_sharded(qf, gf_local, metric, k1, k2, lambda_value, group=group, broadcast_queries=False, ops=ops,
                               gallery_counts=counts)
        keys, cls, ngood, status = ops.partial(d, qp, gp, qc, gc, max_rank, offset)
    elif fused:
        from .metrics.distance import PreparedOperand
        keys, cls, ngood, status = ops.topk_fused(PreparedOperand(qf, metric, ops.split), PreparedOperand(gf_local, metric, ops.split),
                                                  qp, gp, qc, gc, max_rank, offset)
    else:
        d = ops.distance(qf, gf_local, metric)
        keys, cls, ngood, status = ops.partial(d, qp, gp, qc, gc, max_rank, offset)
    if world > 1:
        nq = keys.shape[0]
        keys_all = torch.empty((world * nq, max_rank), dtype=keys.dtype, device=dev)   # rank-major concatenation
        cls_all = torch.empty((world * nq, max_rank), dtype=cls.dtype, device=dev)
        dist.all_gather_into_tensor(keys_all, keys, group=group)
        dist.all_gather_into_tensor(cls_all, cls, group=group)
        keys_all, cls_all = keys_all.view(world, nq, max_rank), cls_all.view(world, nq, max_rank)
        dist.all_reduce(ngood, op=dist.ReduceOp.SUM, group=group)
        or_across_ranks(status, group)
    else:
        keys_all, cls_all = keys.unsqueeze(0), cls.unsqueeze(0)
    return ops.merge(keys_all, cls_all, ngood, max_rank, status)


def evaluate_market1501_sharded(qf, gf_local, q_pids, g_pids_local, q_camids, g_camids_local, metric='euclidean',
                                max_rank=50, group=None, broadcast_queries=True, ops=None, gallery_counts=None):
    """market1501-metric CMC/mAP (rank_cy.pyx:154-241 semantics) of ``qf`` against the union of every
    rank's gallery shard: same arguments as evaluate_mars_sharded, returns (numpy.float32[rank_len], float)
    on every rank, bit-identical to the unsharded evaluator (ties by global gallery index).

    Exchanges: all-reduce(max) of one int, all-gather of the per-query same-pid key lists, all-reduce(sum)
    of their positive / junk counts, all-reduce(sum) of the per-list-item rank counts."""
    world = dist.get_world_size(group) if dist.is_initialized() else 1
    dev = qf.device
    ops = ops or CudaOps()
    qp, qc = _as_dev_i64(q_pids, dev), _as_dev_i64(q_camids, dev)
    gp, gc = _as_dev_i64(g_pids_local, dev), _as_dev_i64(g_camids_local, dev)
    qf = qf.contiguous()
    if world > 1 and broadcast_queries:
        _broadcast_queries(qf, qp, qc, group)
    counts_g, rank = _shard_layout(gf_local.shape[0], dev, world, group, gallery_counts)
    ng_total, offset = sum(counts_g), sum(counts_g[:rank])
    if ng_total < max_rank:
        print('Note: number of gallery samples is quite small, got {}'.format(ng_total))     # rank_cy.pyx:160-162

    max_count, status = ops.market_count(qp, gp, qc, gc)
    if world > 1:
        dist.all_reduce(max_count, op=dist.ReduceOp.MAX, group=group)
    cap = max(8, (int(max_count.cpu()) + 7) // 8 * 8)

    d = ops.distance(qf, gf_local, metric)
    keys, counts, st2 = ops.market_gather(d, qp, gp, qc, gc, offset, cap)
    status = torch.bitwise_or(status, st2)
    nq = keys.shape[0]
    if world > 1:
        keys_all = torch.empty((world * nq, cap), dtype=keys.dtype, device=dev)
        dist.all_gather_into_tensor(keys_all, keys, group=group)
        keys_all = keys_all.view(world, nq, cap)
        dist.all_reduce(counts, op=dist.ReduceOp.SUM, group=group)
        or_across_ranks(status, group)
    else:
        keys_all = keys.unsqueeze(0)
    cnt, srt = ops.market_bin(d, offset, keys_all)
    if world > 1:
        dist.all_reduce(cnt, op=dist.ReduceOp.SUM, group=group)
    return ops.market_finalize(cnt, srt, counts, ng_total, world, cap, max_rank, status)
