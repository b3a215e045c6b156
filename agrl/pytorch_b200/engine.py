"""Device-resident mirror of the reference's ``test()`` (train_vidreid_xent_htri.py:450-542) -- the caller of the
hot path: feature loop over the query / gallery loaders, optional clip pooling (dense / skipdense sampling,
:461-476), distance matrix (:520), optional k-reciprocal re-ranking (:523-527), CMC / mAP with the MARS metric
(:531), the same progress lines and the same return values.

What differs from the reference is where the data lives, not what is computed: features stay on the GPU from the
head to the ranking (the reference copies every batch to the host, :477, and evaluates there), so per call only the
labels go up and ``max_rank + 1`` numbers (or, with ``return_distmat``, the matrix) come down.  The reference reads
its options from a module-global ``args``; here they are keyword arguments with the same names (``test_sample``,
``dist_metric``, ``re_rank``), or an ``args`` namespace carrying them.

Several GPUs (SURVEY.md section 8e): with ``torch.distributed`` initialised (one process per GPU) every rank passes the
loader of ITS gallery shard -- contiguous shards in rank order, e.g. ``sharded.shard_bounds`` -- and the query loader
(rank 0's query features are the ones used); the head runs on each rank's own tracklets without any collective and the
ranking is the gallery-sharded one of ``sharded.evaluate_mars_sharded`` (per-rank distance block and top-``max_rank``,
one all-gather + one all-reduce, merge).  Every rank returns the same ``(cmc[0], mAP)``, bit-identical to the
single-GPU result.  Re-ranking needs the whole gallery on one device and is refused in that mode.

There is no CPU path: ``use_gpu=False`` raises, as every other entry of this package does without a B200.
"""
import time

import numpy as np
import torch

from . import metrics, sharded
from .models import pool_clips
from .utils.re_ranking import re_ranking_dev

__all__ = ['extract_features', 'test']


def _labels(x):
    """pids / camids of one loader batch (a tensor after default collation, :478-479; lists are accepted too)."""
    if isinstance(x, torch.Tensor):
        return x.cpu().numpy()
    return np.asarray(x)


def extract_features(model, loader, pool='avg', test_sample='evenly', device=None):
    """The feature loop of test() (:457-483 for the query set, :487-513 for the gallery).

    ``loader`` yields ``(imgs, pids, camids, adj)``: imgs (n, s, c, h, w) -- or (b, n, s, c, h, w) with
    ``test_sample`` 'dense' / 'skipdense', where the n clips of a tracklet are folded into the batch and pooled
    afterwards ('avg' -> mean, otherwise max, :471-476); adj the dense (.., V, V) pose graph or the compact
    (.., 3) int64 part masks (pose.part_masks).  Returns ``(features, pids, camids, seconds, batches, batch_imgs)``
    with features a (N, D) fp32 tensor on the model's device and seconds the host time spent in model() calls."""
    if device is None:
        device = next(model.parameters()).device
    dense = test_sample in ('dense', 'skipdense')
    feats, pids_all, camids_all = [], [], []
    spent, batches, batch_imgs = 0.0, 0, 0
    for imgs, pids, camids, adj in loader:
        imgs, adj = imgs.to(device, non_blocking=True), adj.to(device, non_blocking=True)
        if dense:
            b, n, s, c, h, w = imgs.size()
            imgs = imgs.view(b * n, s, c, h, w)
            adj = adj.view(b * n, 3) if adj.dtype == torch.int64 and adj.size(-1) == 3 \
                else adj.view(b * n, adj.size(-1), adj.size(-1))
        else:
            n, s, c, h, w = imgs.size()
        batch_imgs = max(batch_imgs, imgs.size(0) * s)
        end = time.time()
        features = model(imgs, adj)
        spent += time.time() - end
        batches += 1
        if dense:
            # the reference's `features.view(n, 1, -1)` + reduction over dim 0 presumes one tracklet per batch
            # (its dense loaders run with test_batch = 1); pool_clips does the same per tracklet for any b
            features = pool_clips(features, n, pool)
        feats.append(features)
        pids_all.extend(_labels(pids))
        camids_all.extend(_labels(camids))
    if feats:
        feats = torch.cat(feats, 0)
    else:
        feats = torch.empty(0, 0, dtype=torch.float32, device=device)
    return feats, np.asarray(pids_all), np.asarray(camids_all), spent, batches, batch_imgs


def _report(say, cmc, mAP, ranks):
    say("Results ----------")
    say("mAP: {:.2%}".format(mAP))
    say("CMC curve")
    for r in ranks:
        say("Rank-{:<3}: {:.2%}".format(r, cmc[r - 1]))
    say("------------------")


def test(model, queryloader, galleryloader, pool='avg', use_gpu=True, ranks=(1, 5, 10, 20), return_distmat=False,
         test_sample='evenly', dist_metric='euclidean', re_rank=False, max_rank=50, args=None, verbose=True,
         group=None, sharded_ops=None, return_ranked=None, aqe=False, qe_k=5, qe_times=1, qe_alpha=3.0):
    """Drop-in for the reference's test(): returns ``(cmc[0], mAP)``, or the (num_query, num_gallery) distance
    matrix as a numpy array with ``return_distmat``.  ``return_ranked=k`` (without ``return_distmat``) returns
    ``(cmc[0], mAP, indices, distances)`` instead, the first k gallery items of every query and their distances as
    (num_query, k) CUDA tensors (metrics.rank_lists on the ranked matrix; with several processes
    sharded.rank_lists_sharded, global gallery indices, the same on every rank).  Raises what the reference raises:
    ``ZeroDivisionError`` for a query without a cross-camera match (rank.py:203), ``ValueError`` for an unknown metric
    (distance.py:50-54).  ``aqe`` applies alpha query expansion (metrics.query_expansion with ``qe_k``, ``qe_times`` and
    ``qe_alpha``; with several processes sharded.query_expansion_sharded) to the extracted features, as FastReID's
    TEST.AQE does before its distance matrix: every later step, re-ranking included, sees the expanded features."""
    if not use_gpu:
        raise RuntimeError('agrl.pytorch_b200 has no CPU path: test() needs use_gpu=True and a B200')
    if args is not None:
        test_sample = getattr(args, 'test_sample', test_sample)
        dist_metric = getattr(args, 'dist_metric', dist_metric)
        re_rank = getattr(args, 're_rank', re_rank)
        aqe = getattr(args, 'aqe', aqe)
        qe_k = getattr(args, 'qe_k', qe_k)
        qe_times = getattr(args, 'qe_times', qe_times)
        qe_alpha = getattr(args, 'qe_alpha', qe_alpha)
    world = torch.distributed.get_world_size(group) if torch.distributed.is_initialized() else 1
    if world > 1 and torch.distributed.get_rank(group) != 0:
        verbose = False                                   # one copy of the progress lines
    say = print if verbose else (lambda *a, **k: None)
    if world > 1 and re_rank:
        raise NotImplementedError('re-ranking needs the whole gallery on one device; run it on one GPU')

    model.eval()
    with torch.no_grad():
        qf, q_pids, q_camids, tq, nq, bq = extract_features(model, queryloader, pool, test_sample)
        say("Extracted features for query set, obtained {}-by-{} matrix".format(qf.size(0), qf.size(1)))
        gf, g_pids, g_camids, tg, ng, bg = extract_features(model, galleryloader, pool, test_sample)
        say("Extracted features for gallery set, obtained {}-by-{} matrix".format(gf.size(0), gf.size(1)))
    say("==> BatchTime(s)/BatchSize(img): {:.3f}/{}".format((tq + tg) / max(nq + ng, 1), max(bq, bg)))

    if aqe:
        say('Applying alpha query expansion (qe_k={}, qe_times={}, alpha={}) ...'.format(qe_k, qe_times, qe_alpha))
        if world > 1:
            qf, gf = sharded.query_expansion_sharded(qf, gf, qe_k, qe_times, qe_alpha, group=group, ops=sharded_ops)
        else:
            qf, gf = metrics.query_expansion(qf, gf, qe_k, qe_times, qe_alpha)

    say('Computing distance matrix with metric={} ...'.format(dist_metric))
    if world > 1:
        # gallery-sharded: this rank's distance block + top-max_rank, merged over the ranks (sharded.py)
        say("Computing CMC and mAP")
        if return_distmat:
            ops = sharded_ops or sharded.CudaOps()
            return ops.distance(qf, gf, dist_metric).cpu().numpy()      # this rank's (num_q, num_g_local) block
        cmc, mAP = sharded.evaluate_mars_sharded(qf, gf, q_pids, g_pids, q_camids, g_camids, metric=dist_metric,
                                                 max_rank=max_rank, group=group, ops=sharded_ops)
        _report(say, cmc, mAP, ranks)
        if return_ranked:
            indices, distances = sharded.rank_lists_sharded(qf, gf, return_ranked, metric=dist_metric, group=group,
                                                            ops=sharded_ops)
            return cmc[0], mAP, indices, distances
        return cmc[0], mAP
    distmat = metrics.compute_distance_matrix(qf, gf, dist_metric)

    if re_rank:
        say('Applying person re-ranking ...')
        distmat_qq = metrics.compute_distance_matrix(qf, qf, dist_metric)
        distmat_gg = metrics.compute_distance_matrix(gf, gf, dist_metric)
        distmat = re_ranking_dev(distmat, distmat_qq, distmat_gg)

    say("Computing CMC and mAP")
    cmc, mAP = metrics.evaluate_rank(distmat, q_pids, g_pids, q_camids, g_camids, max_rank=max_rank,
                                     use_metric_mars=True)

    _report(say, cmc, mAP, ranks)

    if return_distmat:
        return distmat.cpu().numpy() if isinstance(distmat, torch.Tensor) else distmat
    if return_ranked:
        return (cmc[0], mAP) + metrics.rank_lists(distmat, return_ranked)
    return cmc[0], mAP
