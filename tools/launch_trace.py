"""The library kernels every public evaluation entry launches, in order, on one GPU and one process.

For each case: the kernel names _lib.profile records (launch order), the _lib.launch_count() delta, and a SHA-256 of
what the call returned (tensors and arrays by their bytes), so that two trees that must launch the same kernels and
compute the same results can be compared line by line:

    python tools/launch_trace.py [--tree DIR] [--out FILE]     -> one JSON line per case

``--tree`` imports agrl.pytorch_b200 from DIR (default: this script's repository).  The sharded entries run at world
size 1 (no process group).  Sizes are small; the fused routes are reached from sharded.FUSED_MIN_GALLERY (32768) gallery
rows, the size their default switches at."""
import argparse, hashlib, json, os, sys

import numpy as np
import torch

FUSED_ROWS = 32768


def digest(x):
    h = hashlib.sha256()

    def feed(v):
        if isinstance(v, (tuple, list)):
            for e in v:
                feed(e)
        elif isinstance(v, torch.Tensor):
            h.update(v.detach().cpu().contiguous().numpy().tobytes())
        else:
            h.update(np.asarray(v).tobytes())
    feed(x)
    return h.hexdigest()[:16]


def cases(dev):
    from agrl.pytorch_b200 import metrics, sharded
    from agrl.pytorch_b200.utils.re_ranking import re_ranking_dev
    g = torch.Generator(device=dev).manual_seed(5)

    def feats(n, d):
        return torch.randn(n, d, generator=g, device=dev)

    def labels(n, nid=30):
        return (torch.randint(0, nid, (n,), generator=g, device=dev), torch.randint(0, 4, (n,), generator=g, device=dev))

    nq, ng, dim = 120, 900, 128
    qf, gf = feats(nq, dim), feats(ng, dim)
    (qp, qc), (gp, gc) = labels(nq), labels(ng)
    gp[::9] = -1                                                          # distractors
    big = feats(FUSED_ROWS, 64)
    (bp, bc), qbig = labels(FUSED_ROWS, 2000), feats(200, 64)
    qbp, qbc = labels(200, 2000)                                        # few junk items: lists stay <= 256 keys deep
    # overflow: a gallery ordered by decreasing distance to query 0 overflows its fused candidate list
    qo = feats(40, 64)
    u = torch.nn.functional.normalize(feats(1, 64)[0], dim=0)
    go = qo[0][None] + (12000 - torch.arange(12000, device=dev, dtype=torch.float32))[:, None] * 0.01 * u[None]
    d = metrics.compute_distance_matrix(qf, gf)
    qq, gg = metrics.compute_distance_matrix(qf, qf), metrics.compute_distance_matrix(gf, gf)

    yield 'compute_distance_matrix cpu', lambda: metrics.compute_distance_matrix(qf.cpu(), gf.cpu())
    yield 'compute_distance_matrix cuda', lambda: metrics.compute_distance_matrix(qf, gf, 'cosine')
    yield 'evaluate_rank mars', lambda: metrics.evaluate_rank(d, qp, gp, qc, gc, max_rank=50, use_metric_mars=True)
    yield 'evaluate_rank market1501', lambda: metrics.evaluate_rank(d, qp, gp, qc, gc, max_rank=50,
                                                                    use_metric_market1501=True)
    yield 'rank_lists', lambda: metrics.rank_lists(d, 20)
    yield 'rank_lists exclude_junk', lambda: metrics.rank_lists(d, 20, qp, gp, qc, gc, exclude_junk=True)
    yield 'retrieve matrix route', lambda: metrics.retrieve(qf, gf, 20)
    yield 'retrieve fused route', lambda: metrics.retrieve(qbig, big, 20, q_pids=qbp, g_pids=bp, q_camids=qbc,
                                                           g_camids=bc, exclude_junk=True)
    yield 'retrieve forced overflow', lambda: metrics.retrieve(qo, go, 50, fused=True)
    yield 'query_expansion matrix route', lambda: metrics.query_expansion(qf, gf, 5, 2, 3.0)
    yield 'query_expansion fused route', lambda: metrics.query_expansion(qbig, big, 5, 1, 3.0)
    yield 're_ranking_dev', lambda: re_ranking_dev(d, qq, gg)
    yield 'evaluate_mars_sharded unfused', lambda: sharded.evaluate_mars_sharded(qf, gf, qp, gp, qc, gc, fused=False)
    yield 'evaluate_mars_sharded fused', lambda: sharded.evaluate_mars_sharded(qbig, big, qbp, bp, qbc, bc)
    yield 'evaluate_market1501_sharded', lambda: sharded.evaluate_market1501_sharded(qf, gf, qp, gp, qc, gc)
    yield 'rank_lists_sharded', lambda: sharded.rank_lists_sharded(qf, gf, 20, qp, gp, qc, gc, exclude_junk=True)
    yield 'rank_lists_sharded fused', lambda: sharded.rank_lists_sharded(qbig, big, 20, metric='cosine')
    yield 'rank_lists_sharded re_rank', lambda: sharded.rank_lists_sharded(qf, gf, 20, re_rank=True)
    yield 'rank_lists_sharded empty gallery', lambda: sharded.rank_lists_sharded(qf, gf[:0], 20)
    yield 'query_expansion_sharded', lambda: sharded.query_expansion_sharded(qf, gf, 5, 2, 3.0)
    yield 're_ranking_sharded', lambda: sharded.re_ranking_sharded(qf, gf, 'cosine')


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--tree', default=os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    sys.path.insert(0, os.path.abspath(args.tree))
    from agrl.pytorch_b200 import _lib
    _lib.require_device()
    dev = torch.device('cuda')
    lines = []
    for name, fn in cases(dev):
        torch.cuda.synchronize()
        n0 = _lib.launch_count()
        with _lib.profile(torch.cuda.current_stream().cuda_stream) as p:
            res = fn()
            torch.cuda.synchronize()
        lines.append(json.dumps({'case': name, 'launches': _lib.launch_count() - n0,
                                 'kernels': [k for k, _ in p.kernels], 'result_sha256': digest(res)}))
        print(lines[-1], flush=True)
    if args.out:
        with open(args.out, 'w') as f:
            f.write('\n'.join(lines) + '\n')


if __name__ == '__main__':
    main()
