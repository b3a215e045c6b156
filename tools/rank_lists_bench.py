"""Ranked lists on one GPU, one process: wall time per call (CUDA events around the whole call, host syncs included)
and ms per launch of the library's kernels (_lib.profile), k = 50 unless stated.

  matrix_1980x9330       metrics.rank_lists on a resident 1980 x 9330 fp32 matrix (MARS shape), against
                         torch.topk + a stable tie fix-up (re-sort of the k results by (distance, index)) and against
                         evaluate_rank(use_metric_mars=True) on the same matrix
  retrieve_1980x9330     metrics.retrieve, 1980 x 9330 x 4096 features, prepared gallery (matrix route: below
                         sharded.FUSED_MIN_GALLERY)
  retrieve_10kx1m        metrics.retrieve, 10 000 x 1 000 000 x 2048 (the scaled sweep), prepared gallery, fused route;
                         besides, the fused top-k alone (CudaOps.topk_keys) and the lists step alone on its keys

Each timed pass starts after a 512 MB write, so the MARS-shape matrix (74 MB) is not served from L2.
    python tools/rank_lists_bench.py [--reps 10] [--warmup 2] [--out DIR]   -> one JSON line per case (and DIR/*.json)"""
import argparse, json, os, subprocess, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
from agrl.pytorch_b200 import _lib, metrics, sharded, synthetic
from agrl.pytorch_b200.metrics.distance import PreparedOperand

DEV = torch.device('cuda')


def gpu_info():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[torch.cuda.current_device()] if q else torch.cuda.get_device_name()


def timed(fn, args, flush):
    for _ in range(args.warmup):
        fn()
    torch.cuda.synchronize()
    wall, per_kernel = [], {}
    for _ in range(args.reps):
        flush.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with _lib.profile(torch.cuda.current_stream().cuda_stream) as p:
            a.record()
            fn()
            b.record()
        b.synchronize()
        wall.append(a.elapsed_time(b))
        for k, ms in p.kernels:
            per_kernel.setdefault(k, []).append(ms)
    kern = {k: {'launches': len(v) // args.reps, 'ms': round(sum(v) / len(v), 5)} for k, v in per_kernel.items()}
    return {'ms': round(float(np.mean(wall)), 4), 'min_ms': round(float(np.min(wall)), 4),
            'max_ms': round(float(np.max(wall)), 4), 'kernels': kern}


def topk_stable(d, k):
    """torch.topk, then the k results re-sorted by (distance, index): stable among what topk returned (which tied items
    at the k-th place topk keeps is still its own choice)"""
    v, i = torch.topk(d, k, dim=1, largest=False, sorted=True)
    o = torch.argsort(i, dim=1)
    v, i = v.gather(1, o), i.gather(1, o)
    o = torch.sort(v, dim=1, stable=True).indices
    return i.gather(1, o), v.gather(1, o)


def emit(out, case, res):
    res = dict(case=case, gpu=gpu_info(), **res)
    print(json.dumps(res), flush=True)
    if out:
        with open(os.path.join(out, case + '.json'), 'w') as f:
            json.dump(res, f, indent=1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--reps', type=int, default=10)
    ap.add_argument('--warmup', type=int, default=2)
    ap.add_argument('--k', type=int, default=50)
    ap.add_argument('--out', default=None)
    ap.add_argument('--skip-sweep', action='store_true')
    args = ap.parse_args()
    _lib.require_device()
    if args.out:
        os.makedirs(args.out, exist_ok=True)
    flush = torch.empty(128 << 20, dtype=torch.float32, device=DEV)
    k = args.k

    qp, qc, gp, gc = synthetic.eval_labels('mars', seed=7)
    qf, gf = synthetic.eval_features(qp, gp, 4096, seed=7, clustered=True)
    qf, gf = qf.to(DEV), gf.to(DEV)
    d = metrics.compute_distance_matrix(qf, gf)
    ours = metrics.rank_lists(d, k)
    tk = topk_stable(d, k)
    emit(args.out, 'matrix_1980x9330', {
        'k': k,
        'rank_lists': timed(lambda: metrics.rank_lists(d, k), args, flush),
        'torch_topk_stable': timed(lambda: topk_stable(d, k), args, flush),
        'evaluate_rank_mars': timed(lambda: metrics.evaluate_rank(d, qp, gp, qc, gc, max_rank=k, use_metric_mars=True),
                                    args, flush),
        'torch_topk_equal_lists': bool(torch.equal(tk[0], ours[0])),
    })

    gop = PreparedOperand(gf)
    got = metrics.retrieve(qf, gop, k)
    emit(args.out, 'retrieve_1980x9330x4096', {
        'k': k, 'equal_to_rank_lists': bool(torch.equal(got[0], ours[0])),
        'retrieve': timed(lambda: metrics.retrieve(qf, gop, k), args, flush)})
    del d, gop, gf, qf

    if args.skip_sweep:
        return
    g = torch.Generator(device=DEV).manual_seed(1)
    nq, ng, dim = 10000, 1000000, 2048
    gop = PreparedOperand(torch.randn(ng, dim, generator=g, device=DEV))      # the fp32 gallery is freed afterwards
    qf = torch.randn(nq, dim, generator=g, device=DEV)
    ops = sharded.CudaOps()
    qop = PreparedOperand(qf)
    keys = ops.topk_keys(qop, gop, k, 0)
    emit(args.out, 'retrieve_10kx1mx2048', {
        'k': k,
        'retrieve': timed(lambda: metrics.retrieve(qf, gop, k), args, flush),
        'fused_topk_keys_only': timed(lambda: ops.topk_keys(qop, gop, k, 0), args, flush),
        'lists_step_only': timed(lambda: ops.lists(keys.unsqueeze(0), k), args, flush),
        'num_gpus_visible': torch.cuda.device_count(),
    })


if __name__ == '__main__':
    main()
