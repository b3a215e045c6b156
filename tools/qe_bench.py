"""Alpha query expansion on one GPU, one process: wall time per call (CUDA events around the whole call, host syncs
included) and ms per launch of the library's kernels (_lib.profile); k = 5, alpha = 3, one iteration.

  mars_1980+9330x4096       metrics.query_expansion (matrix route: below sharded.FUSED_MIN_GALLERY rows); the mix
                            kernel alone on the lists it used; a torch-on-GPU restatement of FastReID's aqe (fp32
                            torch.mm of the normalised rows, torch.topk, gather + weighted mean)
  fused_10000+100000x2048   the same at a joint set on the fused distance -> top-k route

The mix kernel's bound is its unique HBM traffic over 7.7 TB/s (the HGX B200 data sheet's per-GPU bandwidth): every
feature row read once, every output row written once, plus the lists (12 bytes an entry).  Each timed pass starts
after a 512 MB write, so nothing is served from L2 that a cold call would read from HBM.
    python tools/qe_bench.py [--reps 10] [--warmup 2] [--out DIR]   -> one JSON line per case (and DIR/*.json)"""
import argparse, json, os, subprocess, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
import torch.nn.functional as F
from agrl.pytorch_b200 import _lib, metrics, sharded

DEV = torch.device('cuda')
HBM_BYTES_PER_S = 7.7e12


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


def torch_aqe(qf, gf, qe_k, alpha):
    """FastReID's aqe with one iteration, on the GPU in torch: the N x N fp32 similarity matrix, torch.topk, gather"""
    x = torch.cat([qf, gf])
    n = F.normalize(x, p=2, dim=1)
    s, i = torch.topk(torch.mm(n, n.t()), qe_k, dim=1)
    x = (x[i] * s.pow(alpha).unsqueeze(2)).mean(1)
    return x[:len(qf)], x[len(qf):]


def emit(out, case, res):
    res = dict(case=case, gpu=gpu_info(), **res)
    print(json.dumps(res), flush=True)
    if out:
        with open(os.path.join(out, case + '.json'), 'w') as f:
            json.dump(res, f, indent=1)


def run_case(name, nq, ng, dim, args, flush):
    k, alpha = args.k, 3.0
    g = torch.Generator(device=DEV).manual_seed(nq)
    qf, gf = torch.randn(nq, dim, generator=g, device=DEV), torch.randn(ng, dim, generator=g, device=DEV)
    n = nq + ng
    ops = sharded.CudaOps()
    x = torch.cat([qf, gf])
    idx, d = ops.qe_lists(x, [(0, n)], k)
    q, gq = metrics.query_expansion(qf, gf, k, 1, alpha)
    tq, tg = torch_aqe(qf, gf, k, alpha)
    ref = torch.cat([tq, tg])
    rel = float(((torch.cat([q, gq]) - ref).abs().amax(1) / ref.norm(dim=1)).max())
    mix_bytes = 2 * n * dim * 4 + n * k * 12
    res = {
        'N': n, 'dim': dim, 'k': k, 'alpha': alpha, 'fused_route': n >= sharded.FUSED_MIN_GALLERY,
        'query_expansion': timed(lambda: metrics.query_expansion(qf, gf, k, 1, alpha), args, flush),
        'qe_mix_only': timed(lambda: ops.qe_mix(idx, d, x, alpha), args, flush),
        'mix_unique_bytes': mix_bytes,
        'mix_hbm_bound_ms': round(mix_bytes / HBM_BYTES_PER_S * 1e3, 4),
        'max_row_diff_vs_torch_rel_norm': rel,
    }
    del tq, tg, ref
    torch.cuda.empty_cache()
    try:
        res['torch_mm_topk_gather'] = timed(lambda: torch_aqe(qf, gf, k, alpha), args, flush)
    except torch.cuda.OutOfMemoryError as e:
        res['torch_mm_topk_gather'] = 'out of memory: ' + str(e).splitlines()[0]
    mix = res['qe_mix_only']['kernels'].get('qe_mix', {}).get('ms')
    if mix:
        res['mix_share_of_hbm_bound'] = round(res['mix_hbm_bound_ms'] / mix, 3)
    emit(args.out, name, res)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--reps', type=int, default=10)
    ap.add_argument('--warmup', type=int, default=2)
    ap.add_argument('--k', type=int, default=5)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    _lib.require_device()
    if args.out:
        os.makedirs(args.out, exist_ok=True)
    flush = torch.empty(128 << 20, dtype=torch.float32, device=DEV)
    run_case('mars_1980+9330x4096', 1980, 9330, 4096, args, flush)
    run_case('fused_10000+100000x2048', 10000, 100000, 2048, args, flush)


if __name__ == '__main__':
    main()
