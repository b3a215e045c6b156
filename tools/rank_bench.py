"""Ranking kernels in isolation, one GPU, one process: ms per launch of every rank.cu kernel, from _lib.profile.

  market1501 / mars      agrl_rank_market1501_dev / agrl_rank_mars_dev on a 1980 x 9330 matrix (MARS shape)
  *_sharded              the gallery-sharded kernels over 8 column slices of that matrix, driven as
                         tests/test_gpu_rank.py drives them (single process: the collectives are sums / stacks)
  merge                  rank_mars_merge alone for (queries, shards), K = 50, ascending shard lists
  partial_1m             rank_mars_partial on 2000 queries x 1 000 000 gallery rows (one block of the unfused sweep)
  classify_1m            agrl_rank_mars_classify_dev: 10 000 queries x 1 000 000 gallery labels, valid keys

Each timed pass starts after a 512 MB write, so the inputs (74 MB for the MARS shape) are not served from L2.  Every
case also prints its result (mAP, or a checksum of the class bytes) so two libraries can be compared on outputs.
HV_LIB=path selects another build of the library (tools/build_alt.sh), e.g. -DAGRL_MERGE_SORT for the sorting merge.
    python tools/rank_bench.py [--reps 20] [--warmup 3]   -> one JSON line per case"""
import argparse, json, os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from agrl.pytorch_b200 import _lib
if os.environ.get('HV_LIB'):
    _lib.LIB_PATH = os.path.abspath(os.environ['HV_LIB'])
from agrl.pytorch_b200 import sharded, synthetic
from agrl.pytorch_b200.metrics import rank

DEV = torch.device('cuda')


def timed(name, fn, args, flush):
    for _ in range(args.warmup):
        result = fn()
    per_kernel = {}
    for _ in range(args.reps):
        flush.zero_()
        with _lib.profile(torch.cuda.current_stream().cuda_stream) as p:
            result = fn()
        for k, ms in p.kernels:
            per_kernel.setdefault(k, []).append(ms)
    # launches per pass and ms per launch (mean and min over the passes)
    kern = {k: {'launches': len(v) // args.reps, 'ms': round(sum(v) / len(v), 5), 'min_ms': round(min(v), 5)}
            for k, v in per_kernel.items()}
    print(json.dumps({'lib': os.environ.get('HV_LIB', 'product'), 'case': name, 'kernels': kern, 'result': result}),
          flush=True)


def labels(shape, seed):
    return [torch.as_tensor(x).to(DEV) for x in synthetic.eval_labels(shape, seed=seed)]     # qp, qc, gp, gc


def mars_shape_cases(args, flush):
    qp, qc, gp, gc = labels('mars', 7)
    nq, ng = qp.numel(), gp.numel()
    d = torch.rand(nq, ng, generator=torch.Generator(device=DEV).manual_seed(7), device=DEV)
    K, parts = 50, 8
    timed('market1501', lambda: float(rank.evaluate_cy(d, qp, gp, qc, gc, K)[1]), args, flush)
    timed('mars', lambda: float(rank.evaluate_mars(d, qp, gp, qc, gc, K)[1]), args, flush)

    ops = sharded.CudaOps()
    bounds = sharded.shard_bounds(ng, parts)

    def mars_sharded():
        keys, cls, ngood = [], [], 0
        for lo, hi in bounds:
            k, c, n, st = ops.partial(d[:, lo:hi], qp, gp[lo:hi], qc, gc[lo:hi], K, lo)
            keys.append(k); cls.append(c); ngood = ngood + n
        return float(ops.merge(torch.stack(keys), torch.stack(cls), ngood, K, st)[1])
    timed('mars_sharded', mars_sharded, args, flush)

    slices = [d[:, lo:hi].contiguous() for lo, hi in bounds]

    def market_sharded():
        cap = max(int(ops.market_count(qp, gp[lo:hi], qc, gc[lo:hi])[0].cpu()) for lo, hi in bounds)
        cap = max(8, (cap + 7) // 8 * 8)
        keys, counts = [], 0
        for (lo, hi), s in zip(bounds, slices):
            k, c, st = ops.market_gather(s, qp, gp[lo:hi], qc, gc[lo:hi], lo, cap)
            keys.append(k); counts = counts + c
        keys_all, cnt = torch.stack(keys), 0
        for (lo, hi), s in zip(bounds, slices):
            c, srt = ops.market_bin(s, lo, keys_all)
            cnt = cnt + c
        return float(ops.market_finalize(cnt, srt, counts, ng, parts, cap, K, st)[1])
    timed('market1501_sharded', market_sharded, args, flush)


def merge_cases(args, flush):
    ops = sharded.CudaOps()
    g = torch.Generator(device=DEV).manual_seed(0)
    for nq, parts in ((1980, 8), (10000, 8), (10000, 2)):
        K = 50
        d = torch.rand(parts, nq, K, generator=g, device=DEV)
        idx = torch.arange(parts * nq * K, device=DEV).view(parts, nq, K) % 1000000
        keys = ((d.sort(dim=2).values.view(torch.int32).to(torch.int64) | 0x80000000) << 32) | idx
        keys = keys.sort(dim=2).values.contiguous()
        cls = (torch.rand(parts, nq, K, generator=g, device=DEV) < 0.05).to(torch.uint8)
        ngood = torch.full((nq,), 5, dtype=torch.int32, device=DEV)
        st = torch.zeros(1, dtype=torch.int32, device=DEV)
        timed('merge_%dx%d' % (nq, parts), lambda: float(ops.merge(keys, cls, ngood, K, st)[1]), args, flush)


def gallery_1m_cases(args, flush):
    ng, K = 1000000, 50
    g = torch.Generator(device=DEV).manual_seed(5)
    nid = ng // 20
    gp = torch.randint(0, nid, (ng,), generator=g, device=DEV)
    gc = torch.randint(0, 6, (ng,), generator=g, device=DEV)
    ops = sharded.CudaOps()

    nq = 2000
    qp = torch.randint(0, nid, (nq,), generator=g, device=DEV)
    qc = torch.randint(0, 6, (nq,), generator=g, device=DEV)
    d = torch.rand(nq, ng, generator=g, device=DEV)

    def partial():
        keys, cls, ngood, _ = ops.partial(d, qp, gp, qc, gc, K, 0)
        return [int(keys.sum()), int(cls.to(torch.int64).sum()), int(ngood.sum())]
    timed('partial_1m', partial, args, flush)
    del d

    nq = 10000
    qp = torch.randint(0, nid, (nq,), generator=g, device=DEV)
    qc = torch.randint(0, 6, (nq,), generator=g, device=DEV)
    dist = torch.rand(nq, K, generator=g, device=DEV).sort(dim=1).values
    idx = torch.randint(0, ng, (nq, K), generator=g, device=DEV)
    keys = ((dist.view(torch.int32).to(torch.int64) | 0x80000000) << 32) | idx
    cls = torch.empty(nq, K, dtype=torch.uint8, device=DEV)
    ngood = torch.empty(nq, dtype=torch.int32, device=DEV)
    status = torch.zeros(1, dtype=torch.int32, device=DEV)
    lib = _lib.require_device()
    wsb = lib.agrl_rank_mars_classify_workspace_bytes(nq, ng)
    ws = torch.empty(wsb, dtype=torch.uint8, device=DEV)

    def classify():
        _lib.check(lib.agrl_rank_mars_classify_dev(
            keys.data_ptr(), qp.data_ptr(), gp.data_ptr(), qc.data_ptr(), gc.data_ptr(), nq, ng, K, 0,
            cls.data_ptr(), ngood.data_ptr(), status.data_ptr(), ws.data_ptr(), wsb,
            torch.cuda.current_stream().cuda_stream))
        return [int(cls.to(torch.int64).sum()), int(ngood.to(torch.int64).sum()), int(status.cpu())]
    timed('classify_1m', classify, args, flush)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--reps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=3)
    args = ap.parse_args()
    print(json.dumps({'device': torch.cuda.get_device_name(DEV), 'reps': args.reps, 'warmup': args.warmup}), flush=True)
    flush = torch.empty(512 << 20, dtype=torch.uint8, device=DEV)
    mars_shape_cases(args, flush)
    merge_cases(args, flush)
    gallery_1m_cases(args, flush)


if __name__ == '__main__':
    main()
