"""A/B of two builds of the library on one GPU: output digests and timings of the paths that write GEMM operand planes.
usage: HV_LIB=path python tools/planes_ab.py dump        -> one JSON line {name: sha256 of the output's bytes}
       HV_LIB=path python tools/planes_ab.py time        -> one JSON line: head pass ms, fp16 x 2 distance ms
dump: head `out` and `nodes` at B = 882 and 5 (S = 8) for every head split, low-rank on / off, CTA pairs on / off (fp16 +
E4M3), fp32 / bf16 / fp16 maps and dense / mask pose graphs; the prepared weight buffer of each split; distance matrices
and the written parts of both PreparedOperand buffers at 1980 x 9330 x 4096 (every split, both metrics); the fused top-k
keys at 10 000 x 100 000.  Two builds compute the same thing when every digest agrees.
time: the bench's head pass (11 310 tracklets from a pool of 882, fp32 maps, default mode) and the 1980 x 9330 x 4096
fp16 x 2 distance from prepared operands, CUDA events; the median of HV_REPS timed repetitions each (default 5)."""
import hashlib
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch
import bench
from agrl.pytorch_b200 import _lib
if os.environ.get('HV_LIB'):                      # the build to load (tools/build_alt.sh), instead of the product library
    _lib.LIB_PATH = os.path.abspath(os.environ['HV_LIB'])
from agrl.pytorch_b200.metrics.distance import PreparedOperand, compute_distance_matrix, distance_prepared

METRICS = ('euclidean', 'cosine')


def digest(t):
    return hashlib.sha256(t.contiguous().cpu().view(torch.uint8).numpy().tobytes()).hexdigest()


def operand_parts(op):
    """the bytes agrl_distance_prepare_operand_dev writes: planes, sumsq (euclidean), 1 / scale (fp16 x 2)"""
    k_pad = (op.dim + 63) // 64 * 64
    plane_b = _lib.planes_of_distance_split(op.split) * op.rows * k_pad * 2
    sumsq = (plane_b + 255) // 256 * 256
    unscale = (sumsq + 4 * op.rows + 255) // 256 * 256
    parts = [op.buf[:plane_b]]
    if op.metric == 'euclidean':
        parts.append(op.buf[sumsq:sumsq + 4 * op.rows])
    if op.split == _lib.SPLIT_FP16X2:
        parts.append(op.buf[unscale:unscale + 4 * op.rows])
    return torch.cat(parts)


def dump(dev):
    res = {}
    model = bench.make_model(dev, bench.make_head_weights())
    x1, x2, adj = bench.make_pool(882, dev, seed=1)
    g = torch.Generator(device=dev).manual_seed(2)
    masks = torch.randint(0, 1 << 56, (882, 3), generator=g, device=dev, dtype=torch.int64)
    for dname, dt in (('fp32', torch.float32), ('bf16', torch.bfloat16), ('fp16', torch.float16)):
        m1, m2 = (x1, x2) if dt == torch.float32 else (x1.to(dt), x2.to(dt))
        for split in (1, 2, 3, 4):
            for lr in (1, 0):
                for pair in ((1, 0) if split == 4 else (1,)):
                    model.head_split, model.head_lowrank, model.gemm_pair = split, bool(lr), bool(pair)
                    for gname, graph in (('dense', adj), ('masks', masks)):
                        for B in (882, 5):
                            with torch.no_grad():
                                out, nodes = model.head(m1[:B * bench.S], m2[:B * bench.S], graph[:B], bench.S,
                                                        return_nodes=True)
                            key = 'head/%s/split%d/lr%d/pair%d/%s/B%d' % (dname, split, lr, pair, gname, B)
                            res[key + '/out'], res[key + '/nodes'] = digest(out), digest(nodes)
                    res['prepared/split%d/lr%d/pair%d/%s' % (split, lr, pair, dname)] = digest(model._prep[dev][1])
        del m1, m2
    del x1, x2, adj
    torch.cuda.empty_cache()
    g = torch.Generator(device=dev).manual_seed(3)
    q = torch.randn(1980, 4096, generator=g, device=dev)
    x = torch.randn(9330, 4096, generator=g, device=dev) * torch.logspace(-3, 3, 9330, device=dev)[:, None]
    for split in (2, 3, 5):
        for metric in METRICS:
            key = 'distance/split%d/%s' % (split, metric)
            res[key] = digest(compute_distance_matrix(q, x, metric, split=split))
            qo, go = PreparedOperand(q, metric, split), PreparedOperand(x, metric, split)
            res[key + '/q_operand'], res[key + '/g_operand'] = digest(operand_parts(qo)), digest(operand_parts(go))
    lib = _lib.require_device()
    qf = torch.randn(10000, 512, generator=g, device=dev)
    gf = torch.randn(100000, 512, generator=g, device=dev)
    K = 100
    for split in (2, 3, 5):
        for metric in METRICS:
            qo, go = PreparedOperand(qf, metric, split), PreparedOperand(gf, metric, split)
            keys = torch.empty(10000, K, dtype=torch.int64, device=dev)
            status = torch.zeros(1, dtype=torch.int32, device=dev)
            wsb = lib.agrl_distance_topk_workspace_bytes(10000)
            ws = torch.empty(wsb, dtype=torch.uint8, device=dev)
            _lib.check(lib.agrl_distance_topk_dev(qo.buf.data_ptr(), 10000, go.buf.data_ptr(), 100000, 512,
                                                  _lib.METRIC_EUCLIDEAN if metric == 'euclidean' else _lib.METRIC_COSINE,
                                                  split, K, 0, keys.data_ptr(), status.data_ptr(), ws.data_ptr(), wsb,
                                                  torch.cuda.current_stream(dev).cuda_stream))
            res['topk/split%d/%s' % (split, metric)] = digest(keys) + '/status%d' % int(status.item())
    return res


def timed(fn, reps):
    for _ in range(2):
        fn()
    torch.cuda.synchronize()
    ms = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ms.append(e0.elapsed_time(e1))
    return sorted(ms)[len(ms) // 2]


def time_paths(dev):
    reps = int(os.environ.get('HV_REPS', '5'))
    model = bench.make_model(dev, bench.make_head_weights())
    pool = 882
    x1, x2, adj = bench.make_pool(pool, dev, seed=1)
    J, S = bench.NQ + bench.NG, bench.S
    feats = torch.empty(J, 2 * bench.C, device=dev)

    def head_pass():
        with torch.no_grad():
            for off in range(0, J, pool):
                n = min(pool, J - off)
                model.head(x1[:n * S], x2[:n * S], adj[:n], S, out=feats[off:off + n])
    head_ms = timed(head_pass, reps)
    g = torch.Generator(device=dev).manual_seed(3)
    q = torch.randn(bench.NQ, 4096, generator=g, device=dev)
    x = torch.randn(bench.NG, 4096, generator=g, device=dev)
    qo, go = PreparedOperand(q, 'euclidean', _lib.SPLIT_FP16X2), PreparedOperand(x, 'euclidean', _lib.SPLIT_FP16X2)
    out = torch.empty(bench.NQ, bench.NG, device=dev)

    def dist():
        for _ in range(20):
            distance_prepared(qo, go, out=out)
    dist_ms = timed(dist, reps) / 20
    return {'head_ms': round(head_ms, 3), 'distance_ms': round(dist_ms, 4)}


def main():
    dev = torch.device('cuda', 0)
    torch.cuda.set_device(dev)
    _lib.require_device()
    res = dump(dev) if sys.argv[1] == 'dump' else time_paths(dev)
    print(json.dumps(dict(res, lib=os.environ.get('HV_LIB', 'product'))), flush=True)


if __name__ == '__main__':
    main()
