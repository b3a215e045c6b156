"""Gallery-sharded k-reciprocal re-ranking + MARS ranking, one rank per GPU (NCCL), against the single-device sequence.

    python tools/rerank_sharded_bench.py [--nproc N] [--shape NQ,NG,DIM] [--reps R] [--out FILE]

Wall time per rank from resident features (rank 0's queries, the rank's gallery rows) to CMC/mAP:
evaluate_mars_sharded(re_rank=True), host clock around work that ends in a device synchronise, median and spread over
R passes after a warm-up pass.  A separate instrumented pass splits one run into the feature all-gather, the three
distance GEMM groups, phases A / B / C, the two exchanges and the ranking (synchronise at every boundary, so the
parts add up to more than the pipelined run).  Where N = NQ + NG fits one device (<= 46000) the same run times the
single-device sequence (three distance matrices, re_ranking_dev, evaluate_rank) and checks every rank's block
against it bit for bit.  Prints one JSON line (also written to FILE)."""
import argparse
import json
import os
import socket
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np
import torch
import torch.distributed as dist

from agrl.pytorch_b200 import _lib, metrics, sharded
from agrl.pytorch_b200 import synthetic as synth
from agrl.pytorch_b200.utils.re_ranking import re_ranking_dev


def gpu_conditions():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else torch.cuda.get_device_name()


def sync(world):
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()


def phase_split(ops, qf, gf_own, counts, rank, world, lab, k1=20, k2=6, lam=0.3, max_rank=50):
    """one instrumented pass of re_ranking_sharded + the ranking; seconds per part"""
    t = {}
    clock = [time.perf_counter()]

    def mark(name):
        sync(world)
        now = time.perf_counter()
        t[name] = t.get(name, 0.0) + now - clock[0]
        clock[0] = now
    qp, gp, qc, gc = lab
    nq, ng, n_own, offset = qf.shape[0], sum(counts), counts[rank], sum(counts[:rank])
    mark('start')
    gf_all = sharded._gather_shard_rows(gf_own, 0, counts, rank, None)
    mark('feature_allgather')
    qq = ops.distance(qf, qf, 'euclidean')
    mark('gemm_qq')
    qg = ops.distance(qf, gf_all, 'euclidean')
    mark('gemm_qg')
    width = max(1, sharded.RERANK_SLAB_BYTES // (4 * ng))

    def slabs():
        for s0 in range(0, n_own, width):
            mark('phase_a')                       # the rows call of the previous slab (or of the query rows)
            slab = ops.distance(gf_all, gf_own[s0:s0 + width], 'euclidean')
            mark('gemm_gg')
            yield s0, slab
    st, rank_rows = ops.rerank_rows(qg, qq, slabs(), offset, n_own, max(counts), k1, k2)
    mark('phase_a')
    rank_all = sharded._gather_shard_rows(rank_rows, nq, counts, rank, None)
    mark('exchange_rank')
    v = ops.rerank_expand(st, rank_all)
    mark('phase_b')
    v_all = [sharded._gather_shard_rows(x, nq, counts, rank, None) for x in v]
    mark('exchange_v')
    block = ops.rerank_finish(st, rank_all, v_all[0], v_all[1], v_all[2], lam)
    mark('phase_c')
    keys, cls, ngood, status = ops.partial(block, qp, gp, qc, gc, max_rank, offset)
    if world > 1:
        keys_all = torch.empty((world * nq, max_rank), dtype=keys.dtype, device=keys.device)
        cls_all = torch.empty((world * nq, max_rank), dtype=cls.dtype, device=cls.device)
        dist.all_gather_into_tensor(keys_all, keys)
        dist.all_gather_into_tensor(cls_all, cls)
        keys_all, cls_all = keys_all.view(world, nq, max_rank), cls_all.view(world, nq, max_rank)
        dist.all_reduce(ngood)
        sharded.or_across_ranks(status)
    else:
        keys_all, cls_all = keys.unsqueeze(0), cls.unsqueeze(0)
    ops.merge(keys_all, cls_all, ngood, max_rank, status)
    mark('ranking')
    del t['start']
    return {k: round(v * 1e3, 3) for k, v in t.items()}


def worker(rank, world, port, args, out):
    if world > 1:
        os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port))
        torch.cuda.set_device(rank)
        dist.init_process_group('nccl', rank=rank, world_size=world, device_id=torch.device('cuda', rank))
    dev = torch.device('cuda', torch.cuda.current_device())
    _lib.require_device()
    nq, ng, d = args.shape
    qp, qc, gp, gc = synth.eval_labels((nq, ng, 626, 6), seed=0)
    qf, gf = synth.eval_features(qp, gp, d, seed=0, clustered=True)
    bounds = sharded.shard_bounds(ng, world)
    counts = [hi - lo for lo, hi in bounds]
    lo, hi = bounds[rank]
    qf, gf_own = qf.to(dev), gf[lo:hi].to(dev).contiguous()
    lab = [torch.as_tensor(x).to(dev) for x in (qp, gp[lo:hi], qc, gc[lo:hi])]
    ops = sharded.CudaOps()

    def sharded_pass():
        return sharded.evaluate_mars_sharded(qf, gf_own, lab[0], lab[1], lab[2], lab[3], re_rank=True, ops=ops,
                                             gallery_counts=counts)
    cmc, mAP = sharded_pass()                                               # warm-up: modules, workspaces
    torch.cuda.reset_peak_memory_stats(dev)
    times = []
    for _ in range(args.reps):
        sync(world)
        t0 = time.perf_counter()
        sharded_pass()
        torch.cuda.synchronize()
        times.append(time.perf_counter() - t0)
    peak = torch.cuda.max_memory_allocated(dev)
    phases = phase_split(ops, qf, gf_own, counts, rank, world, lab)
    res = dict(rank=rank, times_ms=[round(x * 1e3, 3) for x in times], peak_gb=round(peak / 1e9, 3), phases_ms=phases,
               mAP=float(mAP), cmc1=float(cmc[0]))
    if nq + ng <= 46000:                                                    # the single-device sequence fits
        cdm = metrics.compute_distance_matrix
        qf_cpu, gf_all = qf, gf.to(dev)
        ref = re_ranking_dev(cdm(qf_cpu, gf_all), cdm(qf_cpu, qf_cpu), cdm(gf_all, gf_all))
        block = sharded.re_ranking_sharded(qf, gf_own, ops=ops, gallery_counts=counts)
        res['bit_identical'] = bool(torch.equal(block.view(torch.int32), ref[:, lo:hi].contiguous().view(torch.int32)))
        rcmc, rmAP = metrics.evaluate_rank(ref, qp, gp, qc, gc, use_metric_mars=True)
        res['metrics_identical'] = bool(np.array_equal(rcmc, cmc) and float(rmAP) == float(mAP))
        if rank == 0:
            single, rr_only = [], []
            for i in range(args.reps + 1):
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                qg = cdm(qf_cpu, gf_all)
                qq = cdm(qf_cpu, qf_cpu)
                gg = cdm(gf_all, gf_all)
                torch.cuda.synchronize()
                t1 = time.perf_counter()
                rr = re_ranking_dev(qg, qq, gg)
                torch.cuda.synchronize()
                t2 = time.perf_counter()
                metrics.evaluate_rank(rr, qp, gp, qc, gc, use_metric_mars=True)
                torch.cuda.synchronize()
                if i:                                                       # the first pass is the warm-up
                    single.append(time.perf_counter() - t0)
                    rr_only.append(t2 - t1)
            res['single_device_ms'] = [round(x * 1e3, 3) for x in single]
            res['single_device_rerank_only_ms'] = [round(x * 1e3, 3) for x in rr_only]
        del ref, gf_all
    if world > 1:
        allres = [None] * world
        dist.all_gather_object(allres, res)
        dist.destroy_process_group()
    else:
        allres = [res]
    if rank == 0:
        per_pass = [max(r['times_ms'][i] for r in allres) for i in range(args.reps)]      # the slowest rank ends a pass
        summary = dict(workload='rerank_sharded', shape=list(args.shape), gpus=world, gpu=gpu_conditions(),
                       reps=args.reps, wall_ms_median=float(np.median(per_pass)), wall_ms_min=min(per_pass),
                       wall_ms_max=max(per_pass), ranks=allres)
        if 'single_device_ms' in res:
            summary['single_device_ms_median'] = float(np.median(res['single_device_ms']))
            summary['single_device_rerank_only_ms_median'] = float(np.median(res['single_device_rerank_only_ms']))
        line = json.dumps(summary)
        print(line)
        if out:
            with open(out, 'a') as f:
                f.write(line + '\n')


def main():
    p = argparse.ArgumentParser()
    p.add_argument('--nproc', type=int, default=1)
    p.add_argument('--shape', default='1980,9330,4096')
    p.add_argument('--reps', type=int, default=10)
    p.add_argument('--out', default='')
    args = p.parse_args()
    args.shape = [int(x) for x in args.shape.split(',')]
    if torch.cuda.device_count() < args.nproc:
        raise SystemExit('needs %d GPUs, %d visible' % (args.nproc, torch.cuda.device_count()))
    if args.nproc == 1:
        worker(0, 1, 0, args, args.out)
        return
    s = socket.socket()
    s.bind(('127.0.0.1', 0))
    port = s.getsockname()[1]
    s.close()
    import torch.multiprocessing as mp
    mp.spawn(worker, args=(args.nproc, port, args, args.out), nprocs=args.nproc, join=True)


if __name__ == '__main__':
    main()
