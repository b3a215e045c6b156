#!/usr/bin/env python
"""bench.py -- the hot path on synthetic MARS-shaped data, one JSON line (see DESIGN.md, "Measurement").

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

Job (BASELINE.json metric "MARS-shape tracklets/s (graph head) + query x gallery eval ms"):
one STEP is a whole MARS-shaped test pass minus the stock backbone -- the graph head over
J = 1980 + 9330 = 11310 tracklets (8 frames, 2048 x 16 x 8 layer4 maps each, fed from a resident
pool that is larger than L2 and cycled), then the 1980 x 9330 distance matrix on the 4096-d
features the head just produced, then CMC/mAP (MARS metric, what the reference's test() calls).
`value` = J / step time with the maps resident in HBM; `eval_ms` carries the distance + ranking
part; `e2e` is the same job through the host-buffer API (maps, features, distance matrix and labels
all start in pinned host memory, results end on the host).  At N > 1 every rank runs the head on
its own J tracklets (no collective) and owns a 9330-row gallery shard of a N x 9330 gallery; the
per-query top-k / good counts are merged with NCCL (weak scaling).

Beside the contract keys the line carries (all measured outside the timed region of `value`):
  roofline         the WHOLE head against the HBM roofline as SURVEY 8(d) defines it, the dominant kernel's own figure,
  kernel_table     per kernel: ms, algorithmic bytes / flops, DRAM bytes (ncu), fraction of its bound,
  energy           NVML energy-counter deltas over the timed region (J per step / per tracklet),
  parity           a feature slice, a distance block and CMC/mAP of this very run checked against the oracle,
  call_size_curve  head time per tracklet at 5 ... 1024 tracklets per call,
  configs          the other BASELINE.json configurations: PRID2011 89 x 89 on one GPU, DukeMTMC-VideoReID 702 x 2636
                   cosine, MARS cosine, MARS with the market1501 metric -- gallery-sharded over the ranks -- and the
                   10 000 x 1 000 000 retrieval sweep (STRONG scaling: the one path that communicates).

`--impl reference` times the reference's CPU implementation of the same path on the host cores
(oracle/: torch-CPU restatement of head and distance, the reference's own compiled rank_cy and the
C restatement of evaluate_mars), on a bounded sample of the job, and prints the same line.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np
import torch

NQ, NG, NIDS, NCAMS = 1980, 9330, 626, 6
S, C, H, W = 8, 2048, 16, 8
V = 56
BYTES_PER_TRACKLET = 2 * S * C * H * W * 4 + 56 * 56 * 4 + 2 * C * 4        # SURVEY 8(d): 16 806 144
FLOPS_PER_TRACKLET = 2 * (2 * 56 * C * C + 2 * 2 * 56 * 56 * C)            # ~0.99 GFLOP
METRIC = 'MARS-shape tracklets/s (graph head) + query×gallery eval ms at 1/2/4/8 B200'
DIST_PRODUCTS = 3          # tensor-core products per distance (AGRL_SPLIT_FP16X2, the default of compute_distance_matrix)
WORKLOAD = ('MARS-shaped test pass: graph head over 11310 tracklets (8 frames, 2048x16x8 maps), 1980x9330 %s distance on '
            'the 4096-d features, MARS-metric CMC/mAP')


def peaks():
    try:
        p = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
        return dict(hbm_gbs=p['hbm_gbs'], bf16_tflops=p['bf16_tflops'], bf16_sustained=p['bf16_tflops_sustained'],
                    source='measured')
    except Exception:
        return dict(hbm_gbs=6650.0, bf16_tflops=1590.0, bf16_sustained=1400.0, source='fallback')


class ClockSampler(object):
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""
    Q = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,'
         'clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
         'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, index):
        self.index, self.proc, self.path = index, None, None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix='.csv')
            os.close(fd)
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.index), '--query-gpu=' + self.Q,
                                          '--format=csv,noheader,nounits', '-lms', '100'],
                                         stdout=open(self.path, 'w'), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = dict(sm_mhz=None, sm_max_mhz=None, reasons=[], samples=0)
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, smax, power, reasons = [], [], [], set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for line in open(self.path):
            f = [x.strip() for x in line.split(',')]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); smax.append(float(f[2]))
            except ValueError:
                continue
            try:
                power.append(float(f[3]))
            except ValueError:
                pass
            for n, v in zip(names, f[5:9]):
                if v.lower().startswith('active'):
                    reasons.add(n)
        os.unlink(self.path)
        if sm:
            out.update(sm_mhz=float(np.median(sm)), sm_max_mhz=float(max(smax)), reasons=sorted(reasons),
                       samples=len(sm), power_w=float(np.median(power)) if power else None)
        return out


class EnergyMeter(object):
    """Board energy from NVML's total-energy counter (millijoules since driver load): joules between start() and
    stop().  The counter ticks every few tens of milliseconds, so only regions of >= ~0.5 s are worth reading."""

    def __init__(self, index):
        self.h = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(self._physical_index(index))
        except Exception:
            self.h = None

    @staticmethod
    def _physical_index(index):
        vis = os.environ.get('CUDA_VISIBLE_DEVICES')
        if vis:
            ids = [v.strip() for v in vis.split(',') if v.strip()]
            if index < len(ids) and ids[index].isdigit():
                return int(ids[index])
        return index

    def read(self):
        if self.h is None:
            return None
        try:
            return self.nv.nvmlDeviceGetTotalEnergyConsumption(self.h) * 1e-3
        except Exception:
            return None

    def start(self):
        self.j0, self.t0 = self.read(), time.perf_counter()

    def stop(self):
        j1, t1 = self.read(), time.perf_counter()
        if self.j0 is None or j1 is None:
            return None
        return dict(joules=j1 - self.j0, seconds=t1 - self.t0)


# ------------------------------------------------------------------------------------------------
# synthetic job
# ------------------------------------------------------------------------------------------------
def make_labels(rank, world):
    from agrl.pytorch_b200 import synthetic as synth
    qp, qc, gp, gc = synth.eval_labels((NQ, NG, NIDS, NCAMS), seed=100 + rank)
    return qp, qc, gp, gc


def make_head_weights(seed=0):
    g = torch.Generator().manual_seed(seed)
    w = {}
    for name in ('global_bottleneck', 'att_bottleneck', 'graph_layers.0.bn', 'graph_layers.1.bn'):
        w[name + '.weight'] = 1.0 + 0.1 * torch.randn(C, generator=g)
        w[name + '.bias'] = 0.1 * torch.randn(C, generator=g)
        w[name + '.running_mean'] = 0.1 * torch.randn(C, generator=g)
        w[name + '.running_var'] = 0.5 + torch.rand(C, generator=g)
    for i in range(2):
        w['graph_layers.%d.linear.weight' % i] = 0.01 * torch.randn(C, C, generator=g)
    return w


def make_model(dev, weights):
    from agrl.pytorch_b200 import models
    m = models.init_model('vmgn', num_classes=625, loss={'xent', 'htri'}, last_stride=1, num_split=4, num_gb=2,
                          num_scale=1, pyramid_part=True, use_pose=True, learn_graph=True, pretrained=False)
    sd = m.state_dict()
    for k, v in weights.items():
        sd[k].copy_(v)
    # only the head's parameters are needed on the device (the backbone is not part of this path)
    for name in ('graph_layers', 'global_bottleneck', 'att_bottleneck'):
        getattr(m, name).to(dev)
    return m.eval()


def make_pool(n, dev, seed, pinned=False):
    """n tracklets of post-ReLU-like layer4 maps + a pose adjacency each; generated on the target."""
    shape = (n * S, C, H, W)
    if pinned:
        g = torch.Generator().manual_seed(seed)
        x1 = torch.empty(shape, pin_memory=True)
        x2 = torch.empty(shape, pin_memory=True)
        blk = 64 * S
        for i in range(0, n * S, blk):             # fill in blocks: keeps the transient small
            x1[i:i + blk] = torch.randn((min(blk, n * S - i), C, H, W), generator=g).clamp_(min=0)
            x2[i:i + blk] = torch.randn((min(blk, n * S - i), C, H, W), generator=g).clamp_(min=0)
    else:
        g = torch.Generator(device=dev).manual_seed(seed)
        x1 = torch.randn(shape, generator=g, device=dev).clamp_(min=0)
        x2 = torch.randn(shape, generator=g, device=dev).clamp_(min=0)
    from agrl.pytorch_b200 import synthetic as synth
    adj = synth.pose_adjacency(n, S, 7, seed=seed)
    adj = adj.pin_memory() if pinned else adj.to(dev)
    return x1, x2, adj


class Ctx(object):
    """Per-process state of the B200 arm: device, rank, collectives."""

    def __init__(self):
        import torch.distributed as dist
        self.dist = dist
        self.world = int(os.environ.get('WORLD_SIZE', '1'))
        self.rank = int(os.environ.get('RANK', '0'))
        self.local = int(os.environ.get('LOCAL_RANK', '0'))
        if self.world > 1:
            import datetime
            dist.init_process_group('nccl', device_id=torch.device('cuda', self.local),
                                    timeout=datetime.timedelta(seconds=180))
        self.dev = torch.device('cuda', self.local)
        torch.cuda.set_device(self.dev)
        self.stream = torch.cuda.current_stream(self.dev)

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        torch.cuda.synchronize(self.dev)

    def max_over_ranks(self, *vals):
        if self.world == 1:
            return [float(v) for v in vals]
        t = torch.tensor([float(v) for v in vals], device=self.dev, dtype=torch.float64)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return [float(v) for v in t.cpu()]

    def timed(self, fn, reps, warm=1):
        """ms per call of fn: CUDA events on the launching stream, barrier + synchronize on both sides, max over ranks."""
        for _ in range(warm):
            fn()
        self.barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(self.stream)
        for _ in range(reps):
            out = fn()
        b.record(self.stream)
        self.barrier()
        return self.max_over_ranks(a.elapsed_time(b) / reps)[0], out


# ------------------------------------------------------------------------------------------------
# B200 arm
# ------------------------------------------------------------------------------------------------
def run_b200(args):
    from agrl.pytorch_b200 import _lib, metrics, sharded
    cx = Ctx()
    dist, world, rank, dev, stream = cx.dist, cx.world, cx.rank, cx.dev, cx.stream
    _lib.require_device()
    pk = peaks()

    J, pool_n = NQ + NG, args.pool
    alloc_n = max(pool_n, 1024) if not args.no_curve else pool_n      # the call-size curve goes up to 1024 per call
    weights = make_head_weights()
    model = make_model(dev, weights)
    x1, x2, adj = make_pool(alloc_n, dev, seed=1 + rank)
    qp, qc, gp, gc = make_labels(rank, world)
    lab = [torch.as_tensor(a).to(dev) for a in (qp, gp, qc, gc)]
    feats = torch.empty(J, 2 * C, device=dev)
    chunks = [(o, min(pool_n, J - o)) for o in range(0, J, pool_n)]
    ev = lambda: torch.cuda.Event(enable_timing=True)

    def head_pass():
        for off, n in chunks:
            model.head(x1[:n * S], x2[:n * S], adj[:n], S, out=feats[off:off + n])

    def eval_pass(metric=args.dist_metric):
        if world == 1:
            d = metrics.compute_distance_matrix(feats[:NQ], feats[NQ:], metric)
            return metrics.evaluate_rank(d, lab[0], lab[1], lab[2], lab[3], use_metric_mars=True)
        return sharded.evaluate_mars_sharded(feats[:NQ], feats[NQ:], lab[0], lab[1], lab[2], lab[3],
                                             metric=metric, max_rank=50, gallery_counts=[NG] * world)

    with torch.no_grad():
        for _ in range(args.warmup):
            head_pass(); result = eval_pass()
        # ---- timed region: exactly K steps, device timed, max over ranks -------------------------
        sampler, energy = ClockSampler(cx.local), EnergyMeter(cx.local)
        if rank == 0:
            sampler.start()
        cx.barrier()
        launches0 = _lib.launch_count()
        energy.start()
        e0, e3 = ev(), ev()
        e0.record(stream)
        marks = []
        for _ in range(args.steps):
            a, b, c = ev(), ev(), ev()
            a.record(stream); head_pass(); b.record(stream); result = eval_pass(); c.record(stream)
            marks.append((a, b, c))
        e3.record(stream)
        cx.barrier()
        joules = energy.stop()
        total_ms = e0.elapsed_time(e3)
        launches = _lib.launch_count() - launches0
        clocks = sampler.stop() if rank == 0 else None
        head_ms = float(np.mean([a.elapsed_time(b) for a, b, c in marks]))
        eval_ms = float(np.mean([b.elapsed_time(c) for a, b, c in marks]))
        total_ms, head_ms, eval_ms = cx.max_over_ranks(total_ms, head_ms, eval_ms)
        ms_per_step = total_ms / args.steps
        value = world * J / (ms_per_step * 1e-3)
        if args.dump_outputs and rank == 0:
            dump_outputs(args.dump_outputs, feats, result)

        # ---- kernel timeline of one more step (CUDA events after every kernel, same stream) ------
        # (every rank runs the pass -- eval_pass holds collectives at N > 1 -- rank 0's timeline is reported)
        cx.barrier()
        with _lib.profile(stream.cuda_stream) as prof:
            head_pass(); eval_pass()
        timeline = prof.totals()
        cx.barrier()

        # ---- parity of THIS run's outputs against the oracle (the checker; never inside a timed region) ----------
        parity = None
        if not args.no_parity and rank == 0:
            parity = guarded(lambda: parity_block(args, model, weights, x1, x2, adj, feats, (qp, qc, gp, gc), result, world))
        cx.barrier()

        # ---- head energy alone: enough passes for the NVML counter (reported per pass) --------------------------
        head_energy = None
        if not args.no_energy:
            head_energy = guarded(lambda: energy_of(cx, head_pass, min_seconds=1.0))

        # ---- the same head pass with the opt-in single-plane fp16 graph-layer GEMM (reported beside, not as `value`) --
        fast = None
        if not args.no_fast_mode:
            default_split = model.head_split

            def fast_mode():
                model.head_split = _lib.SPLIT_FP16X1
                try:
                    ms, _ = cx.timed(head_pass, args.steps, warm=2)
                    with _lib.profile(stream.cuda_stream) as fprof:
                        head_pass()
                    return dict(head_ms=ms, kernels={k: round(t, 4) for k, (n, t) in fprof.totals().items()})
                finally:
                    model.head_split = default_split
            fast = guarded(fast_mode)
            head_pass()                                  # features of the default mode again
            cx.barrier()

        # ---- head time per tracklet against the call size (reference default --test-batch 5 ... 1024) ----------
        curve = None
        if not args.no_curve:
            curve = guarded(lambda: call_size_curve(cx, model, x1, x2, adj, alloc_n))
        cx.barrier()

        # ---- same-box comparator: the reference's module code in stock PyTorch on this GPU (rank 0) ----
        eager = None
        if not args.no_eager and rank == 0:
            eager = guarded(lambda: torch_eager_gpu(args, dev, weights, x1, x2, adj, feats))
            torch.cuda.empty_cache()
        cx.barrier()
        del x1, x2
        torch.cuda.empty_cache()

        # ---- the other BASELINE.json configurations (outside `value`; every rank takes part) -----------------
        configs = None
        if not args.no_configs:
            configs = run_configs(args, cx, model, pool_n)
        cx.barrier()

        # ---- end to end through host buffers -------------------------------------------------
        e2e = None
        if not args.no_e2e:
            e2e = run_e2e(args, model, dev, rank, world, (qp, qc, gp, gc))

    if world > 1:
        dist.barrier()
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    lowrank_on = bool(getattr(model, 'head_lowrank', True))
    passes = {1: 1.0, 2: 3.0, 3: 6.0, 4: 2.0}.get(int(getattr(model, 'head_split', 4)), 2.0)
    table, head_dram = kernel_table(timeline, pk, J, lowrank_on, passes)
    top = max(timeline.items(), key=lambda kv: kv[1][1])[0]
    head_gbs = J * BYTES_PER_TRACKLET / (head_ms * 1e-3) / 1e9
    # `roofline`: the WHOLE head as SURVEY 8(d) defines it -- algorithmic bytes per tracklet (both maps, the pose graph,
    # the output) x tracklets / head time against the measured HBM copy peak.  `traffic` = DRAM bytes of all head kernels
    # per step from the committed ncu --set full capture (profiles/traffic.json), scaled to this run's tracklets.
    roof = dict(scope='whole graph head per step (pool + graph + gemm_graph_layer + graph_mix + attn), SURVEY 8(d)', bound='hbm',
                achieved=head_gbs, peak=pk['hbm_gbs'], unit='GB/s', frac=head_gbs / pk['hbm_gbs'], traffic=head_dram,
                algorithmic_bytes_per_step=J * BYTES_PER_TRACKLET, peak_source=pk['source'],
                dominant_kernel=dict(kernel=top, **{k: table[top][k] for k in ('bound', 'achieved', 'peak', 'unit', 'frac',
                                                                               'launches', 'avg_launch_ms')}))
    gemm_d = timeline.get('gemm_distance', (1, float('nan')))[1]
    line = {
        'metric': METRIC, 'value': value, 'unit': 'tracklets/s', 'n_gpus': world, 'steps': args.steps,
        'warmup': args.warmup, 'ms_per_step': ms_per_step, 'higher_is_better': True, 'scaling': 'weak',
        'vs_baseline': None, 'dtype': 'fp32 (head GEMMs: fp16 + e4m3 correction planes, distance: fp16x2 planes / 3 products, on tcgen05; fp32 accumulate)',
        'data': 'synthetic',
        'config': {'workload': WORKLOAD % args.dist_metric,
                   'tracklets_per_step_per_gpu': J, 'pool_tracklets': pool_n,
                   'head': 'bulk-copy pooling (TMA ring), graph layers on tcgen05 (graph_kernel_tc + split GEMM: fp16 product + one K-concatenated e4m3 correction product; '
                           'first layer on the 32 quarter-strip rows per tracklet); knobs %s' % (
                       {k: getattr(model, k, None) for k in ('head_split', 'head_lowrank', 'pool_tma', 'pool_stages', 'pool_l2_hint')},),
                   'cache': 'input pool %.1f GB per GPU, larger than L2; cycled' % (pool_n * BYTES_PER_TRACKLET / 1e9),
                   'parallelism': 'independent head shards + gallery-sharded eval (NCCL merge)' if world > 1 else 'single GPU'},
        'head_ms': head_ms, 'eval_ms': eval_ms,
        'head_tracklets_per_s_per_gpu': J / (head_ms * 1e-3),
        'roofline': roof, 'kernel_table': table, 'gpu_launches': int(launches),
        'distance': {'ms': gemm_d, 'algorithmic_tflops': 2 * NQ * NG * 2 * C / (gemm_d * 1e-3) / 1e12,
                     'products': DIST_PRODUCTS,
                     'tensor_pipe_frac': DIST_PRODUCTS * 2 * NQ * NG * 2 * C / (gemm_d * 1e-3) / 1e12 / pk['bf16_sustained']},
        'clocks': clocks, 'result': {'mAP': float(result[1]), 'rank1': float(result[0][0])},
    }
    if joules is not None:
        line['energy'] = {'j_per_step': joules['joules'] / args.steps, 'avg_power_w': joules['joules'] / joules['seconds'],
                          'j_per_tracklet': joules['joules'] / args.steps / J,
                          'source': 'nvmlDeviceGetTotalEnergyConsumption deltas around the timed region (rank 0 GPU)',
                          'head_only': head_energy}
    if parity is not None:
        line['parity'] = parity
    if fast is not None:
        if 'head_ms' in fast:
            fgbs = J * BYTES_PER_TRACKLET / (fast['head_ms'] * 1e-3) / 1e9
            fast = {'what': 'opt-in head_split=1: ONE fp16 plane per GEMM operand, pow2-scaled per tracklet / per layer (TF32-class, '
                            '11 significant bits); head error vs the reference 1e-5 norm-relative / 3e-5 max-scaled (bar 1e-4, '
                            'tests/test_gpu_head.py); NOT the configuration `value` is measured in',
                    'head_ms': fast['head_ms'], 'head_tracklets_per_s_per_gpu': J / (fast['head_ms'] * 1e-3),
                    'head_hbm_frac': fgbs / pk['hbm_gbs'], 'kernels_ms': fast['kernels']}
        line['fast_mode'] = fast
    if curve is not None:
        line['call_size_curve'] = curve
    if configs is not None:
        line['configs'] = configs
    if eager is not None:
        if 'head_ms_per_pass' in eager:
            eager['b200_head_speedup'] = eager['head_ms_per_pass'] / head_ms
            eager['b200_distance_speedup'] = eager['distance_ms'] / gemm_d
        line['torch_eager_gpu'] = eager
    if e2e is not None:
        line['e2e'] = e2e
    if not args.no_cpu_baseline:
        line['cpu_baseline'] = cpu_reference(args, steps=1, warmup=0)['cpu_baseline']
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


DUMP_FEATURE_ROWS = 2048        # 2048 x 4096 fp32 = 32 MB of the 11310-row feature matrix (185 MB in full)


def dump_outputs(out_dir, feats, result):
    """What the last timed step handed its caller, as .npy files that two builds can be compared on: `features`, a fixed
    seeded sample of the head's feature rows in ascending row order (float32), and the evaluation's `cmc` and `mAP`
    (float64)."""
    os.makedirs(out_dir, exist_ok=True)
    n = min(DUMP_FEATURE_ROWS, feats.shape[0])
    rows = np.sort(np.random.RandomState(0).choice(feats.shape[0], n, replace=False))
    sample = feats[torch.as_tensor(rows, device=feats.device)].cpu().numpy().astype(np.float32)
    np.save(os.path.join(out_dir, 'features.npy'), sample)
    np.save(os.path.join(out_dir, 'cmc.npy'), np.asarray(result[0], dtype=np.float64))
    np.save(os.path.join(out_dir, 'mAP.npy'), np.asarray(result[1], dtype=np.float64))


def guarded(fn):
    """An extra figure must never cost the bench line: failures are reported as `unavailable`."""
    try:
        return fn()
    except Exception as exc:
        return {'unavailable': '%s: %s' % (type(exc).__name__, exc)}


def energy_of(cx, fn, min_seconds=1.0):
    """Joules per call of fn on this rank's GPU: fn repeated for >= min_seconds between two NVML counter reads."""
    m = EnergyMeter(cx.local)
    if m.h is None:
        return {'unavailable': 'NVML energy counter not readable'}
    fn(); torch.cuda.synchronize(cx.dev)
    t0 = time.perf_counter(); fn(); torch.cuda.synchronize(cx.dev)
    reps = max(3, int(min_seconds / max(time.perf_counter() - t0, 1e-4)))
    time.sleep(0.15)                                   # let the counter settle on the idle board
    m.start()
    for _ in range(reps):
        fn()
    torch.cuda.synchronize(cx.dev)
    r = m.stop()
    return {'j_per_pass': r['joules'] / reps, 'avg_power_w': r['joules'] / r['seconds'], 'passes': reps,
            'ms_per_pass_wall': r['seconds'] / reps * 1e3}


def kernel_table(timeline, pk, J, lowrank_on, gemm_passes=2.0):
    """Per kernel of one step: launches, ms, share, what bounds it, algorithmic bytes or flops per step, achieved rate,
    the peak it is held against and the fraction; `dram_bytes` per step from profiles/traffic.json (ncu --set full,
    dram__bytes_read.sum + dram__bytes_write.sum per launch, scaled by units).  Returns (table, head DRAM bytes)."""
    node_b = V * C * 4                                   # one (V, C) fp32 node tensor: 458 752 B
    q_b = 32 * C * 4
    rows1 = 32 if lowrank_on else V                      # GEMM rows per tracklet in the first layer
    algo = {
        'pool': ('hbm', J * (2 * S * C * H * W * 4 + node_b + C * 4)),
        # read X once, write the operand planes (2 planes x 2 B): layer 1 writes the 32 quarter rows when low-rank
        'graph': ('hbm', J * ((node_b + (q_b if lowrank_on else node_b)) + 2 * node_b)),
        # tensor time in bf16-pass equivalents: 3 for the bf16x2 split, 2 for fp16 + e4m3 (the 8-bit product covers both
        # corrections at twice the rate), 1 for the fp16 plane, 6 for bf16x3
        'gemm_graph_layer': ('tensor', gemm_passes * 2.0 * J * (rows1 + V) * C * C),
        'graph_mix': ('hbm', J * (2 * node_b + q_b)),
        'attn': ('hbm', J * node_b),
        'split_planes': ('hbm', (NQ + NG) * 2 * C * (4 + 4)),
        'gemm_distance': ('tensor', DIST_PRODUCTS * 2.0 * NQ * NG * 2 * C),
        'rank_mars': ('hbm', NQ * NG * 4),
        'rank_mars_partial': ('hbm', NQ * NG * 4),
    }
    try:
        traffic = json.load(open(os.path.join(ROOT, 'profiles', 'traffic.json')))
    except Exception:
        traffic = {}
    step_ms = sum(t for _, t in timeline.values())
    table, head_dram = {}, 0.0
    for k, (n, t) in sorted(timeline.items(), key=lambda kv: -kv[1][1]):
        row = dict(launches=n, ms=round(t, 4), share=round(t / step_ms, 4), avg_launch_ms=t / n)
        if k in algo:
            bound, work = algo[k]
            if bound == 'hbm':
                row.update(bound='hbm', algorithmic_bytes=work, achieved=work / (t * 1e-3) / 1e9, peak=pk['hbm_gbs'], unit='GB/s')
            else:
                row.update(bound='tensor', bf16_flops_issued=work, achieved=work / (t * 1e-3) / 1e12, peak=pk['bf16_sustained'],
                           unit='TFLOP/s')
            row['frac'] = row['achieved'] / row['peak']
        else:
            row.update(bound=None, achieved=None, peak=None, unit=None, frac=None)
        tr = traffic.get(k)
        if tr and 'dram_bytes_per_call' in tr:           # all launches of this name in one head call, summed
            row['dram_bytes'] = tr['dram_bytes_per_call'] / tr['units_per_call'] * (J if tr['unit'] == 'tracklet' else 1)
        elif tr:                                         # round-1 format: one launch
            calls = timeline.get('pool', (n, 0))[0]
            row['dram_bytes'] = tr['dram_bytes_per_launch'] / tr['units_per_launch'] * (
                J * n / max(calls, 1) if tr['unit'] == 'tracklet' else 1)
        else:
            row['dram_bytes'] = None
        if tr and tr['unit'] == 'tracklet':
            head_dram += row['dram_bytes']
        table[k] = row
    return table, (head_dram or None)


def parity_block(args, model, weights, x1, x2, adj, feats, labels, result, world):
    """Outputs of this very run against the oracle (test infrastructure, used here as the checker only): 16 tracklets of
    the feature matrix the timed head passes produced, a block of the distance matrix, and -- one GPU -- CMC/mAP."""
    from oracle import head as ohead, distance as odist, rank as orank
    from agrl.pytorch_b200 import metrics
    n_pool = min(args.pool, x1.shape[0] // S)
    idx = np.unique(np.linspace(0, n_pool - 1, 16).round().astype(np.int64))
    fr = torch.as_tensor((idx[:, None] * S + np.arange(S)[None]).reshape(-1), device=x1.device)
    ref = ohead.head_forward(x1[fr].cpu(), x2[fr].cpu(), adj[torch.as_tensor(idx, device=adj.device)].cpu(), weights,
                             dtype=torch.float64)
    got = feats[torch.as_tensor(idx, device=feats.device)].cpu().double()
    out = {'head_features': {'tracklets_checked': int(len(idx)), 'max_scaled_err': float((got - ref).abs().max() / ref.abs().max()),
                             'norm_rel_err': float((got - ref).norm() / ref.norm()), 'bar': 1e-4,
                             'oracle': 'oracle/head.py fp64 (vmgn.py:296-321)'}}
    qb, gb = feats[:256], feats[NQ:NQ + 512]
    d = metrics.compute_distance_matrix(qb, gb, args.dist_metric).cpu().double()
    ref = odist.distance_matrix(qb.cpu(), gb.cpu(), args.dist_metric, dtype=torch.float64)
    scale = float((qb.double() ** 2).sum(1).max() + (gb.double() ** 2).sum(1).max()) if args.dist_metric == 'euclidean' else 1.0
    out['distance'] = {'block': '256x512x4096', 'max_err_over_norm_scale': float((d - ref).abs().max()) / scale, 'bar': 1e-4,
                       'oracle': 'oracle/distance.py fp64 (distance.py:59-89)'}
    if world == 1:
        qp, qc, gp, gc = labels
        dm = metrics.compute_distance_matrix(feats[:NQ], feats[NQ:], args.dist_metric).cpu().numpy()
        rcmc, rmap = orank.mars_port(dm, qp, gp, qc, gc, 50)
        out['rank'] = {'cmc_bit_exact': bool(np.array_equal(np.asarray(result[0]), rcmc)), 'mAP_bit_exact': bool(result[1] == rmap),
                       'mAP': float(result[1]), 'oracle_mAP': float(rmap),
                       'oracle': 'oracle/rank_oracle.c evaluate_mars restatement (rank.py:160-212) on this run\'s GPU distance matrix'}
    out['ok'] = bool(out['head_features']['max_scaled_err'] < 1e-4 and out['head_features']['norm_rel_err'] < 1e-4 and
                     out['distance']['max_err_over_norm_scale'] < 1e-4 and
                     (world != 1 or (out['rank']['cmc_bit_exact'] and out['rank']['mAP_bit_exact'])))
    return out


def call_size_curve(cx, model, x1, x2, adj, alloc_n):
    """Head time per tracklet at B tracklets per call.  Small calls rotate through the resident pool so that their maps
    are never L2-resident.  Rank 0 times; no collective inside."""
    out = {'note': 'us per tracklet of model.head at B tracklets per call, maps cycled through a %.1f GB pool (> L2)'
                   % (alloc_n * BYTES_PER_TRACKLET / 1e9), 'points': []}
    if cx.rank != 0:
        return None
    best = None
    for B in (5, 16, 64, 128, 256, 512, 882, 1024):
        if B > alloc_n:
            continue
        starts = list(range(0, alloc_n - B + 1, B)) or [0]
        reps = max(3, min(200, int(1500 / B) + 1))
        feats = torch.empty(B, 2 * C, device=cx.dev)

        def once(i):
            o = starts[i % len(starts)]
            model.head(x1[o * S:(o + B) * S], x2[o * S:(o + B) * S], adj[o:o + B], S, out=feats)
        for i in range(3):
            once(i)
        torch.cuda.synchronize(cx.dev)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(cx.stream)
        for i in range(reps):
            once(i)
        b.record(cx.stream)
        torch.cuda.synchronize(cx.dev)
        ms = a.elapsed_time(b) / reps
        t0 = time.perf_counter()
        for i in range(reps):
            once(i)
        host_ms = (time.perf_counter() - t0) / reps * 1e3       # launch path of one call (host side, not waiting)
        torch.cuda.synchronize(cx.dev)
        us = ms * 1e3 / B
        best = us if best is None else min(best, us)
        out['points'].append({'tracklets_per_call': B, 'ms_per_call': ms, 'us_per_tracklet': us, 'host_ms_per_call': host_ms})
    for p in out['points']:
        p['vs_best'] = p['us_per_tracklet'] / best
    return out


# ------------------------------------------------------------------------------------------------
# the other BASELINE.json configurations
# ------------------------------------------------------------------------------------------------
def run_configs(args, cx, model, pool_n):
    """PRID2011 (config 2, one GPU), DukeMTMC-VideoReID cosine (config 4), MARS cosine, MARS + market1501 metric -- the
    gallery sharded over the ranks (STRONG scaling) -- and the 10k x 1M retrieval sweep (config 5).  Features are synthetic
    (clustered, seed fixed); every figure is CUDA-event time, barrier + synchronize both sides, max over ranks."""
    from agrl.pytorch_b200 import metrics, sharded, synthetic as synth
    out = {}
    dev, world, rank = cx.dev, cx.world, cx.rank

    def eval_config(name, nq, ng, nid, ncam, metric, rank_metric, seed, reps=5, dim=2 * C):
        qp, qc, gp, gc = synth.eval_labels((nq, ng, nid, ncam), seed=seed)
        qf, gf = synth.eval_features(qp, gp, dim, seed=seed, clustered=True, num_ids=nid)
        lo, hi = sharded.shard_bounds(ng, world)[rank]
        qf, gfl = qf.to(dev), gf[lo:hi].to(dev)
        qpd, qcd = torch.as_tensor(qp).to(dev), torch.as_tensor(qc).to(dev)
        gpl, gcl = torch.as_tensor(gp[lo:hi]).to(dev), torch.as_tensor(gc[lo:hi]).to(dev)

        def once():
            if world == 1:
                d = metrics.compute_distance_matrix(qf, gfl, metric)
                return metrics.evaluate_rank(d, qpd, gpl, qcd, gcl, **{rank_metric: True})
            fn = sharded.evaluate_mars_sharded if rank_metric == 'use_metric_mars' else sharded.evaluate_market1501_sharded
            return fn(qf, gfl, qpd, gpl, qcd, gcl, metric=metric, max_rank=50, broadcast_queries=False)
        ms, res = cx.timed(once, reps, warm=2)
        return {'queries': nq, 'gallery': ng, 'dim': dim, 'distance': metric, 'rank_metric': rank_metric[len('use_metric_'):],
                'eval_ms': ms, 'gallery_rows_this_rank': hi - lo, 'scaling': 'strong (gallery rows sharded, NCCL merge)' if world > 1 else 'single GPU',
                'mAP': float(res[1]), 'rank1': float(res[0][0])}

    # config 2: PRID2011-shaped test on ONE B200 (rank 0 alone, no collective): head over 178 tracklets + eval
    def prid():
        if rank != 0:
            return None
        n = 89 + 89
        x1, x2, adj = make_pool(n, dev, seed=21)
        feats = torch.empty(n, 2 * C, device=dev)
        qp, qc, gp, gc = synth.eval_labels('prid2011', seed=22)
        lab = [torch.as_tensor(a).to(dev) for a in (qp, gp, qc, gc)]
        st = cx.stream

        def once():
            model.head(x1, x2, adj, S, out=feats)
            d = metrics.compute_distance_matrix(feats[:89], feats[89:], 'euclidean')
            return metrics.evaluate_rank(d, lab[0], lab[1], lab[2], lab[3], use_metric_mars=True)
        for _ in range(3):
            res = once()
        torch.cuda.synchronize(dev)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(st)
        for _ in range(10):
            res = once()
        b.record(st)
        torch.cuda.synchronize(dev)
        ms = a.elapsed_time(b) / 10
        return {'what': 'head over 89 + 89 tracklets -> 89x89 euclidean distance -> MARS-metric CMC/mAP, one GPU, one call each '
                        '(the evaluate_rank result is read back every iteration)', 'ms_per_pass': ms,
                'tracklets_per_s': n / (ms * 1e-3), 'mAP': float(res[1]), 'note': 'maps 3.0 GB > L2'}
    out['prid2011'] = guarded(prid)
    cx.barrier()
    out['dukev_cosine'] = eval_config('dukev', 702, 2636, 702, 8, 'cosine', 'use_metric_mars', seed=23)
    out['mars_cosine'] = eval_config('mars', NQ, NG, NIDS, NCAMS, 'cosine', 'use_metric_mars', seed=24)
    out['mars_euclidean_market1501_metric'] = eval_config('mars', NQ, NG, NIDS, NCAMS, 'euclidean', 'use_metric_market1501', seed=25)
    # BASELINE.json quotes the MARS configuration at d = 2048 (VMGN's eval feature is 4096 wide: SURVEY 8a A8)
    out['mars_euclidean_d2048'] = eval_config('mars', NQ, NG, NIDS, NCAMS, 'euclidean', 'use_metric_mars', seed=26, dim=C)
    if not args.no_sweep:
        torch.cuda.empty_cache()
        out['sweep'] = sweep_measure(args, cx, steps=3, warm=1)
        torch.cuda.empty_cache()
    return out


def sweep_measure(args, cx, steps, warm):
    """Scaled retrieval sweep (BASELINE.json config 5): 10 000 queries x 1 000 000 gallery features (d = 2048), gallery
    rows sharded over the ranks (STRONG scaling), MARS-metric top-50 merged over NCCL.  One step = split the gallery
    shard into operand planes, distance on tcgen05 with the per-shard top-k, one all-gather / all-reduce, the merge."""
    from agrl.pytorch_b200 import _lib, sharded
    from agrl.pytorch_b200.metrics.distance import PreparedOperand, distance_prepared
    dist, world, rank, dev, stream = cx.dist, cx.world, cx.rank, cx.dev, cx.stream
    nq, ng_total, d, K, qchunk = args.sweep_queries, args.sweep_gallery, 2048, 50, 2000
    lo, hi = sharded.shard_bounds(ng_total, world)[rank]
    ng = hi - lo
    g = torch.Generator(device=dev).manual_seed(5)
    qf = torch.randn(nq, d, generator=g, device=dev)                       # same on every rank (same seed)
    g2 = torch.Generator(device=dev).manual_seed(50 + rank)
    gf = torch.randn(ng, d, generator=g2, device=dev)
    nid = max(ng_total // 20, 2)
    qp = torch.randint(0, nid, (nq,), generator=g, device=dev)
    qc = torch.randint(0, 6, (nq,), generator=g, device=dev)
    gp = torch.randint(0, nid, (ng,), generator=g2, device=dev)
    gc = torch.randint(0, 6, (ng,), generator=g2, device=dev)
    if rank == 0:                                                          # every query has a cross-camera match
        n0 = min(nq, ng)
        gp[:n0] = qp[:n0]; gc[:n0] = (qc[:n0] + 1) % 6
    ops = sharded.CudaOps()
    fused = hasattr(ops, 'topk_fused') and not args.sweep_unfused
    keys = torch.empty(nq, K, dtype=torch.int64, device=dev)
    cls = torch.empty(nq, K, dtype=torch.uint8, device=dev)
    ngood = torch.empty(nq, dtype=torch.int32, device=dev)
    dbuf = None if fused else torch.empty(min(qchunk, nq), ng, device=dev)

    def step():
        gop = PreparedOperand(gf, args.dist_metric)
        if fused:
            qop = PreparedOperand(qf, args.dist_metric)
            k, c, n, st = ops.topk_fused(qop, gop, qp, gp, qc, gc, K, lo)
            keys.copy_(k); cls.copy_(c); ngood.copy_(n)
        else:
            st = None
            for q0 in range(0, nq, qchunk):
                q1 = min(nq, q0 + qchunk)
                qop = PreparedOperand(qf[q0:q1], args.dist_metric)
                dm = distance_prepared(qop, gop, out=dbuf[:q1 - q0])
                k, c, n, st = ops.partial(dm, qp[q0:q1], gp, qc[q0:q1], gc, K, lo)
                keys[q0:q1], cls[q0:q1], ngood[q0:q1] = k, c, n
        if world > 1:
            ka = torch.empty(world * nq, K, dtype=keys.dtype, device=dev)
            ca = torch.empty(world * nq, K, dtype=cls.dtype, device=dev)
            dist.all_gather_into_tensor(ka, keys); dist.all_gather_into_tensor(ca, cls)
            nall = ngood.clone(); dist.all_reduce(nall); sharded.or_across_ranks(st)
            return ops.merge(ka.view(world, nq, K), ca.view(world, nq, K), nall, K, st)
        return ops.merge(keys.unsqueeze(0), cls.unsqueeze(0), ngood, K, st)

    ms, res = cx.timed(step, steps, warm=max(1, warm))
    with _lib.profile(stream.cuda_stream) as prof:
        step()
    tl = prof.totals()
    cx.barrier()
    pk = peaks()
    flops = 2.0 * nq * ng_total * d
    gemm_ms = sum(t for k, (n, t) in tl.items() if k.startswith('gemm_distance'))
    kern = {k: dict(launches=n, ms=round(t, 3)) for k, (n, t) in sorted(tl.items(), key=lambda kv: -kv[1][1])}
    other = sorted(((k, t) for k, (n, t) in tl.items() if not k.startswith('gemm_distance')), key=lambda kv: -kv[1])
    return {'what': 'retrieval sweep, gallery rows sharded over the ranks (STRONG scaling), MARS-metric top-50 merged with NCCL; '
                    + ('distance -> top-k fused in the GEMM epilogue (no num_q x num_g matrix)' if fused else
                       'distance blocks of 2000 queries written to HBM and re-read by the top-k kernel'),
            'ms': ms, 'queries': nq, 'gallery': ng_total, 'dim': d, 'gallery_rows_per_gpu': ng, 'distance': args.dist_metric,
            'algorithmic_tflops_per_gpu': flops / world / (ms * 1e-3) / 1e12,
            'gemm_ms_rank0': gemm_ms, 'gemm_share': gemm_ms / max(sum(t for _, (n, t) in tl.items()), 1e-9),
            'gemm_tensor_pipe_frac': DIST_PRODUCTS * flops / world / (max(gemm_ms, 1e-9) * 1e-3) / 1e12 / pk['bf16_sustained'],
            'limiter': 'the tcgen05 distance GEMM (fp16 x 2 operands, 3 products); largest other kernel on rank 0: %s %.2f ms' % (
                other[0] if other else ('-', 0.0)),
            'kernels_rank0': kern, 'mAP': float(res[1]), 'rank1': float(res[0][0])}


def run_sweep(args):
    """`--workload sweep`: the retrieval sweep as the line's own metric (strong scaling over --gpus)."""
    from agrl.pytorch_b200 import _lib
    cx = Ctx()
    _lib.require_device()
    r = sweep_measure(args, cx, steps=args.steps, warm=args.warmup)
    if cx.rank == 0:
        print(json.dumps({
            'metric': 'scaled retrieval sweep: %d queries x %d gallery eval ms' % (r['queries'], r['gallery']), 'value': r['ms'],
            'unit': 'ms', 'n_gpus': cx.world, 'steps': args.steps, 'warmup': max(1, args.warmup), 'ms_per_step': r['ms'],
            'higher_is_better': False, 'scaling': 'strong', 'vs_baseline': None, 'data': 'synthetic',
            'dtype': 'fp32 (fp16x2 split operands, 3 products, on tcgen05; fp32 accumulate)',
            'config': {'workload': r['what'], 'queries': r['queries'], 'gallery': r['gallery'], 'dim': r['dim'],
                       'gallery_rows_per_gpu': r['gallery_rows_per_gpu'], 'metric': r['distance']},
            'algorithmic_tflops_per_gpu': r['algorithmic_tflops_per_gpu'], 'gemm_ms_rank0': r['gemm_ms_rank0'],
            'gemm_tensor_pipe_frac': r['gemm_tensor_pipe_frac'], 'kernels': r['kernels_rank0'], 'limiter': r['limiter'],
            'result': {'mAP': r['mAP'], 'rank1': r['rank1']}}))
    if cx.world > 1:
        cx.dist.destroy_process_group()


def h2d_ceiling(dev, nbytes=1 << 30, reps=3):
    """bandwidthTest-style pinned host -> device copy rate of this rank (GB/s), all ranks copying at the same time."""
    src = torch.empty(nbytes, dtype=torch.uint8, pin_memory=True)
    dst = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    dst.copy_(src, non_blocking=True)
    torch.cuda.synchronize(dev)
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        dst.copy_(src, non_blocking=True)
    b.record()
    torch.cuda.synchronize(dev)
    return nbytes * reps / (a.elapsed_time(b) * 1e-3) / 1e9


def run_e2e(args, model, dev, rank, world, labels):
    """Same job through the host-facing API: maps in pinned host memory, H2D chunk by chunk on two copy
    streams (one per map, double buffered against the head), features back to the host, then the reference's own
    call sequence compute_distance_matrix(CPU tensors) -> .numpy() -> evaluate_rank(numpy)
    (train_vidreid_xent_htri.py:477-531)."""
    import torch.distributed as dist
    from agrl.pytorch_b200 import metrics
    J, n_host, chunk = NQ + NG, args.e2e_pool, args.e2e_chunk
    hx1, hx2, hadj = make_pool(n_host, dev, seed=7 + rank, pinned=True)
    qp, qc, gp, gc = labels
    bufs = [(torch.empty(chunk * S, C, H, W, device=dev), torch.empty(chunk * S, C, H, W, device=dev),
             torch.empty(chunk, 56, 56, device=dev)) for _ in range(2)]
    feats_host = torch.empty(J, 2 * C, pin_memory=True)
    copy1, copy2 = torch.cuda.Stream(dev), torch.cuda.Stream(dev)
    main = torch.cuda.current_stream(dev)
    chunks = [(o, min(chunk, J - o)) for o in range(0, J, chunk)]
    maps_adj = J * (2 * S * C * H * W * 4 + 56 * 56 * 4)
    h2d = maps_adj + J * 2 * C * 4 + NQ * NG * 4 + (NQ + NG) * 16            # maps + adj, features, distmat, labels
    d2h = J * 2 * C * 4 + NQ * NG * 4 + 51 * 8
    if world > 1:
        dist.barrier()
    ceiling = h2d_ceiling(dev)                                              # every rank copies concurrently

    def one_step():
        ready = [(torch.cuda.Event(), torch.cuda.Event()) for _ in chunks]
        freed = [torch.cuda.Event() for _ in chunks]
        for i, (off, n) in enumerate(chunks):
            b1, b2, ba = bufs[i % 2]
            src = (off % n_host)
            if src + n > n_host:
                src = 0
            with torch.cuda.stream(copy1):
                if i >= 2:
                    copy1.wait_event(freed[i - 2])
                b1[:n * S].copy_(hx1[src * S:(src + n) * S], non_blocking=True)
                ba[:n].copy_(hadj[src:src + n], non_blocking=True)
                ready[i][0].record(copy1)
            with torch.cuda.stream(copy2):
                if i >= 2:
                    copy2.wait_event(freed[i - 2])
                b2[:n * S].copy_(hx2[src * S:(src + n) * S], non_blocking=True)
                ready[i][1].record(copy2)
            main.wait_event(ready[i][0]); main.wait_event(ready[i][1])
            f = model.head(b1[:n * S], b2[:n * S], ba[:n], S)
            feats_host[off:off + n].copy_(f, non_blocking=True)
            freed[i].record(main)
        main.synchronize()
        t = time.perf_counter()
        d = metrics.compute_distance_matrix(feats_host[:NQ], feats_host[NQ:], args.dist_metric)   # CPU tensors
        r = metrics.evaluate_rank(d.numpy(), qp, gp, qc, gc, use_metric_mars=True)
        return r, time.perf_counter() - t

    steps = max(1, min(args.steps, args.e2e_steps))
    one_step()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize(dev)
    t0 = time.perf_counter()
    eval_s = 0.0
    for _ in range(steps):
        res, te = one_step()
        eval_s += te
    torch.cuda.synchronize(dev)
    dt = (time.perf_counter() - t0) / steps
    stats = [dt, ceiling]
    if world > 1:
        t = torch.tensor([dt, -ceiling], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        stats = [float(t[0].cpu()), -float(t[1].cpu())]             # slowest rank's step, lowest rank's ceiling
    dt, ceil_min = stats
    del hx1, hx2, bufs
    rate = maps_adj / max(dt - eval_s / steps, 1e-9) / 1e9
    return {'value': world * J / dt, 'unit': 'tracklets/s', 'h2d_bytes_per_step': int(h2d), 'd2h_bytes_per_step': int(d2h),
            'ms_per_step': dt * 1e3, 'steps': steps, 'h2d_gb_per_s': h2d / dt / 1e9,
            'head_phase_h2d_gb_per_s_per_gpu': rate, 'host_eval_ms': eval_s / steps * 1e3,
            'h2d_ceiling_gb_per_s_per_gpu': ceil_min, 'h2d_ceiling_aggregate_gb_per_s': ceil_min * world,
            'fraction_of_h2d_ceiling': rate / ceil_min,
            'note': 'layer4 maps start in pinned host memory (16.8 MB/tracklet over the host link, two copy streams): the step is '
                    'bound by the pinned-copy rate this box gives %d concurrent GPUs (h2d_ceiling_*: 1 GiB cudaMemcpyAsync, all ranks '
                    'at once, slowest rank); eval via the CPU-tensor / numpy API' % world}


# ------------------------------------------------------------------------------------------------
# same-box GPU comparator (SURVEY 8d): the reference's head / distance lines as stock PyTorch modules
# on the same B200 (library kernels: cuDNN/ATen pooling, cuBLAS fp32 GEMMs, elementwise ATen ops)
# ------------------------------------------------------------------------------------------------
def build_eager(dev, weights):
    """(head, distance) callables: the reference's module code for this path, written with the stock torch.nn modules
    it is built from (vmgn.py:104-123,142-172,237-268,270-278,296-321; distance.py:59-73), on device `dev`."""
    import torch.nn as nn
    import torch.nn.functional as F
    pool3d = nn.AdaptiveAvgPool3d(1)
    part_pools = [nn.AdaptiveAvgPool2d((k, 1)) for k in (4, 2, 1)]

    def bn(prefix):
        m = nn.BatchNorm1d(C).to(dev).eval()
        for k in ('weight', 'bias', 'running_mean', 'running_var'):
            getattr(m, k).data.copy_(weights[prefix + '.' + k])
        return m
    g_neck, a_neck = bn('global_bottleneck'), bn('att_bottleneck')
    layers = []
    for i in range(2):
        lin = nn.Linear(C, C, bias=False).to(dev)
        lin.weight.data.copy_(weights['graph_layers.%d.linear.weight' % i])
        layers.append((lin, bn('graph_layers.%d.bn' % i)))
    act = nn.LeakyReLU(0.1)

    def layer(lin, norm, f, a):
        h = lin(f)
        a = F.normalize(a, p=1, dim=2)
        sq = torch.pow(f, 2).sum(dim=2)
        d = sq.unsqueeze(1) + sq.unsqueeze(2)
        d -= 2 * torch.bmm(f, f.transpose(1, 2))
        g = F.normalize(2 / (d.clamp(1e-12).sqrt().exp() + 1), p=1, dim=2)
        hp = torch.bmm((a + g) / 2, h)
        hp = act(norm(hp.view(-1, C)).view(h.shape))
        return 0.9 * f + 0.1 * hp

    def head(m1, m2, a):
        b = a.shape[0]
        g_bn = g_neck(pool3d(m1.view(b, S, C, H, W).transpose(1, 2).contiguous()).view(b, -1))
        f = torch.cat([p(m2).view(b, S, C, k) for p, k in zip(part_pools, (4, 2, 1))], dim=3)
        f = f.transpose(2, 3).contiguous().view(b, S * 7, C)
        for lin, norm in layers:
            f = layer(lin, norm, f, a)
        f = f.view(b, S, 7, C)
        att = F.normalize(f.norm(p=2, dim=3, keepdim=True), p=1, dim=1)
        return torch.cat([g_bn, a_neck(f.mul(att).sum(dim=1).mean(dim=1))], dim=1)

    def distance(q, g):
        d = torch.pow(q, 2).sum(dim=1, keepdim=True).expand(q.shape[0], g.shape[0]) + \
            torch.pow(g, 2).sum(dim=1, keepdim=True).expand(g.shape[0], q.shape[0]).t()
        return d.addmm(q, g.t(), beta=1, alpha=-2)

    return head, distance


def torch_eager_gpu(args, dev, weights, x1, x2, adj, feats):
    """What the reference's own module code costs on this GPU, left in PyTorch's default fp32 mode (TF32 matmuls
    off).  Not a product path and not the oracle: a reported comparator, timed on a bounded sample of the resident
    pool.  The ranking has no GPU form in the reference (numpy / Cython), so it is not part of it."""
    head, distance = build_eager(dev, weights)
    n = min(args.eager_sample, x1.shape[0] // S)

    def timed(fn, reps):
        fn()
        torch.cuda.synchronize(dev)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(reps):
            fn()
        b.record()
        torch.cuda.synchronize(dev)
        return a.elapsed_time(b) / reps

    chunk = min(n, 64)                                     # the transposed copy of 64 tracklets is 0.5 GB
    with torch.no_grad():
        def head_sample():
            for off in range(0, n - chunk + 1, chunk):
                head(x1[off * S:(off + chunk) * S], x2[off * S:(off + chunk) * S], adj[off:off + chunk])
        done = (n // chunk) * chunk
        head_ms = timed(head_sample, 3) / done
        dist_ms = timed(lambda: distance(feats[:NQ], feats[NQ:]), 5)

        def head5():                                       # the reference's default --test-batch 5 (train_...py:49)
            head(x1[:5 * S], x2[:5 * S], adj[:5])
        b5_ms = timed(head5, 20)
    J = NQ + NG
    return {'what': 'the reference head / distance lines as stock torch.nn modules on this GPU, default fp32 (TF32 off), '
                    'maps resident; ranking excluded (numpy / Cython only in the reference)',
            'sample': 'head: %d of %d tracklets in batches of %d, extrapolated; distance %dx%dx%d in full' % (done, J, chunk, NQ, NG, 2 * C),
            'head_ms_per_tracklet': head_ms, 'head_tracklets_per_s': 1e3 / head_ms, 'head_ms_per_pass': head_ms * J,
            'distance_ms': dist_ms, 'head_ms_at_5_tracklets_per_call': b5_ms}


# ------------------------------------------------------------------------------------------------
# reference arm: the reference's CPU implementation of the same path, bounded sample
# ------------------------------------------------------------------------------------------------
def cpu_reference(args, steps, warmup):
    """One step = the head on `cpu_head_sample` tracklets + the 1980 x 9330 x 4096 distance + the MARS-metric ranking in
    full, all really executed `warmup + steps` times with every host core; the job figure extrapolates the head part
    linearly to 11310 tracklets (a tracklet never looks at another, so head time is linear in the count)."""
    from oracle import head as ohead, distance as odist, rank as orank
    cores = len(os.sched_getaffinity(0)) if hasattr(os, 'sched_getaffinity') else (os.cpu_count() or 1)
    torch.set_num_threads(cores)
    J, n_head = NQ + NG, args.cpu_head_sample
    weights = make_head_weights()
    g = torch.Generator().manual_seed(3)
    x1 = torch.randn(n_head * S, C, H, W, generator=g).clamp_(min=0)
    x2 = torch.randn(n_head * S, C, H, W, generator=g).clamp_(min=0)
    from agrl.pytorch_b200 import synthetic as synth
    adj = synth.pose_adjacency(n_head, S, 7, seed=3)
    qp, qc, gp, gc = make_labels(0, 1)
    feats = torch.randn(J, 2 * C, generator=g)
    have_ref_cy = orank.reference_rank_cy() is not None

    def one():
        t0 = time.perf_counter()
        with torch.no_grad():
            ohead.head_forward(x1, x2, adj, weights)
        t1 = time.perf_counter()
        d = odist.distance_matrix(feats[:NQ], feats[NQ:], args.dist_metric)
        t2 = time.perf_counter()
        orank.mars_port(d.numpy(), qp, gp, qc, gc, 50)
        t3 = time.perf_counter()
        return t1 - t0, t2 - t1, t3 - t2

    for _ in range(warmup):
        one()
    runs = [one() for _ in range(max(1, steps))]
    t_cy = None
    if have_ref_cy:                                       # the reference's own compiled evaluator, timed once beside
        d = odist.distance_matrix(feats[:NQ], feats[NQ:], args.dist_metric).numpy()
        t = time.perf_counter()
        orank.reference_evaluate_cy(d, qp, gp, qc, gc, 50, stable=False)
        t_cy = time.perf_counter() - t
    t_head = float(np.mean([r[0] for r in runs]))
    t_dist = float(np.mean([r[1] for r in runs]))
    t_rank = float(np.mean([r[2] for r in runs]))
    step_s = t_head + t_dist + t_rank                      # what one executed step really took
    job_s = J * (t_head / n_head) + t_dist + t_rank        # the whole job, head part extrapolated
    base = {'value': J / job_s, 'unit': 'tracklets/s', 'cores': cores, 'kind': 'port',
            'sample': 'per step: head on %d of %d tracklets (torch-CPU restatement of vmgn.py:296-321, %d threads, %.2f ms/tracklet, '
                      'extrapolated linearly), distance 1980x9330x4096 (%.0f ms) and MARS-metric ranking (C restatement of rank.py:160-212, '
                      '%.0f ms) in full; mean of %d executed steps' % (n_head, J, cores, t_head / n_head * 1e3, t_dist * 1e3, t_rank * 1e3,
                                                                       len(runs)),
            'extrapolated': True, 'steps_executed': len(runs), 'executed_step_ms': step_s * 1e3,
            'head_ms_per_tracklet': t_head / n_head * 1e3, 'distance_ms': t_dist * 1e3, 'rank_mars_ms': t_rank * 1e3,
            'rank_cy_reference_ms': None if t_cy is None else t_cy * 1e3,
            'why_port': 'the reference is a Python package: it is imported in the build container to generate tests/golden (bit-identical '
                        'regeneration checked), but its sources may not be copied into the repo and /root/reference does not exist on the '
                        'GPU box; what travels is the restatement pinned to those goldens and the reference\'s rank_cy.pyx compiled into oracle/_ref'}
    return {'cpu_baseline': base, 'job_s': job_s, 'step_s': step_s, 'eval_ms': (t_dist + t_rank) * 1e3}


def run_reference(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    r = cpu_reference(args, steps=args.steps, warmup=args.warmup)
    base = r['cpu_baseline']
    line = {'impl': 'reference', 'metric': METRIC, 'value': base['value'], 'unit': 'tracklets/s',
            'n_gpus': int(os.environ.get('WORLD_SIZE', '1')), 'steps': args.steps, 'warmup': args.warmup,
            'ms_per_step': r['step_s'] * 1e3, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
            'dtype': 'fp32', 'data': 'synthetic', 'extrapolated': True,
            'job_ms_extrapolated': r['job_s'] * 1e3,
            'config': {'workload': WORKLOAD % args.dist_metric,
                       'sample': 'each executed step runs the head on %d of the 11310 tracklets and the distance + ranking in full; '
                                 '`ms_per_step` is the executed step, `value` = 11310 / job_ms_extrapolated' % args.cpu_head_sample},
            'eval_ms': r['eval_ms'], 'cpu_baseline': base,
            'e2e': {'value': base['value'], 'unit': 'tracklets/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}}
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=5)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--pool', type=int, default=882, help='tracklets per head call = resident input pool (14.8 GB at 882)')
    ap.add_argument('--dist-metric', default='euclidean', choices=['euclidean', 'cosine'])
    ap.add_argument('--e2e-pool', type=int, default=128)
    ap.add_argument('--e2e-chunk', type=int, default=64)
    ap.add_argument('--e2e-steps', type=int, default=2)
    ap.add_argument('--cpu-head-sample', type=int, default=128)
    ap.add_argument('--workload', default='mars', choices=['mars', 'sweep'])
    ap.add_argument('--sweep-queries', type=int, default=10000)
    ap.add_argument('--sweep-gallery', type=int, default=1000000)
    ap.add_argument('--sweep-unfused', action='store_true', help='sweep through distance blocks in HBM + the top-k kernel')
    ap.add_argument('--no-e2e', action='store_true')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-parity', action='store_true', help='skip the oracle check of this run\'s outputs')
    ap.add_argument('--no-energy', action='store_true', help='skip the head-only NVML energy figure')
    ap.add_argument('--no-curve', action='store_true', help='skip the head call-size curve')
    ap.add_argument('--no-configs', action='store_true', help='skip the other BASELINE.json configurations')
    ap.add_argument('--no-sweep', action='store_true', help='skip the 10k x 1M retrieval sweep inside `configs`')
    ap.add_argument('--no-eager', action='store_true', help='skip the stock-PyTorch-on-this-GPU comparator (SURVEY 8d)')
    ap.add_argument('--eager-sample', type=int, default=256, help='tracklets of the pool the comparator head is timed on')
    ap.add_argument('--no-fast-mode', action='store_true', help='skip the extra head pass with the fp16 single-plane GEMM')
    ap.add_argument('--quick', action='store_true', help='only the timed region + kernel table (profiling runs)')
    ap.add_argument('--dump-outputs', metavar='DIR', help='write what the last timed step computed to DIR/<name>.npy '
                                                          '(features sample, cmc, mAP)')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and (args.impl != 'b200' or args.workload != 'mars'):
        ap.error('--dump-outputs applies to the B200 arm of the MARS workload')
    if args.quick:
        args.no_e2e = args.no_cpu_baseline = args.no_parity = args.no_energy = args.no_curve = True
        args.no_configs = args.no_eager = args.no_fast_mode = True
    args.warmup = max(args.warmup, 3) if args.impl == 'b200' else args.warmup
    if args.workload == 'sweep':
        run_sweep(args)
    elif args.impl == 'reference':
        run_reference(args)
    else:
        run_b200(args)


if __name__ == '__main__':
    main()
