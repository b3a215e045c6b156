#!/usr/bin/env python
"""Graph head on bf16 / fp16 layer4 maps (agrl_head_params.maps_dtype) against fp32 maps, one process on one B200.

    python tools/half_maps_bench.py [--rounds 5] [--reps 3] [--out profiles/half_maps_bench.json]

The resident pool of bench.py (882 tracklets, bench.make_pool) is held three times: fp32, bf16 and fp16 copies of the same
values (~30 GB).  A pass is bench.py's head pass: 11 310 tracklets in 13 calls of <= 882.  Routes:
  fp32          fp32 maps (what bench.py times)
  bf16, fp16    16-bit maps read natively by the pooling kernels
  bf16_float    bf16 maps through head(x.float(), ...): what a mixed-precision backbone paid before, conversion included
The routes run alternately, `--rounds` rounds of `--reps` passes each (CUDA events around each round's passes): median and
spread of ms per pass.  A separate pass per route under the library's kernel timeline (_lib.profile) gives per-kernel ms
and the pooling kernel's algorithmic bytes/s (2 maps x S*C*h*w elements per tracklet, 2 or 4 bytes each), then the
ring depth of the 16-bit bulk-copy kernel is swept, and NVML energy per pass is read where the counter is available.
Card name and power limit come from a read-only nvidia-smi query in the same run."""
import argparse
import json
import os
import subprocess
import sys
import time
import types

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np
import torch

import bench

S, C, H, W = bench.S, bench.C, bench.H, bench.W
J = bench.NQ + bench.NG
MAP_ELEMS = S * C * H * W                       # elements of one map per tracklet: 2 097 152


def card():
    try:
        r = subprocess.run(['nvidia-smi', '-i', str(torch.cuda.current_device()), '--query-gpu=name,power.limit',
                            '--format=csv,noheader'], capture_output=True, text=True, timeout=30)
        name, limit = [f.strip() for f in r.stdout.strip().split(',')]
        return dict(name=name, power_limit=limit)
    except Exception as exc:
        return dict(unavailable='%s: %s' % (type(exc).__name__, exc))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--rounds', type=int, default=5)
    ap.add_argument('--reps', type=int, default=3, help='passes per route and round')
    ap.add_argument('--pool', type=int, default=882)
    ap.add_argument('--stages', default='4,8,10,12', help='ring depths of the 16-bit bulk-copy kernel to sweep')
    ap.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'half_maps_bench.json'))
    args = ap.parse_args()

    from agrl.pytorch_b200 import _lib
    _lib.require_device()
    dev = torch.device('cuda', 0)
    torch.cuda.set_device(dev)
    stream = torch.cuda.current_stream(dev)
    info = card()

    model = bench.make_model(dev, bench.make_head_weights())
    x1, x2, adj = bench.make_pool(args.pool, dev, seed=1)
    maps = {'fp32': (x1, x2), 'bf16': (x1.bfloat16(), x2.bfloat16()), 'fp16': (x1.half(), x2.half())}
    maps['bf16_float'] = maps['bf16']
    routes = ['fp32', 'bf16', 'fp16', 'bf16_float']
    elem_bytes = {'fp32': 4, 'bf16': 2, 'fp16': 2, 'bf16_float': 4}     # what the pooling kernel reads per element
    feats = {r: torch.empty(J, 2 * C, device=dev) for r in routes}
    chunks = [(o, min(args.pool, J - o)) for o in range(0, J, args.pool)]

    def head_pass(route):
        m1, m2 = maps[route]
        for off, n in chunks:
            a, b = m1[:n * S], m2[:n * S]
            if route == 'bf16_float':
                a, b = a.float(), b.float()
            model.head(a, b, adj[:n], S, out=feats[route][off:off + n])

    ev = lambda: torch.cuda.Event(enable_timing=True)
    result = dict(card=info, pool_tracklets=args.pool, tracklets_per_pass=J, calls_per_pass=len(chunks),
                  pool_algorithmic_bytes_per_tracklet={r: 2 * MAP_ELEMS * elem_bytes[r] for r in routes})
    with torch.no_grad():
        for r in routes:                                  # warm-up: module load, workspace, prepared weights
            head_pass(r)
        torch.cuda.synchronize()
        # native 16-bit pooling must give the bits of the .float() route on the same 16-bit maps
        result['bf16_native_equals_float_route'] = bool(torch.equal(feats['bf16'], feats['bf16_float']))

        # ---- alternating rounds, CUDA events ----
        times = {r: [] for r in routes}
        for k in range(args.rounds):
            order = routes[k % len(routes):] + routes[:k % len(routes)]
            for r in order:
                torch.cuda.synchronize()
                a, b = ev(), ev()
                a.record(stream)
                for _ in range(args.reps):
                    head_pass(r)
                b.record(stream)
                torch.cuda.synchronize()
                times[r].append(a.elapsed_time(b) / args.reps)
        result['head_ms_per_pass'] = {r: dict(median=float(np.median(t)), min=float(np.min(t)), max=float(np.max(t)),
                                              rounds=[round(v, 3) for v in t]) for r, t in times.items()}

        # ---- per-kernel ms (separate pass, kernel timeline) ----
        kernels = {}
        for r in routes:
            torch.cuda.synchronize()
            with _lib.profile(stream.cuda_stream) as prof:
                head_pass(r)
            tot = prof.totals()
            row = {k: dict(launches=n, ms=round(t, 4)) for k, (n, t) in sorted(tot.items())}
            pool_ms = tot['pool'][1]
            row['pool']['algorithmic_bytes'] = J * 2 * MAP_ELEMS * elem_bytes[r]
            row['pool']['gb_per_s'] = row['pool']['algorithmic_bytes'] / (pool_ms * 1e-3) / 1e9
            kernels[r] = row
        result['kernels_per_pass'] = kernels
        result['pool_rate_16bit_over_fp32'] = {r: kernels[r]['pool']['gb_per_s'] / kernels['fp32']['pool']['gb_per_s']
                                               for r in ('bf16', 'fp16')}

        # ---- ring depth of the bulk-copy kernel (pooling ms per pass under the kernel timeline, alternating) ----
        sweep = {}
        depths = [int(s) for s in args.stages.split(',') if s]
        for _ in range(args.rounds):
            for route in ('fp32', 'bf16'):
                for st in ([4] if route == 'fp32' else depths):
                    model.pool_stages = st
                    with _lib.profile(stream.cuda_stream) as prof:
                        head_pass(route)
                    sweep.setdefault('%s_stages%d' % (route, st), []).append(prof.totals()['pool'][1])
        model.pool_stages = 0
        result['pool_ms_by_stages'] = {k: dict(median=float(np.median(v)), values=[round(x, 3) for x in v])
                                       for k, v in sweep.items()}

        # ---- NVML energy per pass ----
        cx = types.SimpleNamespace(local=0, dev=dev)
        energy = {}
        for r in routes:
            time.sleep(0.3)
            energy[r] = bench.guarded(lambda: bench.energy_of(cx, lambda: head_pass(r), min_seconds=1.5))
        result['energy'] = energy

    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, 'w') as f:
        json.dump(result, f, indent=1)
    print(json.dumps(dict(card=info, head_ms={r: v['median'] for r, v in result['head_ms_per_pass'].items()},
                          pool_gb_s={r: round(kernels[r]['pool']['gb_per_s'], 1) for r in routes},
                          ratio=result['pool_rate_16bit_over_fp32'])))


if __name__ == '__main__':
    main()
