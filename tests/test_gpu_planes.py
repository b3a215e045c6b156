"""GEMM operand planes byte for byte against a torch-CPU restatement of each split format (csrc/planes.cuh).

Distance operands (PreparedOperand.buf, euclidean): the planes of bf16 x 2, bf16 x 3 and fp16 x 2 with the zero padding
up to the 64-element k-block, and fp16 x 2's per-row 1 / scale.  Head weights (the prepared buffer of
agrl_head_prepare_dev): the planes of W for two layers in all four head splits, and the scaled modes' per-layer slots
{2^k, 2^-k, max |W|, 0}.  Where the restatement gives NaN (an Inf input minus its own rounding), the device may write any
NaN encoding; every other byte must match."""
import ctypes
import math

import numpy as np
import pytest
import torch

from oracle import synth

pytestmark = pytest.mark.gpu

E4M3_MAX = 448.0


def _mod():
    from agrl.pytorch_b200 import _lib
    return _lib


def align256(n):
    return (n + 255) // 256 * 256


def bf16_chain(x, P):
    """x = p0 + p1 (+ p2): each plane the bf16 (round to nearest even) of what the planes before it left"""
    planes, r = [], x.clone()
    for _ in range(P):
        b = r.to(torch.bfloat16)
        planes.append(b)
        r = r - b.float()
    return planes


def e4m3(x):
    """SATFINITE conversion: finite and infinite values clamped to +-448 first, NaN kept"""
    return torch.where(torch.isnan(x), x, x.clamp(-E4M3_MAX, E4M3_MAX)).to(torch.float8_e4m3fn)


def f16_scales(bound):
    """2^k that puts bound in [2^13, 2^14), and 2^-k (bound 0: 1)"""
    e = math.frexp(bound)[1] if bound > 0 else 14
    e = max(-100, min(100, e))
    return 2.0 ** (14 - e), 2.0 ** (e - 14)


def f16x2_row_scales(x):
    """per row: 2^k that puts max |x| in [2^7, 2^8), and 2^-k; zero rows and rows with Inf / NaN (or max >= 3e38) keep 1"""
    up, down = [], []
    for row in x:
        mx = float(row.abs().max()) if row.numel() else 0.0
        e = 7
        if 0.0 < mx < 3.0e38 and not bool(torch.isnan(row).any()):
            e = math.frexp(mx)[1] - 1                 # ilogb
        e = max(-110, min(120, e))
        up.append(2.0 ** (7 - e))
        down.append(2.0 ** (e - 7))
    return torch.tensor(up, dtype=torch.float32)[:, None], torch.tensor(down, dtype=torch.float32)


def assert_same_bits(dev, ref, what):
    """dev: device bytes as a tensor of ref's dtype; equal bits except that a NaN of ref may be any NaN"""
    dev = dev.cpu().reshape(ref.shape)
    nan = torch.isnan(ref.float())
    assert bool(torch.isnan(dev[nan].float()).all()), what + ': NaN expected'
    width = {1: torch.uint8, 2: torch.int16, 4: torch.int32}[ref.element_size()]
    a, b = dev.view(width)[~nan], ref.view(width)[~nan]
    bad = (a != b).nonzero()
    assert bad.numel() == 0, '%s: %d of %d differ, first at %s' % (what, bad.size(0), a.numel(), bad[:4].tolist())


# ---- distance operands ------------------------------------------------------------------------------------------------
def operand_rows(rows, dim, seed):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(rows, dim, generator=g)
    x[1] = 0.0                                                            # all-zero row
    sign = torch.where(torch.rand(dim, generator=g) < 0.5, -1.0, 1.0)
    x[2] = sign * torch.logspace(-38, 38, dim)                            # every magnitude in one row
    x[3] = sign * torch.logspace(-45, -39, dim)                           # subnormals (max below fp32's normal range)
    x[4] = sign * torch.linspace(1.0, 3.2e38, dim)                        # max above 3e38: fp16 x 2 leaves it unscaled
    x[5] = x[0] * 1e20
    x[6] = x[0] * 1e-20
    x[7, ::3] = 0.0
    return x


@pytest.mark.parametrize('dim', [63, 64, 65])
@pytest.mark.parametrize('split', [2, 3, 5])               # SPLIT_BF16X2, SPLIT_BF16X3, SPLIT_FP16X2
def test_distance_operand_bytes(split, dim):
    from agrl.pytorch_b200.metrics.distance import PreparedOperand
    rows = 37
    x = operand_rows(rows, dim, seed=100 + dim)
    op = PreparedOperand(x.cuda(), 'euclidean', split)
    torch.cuda.synchronize()
    k_pad = (dim + 63) // 64 * 64
    xp = torch.zeros(rows, k_pad)
    xp[:, :dim] = x
    if split == 5:
        up, down = f16x2_row_scales(x)
        xs = xp * up
        h = xs.to(torch.float16)
        planes = [h, ((xs - h.float()) * 2048.0).to(torch.float16)]
    else:
        planes = bf16_chain(xp, split)
    P = len(planes)
    plane_b = rows * k_pad * 2
    buf = op.buf.cpu()
    for p, ref in enumerate(planes):
        assert_same_bits(buf[p * plane_b:(p + 1) * plane_b].view(ref.dtype), ref, 'split %d plane %d' % (split, p))
    if split == 5:
        off = align256(align256(P * plane_b) + 4 * rows)                  # planes, sumsq, then unscale
        assert_same_bits(buf[off:off + 4 * rows].view(torch.float32), down, 'unscale')


# ---- head weights -----------------------------------------------------------------------------------------------------
def layer_weight(C, seed, with_inf):
    g = torch.Generator().manual_seed(seed)
    w = torch.randn(C, C, generator=g) * 0.02
    w[0] = 0.0
    w[1] = torch.logspace(-30, 2, C) * torch.where(torch.rand(C, generator=g) < 0.5, -1.0, 1.0)
    w[2, :7] = torch.tensor([1e-41, -1e-44, 3.0e-8, 6.1e-5, 65504.0 / 2 ** 14, -2.0 ** -24, 0.5])
    if with_inf:
        w[3, 5], w[4, 70] = float('inf'), -float('inf')                  # ignored by max |W|; saturate the E4M3 copies
    return w


@pytest.mark.parametrize('split', [1, 2, 3, 4])            # SPLIT_FP16X1, SPLIT_BF16X2, SPLIT_BF16X3, SPLIT_FP16_E4M3
def test_head_weight_bytes(split):
    M = _mod()
    lib = M.require_device()
    C, L = 256, 2
    wts = synth.head_weights(C, L, seed=7)
    W = [layer_weight(C, 20 + l, with_inf=(l == 1)) for l in range(L)]
    for l in range(L):
        wts['graph_layers.%d.linear.weight' % l] = W[l]
    dev = {k: v.cuda().contiguous() for k, v in wts.items()}
    P = M.HeadParams()
    P.channels, P.num_layers, P.use_pose, P.learn_graph = C, L, 1, 1
    P.gamma, P.leaky_slope, P.bn_eps, P.split = 0.1, 0.1, 1e-5, split
    for l in range(L):
        pre = 'graph_layers.%d' % l
        P.linear_weight[l] = dev[pre + '.linear.weight'].data_ptr()
        P.bn_weight[l], P.bn_bias[l] = dev[pre + '.bn.weight'].data_ptr(), dev[pre + '.bn.bias'].data_ptr()
        P.bn_mean[l], P.bn_var[l] = dev[pre + '.bn.running_mean'].data_ptr(), dev[pre + '.bn.running_var'].data_ptr()
    for dst, pre in ((P.global_bn, 'global_bottleneck'), (P.att_bn, 'att_bottleneck')):
        for j, k in enumerate(('weight', 'bias', 'running_mean', 'running_var')):
            dst[j] = dev[pre + '.' + k].data_ptr()
    nbytes = lib.agrl_head_prepared_bytes(ctypes.byref(P))
    assert nbytes > 0
    prepared = torch.zeros(nbytes, dtype=torch.uint8, device='cuda')
    M.check(lib.agrl_head_prepare_dev(ctypes.byref(P), prepared.data_ptr(), nbytes, torch.cuda.current_stream().cuda_stream))
    buf = prepared.cpu()

    n_planes = {1: 1, 2: 2, 3: 3, 4: 2}[split]
    plane_b = C * C * 2
    off, w_off = 0, []
    for l in range(L):                                                    # layout of carve_prepared (csrc/head.cu)
        w_off.append(off)
        off = align256(off + n_planes * plane_b)
    for _ in range(L + 2):
        off = align256(align256(off + 4 * C) + 4 * C)                     # folded BN scale, shift
    slots = buf[off:off + 16 * M.HEAD_MAX_LAYERS].view(torch.float32)
    for l in range(L):
        w = W[l]
        base = w_off[l]
        if split in (2, 3):
            planes = bf16_chain(w, split)
            for p, ref in enumerate(planes):
                got = buf[base + p * plane_b:base + (p + 1) * plane_b].view(torch.bfloat16)
                assert_same_bits(got, ref, 'layer %d plane %d' % (l, p))
            continue
        a = w.abs()
        bound = float(a[a < 3.0e38].max())                               # Inf / NaN are not part of the bound
        up, down = f16_scales(bound)
        ref_slot = torch.tensor([up, down, bound, 0.0], dtype=torch.float32)
        assert_same_bits(slots[4 * l:4 * l + 4], ref_slot, 'layer %d scale slots' % l)
        ws = w * up
        h = ws.to(torch.float16)
        assert_same_bits(buf[base:base + plane_b].view(torch.float16), h, 'layer %d fp16 plane' % l)
        if split == 4:
            # B operand: per 64-element k-block 64 value copies e4m3(w s 2^-6), then 64 residuals e4m3((w s - h) 2^6)
            val = e4m3(ws * 0.015625).view(C, C // 64, 1, 64)
            res = e4m3((ws - h.float()) * 64.0).view(C, C // 64, 1, 64)
            ref = torch.cat([val, res], dim=2).reshape(C, 2 * C)
            got = buf[base + plane_b:base + 2 * plane_b].view(torch.float8_e4m3fn)
            assert_same_bits(got, ref, 'layer %d e4m3 plane' % l)
