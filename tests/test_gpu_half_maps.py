"""bf16 / fp16 layer4 maps pooled natively (agrl_head_params.maps_dtype): the kernels convert on load, which is exact, and
sum as they do for fp32, so `head(m16)` must give exactly the bits of `head(m16.float())` -- the route a mixed-precision
backbone took before -- on every pooling kernel and knob.  Also the oracle at bench shape, the absence of an fp32 copy, the
autocast forward and the C ABI of the new field (that last test needs no GPU)."""
import ctypes
import os
import shutil
import subprocess

import numpy as np
import pytest
import torch

from oracle import head as ohead
from oracle import synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TOL = 1e-4
C, H = 2048, 16
HALF = {'bf16': torch.bfloat16, 'fp16': torch.float16}


def make_model(wts, split=None, num_gb=2):
    from agrl.pytorch_b200 import models
    kw = {} if split is None else {'head_split': split}
    m = models.init_model('vmgn', num_classes=8, loss={'xent', 'htri'}, last_stride=1, num_split=4, num_gb=num_gb,
                          num_scale=1, pyramid_part=True, use_pose=True, learn_graph=True, pretrained=False, **kw)
    sd = m.state_dict()
    for k, v in wts.items():
        sd[k].copy_(v)
    for name in ('graph_layers', 'global_bottleneck', 'att_bottleneck'):      # the backbone is not needed here
        getattr(m, name).cuda()
    return m.eval()


def rel_err(got, ref):
    got, ref = got.double(), ref.double()
    return float((got - ref).abs().max() / ref.abs().max()), float((got - ref).norm() / ref.norm())


def device_maps(B, S, w, dtype, seed, scale=2.0):
    """post-ReLU-like maps generated on the device, rounded to `dtype`"""
    g = torch.Generator(device='cuda').manual_seed(seed)
    x1 = torch.randn(B * S, C, H, w, generator=g, device='cuda').clamp_(min=0).mul_(scale).to(dtype)
    x2 = torch.randn(B * S, C, H, w, generator=g, device='cuda').clamp_(min=0).mul_(scale).to(dtype)
    return x1, x2


def offset_copy(x, dtype, offset=1):
    """x as a contiguous tensor of `dtype` that starts `offset` elements into its storage (breaks vector alignment)"""
    buf = torch.empty(x.numel() + offset, dtype=dtype, device=x.device)
    v = buf[offset:].view(x.shape)
    v.copy_(x)
    return v


CASES = [
    dict(split=1), dict(split=2), dict(split=3), dict(split=4),
    dict(lowrank=False), dict(gemm_pair=False), dict(lowrank=False, gemm_pair=False), dict(compact=True),
    dict(stages=2), dict(stages=12), dict(l2_hint=False),
    dict(tma=False), dict(w=2), dict(misaligned=True), dict(nhwc=True), dict(nhwc=True, w=2),
    dict(S=1), dict(S=4), dict(S=9), dict(B=1),
]


def _case_id(c):
    return '-'.join('%s=%s' % kv for kv in sorted(c.items()))


def _run_identity(dtype, B=5, S=8, w=8, split=None, lowrank=True, gemm_pair=True, compact=False, stages=0, l2_hint=True,
                  tma=True, misaligned=False, nhwc=False, seed=300):
    from agrl.pytorch_b200 import pose
    wts = synth.head_weights(C, 2, seed=seed + 1, randomise_bn=True)
    model = make_model(wts, split=split)
    model.head_lowrank, model.gemm_pair, model.pool_stages = lowrank, gemm_pair, stages
    model.pool_l2_hint, model.pool_tma = l2_hint, tma
    m1, m2 = device_maps(B, S, w, dtype, seed=seed + 2 + B + S + w)
    if compact:
        kp, heights, valid = synth.pose_keypoints(B, S, seed=seed + 3)
        adj = pose.part_masks(kp, heights, valid)
    else:
        adj = synth.pose_adjacency(B, S, 7, seed=seed + 3).cuda()
    r1, r2 = m1.float(), m2.float()
    if misaligned:
        # both routes on the scalar-load kernel: a 16-bit map 2 bytes and its fp32 copy 4 bytes past alignment
        m1, m2 = offset_copy(m1, dtype), offset_copy(m2, dtype)
        r1, r2 = offset_copy(r1, torch.float32), offset_copy(r2, torch.float32)
        assert m1.data_ptr() % 8 and r1.data_ptr() % 16
    if nhwc:
        m1, m2 = m1.contiguous(memory_format=torch.channels_last), m2.contiguous(memory_format=torch.channels_last)
        r1, r2 = r1.contiguous(memory_format=torch.channels_last), r2.contiguous(memory_format=torch.channels_last)
    with torch.no_grad():
        ref, ref_nodes = model.head(r1, r2, adj, S, return_nodes=True)
        out, nodes = model.head(m1, m2, adj, S, return_nodes=True)
    torch.cuda.synchronize()
    return out, nodes, ref, ref_nodes


@pytest.mark.gpu
@pytest.mark.parametrize('case', CASES, ids=_case_id)
@pytest.mark.parametrize('dt', ['bf16', 'fp16'])
def test_half_maps_bit_identical_to_the_float_route(dt, case):
    """every pooling kernel (bulk-copy ring at 2 / default / 12 stages, with and without the L2 hint; register loads on
    16x8 maps, narrow 16x2 maps and an unaligned view; channels-last), every GEMM mode and layer variant, S = 1 .. 9"""
    out, nodes, ref, ref_nodes = _run_identity(HALF[dt], **case)
    assert bool(torch.isfinite(out).all())
    assert torch.equal(out, ref), case
    assert torch.equal(nodes, ref_nodes), case


@pytest.mark.gpu
@pytest.mark.parametrize('dt', ['bf16', 'fp16'])
def test_half_maps_bit_identical_at_bench_size(dt):
    """882 tracklets per call: the persistent bulk-copy kernel with many units per CTA"""
    out, nodes, ref, ref_nodes = _run_identity(HALF[dt], B=882, seed=310)
    assert torch.equal(out, ref)
    assert torch.equal(nodes, ref_nodes)


def _oracle_on(idx, x1, x2, adj, wts, S=8, chunk=16):
    outs = []
    for i in range(0, len(idx), chunk):
        sel = idx[i:i + chunk]
        fr = torch.as_tensor((sel[:, None] * S + np.arange(S)[None]).reshape(-1), device=x1.device)
        outs.append(ohead.head_forward(x1[fr].cpu().float(), x2[fr].cpu().float(), adj[torch.as_tensor(sel)].cpu(), wts,
                                       dtype=torch.float64))
    return torch.cat(outs)


@pytest.mark.gpu
@pytest.mark.parametrize('dt,scale', [('bf16', 2.0), ('fp16', 2.0), ('fp16', 9e3)])
def test_half_maps_vs_oracle_at_bench_shape(dt, scale):
    """one 882-tracklet call against the fp64 oracle on the upcast maps (a subsample of tracklets incl. the first and
    the last); fp16 maps also with values up to ~6e4, near the top of the fp16 range"""
    B, S = 882, 8
    wts = synth.head_weights(C, 2, seed=320, randomise_bn=True)
    model = make_model(wts)
    m1, m2 = device_maps(B, S, 8, HALF[dt], seed=321, scale=scale)
    assert bool(torch.isfinite(m1).all() and torch.isfinite(m2).all())
    adj = synth.pose_adjacency(B, S, 7, seed=322)
    with torch.no_grad():
        out = model.head(m1, m2, adj.cuda(), S)
    torch.cuda.synchronize()
    idx = np.unique(np.concatenate([np.linspace(0, B - 1, 24).round().astype(np.int64), [0, B - 1]]))
    ref = _oracle_on(idx, m1, m2, adj, wts)
    emax, enrm = rel_err(out[torch.as_tensor(idx, device='cuda')].cpu(), ref)
    assert emax < TOL and enrm < TOL, (dt, scale, emax, enrm)


@pytest.mark.gpu
def test_half_maps_are_not_copied_to_fp32():
    """after a warm-up call (workspace and prepared weights cached), head() on 64 tracklets of bf16 maps allocates less
    than one fp32 copy of one map"""
    B, S = 64, 8
    wts = synth.head_weights(C, 2, seed=330)
    model = make_model(wts)
    m1, m2 = device_maps(B, S, 8, torch.bfloat16, seed=331)
    adj = synth.pose_adjacency(B, S, 7, seed=332).cuda()
    with torch.no_grad():
        model.head(m1, m2, adj, S)
        torch.cuda.synchronize()
        base = torch.cuda.memory_allocated()
        torch.cuda.reset_peak_memory_stats()
        model.head(m1, m2, adj, S)
        torch.cuda.synchronize()
    growth = torch.cuda.max_memory_allocated() - base
    assert growth < m1.numel() * 4, growth


@pytest.mark.gpu
@pytest.mark.parametrize('dt', [torch.bfloat16, None])
def test_autocast_forward_feeds_16_bit_maps(dt):
    """model(x, adj) under torch.autocast (bf16, and the default fp16): the cuDNN backbone returns 16-bit maps and forward
    hands them to the head as they are; the output stays fp32 and equals head() on those maps"""
    from agrl.pytorch_b200 import models
    torch.manual_seed(0)
    model = models.init_model('vmgn', num_classes=8, loss={'xent', 'htri'}, last_stride=1, num_split=4, num_gb=2,
                              num_scale=1, pyramid_part=True, use_pose=True, learn_graph=True, pretrained=False)
    model = model.cuda().eval()
    B, S = 2, 8
    x = torch.randn(B, S, 3, 256, 128, generator=torch.Generator().manual_seed(1)).cuda()
    adj = synth.pose_adjacency(B, S, 7, seed=2).cuda()
    kw = {} if dt is None else {'dtype': dt}
    want = torch.float16 if dt is None else dt
    det = torch.backends.cudnn.deterministic
    torch.backends.cudnn.deterministic = True
    try:
        with torch.no_grad(), torch.autocast('cuda', **kw):
            m1, m2 = model.featuremaps(x.view(B * S, 3, 256, 128))
            out = model(x, adj)
            direct = model.head(m1, m2, adj, S)
    finally:
        torch.backends.cudnn.deterministic = det
    assert m1.dtype == want and m2.dtype == want
    assert out.dtype == torch.float32 and tuple(out.shape) == (B, 4096)
    assert bool(torch.isfinite(out).all())
    assert torch.equal(out, direct)
    with torch.no_grad():
        assert torch.equal(model.head(m1.float(), m2.float(), adj, S), out)


@pytest.mark.gpu
def test_mixed_16_bit_maps_and_unknown_maps_dtype():
    """bf16 next to fp16 takes the upcast route (same result as upcasting by hand); an unknown maps_dtype is rejected"""
    from agrl.pytorch_b200 import _lib
    B, S = 3, 8
    wts = synth.head_weights(C, 2, seed=340, randomise_bn=True)
    model = make_model(wts)
    m1, _ = device_maps(B, S, 8, torch.bfloat16, seed=341)
    _, m2 = device_maps(B, S, 8, torch.float16, seed=342)
    adj = synth.pose_adjacency(B, S, 7, seed=343).cuda()
    with torch.no_grad():
        mixed = model.head(m1, m2, adj, S)
        ref = model.head(m1.float(), m2.float(), adj, S)
    assert torch.equal(mixed, ref)

    # the same call through the C ABI: maps_dtype selects the kernels' element type, an unknown value is rejected
    lib = _lib.require_device()
    b1, b2 = m1, m2.to(torch.bfloat16)
    with torch.no_grad():
        want = model.head(b1, b2, adj, S)
    stream = torch.cuda.current_stream().cuda_stream
    P, tensors, key = model._head_params()
    P.maps_dtype = _lib.MAPS_BF16
    prepared = model._prepared(lib, P, key, b1.device, stream)
    wsb = lib.agrl_head_workspace_bytes(ctypes.byref(P), B, S)
    ws = torch.empty(wsb, dtype=torch.uint8, device='cuda')
    out = torch.empty(B, 2 * C, device='cuda')

    def call():
        return lib.agrl_head_forward_dev(ctypes.byref(P), prepared.data_ptr(), b1.data_ptr(), b2.data_ptr(), adj.data_ptr(),
                                         out.data_ptr(), out.stride(0), None, B, S, H, 8, ws.data_ptr(), wsb, stream)
    _lib.check(call())
    torch.cuda.synchronize()
    assert torch.equal(out, want)
    P.maps_dtype = 7
    with pytest.raises(ValueError):
        _lib.check(call())


def test_maps_dtype_field_matches_the_c_header(tmp_path):
    """no GPU: the ctypes mirror has the C layout of agrl_head_params (size and the offset of maps_dtype), an unknown
    maps_dtype is rejected, and the prepared-buffer / workspace sizes do not depend on the maps' element type"""
    from agrl.pytorch_b200 import _lib
    gcc = shutil.which('gcc')
    if gcc is None:
        pytest.skip('no gcc')
    src = tmp_path / 'layout.c'
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "agrl_b200.h"\n'
                   'int main(void) { printf("%zu %zu %d %d %d\\n", sizeof(agrl_head_params), '
                   'offsetof(agrl_head_params, maps_dtype), AGRL_MAPS_FP32, AGRL_MAPS_BF16, AGRL_MAPS_FP16); return 0; }\n')
    exe = tmp_path / 'layout'
    r = subprocess.run([gcc, '-std=c99', '-Wall', '-Werror', '-I', os.path.join(ROOT, 'include'), str(src), '-o', str(exe)],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    size, off, f32, b16, f16 = (int(v) for v in subprocess.run([str(exe)], capture_output=True, text=True).stdout.split())
    assert size == ctypes.sizeof(_lib.HeadParams)
    assert off == _lib.HeadParams.maps_dtype.offset
    assert (f32, b16, f16) == (_lib.MAPS_FP32, _lib.MAPS_BF16, _lib.MAPS_FP16)

    lib = _lib.load()
    P = _lib.HeadParams()
    P.channels, P.num_layers, P.use_pose, P.learn_graph, P.split = 2048, 2, 1, 1, _lib.SPLIT_FP16_E4M3
    sizes = set()
    for dt in (_lib.MAPS_FP32, _lib.MAPS_BF16, _lib.MAPS_FP16):
        P.maps_dtype = dt
        sizes.add((lib.agrl_head_prepared_bytes(ctypes.byref(P)), lib.agrl_head_workspace_bytes(ctypes.byref(P), 882, 8)))
    assert len(sizes) == 1 and min(sizes.pop()) > 0
    P.maps_dtype = 7
    assert lib.agrl_head_prepared_bytes(ctypes.byref(P)) == 0
    assert lib.agrl_head_workspace_bytes(ctypes.byref(P), 882, 8) == 0
    with pytest.raises(ValueError):        # rejected before any device is touched
        _lib.check(lib.agrl_head_forward_dev(ctypes.byref(P), None, None, None, None, None, 4096, None, 1, 8, 16, 8,
                                             None, 0, None))
