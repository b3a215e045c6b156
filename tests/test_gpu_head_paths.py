"""Graph head against the fp64 oracle at every size-dependent path boundary, called through the C ABI so that the channel
count is free (the module mirror is built for C = 2048).  Every call runs with guard bands: sentinel-filled space before
and after the workspace and the node output, and an output matrix viewed inside a wider buffer (ld_out > 2C, one odd
ld_out) with sentinels in the row gaps and after the last row.  After each call: every sentinel intact, out and the last
layer's nodes within the oracle's bars (1e-4 max-scaled and norm-relative; 1e-5 norm-relative for the fp32-accurate
splits, as in test_gpu_scale.py), and a second call bit-identical.

Sizes that steer the code (csrc/head.cu): C / 64 Gram k-blocks over three operand buffers / tile stages, C / 128
message-passing blocks over two accumulators, C % 256 (half-empty last column tile of the 256-wide GEMMs; the attention
then computes its own row norms), C % 512 (low-rank first layer and the mixing kernel's grid), 2 C / tile width row-norm
slots of the last GEMM epilogue, h * w (128: the bulk-copy pooling kernel), tracklets per launch (attention slabs at 300 /
600), batch > 32 768 (several launches), and the number of layers (node-buffer ping-pong).

The fp64 oracle (oracle/head.py) runs on the device: the same torch code in float64, so that the wide channel counts cost
milliseconds instead of minutes on the host."""
import ctypes
import gc

import numpy as np
import pytest
import torch

from oracle import head as ohead
from oracle import synth

pytestmark = pytest.mark.gpu

TOL, TOL_FP32 = 1e-4, 1e-5
SENT = -1.2345678e33                       # sentinel: no head output comes near it
GUARD = 1024                               # floats of guard band on each side of a buffer
SPLITS = (1, 2, 3, 4)                      # SPLIT_FP16X1, SPLIT_BF16X2, SPLIT_BF16X3, SPLIT_FP16_E4M3
DTYPES = {'fp32': torch.float32, 'bf16': torch.bfloat16, 'fp16': torch.float16}


def _mod():
    from agrl.pytorch_b200 import _lib
    return _lib


def _lib():
    return _mod().require_device()


def slots_of(C, split):
    """row-norm slots the last layer's GEMM epilogue writes per node row: (column tile, half) pairs"""
    bn = 128 if split == 3 else 256
    return 2 * -(-C // bn)


class Guarded(object):
    """a float32 device buffer of `n` elements with GUARD + `tail` sentinel floats before / after it"""

    def __init__(self, n, tail=GUARD):
        self.n = n
        self.buf = torch.full((GUARD + n + tail,), SENT, dtype=torch.float32, device='cuda')
        self.view = self.buf[GUARD:GUARD + n]

    def ptr(self):
        return self.view.data_ptr()

    def guards_intact(self):
        return bool((self.buf[:GUARD] == SENT).all()) and bool((self.buf[GUARD + self.n:] == SENT).all())


class Head(object):
    """prepared head of C channels and L layers with synthetic weights (BN statistics and affine terms randomised)"""

    def __init__(self, C, L, split, seed, lowrank=True, use_pose=1, learn_graph=1, gemm_pair=True, pool_stages=0):
        M, lib = _mod(), _lib()
        self.C, self.L, self.use_pose, self.learn_graph = C, L, use_pose, learn_graph
        self.split, self.lowrank = split, lowrank
        self.wts = synth.head_weights(C, L, seed=seed, randomise_bn=True)
        self.dev = {k: v.cuda().contiguous() for k, v in self.wts.items()}
        P = M.HeadParams()
        P.channels, P.num_layers, P.use_pose, P.learn_graph = C, L, use_pose, learn_graph
        P.gamma, P.leaky_slope, P.bn_eps, P.split = 0.1, 0.1, 1e-5, split
        P.lowrank_off, P.gemm_no_pair, P.pool_stages = int(not lowrank), int(not gemm_pair), pool_stages
        d = self.dev
        for i in range(min(L, M.HEAD_MAX_LAYERS)):
            pre = 'graph_layers.%d' % i
            P.linear_weight[i] = d[pre + '.linear.weight'].data_ptr()
            P.bn_weight[i], P.bn_bias[i] = d[pre + '.bn.weight'].data_ptr(), d[pre + '.bn.bias'].data_ptr()
            P.bn_mean[i], P.bn_var[i] = d[pre + '.bn.running_mean'].data_ptr(), d[pre + '.bn.running_var'].data_ptr()
        for dst, pre in ((P.global_bn, 'global_bottleneck'), (P.att_bn, 'att_bottleneck')):
            for j, k in enumerate(('weight', 'bias', 'running_mean', 'running_var')):
                dst[j] = d[pre + '.' + k].data_ptr()
        self.P = P
        self.prepared = None
        nbytes = lib.agrl_head_prepared_bytes(ctypes.byref(P))
        if nbytes:
            self.prepared = torch.empty(nbytes, dtype=torch.uint8, device='cuda')
            M.check(lib.agrl_head_prepare_dev(ctypes.byref(P), self.prepared.data_ptr(), nbytes,
                                                torch.cuda.current_stream().cuda_stream))

    def oracle(self, x1, x2, adj, S):
        """fp64 oracle on the device: (B*S, C, h, w) maps (any layout / dtype), dense (B, V, V) graph"""
        out, _, nodes = ohead.head_forward(x1.cuda(), x2.cuda(), adj.cuda(), self.dev, S=S, num_gb=self.L,
                                           use_pose=bool(self.use_pose), learn_graph=bool(self.learn_graph),
                                           dtype=torch.float64, return_nodes=True)
        return out, nodes


class Call(object):
    """one guarded call of agrl_head_forward_dev (dense adj) or agrl_head_forward_compact_dev (int64 (B, 3) masks)"""

    def __init__(self, head, x1, x2, graph, B, S, h, w, pad=4, with_nodes=True, nhwc=False, maps_dtype=None):
        M, lib = _mod(), _lib()
        self.head, self.B, self.S, self.h, self.w = head, B, S, h, w
        self.x1, self.x2, self.graph = x1, x2, graph
        C, V = head.C, S * 7
        head.P.maps_nhwc = int(nhwc)
        head.P.maps_dtype = maps_dtype if maps_dtype is not None else {
            torch.float32: M.MAPS_FP32, torch.bfloat16: M.MAPS_BF16, torch.float16: M.MAPS_FP16}[x1.dtype]
        self.compact = graph is not None and graph.dtype == torch.int64
        self.wsb = lib.agrl_head_workspace_bytes(ctypes.byref(head.P), B, S)
        # room after the workspace for the whole row-norm region: a library that sizes it too small writes into the band
        self.ws = Guarded(-(-self.wsb // 4), tail=GUARD + B * V * slots_of(C, head.split))
        self.ld = 2 * C + pad
        self.out = Guarded(B * self.ld)
        self.nodes = Guarded(B * V * C) if with_nodes else None

    def __call__(self):
        lib = _lib()
        entry = lib.agrl_head_forward_compact_dev if self.compact else lib.agrl_head_forward_dev
        return entry(ctypes.byref(self.head.P), self.head.prepared.data_ptr() if self.head.prepared is not None else None,
                     self.x1.data_ptr(), self.x2.data_ptr(), self.graph.data_ptr() if self.graph is not None else None,
                     self.out.ptr(), self.ld, self.nodes.ptr() if self.nodes is not None else None,
                     self.B, self.S, self.h, self.w, self.ws.ptr(), self.wsb, torch.cuda.current_stream().cuda_stream)

    def result(self):
        C = self.head.C
        out = self.out.view.view(self.B, self.ld)[:, :2 * C]
        nodes = self.nodes.view.view(self.B, self.S * 7, C) if self.nodes is not None else None
        return out, nodes

    def sentinels_intact(self):
        C = self.head.C
        gaps = self.out.view.view(self.B, self.ld)[:, 2 * C:]
        ok = self.ws.guards_intact() and self.out.guards_intact() and bool((gaps == SENT).all())
        return ok and (self.nodes is None or self.nodes.guards_intact())

    def untouched(self):
        """nothing at all was written: the whole output and node buffers still hold the sentinel"""
        ok = bool((self.ws.buf == SENT).all()) and bool((self.out.buf == SENT).all())
        return ok and (self.nodes is None or bool((self.nodes.buf == SENT).all()))


def rel(got, ref):
    got, ref = got.double(), ref.double()
    return float((got - ref).abs().max() / ref.abs().max()), float((got - ref).norm() / ref.norm())


def check_call(call, adj_dense, sel=None):
    """run `call` twice; sentinels, oracle bars (on the tracklets `sel`, default all) and bit-identity of the repeat"""
    _mod().check(call())
    torch.cuda.synchronize()
    assert call.sentinels_intact(), 'a guard band or an output row gap was written'
    out, nodes = call.result()
    first_out = out.clone()
    first_nodes = nodes.clone() if nodes is not None else None
    assert bool(torch.isfinite(out).all())
    head, S = call.head, call.S
    idx = torch.arange(call.B, device='cuda') if sel is None else torch.as_tensor(sel, device='cuda')
    fr = (idx[:, None] * S + torch.arange(S, device='cuda')[None]).reshape(-1)
    ref, ref_nodes = head.oracle(call.x1[fr], call.x2[fr], adj_dense[idx], S)
    emax, enrm = rel(out[idx], ref)
    assert emax < TOL and enrm < TOL, ('out', emax, enrm)
    if head.split != 1:
        assert enrm < TOL_FP32, ('out', enrm)
    if nodes is not None:
        nmax, nnrm = rel(nodes[idx], ref_nodes)
        assert nmax < TOL and nnrm < TOL, ('nodes', nmax, nnrm)
        if head.split != 1:
            assert nnrm < TOL_FP32, ('nodes', nnrm)
    _mod().check(call())
    torch.cuda.synchronize()
    assert call.sentinels_intact(), 'a guard band or an output row gap was written (second call)'
    out, nodes = call.result()
    assert torch.equal(out, first_out), 'second call differs'
    if nodes is not None:
        assert torch.equal(nodes, first_nodes), 'second call differs (nodes)'


def device_maps(B, S, C, h, w, seed, dtype=torch.float32, nhwc=False, misaligned=False):
    """post-ReLU-like maps generated on the device, rounded to `dtype`"""
    g = torch.Generator(device='cuda').manual_seed(seed)
    maps = []
    for _ in range(2):
        x = torch.randn(B * S, C, h, w, generator=g, device='cuda').clamp_(min=0).mul_(2.0).to(dtype)
        if nhwc:
            x = x.contiguous(memory_format=torch.channels_last)
        elif misaligned:                   # one element past the start of its storage: off every vector alignment
            buf = torch.empty(x.numel() + 1, dtype=dtype, device='cuda')
            v = buf[1:].view(x.shape)
            v.copy_(x)
            x = v
        maps.append(x)
    return maps


def pose_graph(B, S, seed, compact):
    """(graph handed to the library, dense (B, V, V) graph for the oracle)"""
    if not compact:
        adj = synth.pose_adjacency(B, S, 7, seed=seed).cuda()
        return adj, adj
    from agrl.pytorch_b200 import pose
    kp, heights, valid = synth.pose_keypoints(B, S, seed=seed)
    masks = pose.part_masks(kp, heights, valid)
    return masks, pose.expand_adjacency(masks, S)


def run_case(C, split, L=2, B=4, S=8, h=4, w=3, seed=0, lowrank=True, use_pose=1, learn_graph=1, gemm_pair=True,
             compact=False, pad=4, with_nodes=True, dtype=torch.float32, nhwc=False, misaligned=False, pool_stages=0):
    head = Head(C, L, split, seed, lowrank=lowrank, use_pose=use_pose, learn_graph=learn_graph, gemm_pair=gemm_pair,
                pool_stages=pool_stages)
    x1, x2 = device_maps(B, S, C, h, w, seed + 1, dtype=dtype, nhwc=nhwc, misaligned=misaligned)
    graph, dense = pose_graph(B, S, seed + 2, compact)
    call = Call(head, x1, x2, graph, B, S, h, w, pad=pad, with_nodes=with_nodes, nhwc=nhwc)
    check_call(call, dense)


# ---------------------------------------------------------------------------------------------------------------------
# 1. channel widths
# ---------------------------------------------------------------------------------------------------------------------
WIDTHS = [128, 256, 384, 512, 640, 1024, 1536, 2048, 2176, 2560, 4096, 4352]
WIDTH_CASES = [(C, s, lr) for C in WIDTHS for s in SPLITS for lr in ((True, False) if C % 512 == 0 else (True,))]


@pytest.mark.parametrize('C,split,lowrank', WIDTH_CASES)
def test_channel_widths(C, split, lowrank):
    """Four splits at each width, the low-rank first layer on and off where C % 512 == 0 allows it.
    * Gram k-blocks C / 64: 2 at C = 128 (fewer than the 3 stages); = 0 mod 3 at 384, 1536; = 1 mod 3 at 256, 640, 1024,
      2176, 2560, 4096; = 2 mod 3 at 512, 2048, 4352.
    * Message-passing blocks C / 128: 1 at C = 128 (fewer than the 2 accumulators); odd at 384, 640, 2176; even elsewhere.
    * C % 256 != 0 at 128, 384, 640, 2176: the 256-wide GEMMs' last column tile is half empty and the attention computes
      its own row norms.
    * C % 512 != 0 (low-rank layer off by geometry) at 128, 256, 384, 640, 2176, 4352.
    * Row-norm slots of the last GEMM epilogue (2 C / tile width, with C a multiple of the width): below 32 at most
      widths; 32 at 2048 split 3 and 4096 256-wide; above 32 at 2176 / 2560 / 4096 / 4352 split 3 (34 / 40 / 64 / 68)
      and 4352 256-wide (34).  Above 32 with the low-rank layer off, a 32-slot region overflowed the workspace."""
    B = 3 if C >= 2048 else 5
    run_case(C, split, B=B, S=8 if C <= 2048 else 4, lowrank=lowrank, seed=1000 + C + 10 * split + int(lowrank),
             pad=4 if C != 640 else 7)


@pytest.mark.parametrize('C', [384, 2048])
@pytest.mark.parametrize('use_pose,learn_graph', [(1, 0), (0, 1)])
def test_graph_kinds(C, use_pose, learn_graph):
    """pose graph alone (no Gram phase: the message-passing loader starts its barrier phases at 0) and learnt graph alone"""
    run_case(C, 2, B=4, use_pose=use_pose, learn_graph=learn_graph, seed=2000 + C + 2 * use_pose)


@pytest.mark.parametrize('C', [128, 384])
def test_fp8_single_cta_tiles(C):
    """split 4 without CTA pairs where one CTA of a pair would hold a W half that lies wholly past N"""
    run_case(C, 4, B=5, gemm_pair=False, seed=2100 + C)


# ---------------------------------------------------------------------------------------------------------------------
# 2. map geometry
# ---------------------------------------------------------------------------------------------------------------------
GEOMS = [(4, 1), (4, 3), (8, 3), (8, 4), (12, 4), (16, 8), (32, 4), (24, 8), (16, 16), (32, 16)]
GEOM_CASES = [(h, w, C, nhwc) for (h, w) in GEOMS for C in (128, 384, 2048) for nhwc in (False, True)]


@pytest.mark.parametrize('h,w,C,nhwc', GEOM_CASES)
def test_map_geometry(h, w, C, nhwc):
    """(8, 4) is last_stride = 2 at 256 x 128 input; h * w = 128 takes the bulk-copy kernel ((16, 8) and (32, 4)); every
    other size the register kernel's quarter strips of qlen = h * w / 4; channels-last beside NCHW"""
    run_case(C, 2 if C != 384 else 3, L=2, B=3, S=4, h=h, w=w, nhwc=nhwc, seed=3000 + 7 * h + w + C)


@pytest.mark.parametrize('dt', ['bf16', 'fp16'])
@pytest.mark.parametrize('h,w,C,layout', [(16, 8, 384, 'nchw'), (32, 4, 128, 'nchw'), (12, 4, 2048, 'nchw'),
                                          (8, 3, 384, 'nhwc'), (16, 8, 128, 'nhwc'), (16, 8, 384, 'misaligned'),
                                          (4, 3, 128, 'misaligned')])
def test_map_geometry_16_bit(dt, h, w, C, layout):
    """bf16 / fp16 maps on both pooling kernels and channels-last, and maps one element past vector alignment"""
    run_case(C, 4, B=3, S=4, h=h, w=w, dtype=DTYPES[dt], nhwc=layout == 'nhwc', misaligned=layout == 'misaligned',
             seed=3500 + h + w + C)


@pytest.mark.parametrize('h,w,C', [(16, 8, 384), (4, 3, 128), (32, 4, 2048)])
def test_map_geometry_fp32_misaligned(h, w, C):
    run_case(C, 2, B=3, S=4, h=h, w=w, misaligned=True, seed=3600 + h + w + C)


# ---------------------------------------------------------------------------------------------------------------------
# 3. layer counts
# ---------------------------------------------------------------------------------------------------------------------
LAYER_CASES = ([(512, 2, L, nodes, lr) for L in range(5) for nodes in (True, False) for lr in (True, False)
                if L > 0 or lr] +
               [(2176, 3, L, True, True) for L in (3, 4)] + [(128, 4, 4, True, True), (384, 1, 3, False, True)])


@pytest.mark.parametrize('C,split,L,nodes,lowrank', LAYER_CASES)
def test_layer_counts(C, split, L, nodes, lowrank):
    """0 .. AGRL_HEAD_MAX_LAYERS layers: node buffers x[0] / x[1] / nodes_out in ping-pong after the low-rank first layer,
    the last layer into nodes_out or not, and no layer (pooled nodes copied out)"""
    run_case(C, split, L=L, B=4, with_nodes=nodes, lowrank=lowrank, seed=4000 + 10 * L + C + int(nodes) + 2 * int(lowrank))


# ---------------------------------------------------------------------------------------------------------------------
# 4. attention slabs
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('n', [299, 300, 599, 600])
@pytest.mark.parametrize('C,split', [(2048, 2), (2176, 3), (384, 2)])
def test_attention_slabs(C, split, n):
    """8 / 4 / 2 channel slabs per tracklet at n < 300 / >= 300 / >= 600 when the attention reads the epilogue's row
    norms (2048 split 2; 2176 split 3, whose 34 slots overflowed a 32-slot region); 384 split 2 computes its own.
    Two frames per tracklet: with one, every attention weight is |x| / |x| = 1 and the norms could be anything."""
    run_case(C, split, B=n, S=2, h=4, w=1, seed=5000 + C + n + split, pad=5)


# ---------------------------------------------------------------------------------------------------------------------
# 5. launch split
# ---------------------------------------------------------------------------------------------------------------------
SPLIT_CFGS = {'c128': dict(C=128, S=1, h=4, w=1, split=2, lowrank=True),
              'c512s9': dict(C=512, S=9, h=4, w=1, split=4, lowrank=True),
              'c128tma': dict(C=128, S=1, h=16, w=8, split=3, lowrank=True)}


def _bytes_needed(head, cfg, B):
    """maps, workspace, nodes and their copy from the first call, dense graph, output, and 1 GB for the rest"""
    C, S, h, w = cfg['C'], cfg['S'], cfg['h'], cfg['w']
    V = 7 * S
    wsb = _lib().agrl_head_workspace_bytes(ctypes.byref(head.P), B, S)
    return 2 * B * S * C * h * w * 4 + wsb + 2 * B * V * C * 4 + B * V * V * 4 + 4 * B * (2 * C + 3) * 4 + (1 << 30)


@pytest.mark.parametrize('compact', [False, True], ids=['dense', 'masks'])
@pytest.mark.parametrize('B', [32767, 32768, 32769, 40000])
@pytest.mark.parametrize('cfg', sorted(SPLIT_CFGS))
def test_launch_split(cfg, B, compact):
    """above 32 768 tracklets the call runs in several launches, each offsetting adj / masks, node rows, operand planes,
    z, G.T, y_unscale and out by its first tracklet; the oracle checks the tracklets on both sides of each seam"""
    c = SPLIT_CFGS[cfg]
    C, S, h, w = c['C'], c['S'], c['h'], c['w']
    seed = 6000 + B + C + S
    head = Head(C, 2, c['split'], seed, lowrank=c['lowrank'])
    gc.collect()
    torch.cuda.empty_cache()                   # what the caching allocator holds does not count as free
    free, _ = torch.cuda.mem_get_info()
    need = _bytes_needed(head, c, B)
    if free < need:
        pytest.skip('needs about %.1f GB of free device memory, %.1f GB free' % (need / 1e9, free / 1e9))
    x1, x2 = device_maps(B, S, C, h, w, seed + 1)
    from agrl.pytorch_b200 import pose
    kp, heights, valid = synth.pose_keypoints(B, S, seed=seed + 2)
    masks = pose.part_masks(kp, heights, valid)
    dense = pose.expand_adjacency(masks, S)
    call = Call(head, x1, x2, masks if compact else dense, B, S, h, w, pad=3)
    sel = sorted({0, 32766, 32767, 32768, 32769, B - 1} & set(range(B)))
    check_call(call, dense, sel=sel)


# ---------------------------------------------------------------------------------------------------------------------
# 6. limits
# ---------------------------------------------------------------------------------------------------------------------
def _limit_call(C=128, S=2, h=16, w=8, L=2, pool_stages=0, B=2):
    head = Head(C, L, 2, seed=7000 + C + S + h + L + pool_stages, pool_stages=pool_stages)
    if head.prepared is None:                  # params rejected: prepare a valid twin so the forward call has a buffer
        valid = Head(128, 2, 2, seed=7000)
        head.prepared = valid.prepared
        head.keep = valid
    x1, x2 = device_maps(B, S, C, h, w, seed=7100)
    adj = synth.pose_adjacency(B, S, 7, seed=7200).cuda()
    call = Call(head, x1, x2, adj, B, S, h, w)
    if call.wsb == 0:                          # rejected params: give the call a workspace anyway
        call.wsb = 1 << 20
        call.ws = Guarded(call.wsb // 4)
    return call, adj


@pytest.mark.parametrize('kw,code', [
    (dict(C=64), 'E_UNSUPPORTED'), (dict(C=192), 'E_UNSUPPORTED'), (dict(C=128), 'OK'),
    (dict(h=2, w=4), 'E_UNSUPPORTED'), (dict(h=6, w=4), 'E_UNSUPPORTED'), (dict(h=4, w=4), 'OK'),
    (dict(S=10, h=4, w=1), 'E_UNSUPPORTED'), (dict(S=9, h=4, w=1), 'OK'),
    (dict(L=4), 'OK'), (dict(L=5), 'E_INVALID'),
    (dict(pool_stages=1), 'E_INVALID'), (dict(pool_stages=13), 'E_INVALID'),
    (dict(pool_stages=2), 'OK'), (dict(pool_stages=12), 'OK'),
], ids=lambda v: v if isinstance(v, str) else '-'.join('%s=%s' % kv for kv in sorted(v.items())))
def test_limits(kw, code):
    """both sides of each limit of agrl_head_params / the forward call; a rejected call writes nothing at all"""
    M = _mod()
    call, adj = _limit_call(**kw)
    want = getattr(M, code)
    if want != M.OK:
        if kw.get('C') is not None or kw.get('L', 2) > 4 or kw.get('pool_stages', 0):
            assert _lib().agrl_head_workspace_bytes(ctypes.byref(call.head.P), 2, 2) == 0
        assert call() == want
        torch.cuda.synchronize()
        assert call.untouched()
    else:
        check_call(call, adj)


# ---------------------------------------------------------------------------------------------------------------------
# 7. the module mirror's argument checks
# ---------------------------------------------------------------------------------------------------------------------
def _model():
    from agrl.pytorch_b200 import models
    m = models.init_model('vmgn', num_classes=8, loss={'xent', 'htri'}, last_stride=1, num_split=4, num_gb=2, num_scale=1,
                          pyramid_part=True, use_pose=True, learn_graph=True, pretrained=False)
    for name in ('graph_layers', 'global_bottleneck', 'att_bottleneck'):
        getattr(m, name).cuda()
    return m.eval()


@pytest.mark.parametrize('case', ['channels', 'x4_2_shape', 'partial_tracklet'])
def test_mirror_rejects_mismatched_maps(case):
    """VMGN.head takes C from the module: maps of another width, an x4_2 unlike x4_1, or B*S not a multiple of seq_len
    raise ValueError before anything is launched"""
    M = _mod()
    model = _model()
    B, S, C = 2, 8, model.feature_dim
    shape1 = (B * S, 2 * C if case == 'channels' else C, 16, 8)
    shape2 = (B * S, shape1[1], 8 if case == 'x4_2_shape' else 16, 8)
    if case == 'partial_tracklet':
        shape1 = shape2 = (B * S + 1, C, 16, 8)
    x1 = torch.rand(shape1, device='cuda')
    # x4_2 lives at the start of a buffer of x4_1's size: a library that read it with x4_1's geometry stays in bounds
    x2 = torch.rand(x1.numel(), device='cuda')[:int(np.prod(shape2))].view(shape2)
    adj = synth.pose_adjacency(B, S, 7, seed=8000).cuda()
    torch.cuda.synchronize()
    before = M.launch_count()
    with pytest.raises(ValueError):
        with torch.no_grad():
            model.head(x1, x2, adj, S)
    assert M.launch_count() == before
