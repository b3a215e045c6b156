"""VMGN with the B200 graph head -- mirror of torchreid/models/vmgn.py (class GSTA, factory vmgn()).

Same constructor arguments, same parameter / buffer names and shapes (so the reference's
size-filtered ``--load-weights`` path, train_vidreid_xent_htri.py:279-287, loads unchanged), same
eval-mode ``forward(x, adj) -> (B, 4096)``.  The ResNet-50 frame backbone (``featuremaps``,
vmgn.py:280-290) stays on stock ``nn.Conv2d`` / ``nn.BatchNorm2d`` (cuDNN) exactly as in the
reference; everything after it (vmgn.py:296-321) is one call into libagrl_b200
(``agrl_head_forward_dev``, csrc/head.cu).

Out of scope (SURVEY.md section 8a): the training-mode tail of forward (classifiers, consistency
sub-sampling, vmgn.py:323-357) raises NotImplementedError; GraphLayer's unused 'dot' affinity is
not provided.  There is no CPU path: a CPU input raises.
"""
import ctypes
import warnings

import torch
from torch import nn

from .. import _lib

__all__ = ['vmgn', 'VMGN', 'pool_clips']

RESNET50_URL = 'https://download.pytorch.org/models/resnet50-19c8e357.pth'
_MAPS_DTYPES = {torch.bfloat16: _lib.MAPS_BF16, torch.float16: _lib.MAPS_FP16}


def pyramid_splits(num_split):
    """calc_splits (utils/reidtools.py:13-15)."""
    assert (num_split & (num_split - 1)) == 0, \
        'num_split must be the power of 2, {} is not supported'.format(num_split)
    return [n for n in range(num_split, 0, -1) if num_split % n == 0]


class _Block(nn.Module):
    """ResNet bottleneck; attribute names follow torchvision / the reference checkpoint keys."""
    expansion = 4

    def __init__(self, cin, width, stride=1, downsample=None):
        super().__init__()
        cout = width * self.expansion
        self.conv1 = nn.Conv2d(cin, width, 1, bias=False)
        self.bn1 = nn.BatchNorm2d(width)
        self.conv2 = nn.Conv2d(width, width, 3, stride=stride, padding=1, bias=False)
        self.bn2 = nn.BatchNorm2d(width)
        self.conv3 = nn.Conv2d(width, cout, 1, bias=False)
        self.bn3 = nn.BatchNorm2d(cout)
        self.relu = nn.ReLU(inplace=True)
        self.downsample = downsample
        self.stride = stride

    def forward(self, x):
        y = self.relu(self.bn1(self.conv1(x)))
        y = self.relu(self.bn2(self.conv2(y)))
        y = self.bn3(self.conv3(y))
        skip = x if self.downsample is None else self.downsample(x)
        return self.relu(y + skip)


def _stage(cin, width, depth, stride):
    cout = width * _Block.expansion
    down = None
    if stride != 1 or cin != cout:
        down = nn.Sequential(nn.Conv2d(cin, cout, 1, stride=stride, bias=False), nn.BatchNorm2d(cout))
    blocks = [_Block(cin, width, stride, down)] + [_Block(cout, width) for _ in range(depth - 1)]
    return nn.Sequential(*blocks), cout


class _GraphLayerParams(nn.Module):
    """Parameter holder with GraphLayer's names (vmgn.py:93-94, init :125-140): linear + bn."""

    def __init__(self, channels, use_pose, learn_graph, gamma=0.1):
        super().__init__()
        assert use_pose or learn_graph                                   # vmgn.py:92
        self.use_pose, self.learn_graph, self.gamma = use_pose, learn_graph, gamma
        self.linear = nn.Linear(channels, channels, bias=False)
        self.bn = nn.BatchNorm1d(channels)
        nn.init.normal_(self.linear.weight, 0, 0.01)
        nn.init.constant_(self.bn.weight, 1)
        nn.init.constant_(self.bn.bias, 0)


def _neck(channels):
    bn = nn.BatchNorm1d(channels)
    bn.bias.requires_grad_(False)                                        # vmgn.py:239, :265
    return bn


def _init_neck(bn, fc):
    nn.init.normal_(bn.weight, 1.0, 0.001)                               # weights_init_kaiming, torchtools.py:61-64
    nn.init.constant_(bn.bias, 0.0)
    nn.init.normal_(fc.weight, std=0.001)                                # weights_init_classifier, torchtools.py:83-88


class VMGN(nn.Module):
    """GSTA of the reference (vmgn.py:214-357) with the graph head on libagrl_b200."""

    def __init__(self, num_classes, loss, num_split, pyramid_part, num_gb, use_pose, learn_graph,
                 consistent_loss=False, pretrained=True, head_split=_lib.SPLIT_FP16_E4M3, **kwargs):
        super().__init__()
        self.loss = loss
        self.feature_dim = 512 * _Block.expansion
        # backbone, last stride forced to 1 (vmgn.py:224) -> 16x8 maps for 256x128 frames
        self.conv1 = nn.Conv2d(3, 64, 7, stride=2, padding=3, bias=False)
        self.bn1 = nn.BatchNorm2d(64)
        self.relu = nn.ReLU(inplace=True)
        self.maxpool = nn.MaxPool2d(3, stride=2, padding=1)
        self.layer1, c = _stage(64, 64, 3, 1)
        self.layer2, c = _stage(c, 128, 4, 2)
        self.layer3, c = _stage(c, 256, 6, 2)
        self.layer4_1, c = _stage(c, 512, 3, 1)
        if pretrained:
            self._load_imagenet()
        import copy
        self.layer4_2 = copy.deepcopy(self.layer4_1)                      # vmgn.py:234

        self.global_bottleneck = _neck(self.feature_dim)
        self.global_classifier = nn.Linear(self.feature_dim, num_classes, bias=False)
        _init_neck(self.global_bottleneck, self.global_classifier)

        self.num_split = num_split
        self.total_split_list = pyramid_splits(num_split) if pyramid_part else [num_split]
        self.total_split = sum(self.total_split_list)
        self.num_gb = num_gb
        self.graph_layers = nn.ModuleList(
            _GraphLayerParams(self.feature_dim, use_pose, learn_graph) for _ in range(num_gb))
        self.use_pose, self.learn_graph = use_pose, learn_graph
        self.consistent_loss = consistent_loss

        self.att_bottleneck = _neck(self.feature_dim)
        self.att_classifier = nn.Linear(self.feature_dim, num_classes, bias=False)
        _init_neck(self.att_bottleneck, self.att_classifier)

        self.head_split = head_split
        # tuning knobs of the head, per module (they travel in agrl_head_params; the library has no global state)
        self.head_lowrank = True         # first layer's X.W^T on the 4S quarter-strip rows (False: on all 7S node rows)
        self.pool_tma = True             # bulk-copy (TMA ring) pooling kernel where it applies (False: register loads)
        self.pool_stages = 0             # ring stages per pooling CTA (0 = library default)
        self.pool_l2_hint = True         # evict-first hint on the pooling bulk copies
        self.gemm_pair = True            # fp16 + e4m3 mode: layer GEMMs as CTA pairs (cta_group::2); False: one CTA per tile
        self._prep = {}                  # device -> (key, prepared buffer): what the cached buffer was built from
        self._ws = {}                    # (device, stream) -> workspace

    # -- weights ---------------------------------------------------------------------------------
    def _load_imagenet(self):
        """init_pretrained_weights (vmgn.py:360-370): name-and-size filtered ImageNet ResNet-50."""
        try:
            import torch.utils.model_zoo as model_zoo
            pre = model_zoo.load_url(RESNET50_URL)
        except Exception as e:                       # no network in this environment
            warnings.warn('ImageNet weights unavailable ({}); backbone keeps its random init'.format(type(e).__name__))
            return
        own = self.state_dict()
        remap = {k.replace('layer4.', 'layer4_1.'): v for k, v in pre.items()}
        own.update({k: v for k, v in remap.items() if k in own and own[k].size() == v.size()})
        self.load_state_dict(own)

    # -- backbone (stock cuDNN) -------------------------------------------------------------------
    def featuremaps(self, x):
        x = self.maxpool(self.relu(self.bn1(self.conv1(x))))
        x = self.layer3(self.layer2(self.layer1(x)))
        return self.layer4_1(x), self.layer4_2(x)

    # -- graph head (libagrl_b200) ------------------------------------------------------------------
    def _head_params(self):
        P = _lib.HeadParams()
        P.channels, P.num_layers = self.feature_dim, self.num_gb
        P.use_pose, P.learn_graph = int(self.use_pose), int(self.learn_graph)
        P.gamma = self.graph_layers[0].gamma if self.num_gb else 0.1
        P.leaky_slope, P.bn_eps, P.split = 0.1, 1e-5, self.head_split
        P.lowrank_off, P.pool_register_loads = int(not self.head_lowrank), int(not self.pool_tma)
        P.pool_stages, P.pool_no_l2_hint = int(self.pool_stages), int(not self.pool_l2_hint)
        P.gemm_no_pair = int(not self.gemm_pair)
        tensors, key = [], []

        def ptr(t):
            # the cache key describes the module's OWN parameter / buffer (a converted temporary has _version 0 and an
            # address the allocator may recycle: it cannot tell a reloaded weight from the old one)
            key.append((id(t), t.data_ptr(), t._version, t.dtype))
            t = t.detach()
            if t.dtype != torch.float32 or not t.is_contiguous():
                t = t.float().contiguous()
            tensors.append(t)
            return t.data_ptr()

        for i, gl in enumerate(self.graph_layers):
            P.linear_weight[i] = ptr(gl.linear.weight)
            P.bn_weight[i], P.bn_bias[i] = ptr(gl.bn.weight), ptr(gl.bn.bias)
            P.bn_mean[i], P.bn_var[i] = ptr(gl.bn.running_mean), ptr(gl.bn.running_var)
        for dst, bn in ((P.global_bn, self.global_bottleneck), (P.att_bn, self.att_bottleneck)):
            dst[0], dst[1], dst[2], dst[3] = ptr(bn.weight), ptr(bn.bias), ptr(bn.running_mean), ptr(bn.running_var)
        return P, tensors, tuple(key)

    def _prepared(self, lib, P, key, dev, stream):
        """bf16 planes of W + folded BN, rebuilt when a parameter is replaced or modified in place.  nn.DataParallel
        replicas are rebuilt on every forward (fresh tensors at possibly recycled addresses), so a replica never trusts a
        cached buffer: one process per GPU (or one module per device) is the supported way to scale."""
        key = (self.head_split,) + key
        hit = self._prep.get(dev)
        if hit is None or hit[0] != key or getattr(self, '_is_replica', False):
            nbytes = lib.agrl_head_prepared_bytes(ctypes.byref(P))
            if nbytes == 0:
                _lib.check(_lib.E_UNSUPPORTED)
            buf = torch.empty(nbytes, dtype=torch.uint8, device=dev)
            _lib.check(lib.agrl_head_prepare_dev(ctypes.byref(P), buf.data_ptr(), nbytes, stream))
            hit = (key, buf)
            if not getattr(self, '_is_replica', False):
                self._prep[dev] = hit
        return hit[1]

    def head(self, x4_1, x4_2, adj, seq_len, return_nodes=False, out=None):
        """vmgn.py:296-321 on the GPU: (B*S,C,h,w) x2 + (B,V,V) -> (B, 2C) fp32.  The maps may be fp32, or both bf16 /
        both fp16 (a backbone under torch.autocast): those are read without an fp32 copy, same result as ``.float()``.
        ``out``: optional preallocated (B, 2C) fp32 CUDA tensor (unit column stride) to write into."""
        lib = _lib.require_device()
        if not x4_1.is_cuda:
            raise RuntimeError('agrl.pytorch_b200 has no CPU path: move the model and inputs to a B200')
        if self.total_split_list != [4, 2, 1]:
            _lib.check(_lib.E_UNSUPPORTED)
        dev = x4_1.device
        BS, C, h, w = x4_1.shape
        # the library takes C from the module and reads both maps with x4_1's geometry: a mismatch would be read with the
        # wrong layout (or past the end of x4_2), and frames beyond the last whole tracklet would be dropped
        if C != self.feature_dim:
            raise ValueError('x4_1 has %d channels; this module is built for %d' % (C, self.feature_dim))
        if tuple(x4_2.shape) != tuple(x4_1.shape):
            raise ValueError('x4_2 must have the shape of x4_1: %s vs %s' % (tuple(x4_2.shape), tuple(x4_1.shape)))
        if BS % seq_len != 0:
            raise ValueError('B*S = %d maps is not a multiple of seq_len = %d' % (BS, seq_len))
        B, V = BS // seq_len, seq_len * self.total_split
        if B == 0:                                                   # empty loader batch: nothing to launch
            empty = torch.empty(0, 2 * C, dtype=torch.float32, device=dev) if out is None else out
            return (empty, torch.empty(0, V, C, dtype=torch.float32, device=dev)) if return_nodes else empty
        # a torch.channels_last backbone hands over (B*S, h, w, C)-ordered memory: pooled as is (no NCHW copy)
        nhwc = (x4_1.dim() == 4 and C % 4 == 0 and not x4_1.is_contiguous()
                and x4_1.is_contiguous(memory_format=torch.channels_last)
                and x4_2.is_contiguous(memory_format=torch.channels_last))
        # bf16 / fp16 maps (a backbone under torch.autocast) are pooled as they are, without an fp32 copy: the kernels
        # convert exactly on load, so the result has the bits of the .float() route.  Channels-last pooling needs maps
        # aligned to four elements; every other case keeps the .float() route.
        maps_dtype = _MAPS_DTYPES.get(x4_1.dtype) if x4_2.dtype == x4_1.dtype else None
        if nhwc:
            native = (x4_1.data_ptr() | x4_2.data_ptr()) % 8 == 0
        else:
            native = x4_1.is_contiguous() and x4_2.is_contiguous()
        if maps_dtype is None or not native:
            maps_dtype = _lib.MAPS_FP32
            if nhwc:
                x4_1, x4_2 = x4_1.float(), x4_2.float()              # .float() keeps the memory format
            else:
                x4_1 = x4_1.float().contiguous()
                x4_2 = x4_2.float().contiguous()
        compact = False
        if self.use_pose:
            # adj: the reference's dense (B, V, V) fp32 graph, or the three part-membership masks per tracklet it is
            # made of (int64 (B, 3), agrl.pytorch_b200.pose.part_masks) -- the compact wire format
            compact = adj is not None and adj.dtype == torch.int64 and tuple(adj.shape) == (B, 3)
            if compact:
                adj = adj.to(device=dev).contiguous()
            else:
                assert adj is not None and tuple(adj.shape) == (B, V, V), 'adj must be (B, V, V) with V = S * P'
                adj = adj.to(device=dev, dtype=torch.float32).contiguous()
        with torch.cuda.device(dev):
            stream = torch.cuda.current_stream(dev).cuda_stream
            P, tensors, key = self._head_params()
            P.maps_nhwc, P.maps_dtype = int(nhwc), maps_dtype
            prepared = self._prepared(lib, P, key, dev, stream)
            wsb = lib.agrl_head_workspace_bytes(ctypes.byref(P), B, seq_len)
            ws = self._ws.get((dev, stream))                         # one workspace per (device, stream)
            if ws is None or ws.numel() < wsb:
                ws = self._ws[(dev, stream)] = torch.empty(wsb, dtype=torch.uint8, device=dev)
            if out is None:
                out = torch.empty(B, 2 * C, dtype=torch.float32, device=dev)
            else:
                assert out.dtype == torch.float32 and out.device == dev and tuple(out.shape) == (B, 2 * C) \
                    and out.stride(1) == 1, 'out must be a (B, 2C) fp32 tensor on the input device'
            nodes = torch.empty(B, V, C, dtype=torch.float32, device=dev) if return_nodes else None
            entry = lib.agrl_head_forward_compact_dev if compact else lib.agrl_head_forward_dev
            _lib.check(entry(
                ctypes.byref(P), prepared.data_ptr(), x4_1.data_ptr(), x4_2.data_ptr(),
                adj.data_ptr() if self.use_pose else None, out.data_ptr(), out.stride(0),
                nodes.data_ptr() if return_nodes else None, B, seq_len, h, w,
                ws.data_ptr(), wsb, stream))
        return (out, nodes) if return_nodes else out

    def forward_clips(self, imgs, adj, pool='avg'):
        """The dense / skipdense branch of the reference's test() (train_vidreid_xent_htri.py:461-476):
        imgs (b, n, s, c, h, w), adj (b, n, V, V) -> clip-pooled features (b, 4096)."""
        b, n, s, c, h, w = imgs.size()
        feats = self.forward(imgs.view(b * n, s, c, h, w), adj.view(b * n, adj.size(-1), adj.size(-1)))
        return pool_clips(feats, n, pool)

    def forward(self, x, adj, *args):
        if self.training:
            raise NotImplementedError('agrl.pytorch_b200 covers the test-time path only (model.eval()); '
                                      'the training branches of vmgn.py:323-357 are out of scope')
        B, S, C, H, W = x.size()
        x4_1, x4_2 = self.featuremaps(x.view(B * S, C, H, W))
        return self.head(x4_1, x4_2, adj, S)


def pool_clips(features, num_clips, pool='avg'):
    """Clip pooling of the reference's dense / skipdense test sampling (train_vidreid_xent_htri.py:471-476):
    features (tracklets * num_clips, D) on a CUDA device, the clips of a tracklet consecutive ->
    (tracklets, D); ``pool='avg'`` is torch.mean over the clips, anything else torch.max (as in the reference)."""
    lib = _lib.require_device()
    if not features.is_cuda:
        raise RuntimeError('agrl.pytorch_b200 has no CPU path: move the features to a B200')
    assert features.dim() == 2 and features.size(0) % num_clips == 0
    f = features.detach().float()
    if f.stride(1) != 1:
        f = f.contiguous()
    t, d = f.size(0) // num_clips, f.size(1)
    out = torch.empty(t, d, dtype=torch.float32, device=f.device)
    with torch.cuda.device(f.device):
        _lib.check(lib.agrl_clip_pool_dev(f.data_ptr(), f.stride(0), t, num_clips, d,
                                          _lib.CLIP_POOL_AVG if pool == 'avg' else _lib.CLIP_POOL_MAX,
                                          out.data_ptr(), out.stride(0), torch.cuda.current_stream(f.device).cuda_stream))
    return out


def vmgn(num_classes, loss, last_stride, num_split, num_gb, num_scale, pyramid_part, use_pose, learn_graph,
         consistent_loss=False, **kwargs):
    """Factory with the reference's signature (vmgn.py:373-389); ``last_stride`` and ``num_scale``
    are accepted and ignored there too (:224)."""
    return VMGN(num_classes=num_classes, loss=loss, num_split=num_split, pyramid_part=pyramid_part,
                num_gb=num_gb, use_pose=use_pose, learn_graph=learn_graph,
                consistent_loss=consistent_loss, **kwargs)
