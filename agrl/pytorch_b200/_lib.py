"""ctypes binding of libagrl_b200.so (the C ABI declared in include/agrl_b200.h).

The library is the product; this module only loads it and declares argument types.  There is no
CPU fallback anywhere in agrl.pytorch_b200: if the shared library is missing, or no sm_100 device
is present, every compute call raises.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, 'libagrl_b200.so')

OK = 0
E_INVALID, E_NO_DEVICE, E_CUDA, E_WORKSPACE, E_UNSUPPORTED = -1, -2, -3, -4, -5
E_NO_VALID_QUERY, E_ZERO_DIVISION, E_LABEL_RANGE = -6, -7, -8
ST_NO_VALID_QUERY, ST_ZERO_DIVISION, ST_LABEL_RANGE, ST_TOPK_OVERFLOW = 1, 2, 4, 8
METRIC_EUCLIDEAN, METRIC_COSINE = 0, 1
SPLIT_BF16X3, SPLIT_BF16X2, SPLIT_FP16X1, SPLIT_FP16_E4M3, SPLIT_FP16X2 = 3, 2, 1, 4, 5
CLIP_POOL_AVG, CLIP_POOL_MAX = 0, 1
MAPS_FP32, MAPS_BF16, MAPS_FP16 = 0, 1, 2
HEAD_MAX_LAYERS = 4

c_i64, c_i32, c_sz, c_vp, c_int = ctypes.c_int64, ctypes.c_int32, ctypes.c_size_t, ctypes.c_void_p, ctypes.c_int


class HeadParams(ctypes.Structure):
    """struct agrl_head_params (include/agrl_b200.h)."""
    _fields_ = [
        ('channels', c_i32), ('num_layers', c_i32), ('use_pose', c_i32), ('learn_graph', c_i32),
        ('gamma', ctypes.c_float), ('leaky_slope', ctypes.c_float), ('bn_eps', ctypes.c_float),
        ('split', c_i32),
        ('linear_weight', c_vp * HEAD_MAX_LAYERS),
        ('bn_weight', c_vp * HEAD_MAX_LAYERS), ('bn_bias', c_vp * HEAD_MAX_LAYERS),
        ('bn_mean', c_vp * HEAD_MAX_LAYERS), ('bn_var', c_vp * HEAD_MAX_LAYERS),
        ('global_bn', c_vp * 4), ('att_bn', c_vp * 4),
        ('maps_nhwc', c_i32),
        ('lowrank_off', c_i32), ('pool_register_loads', c_i32), ('pool_stages', c_i32), ('pool_no_l2_hint', c_i32),
        ('gemm_no_pair', c_i32), ('maps_dtype', c_i32),
    ]


_SIGNATURES = {
    'agrl_abi_version': (c_int, []),
    'agrl_status_string': (ctypes.c_char_p, [c_int]),
    'agrl_last_cuda_error': (ctypes.c_char_p, []),
    'agrl_device_ok': (c_int, []),
    'agrl_launch_count': (ctypes.c_uint64, []),
    'agrl_profile_begin': (c_int, [c_vp]),
    'agrl_profile_end': (c_int, [ctypes.c_char_p, c_sz]),
    'agrl_rank_workspace_bytes': (c_sz, [c_i64, c_i64, c_i64]),
    'agrl_rank_market1501_dev': (c_int, [c_vp, c_i64, c_vp, c_vp, c_vp, c_vp, c_i64, c_i64, c_i64,
                                         c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_sz, c_vp]),
    'agrl_rank_mars_dev': (c_int, [c_vp, c_i64, c_vp, c_vp, c_vp, c_vp, c_i64, c_i64, c_i64,
                                   c_vp, c_vp, c_vp, c_vp, c_vp, c_sz, c_vp]),
    'agrl_rank_mars_partial_dev': (c_int, [c_vp, c_i64, c_vp, c_vp, c_vp, c_vp, c_i64, c_i64, c_i64, c_i64,
                                           c_vp, c_vp, c_vp, c_vp, c_vp, c_sz, c_vp]),
    'agrl_rank_mars_merge_dev': (c_int, [c_vp, c_vp, c_vp, c_i64, c_i64, c_i64, c_vp, c_vp, c_vp, c_vp,
                                         c_vp, c_sz, c_vp]),
    'agrl_rank_market1501_count_dev': (c_int, [c_vp, c_vp, c_vp, c_vp, c_i64, c_i64, c_vp, c_vp, c_vp, c_sz, c_vp]),
    'agrl_rank_market1501_gather_dev': (c_int, [c_vp, c_i64, c_vp, c_vp, c_vp, c_vp, c_i64, c_i64, c_i64, c_i64,
                                                c_vp, c_vp, c_vp, c_vp, c_vp, c_sz, c_vp]),
    'agrl_rank_market1501_list_len': (c_i64, [c_i64, c_i64]),
    'agrl_rank_market1501_bin_dev': (c_int, [c_vp, c_i64, c_i64, c_i64, c_i64, c_vp, c_i64, c_i64, c_vp, c_vp, c_vp]),
    'agrl_rank_market1501_finalize_workspace_bytes': (c_sz, [c_i64, c_i64, c_i64, c_i64]),
    'agrl_rank_market1501_finalize_dev': (c_int, [c_vp, c_vp, c_vp, c_vp, c_i64, c_i64, c_i64, c_i64, c_i64,
                                                  c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_sz, c_vp]),
    'agrl_rank_market1501_host': (c_int, [c_vp, c_vp, c_vp, c_vp, c_vp, c_i64, c_i64, c_i64,
                                          c_vp, c_vp, c_vp, c_vp, c_vp]),
    'agrl_rank_mars_host': (c_int, [c_vp, c_vp, c_vp, c_vp, c_vp, c_i64, c_i64, c_i64, c_vp, c_vp, c_vp]),
    'agrl_distance_workspace_bytes': (c_sz, [c_i64, c_i64, c_i64, c_int]),
    'agrl_distance_dev': (c_int, [c_vp, c_i64, c_vp, c_i64, c_vp, c_i64, c_i64, c_i64, c_i64, c_int, c_int,
                                  c_vp, c_sz, c_vp]),
    'agrl_distance_operand_bytes': (c_sz, [c_i64, c_i64, c_int]),
    'agrl_distance_prepare_operand_dev': (c_int, [c_vp, c_i64, c_i64, c_i64, c_int, c_int, c_vp, c_sz, c_vp]),
    'agrl_distance_prepared_dev': (c_int, [c_vp, c_i64, c_vp, c_i64, c_i64, c_int, c_int, c_vp, c_i64, c_vp]),
    'agrl_distance_host': (c_int, [c_vp, c_vp, c_vp, c_i64, c_i64, c_i64, c_int, c_int]),
    'agrl_distance_topk_workspace_bytes': (c_sz, [c_i64]),
    'agrl_distance_topk_dev': (c_int, [c_vp, c_i64, c_vp, c_i64, c_i64, c_int, c_int, c_i64, c_i64, c_vp, c_vp, c_vp, c_sz, c_vp]),
    'agrl_rank_mars_classify_workspace_bytes': (c_sz, [c_i64, c_i64]),
    'agrl_rank_mars_classify_dev': (c_int, [c_vp, c_vp, c_vp, c_vp, c_vp, c_i64, c_i64, c_i64, c_i64, c_vp, c_vp, c_vp,
                                            c_vp, c_sz, c_vp]),
    'agrl_pose_part_masks_dev': (c_int, [c_vp, c_vp, c_vp, c_i64, c_i32, c_i32, ctypes.c_double, c_vp, c_vp]),
    'agrl_pose_adjacency_dev': (c_int, [c_vp, c_i64, c_i32, c_vp, c_vp]),
    'agrl_head_forward_compact_dev': (c_int, [ctypes.POINTER(HeadParams), c_vp, c_vp, c_vp, c_vp, c_vp, c_i64, c_vp,
                                              c_i64, c_i32, c_i32, c_i32, c_vp, c_sz, c_vp]),
    'agrl_rerank_workspace_bytes': (c_sz, [c_i64, c_i64, c_i64, c_i64]),
    'agrl_rerank_dev': (c_int, [c_vp, c_i64, c_vp, c_i64, c_vp, c_i64, c_i64, c_i64, c_i64, c_i64, ctypes.c_double,
                                c_vp, c_i64, c_vp, c_sz, c_vp]),
    'agrl_rerank_shard_workspace_bytes': (c_sz, [c_i64, c_i64, c_i64, c_i64, c_i64]),
    'agrl_rerank_shard_rows_dev': (c_int, [c_vp, c_i64, c_vp, c_i64, c_vp, c_i64, c_i64, c_i64, c_i64, c_i64, c_i64, c_i64,
                                           c_i64, c_i64, c_vp, c_vp, c_sz, c_vp]),
    'agrl_rerank_shard_expand_dev': (c_int, [c_vp, c_i64, c_i64, c_i64, c_i64, c_i64, c_i64, c_vp, c_vp, c_vp,
                                             c_vp, c_sz, c_vp]),
    'agrl_rerank_shard_finish_dev': (c_int, [c_vp, c_vp, c_vp, c_vp, c_i64, c_i64, c_i64, c_i64, c_i64, c_i64,
                                             ctypes.c_double, c_vp, c_i64, c_vp, c_sz, c_vp]),
    'agrl_clip_pool_dev': (c_int, [c_vp, c_i64, c_i64, c_i64, c_i64, c_int, c_vp, c_i64, c_vp]),
    'agrl_head_prepared_bytes': (c_sz, [ctypes.POINTER(HeadParams)]),
    'agrl_head_prepare_dev': (c_int, [ctypes.POINTER(HeadParams), c_vp, c_sz, c_vp]),
    'agrl_head_workspace_bytes': (c_sz, [ctypes.POINTER(HeadParams), c_i64, c_i32]),
    'agrl_head_forward_dev': (c_int, [ctypes.POINTER(HeadParams), c_vp, c_vp, c_vp, c_vp, c_vp, c_i64, c_vp,
                                      c_i64, c_i32, c_i32, c_i32, c_vp, c_sz, c_vp]),
}

_lib = None


class AgrlError(RuntimeError):
    def __init__(self, code, text):
        super().__init__('libagrl_b200: %s (code %d)' % (text, code))
        self.code = code


def load(build_if_missing=True):
    """Load libagrl_b200.so (building it in-tree with nvcc when absent).  Raises if it cannot."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH) and build_if_missing:
        from . import build as _build
        _build.build()
    if not os.path.exists(LIB_PATH):
        raise ImportError('libagrl_b200.so is not built (python -m agrl.pytorch_b200.build); '
                          'agrl.pytorch_b200 has no CPU fallback')
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in _SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError if the ABI and this table ever diverge
        fn.restype, fn.argtypes = res, args
    if lib.agrl_abi_version() != 2:
        raise ImportError('libagrl_b200.so ABI version mismatch')
    _lib = lib
    return lib


def planes_of_distance_split(split):
    """16-bit planes per row of a prepared distance operand (csrc/distance.cu planes_of)."""
    return 2 if split == SPLIT_FP16X2 else int(split)


def exported_names():
    return sorted(_SIGNATURES)


def check(code):
    """Translate an ABI return code into the exception the reference would raise."""
    if code == OK:
        return
    lib = load()
    text = lib.agrl_status_string(code).decode()
    if code == E_NO_VALID_QUERY:
        raise AssertionError(text)                      # rank_cy.pyx:227 / rank.py:144
    if code == E_ZERO_DIVISION:
        raise ZeroDivisionError('division by zero')     # rank.py:203
    if code == E_CUDA:
        text += ': ' + lib.agrl_last_cuda_error().decode()
    if code == E_INVALID:
        raise ValueError(text)
    raise AgrlError(code, text)


def require_device():
    """Fail loudly when the CUDA path cannot run (no silent fallback)."""
    lib = load()
    rc = lib.agrl_device_ok()
    if rc != OK:
        raise AgrlError(rc, lib.agrl_status_string(rc).decode())
    return lib


def launch_count():
    return int(load().agrl_launch_count())


class profile(object):
    """Context manager around agrl_profile_begin/_end: ``with profile(stream) as p: ...`` then
    ``p.kernels`` is a list of (kernel name, milliseconds) in launch order."""

    def __init__(self, stream=None):
        self.stream, self.kernels = stream, []

    def __enter__(self):
        check(load().agrl_profile_begin(self.stream))
        return self

    def __exit__(self, *exc):
        buf = ctypes.create_string_buffer(1 << 20)
        rc = load().agrl_profile_end(buf, len(buf))
        if exc[0] is None:
            check(rc)
        self.kernels = [(k, float(v)) for k, v in (item.split(':') for item in buf.value.decode().split(';') if item)]
        return False

    def totals(self):
        out = {}
        for k, ms in self.kernels:
            n, t = out.get(k, (0, 0.0))
            out[k] = (n + 1, t + ms)
        return out
