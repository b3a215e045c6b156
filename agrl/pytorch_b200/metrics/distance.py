"""Mirror of torchreid/metrics/distance.py: ``compute_distance_matrix`` with the reference's
signature, checks and error behaviour (distance.py:11-56), computed by the tcgen05 GEMM of
libagrl_b200 (csrc/distance.cu).

CPU tensors in -> CPU tensor out (the reference's test() passes CPU tensors,
train_vidreid_xent_htri.py:477,507,520); the work still happens on the GPU, through the
host-buffer entry point.  CUDA tensors in -> CUDA tensor out with no host round trip.
"""
import torch

from .. import _lib

_METRICS = {'euclidean': _lib.METRIC_EUCLIDEAN, 'cosine': _lib.METRIC_COSINE}
_ws_cache = {}


def _workspace(dev, nbytes):
    """Operand-plane scratch, one buffer per (device, stream): two streams (or DataParallel threads) working on the same
    device never share planes, and a buffer is only ever reused / released in the order of the stream that uses it."""
    key = (dev, torch.cuda.current_stream(dev).cuda_stream)
    ws = _ws_cache.get(key)
    if ws is None or ws.numel() < nbytes:
        ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)       # allocated on (and tied to) the current stream
        _ws_cache[key] = ws
    return ws


def _check_metric(metric):
    """The library's code of a metric name; ValueError as distance.py:50-54 for any other name."""
    if metric not in _METRICS:
        raise ValueError(
            'Unknown distance metric: {}. '
            'Please choose either "euclidean" or "cosine"'.format(metric)
        )
    return _METRICS[metric]


def compute_distance_matrix(input1, input2, metric='euclidean', split=_lib.SPLIT_FP16X2):
    """A wrapper function for computing distance matrix (distance.py:11).

    Args:
        input1 (torch.Tensor): 2-D feature matrix.
        input2 (torch.Tensor): 2-D feature matrix.
        metric (str, optional): "euclidean" or "cosine".  Default is "euclidean".
    Returns:
        torch.Tensor: distance matrix (squared euclidean, or 1 - cosine similarity).
    """
    # check input (distance.py:39-44)
    assert isinstance(input1, torch.Tensor)
    assert isinstance(input2, torch.Tensor)
    assert input1.dim() == 2, 'Expected 2-D tensor, but got {}-D'.format(input1.dim())
    assert input2.dim() == 2, 'Expected 2-D tensor, but got {}-D'.format(input2.dim())
    assert input1.size(1) == input2.size(1)
    code = _check_metric(metric)
    lib = _lib.require_device()
    m, n, d = input1.size(0), input2.size(0), input1.size(1)
    if input1.is_cuda != input2.is_cuda:
        raise RuntimeError('Expected all tensors to be on the same device')
    if not input1.is_cuda:
        a = input1.detach().to(torch.float32).contiguous()
        b = input2.detach().to(torch.float32).contiguous()
        out = torch.empty(m, n, dtype=torch.float32)
        if m and n:
            _lib.check(lib.agrl_distance_host(a.data_ptr(), b.data_ptr(), out.data_ptr(), m, n, d, code, split))
        return out
    dev = input1.device
    a = input1.detach().to(torch.float32)
    b = input2.detach().to(device=dev, dtype=torch.float32)
    if a.stride(1) != 1:
        a = a.contiguous()
    if b.stride(1) != 1:
        b = b.contiguous()
    out = torch.empty(m, n, dtype=torch.float32, device=dev)
    if m == 0 or n == 0:
        return out
    wsb = lib.agrl_distance_workspace_bytes(m, n, d, split)
    ws = _workspace(dev, wsb)
    _lib.call(dev, lib.agrl_distance_dev, a.data_ptr(), a.stride(0), b.data_ptr(), b.stride(0),
              out.data_ptr(), out.stride(0), m, n, d, code, split, ws.data_ptr(), wsb)
    return out


class PreparedOperand(object):
    """A feature matrix already split into the GEMM's bf16 operand planes (+ norms) on its device.

    Retrieval against a fixed gallery prepares the gallery once and reuses it for every query batch
    (``agrl_distance_prepare_operand_dev`` / ``agrl_distance_prepared_dev``)."""

    def __init__(self, x, metric='euclidean', split=_lib.SPLIT_FP16X2):
        assert isinstance(x, torch.Tensor) and x.dim() == 2 and x.is_cuda
        code = _check_metric(metric)
        lib = _lib.require_device()
        x = x.detach().to(torch.float32)
        if x.stride(1) != 1:
            x = x.contiguous()
        self.rows, self.dim, self.metric, self.split, self.device = x.size(0), x.size(1), metric, split, x.device
        nbytes = lib.agrl_distance_operand_bytes(self.rows, self.dim, split)
        self.buf = torch.empty(max(nbytes, 16), dtype=torch.uint8, device=x.device)
        _lib.call(x.device, lib.agrl_distance_prepare_operand_dev, x.data_ptr(), x.stride(0), self.rows, self.dim, code,
                  split, self.buf.data_ptr(), nbytes)


    def rows_view(self, r0, r1):
        """Rows [r0, r1) as an operand of their own (a copy of those rows' planes and norms; the plane layout
        [P][rows][K_pad] is not sliceable in place)."""
        lib = _lib.require_device()
        k_pad = (self.dim + 63) // 64 * 64
        n = r1 - r0
        v = object.__new__(PreparedOperand)
        v.rows, v.dim, v.metric, v.split, v.device = n, self.dim, self.metric, self.split, self.device
        nbytes = lib.agrl_distance_operand_bytes(n, self.dim, self.split)
        v.buf = torch.empty(max(nbytes, 16), dtype=torch.uint8, device=self.device)
        P = _lib.planes_of_distance_split(self.split)
        plane_b = self.rows * k_pad * 2
        src = self.buf[:P * plane_b].view(P, self.rows, k_pad * 2)
        v.buf[:P * n * k_pad * 2].view(P, n, k_pad * 2).copy_(src[:, r0:r1])
        # after the planes: squared norms, then the per-row 1 / scale of the fp16 x 2 split (256-byte aligned arrays)
        off_src = (P * plane_b + 255) // 256 * 256
        off_dst = (P * n * k_pad * 2 + 255) // 256 * 256
        for _ in range(2):
            v.buf[off_dst:off_dst + 4 * n].copy_(self.buf[off_src + 4 * r0:off_src + 4 * r1])
            off_src = (off_src + 4 * self.rows + 255) // 256 * 256
            off_dst = (off_dst + 4 * n + 255) // 256 * 256
        return v


def distance_prepared(q, g, out=None):
    """Distance matrix between two PreparedOperand (same metric, split, dim, device)."""
    assert isinstance(q, PreparedOperand) and isinstance(g, PreparedOperand)
    assert (q.metric, q.split, q.dim, q.device) == (g.metric, g.split, g.dim, g.device)
    lib = _lib.require_device()
    if out is None:
        out = torch.empty(q.rows, g.rows, dtype=torch.float32, device=q.device)
    assert out.shape == (q.rows, g.rows) and out.stride(1) == 1 and out.dtype == torch.float32
    if q.rows and g.rows:
        _lib.call(q.device, lib.agrl_distance_prepared_dev, q.buf.data_ptr(), q.rows, g.buf.data_ptr(), g.rows, q.dim,
                  _METRICS[q.metric], q.split, out.data_ptr(), out.stride(0))
    return out
