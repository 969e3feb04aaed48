"""array interchange: torch CUDA tensors and DLPack exporters stay on the device; host arrays
(numpy, CPU torch) are staged through pinned memory and results come back in the caller's kind.

This is the equivalent of the reference's ``array_namespace`` switch
(/root/reference/src/iqwaveform/util.py:198-214): unknown objects raise
``TypeError('unrecognized object type')``.
"""
from __future__ import annotations

import numpy as np
import torch


class Residence:
    """remembers where the caller's array lived so that results can be returned alike"""

    def __init__(self, kind: str):
        self.kind = kind  # 'torch_cuda' | 'torch_cpu' | 'numpy'

    def give_back(self, t: torch.Tensor):
        if self.kind == 'torch_cuda':
            return t
        host = torch.empty(t.shape, dtype=t.dtype, pin_memory=True)
        host.copy_(t, non_blocking=True)
        torch.cuda.current_stream(t.device).synchronize()
        return host.numpy() if self.kind == 'numpy' else host


def from_numpy_readonly_ok(a: np.ndarray) -> torch.Tensor:
    """torch.from_numpy without the warning about read-only arrays (memory-mapped captures): the tensor is
    only ever the SOURCE of a host->device copy"""
    import warnings
    with warnings.catch_warnings():
        warnings.simplefilter('ignore', UserWarning)
        return torch.from_numpy(a)


def _device() -> torch.device:
    if not torch.cuda.is_available():
        raise RuntimeError('iqwaveform_b200 needs a CUDA device (there is no CPU fallback)')
    return torch.device('cuda', torch.cuda.current_device())


def to_device(x) -> tuple[torch.Tensor, Residence]:
    """return (device tensor, residence).  Host data is copied host->device on the current stream."""
    if isinstance(x, torch.Tensor):
        if x.is_cuda:
            return x, Residence('torch_cuda')
        dev = _device()
        src = x if x.is_pinned() else x.contiguous()
        return src.to(dev, non_blocking=True), Residence('torch_cpu')
    if isinstance(x, np.ndarray):
        dev = _device()
        return from_numpy_readonly_ok(np.ascontiguousarray(x)).to(dev, non_blocking=True), Residence('numpy')
    if hasattr(x, '__dlpack__'):
        t = torch.from_dlpack(x)
        if not t.is_cuda:
            return t.to(_device()), Residence('torch_cpu')
        return t, Residence('torch_cuda')
    raise TypeError('unrecognized object type')


def as_channels(x: torch.Tensor, axis: int) -> tuple[torch.Tensor, tuple, tuple]:
    """move `axis` last and flatten the rest into a channel axis -> (C, N) contiguous view/copy.
    Returns (x2d, leading_shape, trailing_shape) of the original layout around `axis`."""
    if axis < 0:
        axis += x.ndim
    if not 0 <= axis < x.ndim:
        raise ValueError(f'axis {axis} exceeds the number of dimensions')
    lead, trail = tuple(x.shape[:axis]), tuple(x.shape[axis + 1:])
    if trail:
        t = _transpose_time_last(x, axis, lead, trail)
        if t is not None:
            return t, lead, trail
        x = x.movedim(axis, -1)
    return unit_stride_rows(x.reshape(-1, x.shape[-1])), lead, trail


def unit_stride_rows(x2: torch.Tensor) -> torch.Tensor:
    """(C, N) rows of unit stride that do not overlap, as the kernels read them: `x2` itself when it is so laid
    out (any row pitch >= N), else a contiguous copy"""
    if x2.stride(-1) != 1 or (x2.shape[0] > 1 and x2.stride(0) < x2.shape[-1]):
        return x2.contiguous()
    return x2


def _transpose_time_last(x: torch.Tensor, axis: int, lead: tuple, trail: tuple):
    """(lead..., N, trail...) contiguous complex64 on the device -> (prod(lead) * prod(trail), N) through the
    library's tiled transpose (csrc/iqw_elementwise.cu); None when the tensor does not qualify (the caller then
    lets torch make the copy)"""
    import ctypes
    import math
    from . import _lib
    if not (x.is_cuda and x.dtype == torch.complex64 and x.is_contiguous()):
        return None
    n = x.shape[axis]
    batch, cols = math.prod(lead), math.prod(trail)
    if batch > 65535 or cols > 65535 * 32 or n == 0 or cols == 0 or batch == 0:
        return None
    out = torch.empty((batch * cols, n), dtype=torch.complex64, device=x.device)
    _lib.check(_lib.lib.iqw_transpose_c64(ctypes.c_void_p(x.data_ptr()), batch, n, cols, ctypes.c_void_p(out.data_ptr()),
                                          ctypes.c_void_p(torch.cuda.current_stream(x.device).cuda_stream)))
    return out


def restore_layout(y: torch.Tensor, lead: tuple, trail: tuple, new_axes: int) -> torch.Tensor:
    """inverse of as_channels for a result whose last `new_axes` axes replace the time axis:
    (C, *new) -> lead + new + trail"""
    new_shape = tuple(y.shape[1:])
    if not trail:
        return y.reshape(lead + new_shape)
    y = y.reshape(lead + trail + new_shape)
    nl, nt = len(lead), len(trail)
    # axes order now: lead, trail, new  ->  lead, new, trail
    perm = tuple(range(nl)) + tuple(range(nl + nt, nl + nt + new_axes)) + tuple(range(nl, nl + nt))
    return y.permute(perm)
