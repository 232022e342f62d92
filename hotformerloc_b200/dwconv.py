"""Octree depth-wise convolution with backward: a drop-in for the reference's
``dwconv`` package (libs/dwconv: ``dwconv.core`` + ``dwconv/nn.py``), fp32 on
the kernels of csrc/dwconv.cu.

The three ``core`` ops keep the reference's pybind signatures and also take
int32 neighbour tables (``Octree.ne_table``).  Replacing the reference's
``from .core import ...`` line (libs/dwconv/dwconv/nn.py) with an import from
this module is enough to run its autograd function and module on these kernels;
:func:`octree_dwconv` and :class:`OctreeDWConv` are the same two on top.
Every op runs on the current torch stream and raises ``HflError`` on bad input.
"""
from __future__ import annotations

import torch

from . import native as N
from .native import HflError
from .octree import LUT_KERNEL

__all__ = ['dwconv_forward_backward', 'dwconv_weight_backward', 'inverse_neigh', 'octree_dwconv',
           'OctreeDWConv', 'OctreeDWConvFunction']

MAX_TAPS = 27


def _require(cond: bool, msg: str):
    if not cond:
        raise HflError(msg)


def _check_f32(name: str, t: torch.Tensor, dim: int):
    _require(isinstance(t, torch.Tensor), f'{name} must be a tensor')
    _require(t.is_cuda, f'{name} must be a CUDA tensor')
    _require(t.dtype == torch.float32, f'{name} must be float32, got {t.dtype}')
    _require(t.dim() == dim, f'{name} must have {dim} dimensions, got shape {tuple(t.shape)}')
    _require(t.is_contiguous(), f'{name} must be contiguous')


def _check_table(neigh: torch.Tensor) -> int:
    """Validates a (rows, K) neighbour table; returns 1 for int64, 0 for int32."""
    _require(isinstance(neigh, torch.Tensor), 'neigh must be a tensor')
    _require(neigh.is_cuda, 'neigh must be a CUDA tensor')
    _require(neigh.dtype in (torch.int64, torch.int32), f'neigh must be int64 or int32, got {neigh.dtype}')
    _require(neigh.dim() == 2 and 1 <= neigh.shape[1] <= MAX_TAPS,
             f'neigh must be (rows, K) with 1 <= K <= {MAX_TAPS}, got shape {tuple(neigh.shape)}')
    _require(neigh.is_contiguous(), 'neigh must be contiguous')
    return int(neigh.dtype == torch.int64)


def _same_device(*ts):
    dev = ts[0].device
    _require(all(t.device == dev for t in ts), 'all tensors must be on the same device')
    return dev


def _check_weight(weight: torch.Tensor, K: int, C: int):
    _check_f32('weight', weight, 3)
    _require(tuple(weight.shape) == (K, 1, C), f'weight must be (K, 1, C) = {(K, 1, C)}, got {tuple(weight.shape)}')


def _dwconv(data, weight, neigh, i64) -> torch.Tensor:
    K, C = neigh.shape[1], data.shape[1]
    out = torch.empty((neigh.shape[0], C), dtype=torch.float32, device=data.device)
    N.check(N.lib().hfl_dwconv(N.ptr(data), N.ptr(neigh), i64, N.ptr(weight), neigh.shape[0], data.shape[0],
                               K, C, N.ptr(out), N.stream()))
    return out


def _inverse(neigh: torch.Tensor, n_data: int, i64: int) -> torch.Tensor:
    out = torch.empty((n_data, neigh.shape[1]), dtype=neigh.dtype, device=neigh.device)
    N.check(N.lib().hfl_dwconv_inverse(N.ptr(neigh), i64, neigh.shape[0], n_data, neigh.shape[1], N.ptr(out),
                                       N.stream()))
    return out


def dwconv_forward_backward(data: torch.Tensor, weight: torch.Tensor, neigh: torch.Tensor) -> torch.Tensor:
    """out[i, c] = sum_k weight[k, 0, c] * data[neigh[i, k], c] over the taps with neigh >= 0.
    data (N_in, C) float32, weight (K, 1, C) float32, neigh (N, K) int64 or int32 -> (N, C) float32.
    With ``inverse_neigh(neigh)`` and the output gradient it is the input gradient."""
    i64 = _check_table(neigh)
    _check_f32('data', data, 2)
    _check_weight(weight, neigh.shape[1], data.shape[1])
    with torch.cuda.device(_same_device(data, weight, neigh)):
        return _dwconv(data, weight, neigh, i64)


def inverse_neigh(neigh: torch.Tensor) -> torch.Tensor:
    """ineigh[neigh[i, k], k] = i, -1 where no row points; same shape and dtype as ``neigh``.
    If several rows point to one (j, k) -- never in a stride-1 octree table -- the largest i wins."""
    i64 = _check_table(neigh)
    with torch.cuda.device(neigh.device):
        return _inverse(neigh, neigh.shape[0], i64)


def _wgrad(grad, data, neigh, i64) -> torch.Tensor:
    L = N.lib()
    n, K, C = neigh.shape[0], neigh.shape[1], data.shape[1]
    dw = torch.empty((K, 1, C), dtype=torch.float32, device=data.device)
    ws_bytes = int(L.hfl_dwconv_wgrad_workspace_bytes(n, K, C))
    ws = torch.empty(max(ws_bytes, 1), dtype=torch.uint8, device=data.device)
    N.check(L.hfl_dwconv_wgrad(N.ptr(grad), N.ptr(data), N.ptr(neigh), i64, n, data.shape[0], K, C, N.ptr(dw),
                               N.ptr(ws), ws_bytes, N.stream()))
    return dw


def dwconv_weight_backward(grad: torch.Tensor, data: torch.Tensor, neigh: torch.Tensor) -> torch.Tensor:
    """dw[k, 0, c] = sum_i grad[i, c] * data[neigh[i, k], c]: grad (N, C), data (N_in, C) float32,
    neigh (N, K) int64 or int32 -> (K, 1, C) float32.  Bit-reproducible run to run and across GPUs."""
    i64 = _check_table(neigh)
    _check_f32('grad', grad, 2)
    _check_f32('data', data, 2)
    _require(grad.shape == (neigh.shape[0], data.shape[1]),
             f'grad must be (N, C) = {(neigh.shape[0], data.shape[1])}, got {tuple(grad.shape)}')
    with torch.cuda.device(_same_device(grad, data, neigh)):
        return _wgrad(grad, data, neigh, i64)


class OctreeDWConvFunction(torch.autograd.Function):
    """Autograd form (libs/dwconv/dwconv/nn.py:17): the input gradient is the forward op over the
    inverse table, the weight gradient the deterministic reduction."""

    @staticmethod
    def forward(ctx, data, weights, neigh):
        data, weights, neigh = data.contiguous(), weights.contiguous(), neigh.contiguous()
        out = dwconv_forward_backward(data, weights, neigh)
        ctx.save_for_backward(data, weights, neigh)
        return out

    @staticmethod
    def backward(ctx, grad):
        data, weights, neigh = ctx.saved_tensors
        grad = grad.contiguous()
        i64 = _check_table(neigh)
        _check_f32('grad', grad, 2)
        grad_d = grad_w = None
        with torch.cuda.device(data.device):
            if ctx.needs_input_grad[0]:
                grad_d = _dwconv(grad, weights, _inverse(neigh, data.shape[0], i64), i64)
            if ctx.needs_input_grad[1]:
                grad_w = _wgrad(grad, data, neigh, i64)
        return grad_d, grad_w, None


octree_dwconv = OctreeDWConvFunction.apply


def _kernel_str(kernel_size) -> str:
    ks = [int(k) for k in kernel_size]
    if len(ks) == 1:
        ks = ks * 3
    return ''.join(str(k) for k in ks)


class OctreeDWConv(torch.nn.Module):
    """``dwconv.OctreeDWConv`` (libs/dwconv/dwconv/nn.py:49): depth-wise octree conv with stride 1.
    Parameters ``weights`` (kdim, 1, C) (xavier-uniform) and, with ``use_bias``, ``bias`` (C,) --
    the state_dict layout of ``ocnn.nn.OctreeDWConv``.  ``forward`` reads the neighbour table through
    ``octree.get_neigh(depth, kernel, 1, nempty)``, so any ocnn-like octree works."""

    def __init__(self, channels: int, kernel_size=[3], nempty: bool = False, use_bias: bool = False):
        super().__init__()
        self.in_channels = self.out_channels = channels
        self.kernel_size = list(kernel_size)
        self.kernel = _kernel_str(kernel_size)
        if self.kernel not in LUT_KERNEL:
            raise ValueError(f'unsupported kernel_size {kernel_size}')
        self.kdim = len(LUT_KERNEL[self.kernel])
        self.stride, self.nempty, self.use_bias = 1, nempty, use_bias
        self.weights = torch.nn.Parameter(torch.empty(self.kdim, 1, channels))
        torch.nn.init.xavier_uniform_(self.weights)
        if use_bias:
            self.bias = torch.nn.Parameter(torch.zeros(channels))

    def forward(self, data: torch.Tensor, octree, depth: int) -> torch.Tensor:
        neigh = octree.get_neigh(depth, self.kernel, self.stride, self.nempty)
        out = octree_dwconv(data, self.weights, neigh)
        if self.use_bias:
            out = out + self.bias
        return out

    def extra_repr(self) -> str:
        return (f'channels={self.in_channels}, kernel_size={self.kernel_size}, nempty={self.nempty}, '
                f'use_bias={self.use_bias}')
