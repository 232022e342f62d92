"""Octree convolution with backward for training: ``ocnn.nn.OctreeConv`` for the two shapes the model uses
(3x3x3 stride 1 in ``PatchEmbed``, 2x2x2 stride 2 in every downsample, both nempty), fp32 on the kernels
of csrc/octree_conv_train.cu.

:func:`octree_conv` is the autograd function; :class:`OctreeConv` keeps ocnn's constructor and
``weights`` / ``bias`` parameters, so the ``*.conv.*`` tensors of a checkpoint load into it.  The input
gradient is the forward kernel over the inverse table (``hfl_dwconv_inverse``) with per-tap transposed
weights; the weight gradient is a fixed-order reduction.  Every op runs on the current torch stream and
raises ``HflError`` on bad input before any launch.
"""
from __future__ import annotations

import torch

from . import native as N
from .dwconv import _check_f32, _inverse, _kernel_str, _require, _same_device
from .octree import LUT_KERNEL, Octree

__all__ = ['octree_conv', 'OctreeConv', 'OctreeConvFunction']

MAX_CHANNELS = 256
SUPPORTED = {('333', 1), ('222', 2)}      # (kernel, stride) of OctreeConvNormRelu and Downsample


def _check_table(neigh: torch.Tensor) -> int:
    """Validates a (rows, K) table with K in {8, 27}; returns 1 for int64, 0 for int32."""
    _require(isinstance(neigh, torch.Tensor), 'neigh must be a tensor')
    _require(neigh.is_cuda, 'neigh must be a CUDA tensor')
    _require(neigh.dtype in (torch.int64, torch.int32), f'neigh must be int64 or int32, got {neigh.dtype}')
    _require(neigh.dim() == 2 and neigh.shape[1] in (8, 27),
             f'neigh must be (rows, K) with K in (8, 27), got shape {tuple(neigh.shape)}')
    _require(neigh.is_contiguous(), 'neigh must be contiguous')
    return int(neigh.dtype == torch.int64)


def _check_args(data, weights, neigh) -> int:
    i64 = _check_table(neigh)
    _check_f32('data', data, 2)
    _check_f32('weights', weights, 3)
    K, Cin, Cout = weights.shape
    _require(K == neigh.shape[1], f'weights must have K = {neigh.shape[1]} taps, got shape {tuple(weights.shape)}')
    _require(1 <= Cin <= MAX_CHANNELS and 1 <= Cout <= MAX_CHANNELS,
             f'Cin and Cout must be in [1, {MAX_CHANNELS}], got {Cin} and {Cout}')
    _require(data.shape[1] == Cin, f'data must have Cin = {Cin} channels, got shape {tuple(data.shape)}')
    _same_device(data, weights, neigh)
    return i64


def _conv(data, w, neigh, i64, n_out) -> torch.Tensor:
    K, Cin, Cout = w.shape
    out = torch.empty((n_out, Cout), dtype=torch.float32, device=data.device)
    N.check(N.lib().hfl_octree_conv_train_fwd(N.ptr(data), N.ptr(neigh), i64, N.ptr(w), n_out, data.shape[0],
                                              K, Cin, Cout, N.ptr(out), N.stream()))
    return out


def _wgrad(data, neigh, i64, grad, K, Cin, Cout) -> torch.Tensor:
    L = N.lib()
    n = neigh.shape[0]
    dw = torch.empty((K, Cin, Cout), dtype=torch.float32, device=data.device)
    ws_bytes = int(L.hfl_octree_conv_train_wgrad_workspace_bytes(n, K, Cin, Cout))
    ws = torch.empty(max(ws_bytes, 1), dtype=torch.uint8, device=data.device)
    N.check(L.hfl_octree_conv_train_wgrad(N.ptr(data), N.ptr(neigh), i64, N.ptr(grad), n, data.shape[0], K, Cin,
                                          Cout, N.ptr(dw), N.ptr(ws), ws_bytes, N.stream()))
    return dw


class OctreeConvFunction(torch.autograd.Function):
    """out[i] = sum_k data[neigh[i, k]] @ weights[k] over the taps with neigh in [0, n_in)."""

    @staticmethod
    def forward(ctx, data, weights, neigh):
        data, weights, neigh = data.contiguous(), weights.contiguous(), neigh.contiguous()
        i64 = _check_args(data, weights, neigh)
        with torch.cuda.device(data.device):
            out = _conv(data, weights, neigh, i64, neigh.shape[0])
        ctx.save_for_backward(data, weights, neigh)
        return out

    @staticmethod
    def backward(ctx, grad):
        data, weights, neigh = ctx.saved_tensors
        grad = grad.contiguous()
        i64 = _check_table(neigh)
        _check_f32('grad', grad, 2)
        K, Cin, Cout = weights.shape
        _require(tuple(grad.shape) == (neigh.shape[0], Cout),
                 f'grad must be {(neigh.shape[0], Cout)}, got {tuple(grad.shape)}')
        grad_d = grad_w = None
        with torch.cuda.device(data.device):
            if ctx.needs_input_grad[0]:
                inv = _inverse(neigh, data.shape[0], i64)
                grad_d = _conv(grad, weights.transpose(1, 2).contiguous(), inv, i64, data.shape[0])
            if ctx.needs_input_grad[1]:
                grad_w = _wgrad(data, neigh, i64, grad, K, Cin, Cout)
        return grad_d, grad_w, None


octree_conv = OctreeConvFunction.apply


class OctreeConv(torch.nn.Module):
    """``ocnn.nn.OctreeConv`` for kernel_size [3] with stride 1 and [2] with stride 2, nempty=True.
    Parameters ``weights`` (kdim, Cin, Cout) (xavier-uniform) and, with ``use_bias``, ``bias`` (Cout,).
    ``direct_method`` and ``max_buffer`` are accepted for ocnn's signature and have no effect.
    ``forward(data, octree, depth)`` takes the input depth; on this project's :class:`Octree` it reads the
    int32 ``ne_table`` / ``child_table``, on an ocnn octree ``get_neigh``."""

    def __init__(self, in_channels: int, out_channels: int, kernel_size=[3], stride: int = 1,
                 nempty: bool = False, direct_method: bool = False, use_bias: bool = False,
                 max_buffer: int = int(2e8)):
        super().__init__()
        self.in_channels, self.out_channels = in_channels, out_channels
        self.kernel_size = list(kernel_size)
        self.kernel = _kernel_str(kernel_size)
        self.stride, self.nempty, self.use_bias = stride, nempty, use_bias
        if (self.kernel, stride) not in SUPPORTED or not nempty:
            raise ValueError(f'unsupported OctreeConv: kernel_size {kernel_size}, stride {stride}, nempty {nempty} '
                             f'(supported: [3] stride 1 and [2] stride 2, nempty=True)')
        if not (1 <= in_channels <= MAX_CHANNELS and 1 <= out_channels <= MAX_CHANNELS):
            raise ValueError(f'in_channels and out_channels must be in [1, {MAX_CHANNELS}]')
        self.kdim = len(LUT_KERNEL[self.kernel])
        self.weights = torch.nn.Parameter(torch.empty(self.kdim, in_channels, out_channels))
        torch.nn.init.xavier_uniform_(self.weights)
        if use_bias:
            self.bias = torch.nn.Parameter(torch.zeros(out_channels))

    def neigh(self, octree, depth: int) -> torch.Tensor:
        if isinstance(octree, Octree):
            return octree.ne_table(depth) if self.stride == 1 else octree.child_table(depth)
        return octree.get_neigh(depth, self.kernel, self.stride, True)

    def forward(self, data: torch.Tensor, octree, depth: int) -> torch.Tensor:
        out = octree_conv(data, self.weights, self.neigh(octree, depth))
        if self.use_bias:
            out = out + self.bias
        return out

    def extra_repr(self) -> str:
        return (f'in_channels={self.in_channels}, out_channels={self.out_channels}, '
                f'kernel_size={self.kernel_size}, stride={self.stride}, nempty={self.nempty}, '
                f'use_bias={self.use_bias}')
