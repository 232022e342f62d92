"""Differentiable relay-token initialiser, fp32 on the kernels of csrc/rt_init_train.cu.

:func:`relay_token_init` is the reference's ``RelayTokenInitialiser.forward`` (hotformerloc_backbone.py:345-363)
together with ``OctreeT.compute_window_stats`` (models/octree.py:285-344) for one pyramid level: each window of
K consecutive padded rows gets the mean of its tokens that share the first token's submap (padding rows count
as zeros), and, with ADaPE, the window statistics of the node centres.  It reads the level's
``Octree.tokens(depth, n_pad)`` table instead of the reference's ``rt_init_mask`` and padded features.  The
op runs on the current torch stream and raises ``HflError`` on bad input, before any launch.
"""
from __future__ import annotations

from typing import Optional, Tuple

import torch

from . import native as N
from .native import HflError

__all__ = ['relay_token_init', 'RelayTokenInitFunction', 'ADAPE_MODES']

ADAPE_MODES = {None: 0, 'pos': 3, 'var': 6, 'cov': 9}
MIN_C, MAX_C = 32, 512
MAX_K = 4096


def _require(cond: bool, msg: str):
    if not cond:
        raise HflError(msg)


def _check_args(src, tokens, K, depth, mode):
    _require(isinstance(K, int) and 1 <= K <= MAX_K, f'K must be an int in [1, {MAX_K}], got {K!r}')
    _require(mode in (0, 3, 6, 9), f'mode must be 0, 3, 6 or 9, got {mode!r}')
    _require(isinstance(depth, int) and 0 <= depth <= 15, f'depth must be an int in [0, 15], got {depth!r}')
    _require(isinstance(src, torch.Tensor) and src.dim() == 2, 'src must be an (n, C) tensor')
    _require(src.dtype == torch.float32, f'src must be torch.float32, got {src.dtype}')
    n, C = src.shape
    _require(MIN_C <= C <= MAX_C and C % 32 == 0, f'C must be a multiple of 32 in [{MIN_C}, {MAX_C}], got {C}')
    _require(isinstance(tokens, torch.Tensor) and tokens.dtype == torch.int16 and tokens.dim() == 2
             and tokens.shape[1] == 4, 'tokens must be an (n_pad, 4) int16 tensor (Octree.tokens)')
    n_pad = tokens.shape[0]
    _require(n_pad % K == 0, f'the token rows ({n_pad}) must be a multiple of K = {K}')
    _require(n <= n_pad, f'src has {n} rows, more than the {n_pad} token rows')
    _require(src.is_cuda and tokens.is_cuda, 'src and tokens must be CUDA tensors')
    _require(src.device == tokens.device, 'src and tokens must be on the same device')
    _require(src.is_contiguous() and tokens.is_contiguous(), 'src and tokens must be contiguous')
    return n, C, n_pad // K


class RelayTokenInitFunction(torch.autograd.Function):
    """rt[w] = masked mean of src over window w (+ ADaPE statistics, not differentiable); gradient for src."""

    @staticmethod
    def forward(ctx, src, tokens, K, depth, mode):
        n, C, n_win = _check_args(src, tokens, K, depth, mode)
        dev = src.device
        with torch.cuda.device(dev):
            rt = torch.empty((n_win, C), dtype=torch.float32, device=dev)
            stats = torch.empty((n_win, mode), dtype=torch.float32, device=dev)
            N.check(N.lib().hfl_rt_init_train_fwd(N.ptr(src), N.ptr(tokens), n, n_win, K, C, depth, mode, N.ptr(rt),
                                                  N.ptr(stats) if mode else None, N.stream()))
        ctx.save_for_backward(tokens)
        ctx.args = (n, C, n_win, K)
        ctx.mark_non_differentiable(stats)
        return rt, stats

    @staticmethod
    def backward(ctx, grad_rt, grad_stats):
        tokens, = ctx.saved_tensors
        n, C, n_win, K = ctx.args
        _require(grad_rt.dtype == torch.float32 and tuple(grad_rt.shape) == (n_win, C), 'grad must match rt')
        grad_rt = grad_rt.contiguous()
        with torch.cuda.device(tokens.device):
            grad_src = torch.empty((n, C), dtype=torch.float32, device=tokens.device)
            N.check(N.lib().hfl_rt_init_train_bwd(N.ptr(grad_rt), N.ptr(tokens), n, n_win, K, C, N.ptr(grad_src),
                                                  N.stream()))
        return grad_src, None, None, None, None


def relay_token_init(src: torch.Tensor, tokens: torch.Tensor, K: int, depth: int,
                     mode: int = 0) -> Tuple[torch.Tensor, Optional[torch.Tensor]]:
    """Relay tokens and ADaPE statistics of one pyramid level.

    src (n, C) float32 CUDA, the level's tokens, C a multiple of 32 in [32, 512]; tokens (n_pad, 4) int16, the
    level's ``Octree.tokens(depth, n_pad)`` with n_pad a multiple of K and n <= n_pad; mode 0 (no statistics) or
    3 / 6 / 9 for ADaPE 'pos' / 'var' / 'cov' (:data:`ADAPE_MODES`).  Returns ``(rt, stats)``: rt (n_pad / K, C),
    the mean over each window's tokens of the first token's submap, padding rows counted as zeros;
    stats (n_pad / K, mode) float32 without gradient, or None for mode 0.  Differentiable in src, with
    outputs and gradient bit-identical run to run."""
    rt, stats = RelayTokenInitFunction.apply(src, tokens, K, depth, mode)
    return rt, (stats if mode else None)
