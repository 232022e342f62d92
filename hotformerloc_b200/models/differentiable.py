"""Differentiable fp32 forward of HOTFormerLoc on the training kernels: the autograd statement of the
reference's ``HOTFormerLoc.forward`` (hotformerloc.py:33-59; backbone hotformerloc_backbone.py:540-723,
octformer_backbone.py:251-299, 451-477), the graph ``oracle.model_ref.forward`` states.

It reads the parameters of the existing module tree (:class:`~.hotformerloc.HOTFormer`,
:class:`~.hotformerloc.PoolingWrapper`): no new parameters and no new ``state_dict`` keys.  The non-standard
ops run on this project's fp32 CUDA kernels -- octree convolution, depth-wise CPE convolution, window
attention with RPE and relay token, relay-token initialisation, relay-token self-attention and attention
pooling -- and LayerNorm, Linear, GELU and the residual adds stay in torch.  Windows are views of the
zero-padded level (dilation d: the transpose of ``OctreeT``'s ``(-1, K, d)`` row grouping), so gathering
and scattering back are reshapes under autograd.  Only the host node counts (``batch_nnum_nempty``) are
read: no host synchronisation after ``Octree.finalize()``.

With ``grad_checkpoint`` and grad enabled, each OctFormer block, each RTSA block and each H-OSA block of each
level is recomputed in backward (``torch.utils.checkpoint``, non-reentrant; the graph has no randomness).
"""
from __future__ import annotations

from functools import partial
from typing import Dict, List, Tuple

import torch
import torch.nn.functional as F
from torch.utils.checkpoint import checkpoint

from ..attention_pool import PyramidAttnPool
from ..dwconv import octree_dwconv
from ..native import HflError
from ..octree import Octree
from ..octree_conv import octree_conv
from ..relay_token_attention import RelayTokenLayout, relay_token_attention, rt_layout
from ..rt_init import ADAPE_MODES, relay_token_init
from ..window_attention import window_attention
from .hotformerloc import _native_octree

__all__ = ['backbone_forward', 'model_forward', 'check_trainable']


def check_trainable(backbone) -> None:
    """Refuse what the differentiable forward does not implement, and a model off the GPU."""
    if backbone.training and backbone.drop_path > 0:
        raise NotImplementedError(
            f'drop_path = {backbone.drop_path} in training mode: OctreeDropPath is not implemented in the '
            f'differentiable forward, and training without it would diverge from the reference; set drop_path = 0 '
            f'in the [MODEL] config or call .eval()')
    p = next(backbone.parameters())
    if not p.is_cuda:
        raise HflError('the differentiable forward runs on the GPU only (there is no CPU path): move the model '
                       'to a CUDA device')


class _Level:
    """One level of the octree: its tokens padded to a multiple of K * dilation (``make_level``), the depth-wise
    conv table and, per window shape, the window coordinates and submap ids (shared by all the level's blocks)."""

    def __init__(self, octree: Octree, depth: int, K: int, dilation: int):
        blk = K * dilation
        self.depth, self.K = depth, K
        self.n = octree.n(depth)
        self.n_pad = -(-self.n // blk) * blk
        self.ne = octree.ne_table(depth)
        self.tok = octree.tokens(depth, self.n_pad)           # (n_pad, 4) int16 (x, y, z, submap)
        self._win = {}

    def windows(self, x: torch.Tensor, dil: int) -> torch.Tensor:
        """(n, C) -> (n_pad / K, K, C): window g * dil + a holds rows g K dil + k dil + a, k < K."""
        C, K = x.shape[-1], self.K
        xp = F.pad(x, (0, 0, 0, self.n_pad - x.shape[0]))
        if dil == 1:
            return xp.view(-1, K, C)
        return xp.view(-1, K, dil, C).transpose(1, 2).reshape(-1, K, C)

    def unwindows(self, w: torch.Tensor, dil: int) -> torch.Tensor:
        """Inverse of :meth:`windows`, without the padding rows: (n_pad / K, K, C) -> (n, C)."""
        C, K = w.shape[-1], self.K
        if dil > 1:
            w = w.view(-1, dil, K, C).transpose(1, 2)
        return w.reshape(self.n_pad, C)[:self.n]

    def coords(self, dil: int, hat: bool) -> Tuple[torch.Tensor, torch.Tensor]:
        """int32 (N_win, K, 3) token coordinates and (N_win, K + hat) submap ids of the windows; with ``hat``
        the relay token at position 0 takes the first token's id (hotformerloc_backbone.py:197-236)."""
        key = (dil, hat)
        if key not in self._win:
            t = self.tok.to(torch.int32)
            xyz = self.windows(t[:, :3], dil).contiguous()
            ids = self.windows(t[:, 3:], dil)[..., 0]
            if hat:
                ids = torch.cat([ids[:, :1], ids], 1)
            self._win[key] = (xyz, ids.contiguous())
        return self._win[key]


def _mlp(m, x):
    return m.fc2(F.gelu(m.fc1(x)))


def _conv_norm(cn, x, table, relu: bool):
    """OctreeConvNormRelu / Downsample (octformer_layers.py:80-98, octformer_backbone.py:464-477)."""
    y = octree_conv(x, cn.conv.weights, table)
    if hasattr(cn.conv, 'bias'):
        y = y + cn.conv.bias
    y = cn.norm(y)
    return F.relu(y) if relu else y


def _cpe(cn, x, ne):
    """CPE without the residual: LayerNorm(OctreeDWConv(x)) (octformer_layers.py:177-190)."""
    return cn.norm(octree_dwconv(x, cn.conv.weights, ne))


def _attend(att, y, xyz, ids, hat: bool, H: int):
    rpe = getattr(att, 'rpe', None)
    o = window_attention(att.qkv(y), xyz, ids, rpe.rpe_table if rpe is not None else None,
                         rpe.pos_bnd if rpe is not None else 0, hat, H)
    return att.proj(o)


def _octf_block(b, x, lv: _Level, H: int):
    """OctFormerBlock.forward without drop path (octformer_backbone.py:251-299)."""
    x = x + _cpe(b.cpe, x, lv.ne)
    xyz, ids = lv.coords(b.dilation, False)
    w = lv.windows(x, b.dilation)
    w = w + _attend(b.attention, b.norm1(w), xyz, ids, False, H)
    w = w + _mlp(b.mlp, b.norm2(w))
    return lv.unwindows(w, b.dilation)


def _hosa_block(b, x, rt, lv: _Level, H: int):
    """HOTFormerBlock.forward without drop path (hotformerloc_backbone.py:197-236): the level's relay token
    joins each window at position 0."""
    x = x + _cpe(b.cpe, x, lv.ne)
    xyz, ids = lv.coords(1, True)
    w = torch.cat([rt.unsqueeze(1), lv.windows(x, 1)], 1)
    w = w + _attend(b.attention, b.norm1(w), xyz, ids, True, H)
    w = w + _mlp(b.mlp, b.norm2(w))
    return lv.unwindows(w[:, 1:], 1), w[:, 0]


def _rtsa_block(b, x, layout: RelayTokenLayout, H: int):
    """RelayTokenTransformerBlock.forward without drop path (hotformerloc_backbone.py:275-295) on packed rows."""
    att = b.rt_attention
    x = x + att.proj(relay_token_attention(att.qkv(b.norm1(x)), layout, H))
    return x + _mlp(b.mlp, b.norm2(x))


def _run(ckpt: bool, fn, *args):
    if ckpt:
        return checkpoint(fn, *args, use_reentrant=False, preserve_rng_state=False)
    return fn(*args)


def backbone_forward(model, data: torch.Tensor, octree: Octree
                     ) -> Tuple[Dict[int, torch.Tensor], Dict[int, torch.Tensor]]:
    """PatchEmbed -> OctFormer stage -> HOTFormer stage (hotformerloc_backbone.py:702-723) of ``model``, a
    :class:`~.hotformerloc.HOTFormer`, with ``data`` (n_leaf, 3) float32 as the stem input.  Returns
    ``({depth: (n_d, C)}, {depth: (N_win_d, C)})``, the local features and relay tokens of the pyramid levels."""
    check_trainable(model)
    cfg, bb = model.cfg, model.backbone
    octree.finalize()
    K, dil, L = cfg['patch_size'], cfg['dilation'], cfg['num_pyramid_levels']
    H0, H1 = cfg['num_heads']
    ckpt = bool(model.grad_checkpoint) and torch.is_grad_enabled()

    # PatchEmbed (octformer_backbone.py:451-461)
    pe, d, x = bb.patch_embed, octree.depth, data
    for i in range(cfg['stem_down']):
        x = _conv_norm(pe.convs[i], x, octree.ne_table(d), relu=True)
        x = _conv_norm(pe.downsamples[i], x, octree.child_table(d), relu=True)
        d -= 1
    x = _conv_norm(pe.proj, x, octree.ne_table(d), relu=True)

    # OctFormer stage + downsample (hotformerloc_backbone.py:715-718)
    lv0 = _Level(octree, d, K, dil)
    for b in bb.octf_stage[0].blocks:
        x = _run(ckpt, partial(_octf_block, b, lv=lv0, H=H0), x)
    x = _conv_norm(bb.downsample[0], x, octree.child_table(d), relu=False)
    d -= 1

    # relay-token initialisation + pyramid downsamples (hotformerloc_backbone.py:540-572)
    hs = bb.hotf_stage
    levels = [_Level(octree, d - j, K, dil) for j in range(L)]
    mode = ADAPE_MODES[cfg['ADaPE_mode']]
    feats: List[torch.Tensor] = [x]
    rts: List[torch.Tensor] = []
    for j, lv in enumerate(levels):
        src = feats[j] if mode else _cpe(hs.relay_tokeniser.cpe, feats[j], lv.ne)
        rt, stats = relay_token_init(src, lv.tok, K, lv.depth, mode)
        if mode:
            rt = rt + _mlp(hs.rt_adape.mlp, stats)
        rts.append(rt)
        if j < L - 1:
            feats.append(_conv_norm(hs.downsamples[j], feats[j], octree.child_table(lv.depth), relu=False))

    # M x [RTSA ; H-OSA per level] (hotformerloc_backbone.py:593-633)
    layout = rt_layout([octree.batch_nnum_nempty[lv.depth] for lv in levels], K, dil, x.device)
    for i in range(cfg['num_blocks'][-1]):
        rts = layout.unpack(_run(ckpt, partial(_rtsa_block, hs.rtsa_blocks[i], layout=layout, H=H1), layout.pack(rts)))
        for j, lv in enumerate(levels):
            feats[j], rts[j] = _run(ckpt, partial(_hosa_block, hs.hosa_blocks[j][i], lv=lv, H=H1), feats[j], rts[j])
    return ({lv.depth: f for lv, f in zip(levels, feats)}, {lv.depth: r for lv, r in zip(levels, rts)})


def model_forward(model, octree) -> torch.Tensor:
    """``HOTFormerLoc.forward(batch)['global']`` of ``model``, a :class:`~.hotformerloc.HOTFormerLoc`, for a native
    or ocnn octree: the backbone above, the pyramid attention-pooling head (``PyramidAttnPool.forward`` over the
    ``PyramidAttnPoolWrapper``'s parameters) and, with ``normalize_embeddings``, F.normalize."""
    if model.pooling.pool_method != 'PyramidAttnPoolMixer':
        raise NotImplementedError(f'pooling = {model.pooling.pool_method}: the differentiable forward implements '
                                  f'pooling = PyramidAttnPoolMixer only')
    check_trainable(model.backbone)
    octree = _native_octree(octree)
    local, _ = backbone_forward(model.backbone, model.get_input_feature(octree), octree)
    g = PyramidAttnPool.forward(model.pooling.pooling, local, octree)
    return F.normalize(g, dim=1) if model.normalize_embeddings else g
