"""Autograd entry to the oracle graph (test infrastructure): ``oracle.model_ref.forward`` with autograd enabled,
computed in the dtype of the state dict's floating-point tensors.

``model_ref.forward`` runs under ``torch.inference_mode``, reads the input feature as float32 and computes the
ADaPE window statistics in float32, so it can give neither gradients nor a float64 statement.  :func:`forward_autograd`
issues the same sequence of ``model_ref`` layer functions; only the input feature and the window statistics
follow the state dict's dtype.  (``model_ref._attention``'s float32 mask bias holds 0 and -1000, both exact, and
is promoted to the scores' dtype.)  For a float32 state dict the result equals ``model_ref.forward`` bit for bit,
which tests/test_differentiable_model_cpu.py pins; with float64 tensors that require grad, ``backward`` gives the
float64 reference for every parameter gradient."""
from __future__ import annotations

from typing import Dict

import torch
import torch.nn.functional as F

from oracle import model_ref as M
from oracle import octree_ref as R


def window_stats(lv: M.Level, K, mode='cov', dtype=torch.float32):
    """``model_ref.window_stats`` (models/octree.py:285-344) in ``dtype``: the same operations, so float32 gives
    the same bits."""
    d = lv.depth
    pts = lv.xyz.to(dtype) * (2 ** (1 - d)) - 1.0
    pts[lv.n:] = 0.0                                           # padded AFTER rescale
    pts = pts.view(-1, K, 3)
    bid = lv.bid.view(-1, K)
    valid = (bid == bid[:, :1])
    cnt = valid.sum(1, keepdim=True).to(dtype)
    v = valid.unsqueeze(-1).to(dtype)
    mu = (pts * v).sum(1) / cnt.clamp(min=1.0)
    if mode == 'pos':
        return mu
    cen = (pts - mu.unsqueeze(1)) * v
    den = (cnt - 1).clamp(min=1.0)
    ok = (cnt >= 2).to(dtype)
    if mode == 'var':
        return torch.cat([mu, (cen ** 2).sum(1) / den * ok], 1)
    cov = torch.bmm(cen.transpose(1, 2), cen) / den.unsqueeze(-1) * ok.unsqueeze(-1)
    iu = torch.triu_indices(3, 3)
    return torch.cat([mu, cov[:, iu[0], iu[1]]], 1)


def forward_autograd(sd: Dict[str, torch.Tensor], oct: R.RefOctree, hp: M.HParams) -> torch.Tensor:
    """HOTFormerLoc.forward -> (B, output_dim) in the state dict's dtype, with autograd (the order of
    ``model_ref.forward``)."""
    with torch.enable_grad():
        cx = M._Ctx(sd, oct, hp)
        B, D, K = oct.batch_size, oct.depth, hp.patch_size
        BB = 'backbone.backbone'
        dtype = next(v.dtype for v in sd.values() if v.is_floating_point())
        x = torch.from_numpy(oct.input_feature_P()).to(dtype)
        d = D
        for i in range(hp.stem_down):
            x = cx.conv_norm_relu(x, f'{BB}.patch_embed.convs.{i}', d, '333', 1)
            x = cx.conv_norm_relu(x, f'{BB}.patch_embed.downsamples.{i}', d, '222', 2)
            d -= 1
        x = cx.conv_norm_relu(x, f'{BB}.patch_embed.proj', d, '333', 1)
        for i in range(hp.num_octf_levels):
            lv = M.make_level(oct, d, K, hp.dilation)
            for blk in range(hp.num_blocks[i]):
                dil = 1 if blk % 2 == 0 else hp.dilation
                x = M.octformer_block(cx, x, f'{BB}.octf_stage.{i}.blocks.{blk}', lv, hp.num_heads[i], K, dil)
            x = cx.downsample(x, f'{BB}.downsample.{i}', d)
            d -= 1
        HS = f'{BB}.hotf_stage'
        H, L = hp.num_heads[-1], hp.num_pyramid_levels
        levels = [M.make_level(oct, d - j, K, hp.dilation) for j in range(L)]
        feats, rts = [x], []
        for j, lv in enumerate(levels):
            src = feats[j]
            if hp.ADaPE_mode is None:
                src = cx.cpe(src, f'{HS}.relay_tokeniser.cpe', lv.depth)
            rt = M.rt_init(src, lv, K)
            if hp.ADaPE_mode is not None:
                rt = rt + M._mlp(window_stats(lv, K, hp.ADaPE_mode, dtype), sd, f'{HS}.rt_adape.mlp')
            rts.append(rt)
            if j < L - 1:
                feats.append(cx.downsample(feats[j], f'{HS}.downsamples.{j}', lv.depth))
        index, ids = M.rt_layout(levels, B)
        for i in range(hp.num_blocks[-1]):
            rts = M.rtsa_block(cx, rts, f'{HS}.rtsa_blocks.{i}', index, ids, H)
            for j, lv in enumerate(levels):
                feats[j], rts[j] = M.hosa_block(cx, feats[j], rts[j], f'{HS}.hosa_blocks.{j}.{i}', lv, H, K)
        if hp.pooling != 'PyramidAttnPoolMixer':
            raise NotImplementedError(hp.pooling)
        g = M.attn_pool_mixer(cx, feats, levels)
        return F.normalize(g, dim=1) if hp.normalize_embeddings else g
