"""HOTFormerLoc -- drop-in for the reference's ``models/hotformerloc.py`` /
``models/hotformerloc_backbone.py`` on the inference path.

The module tree below only *holds parameters*, under exactly the reference's
``state_dict`` names (SURVEY.md section 8b), so pretrained ``.pth`` / ``.ckpt``
files load unchanged.  The computation is issued by :class:`_Engine` as a
fixed sequence of libhfl_b200.so kernels (include/hfl.h): there is no CPU path
in ``forward`` and PyTorch only provides the device buffers.

Reference anchors: HOTFormerLoc.forward models/hotformerloc.py:33-59;
HOTFormerBase.forward hotformerloc_backbone.py:702-723; HOTFormerStage.forward
:574-635; PatchEmbed octformer_backbone.py:451-461; PyramidAttnPoolWrapper
models/layers/pooling.py:183-233.
"""
from __future__ import annotations

from typing import Dict, List, Optional, Sequence

import numpy as np
import torch
import torch.nn as nn

from .. import native as N
from .. import ops
from ..octree import Octree, from_ocnn


# ----------------------------------------------------------------------------
# parameter containers (names == reference state_dict keys)
# ----------------------------------------------------------------------------
def _trunc(t, std=0.02):
    return nn.init.trunc_normal_(t, std=std)


def _native_octree(octree) -> Octree:
    """The model runs on the native Octree; an ocnn octree (what the reference's callers pass) is
    imported on the device.  Anything else raises TypeError naming the missing attributes."""
    return octree if isinstance(octree, Octree) else from_ocnn(octree)


class _OctConv(nn.Module):
    """holds ``weights`` (kdim, Cin, Cout) [+ ``bias``] like ocnn.nn.OctreeConv/OctreeDWConv"""

    def __init__(self, kdim, cin, cout, bias=False):
        super().__init__()
        self.weights = nn.Parameter(torch.empty(kdim, cin, cout))
        nn.init.xavier_uniform_(self.weights)
        if bias:
            self.bias = nn.Parameter(torch.zeros(cout))


class _ConvNorm(nn.Module):
    def __init__(self, kdim, cin, cout, bias=False):
        super().__init__()
        self.conv = _OctConv(kdim, cin, cout, bias)
        self.norm = nn.LayerNorm(cout)


class _RPE(nn.Module):
    def __init__(self, patch_size, num_heads, dilation):
        super().__init__()
        self.pos_bnd = int(0.8 * patch_size * dilation ** 0.5)
        self.rpe_table = nn.Parameter(_trunc(torch.zeros(3 * (2 * self.pos_bnd + 1), num_heads)))


class _Attention(nn.Module):
    def __init__(self, dim, patch_size, num_heads, dilation, use_rpe=True):
        super().__init__()
        self.qkv = nn.Linear(dim, dim * 3)
        self.proj = nn.Linear(dim, dim)
        if use_rpe:
            self.rpe = _RPE(patch_size, num_heads, dilation)


class _RTAttention(nn.Module):
    def __init__(self, dim):
        super().__init__()
        self.qkv = nn.Linear(dim, dim * 3)
        self.proj = nn.Linear(dim, dim)


class _MLP(nn.Module):
    def __init__(self, cin, hidden, cout):
        super().__init__()
        self.fc1 = nn.Linear(cin, hidden)
        self.fc2 = nn.Linear(hidden, cout)


class _Block(nn.Module):
    """OctFormerBlock / HOTFormerBlock parameters."""

    def __init__(self, dim, num_heads, patch_size, dilation, use_rpe=True):
        super().__init__()
        self.dilation = dilation
        self.norm1 = nn.LayerNorm(dim)
        self.attention = _Attention(dim, patch_size, num_heads, dilation, use_rpe)
        self.norm2 = nn.LayerNorm(dim)
        self.mlp = _MLP(dim, 4 * dim, dim)
        self.cpe = _ConvNorm(27, 1, dim)


class _RTSABlock(nn.Module):
    def __init__(self, dim):
        super().__init__()
        self.norm1 = nn.LayerNorm(dim)
        self.rt_attention = _RTAttention(dim)
        self.norm2 = nn.LayerNorm(dim)
        self.mlp = _MLP(dim, 4 * dim, dim)


class _Stage(nn.Module):
    def __init__(self, dim, num_heads, patch_size, dilation, num_blocks, use_rpe):
        super().__init__()
        self.blocks = nn.ModuleList([
            _Block(dim, num_heads, patch_size, 1 if i % 2 == 0 else dilation, use_rpe)
            for i in range(num_blocks)])


class _PatchEmbed(nn.Module):
    def __init__(self, cin, dim, num_down):
        super().__init__()
        ch = [int(dim * 2 ** i) for i in range(-num_down, 1)]
        self.convs = nn.ModuleList([_ConvNorm(27, cin if i == 0 else ch[i], ch[i])
                                    for i in range(num_down)])
        self.downsamples = nn.ModuleList([_ConvNorm(8, ch[i], ch[i + 1]) for i in range(num_down)])
        self.proj = _ConvNorm(27, ch[-1], dim)


class _ADaPE(nn.Module):
    def __init__(self, dim, mode):
        super().__init__()
        self.mlp = _MLP({'pos': 3, 'var': 6, 'cov': 9}[mode], dim, dim)


class _RelayTokeniser(nn.Module):
    def __init__(self, dim, use_cpe):
        super().__init__()
        if use_cpe:
            self.cpe = _ConvNorm(27, 1, dim)


class _HOTFStage(nn.Module):
    def __init__(self, dim, num_heads, num_blocks, levels, patch_size, adape_mode, use_rpe):
        super().__init__()
        self.hosa_blocks = nn.ModuleList([
            nn.ModuleList([_Block(dim, num_heads, patch_size, 1, use_rpe) for _ in range(num_blocks)])
            for _ in range(levels)])
        self.rtsa_blocks = nn.ModuleList([_RTSABlock(dim) for _ in range(num_blocks)])
        self.relay_tokeniser = _RelayTokeniser(dim, use_cpe=adape_mode is None)
        if adape_mode is not None:
            self.rt_adape = _ADaPE(dim, adape_mode)
        self.downsamples = nn.ModuleList([_ConvNorm(8, dim, dim, bias=True)
                                          for _ in range(levels - 1)])


class HOTFormerBase(nn.Module):
    def __init__(self, in_channels, channels, num_blocks, num_heads, num_pyramid_levels,
                 num_octf_levels, patch_size, dilation, stem_down, ADaPE_mode, disable_RPE):
        super().__init__()
        self.patch_embed = _PatchEmbed(in_channels, channels[0], stem_down)
        self.octf_stage = nn.ModuleList([
            _Stage(channels[i], num_heads[i], patch_size, dilation, num_blocks[i], not disable_RPE)
            for i in range(num_octf_levels)])
        self.downsample = nn.ModuleList([_ConvNorm(8, channels[i], channels[i + 1], bias=True)
                                         for i in range(num_octf_levels)])
        self.hotf_stage = _HOTFStage(channels[-1], num_heads[-1], num_blocks[-1],
                                     num_pyramid_levels, patch_size, ADaPE_mode, not disable_RPE)


class HOTFormer(nn.Module):
    """Backbone container (reference: hotformerloc_backbone.py:726-849)."""

    def __init__(self, in_channels: int, channels=(128, 256), num_blocks=(4, 10),
                 num_heads=(8, 16), num_pyramid_levels: int = 3, num_octf_levels: int = 1,
                 patch_size: int = 32, dilation: int = 4, drop_path: float = 0.5,
                 nempty: bool = True, stem_down: int = 2, rt_size: int = 1,
                 rt_propagation: bool = False, rt_propagation_scale=None,
                 disable_rt: bool = False, ADaPE_mode: Optional[str] = None,
                 grad_checkpoint: bool = True, downsample_input_embeddings: bool = True,
                 disable_RPE: bool = False, conv_norm: str = 'layernorm', layer_scale=None,
                 qkv_init=('trunc_normal', 0.02), xcpe: bool = False, **kwargs):
        super().__init__()
        unsupported = []
        if in_channels != 3: unsupported.append("input_features other than 'P'")
        if conv_norm != 'layernorm': unsupported.append(f'conv_norm={conv_norm}')
        if disable_rt: unsupported.append('disable_rt')
        if rt_propagation: unsupported.append('ct_propagation')
        if rt_size != 1: unsupported.append('ct_size != 1')
        if layer_scale is not None: unsupported.append('layer_scale')
        if xcpe: unsupported.append('xCPE')
        if not downsample_input_embeddings: unsupported.append('downsample_input_embeddings=False')
        if len(set(channels[num_octf_levels:])) != 1: unsupported.append('per-level channels')
        if num_octf_levels != 1 or len(channels) != 2: unsupported.append('num_octf_levels != 1')
        if channels[0] not in (128, 256) or channels[1] not in (128, 256):
            unsupported.append('channels outside {128,256}')
        if unsupported:
            raise NotImplementedError('not on the B200 hot path (no shipped cfg uses it): '
                                      + ', '.join(unsupported))
        assert all(c // h == 16 for c, h in zip(channels, num_heads)), 'head_dim must be 16'
        self.cfg = dict(channels=tuple(channels), num_blocks=tuple(num_blocks),
                        num_heads=tuple(num_heads), num_pyramid_levels=num_pyramid_levels,
                        num_octf_levels=num_octf_levels, patch_size=patch_size, dilation=dilation,
                        stem_down=stem_down, ADaPE_mode=ADaPE_mode, disable_RPE=disable_RPE)
        self.backbone = HOTFormerBase(in_channels, tuple(channels), tuple(num_blocks),
                                      tuple(num_heads), num_pyramid_levels, num_octf_levels,
                                      patch_size, dilation, stem_down, ADaPE_mode, disable_RPE)
        for m in self.modules():                       # hotformerloc_backbone.py:817-843
            if isinstance(m, nn.Linear):
                _trunc(m.weight)
                nn.init.zeros_(m.bias)
        self._own_engine = None

    def forward(self, data, octree: Octree, depth: int):
        """Reference signature (hotformerloc_backbone.py:845-849):
        ``(local_feat_dict {depth: (n_d, C)}, relay_token_dict {depth: (N_win_d, C)}, octree)``.
        ``data`` must be ``InputFeature('P', nempty=True)(octree)`` -- the leaf point means the first
        kernel reads straight from the octree (only input_features='P' is on the hot path): it is
        checked for shape and otherwise not re-read.  ``octree`` may be an ocnn octree; the third
        output is then the native Octree imported from it."""
        octree = _native_octree(octree)
        assert depth == octree.depth, 'the backbone starts at the leaf depth of the octree'
        if data is not None:
            assert tuple(data.shape) == (octree.n(octree.depth), 3), \
                "data must be the (n_leaf, 3) 'P' input feature of this octree"
        if self._own_engine is None:
            self._own_engine = _Engine(self)
        return self._outputs(self._own_engine.backbone(octree), octree)

    @staticmethod
    def _outputs(ctx, octree):
        K = ctx['K']
        local = {d: ctx['Xl'][j][ctx['hat_rows'][j].long()] for j, d in enumerate(ctx['depths'])}
        relay = {d: ctx['Xl'][j][::K + 1] for j, d in enumerate(ctx['depths'])}
        return local, relay, octree


class _AdaptivePooling(nn.Module):
    def __init__(self, dim, k):
        super().__init__()
        self.query = nn.Parameter(torch.randn(k, dim))


class _MixerLayer(nn.Module):
    def __init__(self, dim):
        super().__init__()
        self.mix = nn.Sequential(nn.LayerNorm(dim), nn.Linear(dim, dim), nn.GELU(),
                                 nn.Linear(dim, dim))
        for m in self.mix:
            if isinstance(m, nn.Linear):
                _trunc(m.weight)
                nn.init.zeros_(m.bias)


class _Mixer(nn.Module):
    def __init__(self, k_in, k_out, dim, out_d, depth=4):
        super().__init__()
        self.mix = nn.Sequential(*[_MixerLayer(dim) for _ in range(depth)])
        self.row_proj = nn.Linear(dim, out_d)
        self.channel_proj = nn.Linear(k_in, k_out)


class PyramidAttnPoolWrapper(nn.Module):
    def __init__(self, feature_size, output_dim, num_pyramid_levels, k_pooled_tokens):
        super().__init__()
        assert len(k_pooled_tokens) == num_pyramid_levels
        self.k_pooled_tokens = tuple(k_pooled_tokens)
        ktot = sum(k_pooled_tokens)
        k_out = ktot // 4
        out_d = output_dim // k_out
        assert k_out * out_d == output_dim, 'k_pooled_tokens incompatible with output_dim'
        self.attpool = nn.ModuleList([_AdaptivePooling(feature_size, k) for k in k_pooled_tokens])
        self.descriptor_extractor = _Mixer(ktot, k_out, feature_size, out_d)


class PyramidOctGeMWrapper(nn.Module):
    def __init__(self, input_dim, output_dim, num_pyramid_levels, p=3.0, eps=1e-6):
        super().__init__()
        self.p = nn.Parameter(torch.ones(num_pyramid_levels) * p)
        self.eps = eps
        self.linear_bn = nn.Sequential(
            nn.Linear(input_dim * num_pyramid_levels, output_dim, bias=False),
            nn.BatchNorm1d(input_dim))


class PoolingWrapper(nn.Module):
    """models/layers/pooling_wrapper.py:11-79 (methods reachable from shipped cfgs)."""

    def __init__(self, pool_method, in_dim, output_dim, num_pyramid_levels=None, channels=None,
                 k_pooled_tokens=None):
        super().__init__()
        self.pool_method, self.in_dim, self.output_dim = pool_method, in_dim, output_dim
        self.pooled_feats = 'local'
        if pool_method == 'PyramidAttnPoolMixer':
            self.pooling = PyramidAttnPoolWrapper(in_dim, output_dim, num_pyramid_levels,
                                                  k_pooled_tokens)
        elif pool_method == 'PyramidOctGeM':
            self.pooling = PyramidOctGeMWrapper(in_dim, output_dim, num_pyramid_levels)
        else:
            raise NotImplementedError(f'pooling={pool_method} is not on the B200 hot path')


# ----------------------------------------------------------------------------
# the kernel schedule
# ----------------------------------------------------------------------------
def _fused_mlp(C: int) -> bool:
    """Which MLP path a stage uses: HFL_FUSED_MLP = comma list of channel counts (default
    '128,256': the fused kernel, which keeps the hidden activation in tensor memory, beats the
    two-GEMM path at both widths -- see DESIGN.md section 4; '' selects the two-GEMM path)."""
    import os
    return str(C) in os.environ.get('HFL_FUSED_MLP', '128,256').split(',')


def _fused_attn() -> bool:
    """HFL_FUSED_ATTN=0 selects the qkv GEMM + stand-alone window attention kernels; default: the fused
    tensor-core kernel (hfl_qkv_attn) wherever it supports the window shape."""
    import os
    return os.environ.get('HFL_FUSED_ATTN', '1') != '0'


def _fused_proj_mlp() -> bool:
    """HFL_FUSED_PROJ=0 selects the round-1 schedule (proj GEMM with residual + LayerNorm epilogue,
    then the MLP kernel); default: one kernel for proj + residual + norm2 + MLP + residual."""
    import os
    return os.environ.get('HFL_FUSED_PROJ', '1') != '0'


def _bf(t):
    return t.detach().to(torch.bfloat16).contiguous()


def _f(t):
    return t.detach().float().contiguous()


def _conv_w(conv: _OctConv):
    return _bf(conv.weights.detach().flatten(0, 1).t())          # [Cout, kdim*Cin]


class _Engine:
    """Issues the kernel schedule for a backbone (``HOTFormer``) and, when given, its pooling head."""

    def __init__(self, backbone: 'HOTFormer', pooling: Optional['PoolingWrapper'] = None,
                 normalize_embeddings: bool = False):
        self.bb_module = backbone
        self.pooling = pooling
        self.normalize_embeddings = normalize_embeddings
        self.sig = None
        self.w: Dict[str, object] = {}

    def _modules(self):
        return [self.bb_module] + ([self.pooling] if self.pooling is not None else [])

    def invalidate(self):
        """Forget the repacked weights (call after writing parameters through ``.data``)."""
        self.sig = None

    def _level_streams(self, dev, L):
        """HFL_LEVEL_STREAMS=1: run the pyramid levels of an H-OSA block on separate streams."""
        import os
        if os.environ.get('HFL_LEVEL_STREAMS', '0') != '1':
            return None
        if getattr(self, '_streams', None) is None or len(self._streams) < L:
            self._streams = [torch.cuda.Stream(device=dev) for _ in range(L)]
        return self._streams[:L]

    def _signature(self):
        # (storage pointer, version counter) of every parameter / buffer: any in-place update through
        # the autograd-visible API, a load_state_dict, a .to() or a re-assignment changes it.  Writes
        # through ``p.data`` bump neither: call model.refresh_weights() after those.
        ps = [t for m in self._modules() for t in list(m.parameters()) + list(m.buffers())]
        return tuple((t.data_ptr(), t._version) for t in ps)

    def prepare(self):
        sig = self._signature()
        if sig == self.sig:
            return self.w
        bb = self.bb_module.backbone
        w: Dict[str, object] = {}

        def block(b):
            d = dict(n1=(_f(b.norm1.weight), _f(b.norm1.bias)),
                     n2=(_f(b.norm2.weight), _f(b.norm2.bias)),
                     fc1=(_bf(b.mlp.fc1.weight), _f(b.mlp.fc1.bias)),
                     fc2=(_bf(b.mlp.fc2.weight), _f(b.mlp.fc2.bias)))
            att = b.attention if hasattr(b, 'attention') else b.rt_attention
            d['qkv'] = (_bf(att.qkv.weight), _f(att.qkv.bias))
            if hasattr(b, 'cpe') and att.qkv.weight.shape[1] % 64 == 0:
                d['qkv_g'] = ops.regroup_qkv(*d['qkv'])          # per-4-head [q | k | v] rows (hfl_qkv_attn)
            d['proj'] = (_bf(att.proj.weight), _f(att.proj.bias))
            if hasattr(att, 'rpe'):
                d['rpe'] = _f(att.rpe.rpe_table)
                d['bnd'] = att.rpe.pos_bnd
            else:
                d['rpe'], d['bnd'] = None, 0
            if hasattr(b, 'cpe'):
                d['cpe'] = (_bf(b.cpe.conv.weights[:, 0, :]), _f(b.cpe.norm.weight),
                            _f(b.cpe.norm.bias))
                d['dil'] = b.dilation
            return d

        def convnorm(c):
            return dict(w=_conv_w(c.conv), b=_f(c.conv.bias) if hasattr(c.conv, 'bias') else None,
                        ln=(_f(c.norm.weight), _f(c.norm.bias)))
        pe = bb.patch_embed
        w['stem0'] = dict(w=_f(pe.convs[0].conv.weights.flatten(0, 1)),
                          ln=(_f(pe.convs[0].norm.weight), _f(pe.convs[0].norm.bias)))
        w['convs'] = [convnorm(c) for c in pe.convs]
        w['stem_down'] = [convnorm(c) for c in pe.downsamples]
        w['stem_proj'] = convnorm(pe.proj)
        w['octf'] = [block(b) for b in bb.octf_stage[0].blocks]
        w['down0'] = convnorm(bb.downsample[0])
        hs = bb.hotf_stage
        w['hosa'] = [[block(b) for b in lvl] for lvl in hs.hosa_blocks]
        w['rtsa'] = [block(b) for b in hs.rtsa_blocks]
        w['hdown'] = [convnorm(c) for c in hs.downsamples]
        if hasattr(hs, 'rt_adape'):
            a = hs.rt_adape.mlp
            w['adape'] = dict(w1=_f(a.fc1.weight), b1=_f(a.fc1.bias), w2=_bf(a.fc2.weight),
                              b2=_f(a.fc2.bias), mode=a.fc1.weight.shape[1])
        else:
            c = hs.relay_tokeniser.cpe
            w['rt_cpe'] = (_bf(c.conv.weights[:, 0, :]), _f(c.norm.weight), _f(c.norm.bias))
        pool = self.pooling.pooling if self.pooling is not None else None
        if pool is None:
            pass
        elif isinstance(pool, PyramidAttnPoolWrapper):
            qs = []
            for ap in pool.attpool:
                k, C = ap.query.shape
                npad = (k + 63) // 64 * 64
                q = torch.zeros(npad, C, dtype=torch.bfloat16, device=ap.query.device)
                q[:k] = ap.query.detach().to(torch.bfloat16)
                qs.append((q, k, npad))
            w['queries'] = qs
            de = pool.descriptor_extractor
            w['mixer'] = [dict(ln=(_f(l.mix[0].weight), _f(l.mix[0].bias)),
                               fc1=(_bf(l.mix[1].weight), _f(l.mix[1].bias)),
                               fc2=(_bf(l.mix[3].weight), _f(l.mix[3].bias))) for l in de.mix]
            w['tail'] = dict(wc=_f(de.channel_proj.weight), bc=_f(de.channel_proj.bias),
                             wr=_f(de.row_proj.weight), br=_f(de.row_proj.bias))
        else:
            bn = pool.linear_bn[1]
            w['gem'] = dict(p=[float(v) for v in pool.p.detach().cpu()], eps=pool.eps,
                            w=_f(pool.linear_bn[0].weight), bn=(
                                _f(bn.weight), _f(bn.bias), _f(bn.running_mean),
                                _f(bn.running_var), bn.eps))
        self.w, self.sig = w, sig
        return w

    # ------------------------------------------------------------------
    def _block(self, bw, x, xb, ne, tok, n, rows, n_win, C, H, K, hat, bufs, out_rows=None):
        """One OctFormer / H-OSA block on a level (6 kernels)."""
        y, qkv, o = (t.view(-1)[:rows * c].view(rows, c) for t, c in
                     ((bufs['y'], C), (bufs['qkv'], 3 * C), (bufs['o'], C)))
        cw, cg, cb = bw['cpe']
        ops.cpe_ln(x, xb, ne, cw, cg, cb, bw['n1'][0], bw['n1'][1], y, None, n, rows, C,
                   K if hat else 0)
        if _fused_attn() and 'qkv_g' in bw and ops.qkv_attn_supported(H, C, K, bw['dil'], hat, bw['bnd']):
            # the (query, key) pair codes depend on the token positions only: one array per level and window shape,
            # shared by all its blocks in this forward
            ck = ('codes', tok.data_ptr(), K, bw['dil'], hat, bw['bnd'], bw['rpe'] is None)
            if ck not in bufs:
                bufs[ck] = ops.qkv_attn_codes(tok, n_win, K, bw['dil'], hat, bw['bnd'], bw['rpe'] is not None)
            ops.qkv_attn(y, bw['qkv_g'][0], bw['qkv_g'][1], o, tok, bw['rpe'], n_win, H, C, K, bw['dil'],
                         hat, bw['bnd'], 0.25, codes=bufs[ck])
        else:
            ops.gather_gemm(y, bw['qkv'][0], bias=bw['qkv'][1], out_v_bf16=qkv)
            ops.window_attn(qkv, o, tok, bw['rpe'], n_win, H, C, K, bw['dil'], hat, bw['bnd'], 0.25)
        if _fused_proj_mlp():
            ops.proj_mlp_fused(o, bw['proj'][0], bw['proj'][1], bw['n2'][0], bw['n2'][1], bw['fc1'][0],
                               bw['fc1'][1], bw['fc2'][0], bw['fc2'][1], res=x, out_f32=x, out_bf16=xb)
            return
        ops.gather_gemm(o, bw['proj'][0], bias=bw['proj'][1], res=x, out_v_f32=x, ln=bw['n2'],
                        out_y_bf16=y)
        if _fused_mlp(C):
            ops.mlp_fused(y, bw['fc1'][0], bw['fc1'][1], bw['fc2'][0], bw['fc2'][1], res=x, out_f32=x,
                          out_bf16=xb)
        else:
            h = bufs['h'].view(-1)[:rows * 4 * C].view(rows, 4 * C)
            ops.gather_gemm(y, bw['fc1'][0], bias=bw['fc1'][1], act=1, out_v_bf16=h)
            ops.gather_gemm(h, bw['fc2'][0], bias=bw['fc2'][1], res=x, out_v_f32=x, out_v_bf16=xb)

    @torch.no_grad()
    def forward(self, octree: Octree, return_intermediates: bool = False):
        ctx = self.backbone(octree, return_intermediates)
        out = self.head(ctx)
        return (out, ctx['inter']) if return_intermediates else out

    @torch.no_grad()
    def backbone(self, octree: Octree, return_intermediates: bool = False):
        """PatchEmbed -> OctFormer stage -> HOTFormer stage (hotformerloc_backbone.py:702-723).  Returns the
        per-level buffers in the hat layout (relay token first in every window) and their row tables."""
        w = self.prepare()
        cfg = self.bb_module.cfg
        octree.finalize()
        dev = octree.device
        B, D, K, dil = octree.batch_size, octree.depth, cfg['patch_size'], cfg['dilation']
        C0, C1 = cfg['channels']
        H0, H1 = cfg['num_heads']
        L = cfg['num_pyramid_levels']
        sd = cfg['stem_down']
        d0 = D - sd
        assert d0 - L >= octree.full_depth, 'octree not deep enough for the model'
        n = [octree.n(d) for d in range(D + 1)]
        bf, f32, i32 = torch.bfloat16, torch.float32, torch.int32
        E = lambda *s, dt=bf: torch.empty(*s, dtype=dt, device=dev)
        Z = lambda *s, dt=bf: torch.zeros(*s, dtype=dt, device=dev)
        inter = {}

        # ---------------- PatchEmbed ----------------
        d = D
        f = E(n[d], w['stem0']['w'].shape[1])
        ops.stem_conv(octree._leaf_points, octree.ne_table(d), n[d], d, w['stem0']['w'],
                      w['stem0']['ln'][0], w['stem0']['ln'][1], f)
        for i in range(sd):
            if i > 0:
                c = w['convs'][i]
                g = E(n[d], c['w'].shape[0])
                ops.gather_gemm(f, c['w'], idx=octree.ne_table(d), KD=27, ln=c['ln'], relu=True,
                                out_y_bf16=g)
                f = g
            c = w['stem_down'][i]
            g = E(n[d - 1], c['w'].shape[0])
            ops.gather_gemm(f, c['w'], idx=octree.child_table(d), KD=8, ln=c['ln'], relu=True,
                            out_y_bf16=g)
            f, d = g, d - 1
        blk = K * dil
        npad0 = -(-n[d0] // blk) * blk
        x0, xb0 = E(npad0, C0, dt=f32), E(npad0, C0)
        x0[n[d0]:].zero_()                     # padding tokens must stay finite (they are keys/values)
        c = w['stem_proj']
        ops.gather_gemm(f, c['w'], idx=octree.ne_table(d0), KD=27, ln=c['ln'], relu=True,
                        out_y_f32=x0, out_y_bf16=xb0)
        if return_intermediates:
            inter['stem'] = x0[:n[d0]].clone()

        # ---------------- level geometry ----------------
        depths = [d0 - 1 - j for j in range(L)]
        nl = [n[dj] for dj in depths]
        npad = [-(-v // blk) * blk for v in nl]
        nwin = [v // K for v in npad]
        rows = [v * (K + 1) for v in nwin]
        R = np.concatenate([[0], np.cumsum(rows)]).astype(np.int64)
        max_rows = max([npad0] + rows)
        Cm = max(C0, C1)
        bufs = dict(y=E(max_rows * Cm), qkv=E(max_rows * 3 * Cm), o=E(max_rows * Cm))
        if not (_fused_mlp(C0) and _fused_mlp(C1)):
            bufs['h'] = E(max_rows * 4 * Cm)

        # ---------------- OctFormer stage ----------------
        tok0 = octree.tokens(d0, npad0)
        ne0 = octree.ne_table(d0)
        for bw in w['octf']:
            self._block(bw, x0, xb0, ne0, tok0, n[d0], npad0, npad0 // K, C0, H0, K, False, bufs)
        if return_intermediates:
            inter['octf0'] = x0[:n[d0]].clone()

        # ---------------- host tables for the pyramid (from the node counts) ----------------
        tabs = self._host_tables(octree, depths, nl, npad, nwin, R, K, B)
        X, Xb = E(int(R[-1]), C1, dt=f32), E(int(R[-1]), C1)
        Xl = [X[R[j]:R[j + 1]] for j in range(L)]
        for j in range(L):                     # zero only the padding tail of each level
            Xl[j][nl[j] + nl[j] // K + 1:].zero_()
        Xbl = [Xb[R[j]:R[j + 1]] for j in range(L)]
        tok = [octree.tokens(depths[j], npad[j]) for j in range(L)]
        ne = [octree.ne_table(dj) for dj in depths]
        hat_rows = []
        for j in range(L):
            r = E(nl[j], dt=i32)
            ops.hat_rows(r, nl[j], K, 0)
            hat_rows.append(r)

        # downsample d0 -> level 0 (octformer_backbone.py:464-477)
        c = w['down0']
        ops.gather_gemm(xb0, c['w'], idx=octree.child_table(d0), KD=8, bias=c['b'], ln=c['ln'],
                        y_mapped=True, out_y_f32=Xl[0], out_y_bf16=Xbl[0], out_rows=hat_rows[0])

        # ---------------- relay-token init + pyramid downsamples (:540-572) ----------------
        for j in range(L):
            if 'adape' in w:
                a = w['adape']
                hbuf = E(nwin[j], C1)
                ops.rt_init(Xl[j], None, tok[j], nl[j], nwin[j], K, C1, depths[j], a['mode'],
                            a['w1'], a['b1'], hbuf)
                ops.gather_gemm(hbuf, a['w2'], bias=a['b2'], res=Xl[j], out_v_f32=Xl[j],
                                out_rows=tabs['rt_local'][j])
            else:
                cw, cg, cb = w['rt_cpe']
                tmp = E(max(nl[j], 1), C1, dt=f32)
                ops.cpe_ln(Xl[j], Xbl[j], ne[j], cw, cg, cb, None, None, None, tmp, nl[j], rows[j],
                           C1, K)
                ops.rt_init(Xl[j], tmp, tok[j], nl[j], nwin[j], K, C1, depths[j], 0, None, None,
                            None)
            if j < L - 1:
                c = w['hdown'][j]
                ct = octree.child_table(depths[j])
                idx = E(ct.shape[0], 8, dt=i32)
                ops.remap_hat(ct, idx, ct.numel(), K)
                ops.gather_gemm(Xbl[j], c['w'], idx=idx, KD=8, bias=c['b'], ln=c['ln'],
                                y_mapped=True, out_y_f32=Xl[j + 1], out_y_bf16=Xbl[j + 1],
                                out_rows=hat_rows[j + 1])
        if return_intermediates:
            inter['rt_init'] = [Xl[j][::K + 1].clone() for j in range(L)]

        # ---------------- M x [RTSA ; H-OSA per level] (:593-633) ----------------
        T = tabs['total_rt']
        yr, qkvr, orr = E(T, C1), E(T, 3 * C1), E(T, C1)
        lvl_streams = self._level_streams(dev, L)
        if lvl_streams is not None:
            main_stream = torch.cuda.current_stream()
            lvl_bufs = [bufs] + [dict(y=E(rows[j] * C1), qkv=E(rows[j] * 3 * C1), o=E(rows[j] * C1))
                                 for j in range(1, L)]
            if 'h' in bufs:
                for j in range(1, L):
                    lvl_bufs[j]['h'] = E(rows[j] * 4 * C1)
        for i in range(cfg['num_blocks'][-1]):
            bw = w['rtsa'][i]
            ops.ln_rows(X, tabs['rt_rows'], T, C1, bw['n1'][0], bw['n1'][1], yr)
            ops.gather_gemm(yr, bw['qkv'][0], bias=bw['qkv'][1], out_v_bf16=qkvr)
            ops.varlen_attn(qkvr, orr, tabs['cu'], tabs['ids'], B, tabs['max_len'], H1, C1, 0.25)
            if _fused_proj_mlp():
                ops.proj_mlp_fused(orr, bw['proj'][0], bw['proj'][1], bw['n2'][0], bw['n2'][1],
                                   bw['fc1'][0], bw['fc1'][1], bw['fc2'][0], bw['fc2'][1], res=X,
                                   out_f32=X, out_rows=tabs['rt_rows'])
            else:
                ops.gather_gemm(orr, bw['proj'][0], bias=bw['proj'][1], res=X, out_v_f32=X,
                                ln=bw['n2'], out_y_bf16=yr, out_rows=tabs['rt_rows'])
                if _fused_mlp(C1):
                    ops.mlp_fused(yr, bw['fc1'][0], bw['fc1'][1], bw['fc2'][0], bw['fc2'][1], res=X,
                                  out_f32=X, out_rows=tabs['rt_rows'])
                else:
                    hr = E(T, 4 * C1)
                    ops.gather_gemm(yr, bw['fc1'][0], bias=bw['fc1'][1], act=1, out_v_bf16=hr)
                    ops.gather_gemm(hr, bw['fc2'][0], bias=bw['fc2'][1], res=X, out_v_f32=X,
                                    out_rows=tabs['rt_rows'])
            if lvl_streams is None:
                for j in range(L):
                    self._block(w['hosa'][j][i], Xl[j], Xbl[j], ne[j], tok[j], nl[j], rows[j], nwin[j],
                                C1, H1, K, True, bufs)
            else:
                # the levels of one H-OSA block are independent (the reference runs them on three
                # streams too, hotformerloc_backbone.py:596-618); only RTSA couples them
                fork = main_stream.record_event()
                for j in range(L):
                    lvl_streams[j].wait_event(fork)
                    with torch.cuda.stream(lvl_streams[j]):
                        self._block(w['hosa'][j][i], Xl[j], Xbl[j], ne[j], tok[j], nl[j], rows[j],
                                    nwin[j], C1, H1, K, True, lvl_bufs[j])
                        main_stream.wait_event(lvl_streams[j].record_event())
        if return_intermediates:
            inter['feats'] = [Xl[j][hat_rows[j].long()].clone() for j in range(L)]
            inter['rts'] = [Xl[j][::K + 1].clone() for j in range(L)]

        return dict(Xl=Xl, Xbl=Xbl, hat_rows=hat_rows, tabs=tabs, rows=rows, nl=nl, nwin=nwin, depths=depths,
                    K=K, B=B, C1=C1, L=L, inter=inter, dev=dev)

    @torch.no_grad()
    def head(self, ctx):
        """Pooling head (pooling.py:183-233 / :87-103) + F.normalize (hotformerloc.py:55-56)."""
        w = self.w
        Xl, Xbl, tabs, rows, K, B, C1, L, dev = (ctx[k] for k in ('Xl', 'Xbl', 'tabs', 'rows', 'K', 'B', 'C1', 'L',
                                                                  'dev'))
        bf, f32 = torch.bfloat16, torch.float32
        E = lambda *s, dt=bf: torch.empty(*s, dtype=dt, device=dev)
        if 'queries' in w:
            ktot = sum(k for _, k, _ in w['queries'])
            Tk = E(B, ktot, C1, dt=f32)
            qoff = 0
            for j, (q, k, npd) in enumerate(w['queries']):
                logits = E(rows[j], npd, dt=f32)
                ops.gather_gemm(Xbl[j], q, out_v_f32=logits)
                stat = E(B, k, 2, dt=f32)
                ops.attn_pool(logits, Xl[j], Xbl[j], tabs['tok_off'][j], stat, Tk, B, k, npd, K, C1, ktot,
                              qoff, C1 ** -0.5)
                qoff += k
            T2 = Tk.view(B * ktot, C1)
            ty, th = E(B * ktot, C1), E(B * ktot, C1)
            for lw in w['mixer']:
                ops.ln_rows(T2, None, B * ktot, C1, lw['ln'][0], lw['ln'][1], ty)
                ops.gather_gemm(ty, lw['fc1'][0], bias=lw['fc1'][1], act=1, out_v_bf16=th)
                ops.gather_gemm(th, lw['fc2'][0], bias=lw['fc2'][1], res=T2, out_v_f32=T2)
            t = w['tail']
            kout, od = t['wc'].shape[0], t['wr'].shape[0]
            out = E(B, kout * od, dt=f32)
            ops.mixer_tail(Tk, t['wc'], t['bc'], t['wr'], t['br'], out, B, ktot, kout, C1, od,
                           self.normalize_embeddings)
        else:
            gw = w['gem']
            pooled = E(B, L * C1, dt=f32)
            for j in range(L):
                ops.gem_pool(Xl[j], tabs['tok_off'][j], B, K, C1, gw['p'][j], gw['eps'], pooled,
                             L * C1, j * C1)
            g, b, mu, var, eps = gw['bn']
            out = E(B, gw['w'].shape[0], dt=f32)
            ops.gem_head(pooled, gw['w'], g, b, mu, var, eps, self.normalize_embeddings, out)
        return out

    def _host_tables(self, octree, depths, nl, npad, nwin, R, K, B):
        """Relay-token ownership / sequence tables (models/octree.py:156-184, 229-265;
        relay_token_utils.py:12-40) from the host copy of the node counts; one
        pinned staging buffer, one H2D copy."""
        L = len(depths)
        counts = [octree.batch_nnum_nempty[dj].numpy().astype(np.int64) for dj in depths]
        nws, starts = [], []
        for j in range(L):
            cum = np.cumsum(counts[j])
            cum[-1] += npad[j] - nl[j]
            boundary = -(-cum // K)
            nw = np.diff(np.concatenate([[0], boundary]))
            nws.append(nw)
            starts.append(np.cumsum(nw) - nw)
        tot = np.sum(nws, axis=0)
        cu = np.concatenate([[0], np.cumsum(tot)]).astype(np.int32)
        total_rt = int(cu[-1])
        rt_rows = np.empty(total_rt, dtype=np.int32)
        ids = np.empty(total_rt, dtype=np.int32)
        prefix = np.zeros(B, dtype=np.int64)
        for j in range(L):
            wi = np.arange(nwin[j], dtype=np.int64)
            owner = np.repeat(np.arange(B, dtype=np.int64), nws[j])
            pos = cu[owner] + prefix[owner] + (wi - starts[j][owner])
            rt_rows[pos] = R[j] + wi * (K + 1)
            first_pad = -(-nl[j] // K)                  # windows >= this hold only padding
            ids[pos] = np.where(wi >= first_pad, B, owner)
            prefix += nws[j]
        tok_off = [np.concatenate([[0], np.cumsum(c)]).astype(np.int32) for c in counts]
        rt_local = [(np.arange(nwin[j], dtype=np.int64) * (K + 1)).astype(np.int32) for j in range(L)]
        parts = [rt_rows, ids, cu] + tok_off + rt_local
        sizes = [p.size for p in parts]
        stage = N.pinned.take(4 * sum(sizes)).view(torch.int32)
        o = 0
        for p in parts:
            stage[o:o + p.size] = torch.from_numpy(np.ascontiguousarray(p, dtype=np.int32))
            o += p.size
        devbuf = stage.to(octree.device, non_blocking=True)
        N.pinned.mark()
        views, o = [], 0
        for s in sizes:
            views.append(devbuf[o:o + s])
            o += s
        return dict(rt_rows=views[0], ids=views[1], cu=views[2], tok_off=views[3:3 + L],
                    rt_local=views[3 + L:3 + 2 * L], total_rt=total_rt,
                    max_len=int(tot.max()), num_windows=nws)


class HOTFormerLoc(nn.Module):
    """Same constructor and ``forward(batch) -> {'global': (B, output_dim)}`` as the
    reference (models/hotformerloc.py:18-59); ``batch['octree']`` is a native Octree or an ocnn
    octree."""

    def __init__(self, backbone: nn.Module, pooling: PoolingWrapper,
                 normalize_embeddings: bool = False, input_features='P'):
        super().__init__()
        assert input_features == 'P', "only input_features='P' is on the hot path"
        self.backbone = backbone
        self.pooling = pooling
        self.normalize_embeddings = normalize_embeddings
        self.input_features = input_features
        self.stats = {}
        self._engine = _Engine(backbone, pooling, normalize_embeddings)

    def get_input_feature(self, octree):
        """InputFeature('P', nempty=True) (hotformerloc.py:28-31): leaf point means in [-1, 1]."""
        D = octree.depth
        return octree.points[D] * (2.0 ** (1 - D)) - 1.0

    def refresh_weights(self):
        """Re-read the parameters on the next forward (needed only after writes through ``.data``)."""
        self._engine.invalidate()

    def forward(self, batch):
        octree = _native_octree(batch['octree'])
        self._engine.normalize_embeddings = self.normalize_embeddings
        x = self._engine.forward(octree)
        assert x.dim() == 2 and x.shape[1] == self.pooling.output_dim
        return {'global': x}

    def forward_debug(self, batch):
        return self._engine.forward(_native_octree(batch['octree']), return_intermediates=True)

    def print_info(self):
        print('Model class: HOTFormerLoc (B200-native)')
        print(f'Total parameters: {sum(p.nelement() for p in self.parameters())}')
        base = self.backbone.backbone
        print(f'Backbone: {type(self.backbone).__name__}\t#parameters: '
              f'{sum(p.nelement() for p in self.backbone.parameters())}')
        print(f'  ConvEmbed:\t#parameters: {sum(p.nelement() for p in base.patch_embed.parameters())}')
        print(f'Pooling method: {self.pooling.pool_method}\t#parameters: '
              f'{sum(p.nelement() for p in self.pooling.parameters())}')
        print(f'# output channels : {self.pooling.output_dim}')
        print(f'Embedding normalization: {self.normalize_embeddings}')
