"""The HOTFormer-stage and pooling-head kernels against float64, at every preset's shapes.

Every output element is held to the bound of tests/test_hotf_bounds_cpu.py (which shows on the CPU that an
emulation of each kernel's arithmetic fits it and that one-defect mutants do not).  The references are float64
statements on the kernel's own operands: the bf16 qkv, the fp32 logits of gather_gemm, the bf16 shadow xb.

| preset         | depth / levels | K                         | ADaPE                       | pooling kq (ktot)  | mixer kin->kout, od |
|----------------|----------------|---------------------------|-----------------------------|--------------------|---------------------|
| oxford         | 9 / 6,5,4      | 48 (fused attention)      | cov                         | 74, 36, 18 (128)   | 128->32, 8          |
| cs-wild-places | 7 / 4,3,2      | 64 + RT -> hfl_window_attn | cov                         | 74, 36, 18 (128)   | 128->32, 8          |
| cs-campus3d    | 7 / 4,3,2      | 64 + RT -> hfl_window_attn | cov                         | 148, 72, 36 (256)  | 256->64, 4          |
| wild-places    | 7 / 4,3,2      | 48                        | off -> rt_init mode 0 + src | 148, 72, 36 (256)  | 256->64, 4          |

hfl_window_attn also runs at K = 96 + RT (the sweep shape, compact shared-memory layout).  Each batch has
submaps shorter than a window (windows spanning 2-3 submaps), padding-only windows and a submap that owns no
relay token at a coarse level.
"""
import functools

import numpy as np
import pytest
import torch

from hotformerloc_b200 import native as N
from hotformerloc_b200 import ops
from tests.test_hotf_bounds_cpu import (DIL, LENS, MODE_NAMES, PRESETS, bf16r, gem_head_ref, gem_ref, hat_row,
                                        level_from_tokens, ln_ref, mixer_ref, pool_ref, pool_segments, ratio,
                                        rt_ref, small_clouds, varlen_check, varlen_layout, wide_windows,
                                        window_check, window_ids)

pytestmark = pytest.mark.gpu
DEV = 'cuda'
H1, C1 = 16, 256                # HOTFormer stage of every preset


@functools.lru_cache(maxsize=None)
def _octree(depth):
    from hotformerloc_b200.octree import build_batch
    return build_batch(small_clouds(depth), depth, 2, DEV).finalize()


def _level(depth, d, K):
    """(Level on the device, token table int16) of depth d, padded as the model pads (K * DIL)."""
    o = _octree(depth)
    n = o.n(d)
    n_pad = -(-n // (K * DIL)) * K * DIL
    tok = o.tokens(d, n_pad)
    counts = o.batch_nnum_nempty[d].numpy().astype(np.int64)
    return level_from_tokens(tok, n, d, counts), tok


def _report(name, r):
    print(f'{name}: max err/bound = {r:.3f}')
    assert r <= 1.0, f'{name}: max err/bound = {r:.3f}'


# ---------------------------------------------------------------------------
# hfl_window_attn (k_window_attn3): K = 64 and 96 plus the relay token
# ---------------------------------------------------------------------------
def _run_window(xyz, bid, tok, K, table, seed):
    W = bid.shape[0]
    L = K + 1
    g = torch.Generator(device=DEV).manual_seed(seed)
    qkv = bf16r(torch.randn(W * L, 3 * C1, device=DEV, generator=g)).to(torch.bfloat16)
    out = torch.zeros(W * L, C1, device=DEV, dtype=torch.bfloat16)
    rpe = None if table is None else table.float().contiguous()
    ops.window_attn(qkv, out, tok, rpe, W, H1, C1, K, 1, True, int(0.8 * K), 0.25)
    return window_check(out.view(W, L, C1), qkv.view(W, L, 3 * C1), window_ids(bid, True), xyz,
                        table, K, True, H1)


@pytest.mark.parametrize('table', ['rpe', 'no_rpe', 'rpe_large'])
@pytest.mark.parametrize('preset', ['cs-wild-places', 'cs-campus3d', 'sweep-k96'])
def test_window_attn(preset, table):
    K = 96 if preset == 'sweep-k96' else 64
    P = PRESETS['cs-wild-places']
    std = {'rpe': 0.5, 'no_rpe': None, 'rpe_large': 16.0}[table]
    bnd = int(0.8 * K)
    seed = 11 if preset == 'cs-campus3d' else 7
    g = torch.Generator(device=DEV).manual_seed(seed)
    tab = None if std is None else torch.randn(3 * (2 * bnd + 1), H1, device=DEV, generator=g, dtype=torch.float64) * std
    if tab is not None:
        tab = tab.float().double()                       # the fp32 table the kernel reads
    for d in P['levels']:
        lv, tok = _level(P['depth'], d, K)
        r = _run_window(lv.xyz.view(-1, K, 3), lv.bid.view(-1, K), tok, K, tab, seed + d)
        _report(f'window_attn {preset} K={K} level {d} {table}', r)
    # coordinates spanning 128 cells: offsets reach the RPE clamp
    xyz, bid = wide_windows(24, K)
    tok = torch.cat([xyz.reshape(-1, 3), bid.reshape(-1, 1)], 1).to(torch.int16).to(DEV).contiguous()
    r = _run_window(xyz.to(DEV), bid.to(DEV), tok, K, tab, seed)
    _report(f'window_attn {preset} K={K} wide coordinates {table}', r)


# ---------------------------------------------------------------------------
# hfl_varlen_attn
# ---------------------------------------------------------------------------
def _rt_layout(preset):
    """cu, ids (int32, device) and T of the preset batch's relay-token sequences (padding windows: id B)."""
    from hotformerloc_b200.models.hotformerloc import rt_ownership
    P = PRESETS[preset]
    K, o = P['K'], _octree(P['depth'])
    counts = [o.batch_nnum_nempty[d].numpy().astype(np.int64) for d in P['levels']]
    n_pad = [-(-int(c.sum()) // (K * DIL)) * K * DIL for c in counts]
    own = rt_ownership(counts, K, n_pad)
    assert bool((own.ids == o.batch_size).any())
    return (torch.from_numpy(own.cu.astype(np.int32)).to(DEV), torch.from_numpy(own.ids.astype(np.int32)).to(DEV),
            own.total, own.max_len)


@pytest.mark.parametrize('H', [16, 8])
@pytest.mark.parametrize('layout', ['lengths', 'oxford', 'cs-wild-places'])
def test_varlen_attn(layout, H):
    C = 16 * H
    if layout == 'lengths':
        cu, ids = varlen_layout(LENS, pad_tail=5, device=DEV)
        T, max_len = int(cu[-1]), max(LENS)
    else:
        cu, ids, T, max_len = _rt_layout(layout)
    g = torch.Generator(device=DEV).manual_seed(H)
    qkv = torch.randn(T, 3 * C, device=DEV, generator=g).to(torch.bfloat16)
    out = torch.zeros(T, C, device=DEV, dtype=torch.bfloat16)
    ops.varlen_attn(qkv, out, cu, ids, cu.numel() - 1, max_len, H, C, 0.25)
    _report(f'varlen_attn {layout} H={H}', varlen_check(out, qkv, cu.cpu(), ids, H))


# ---------------------------------------------------------------------------
# hfl_rt_init
# ---------------------------------------------------------------------------
def _run_rt_init(depth, d, K, C, mode, use_src, seed):
    lv, tok = _level(depth, d, K)
    n, W = lv.n, lv.n_pad // K
    g = torch.Generator(device=DEV).manual_seed(seed)
    feat = torch.randn(n, C, device=DEV, generator=g)
    x = torch.zeros(W * (K + 1), C, device=DEV)
    tr = hat_row(torch.arange(n, device=DEV), K)
    # src path: the token rows of x hold something else, the statistics come from src
    x[tr] = torch.randn(n, C, device=DEV, generator=g) if use_src else feat
    x[::K + 1] = 7.0
    x0 = x.clone()
    src = feat.clone() if use_src else None
    w1 = torch.randn(C, max(mode, 1), device=DEV, generator=g) * 0.5
    b1 = torch.randn(C, device=DEV, generator=g) * 0.1
    h = torch.zeros(W, C, device=DEV, dtype=torch.bfloat16)
    stats = torch.zeros(W, 9, device=DEV)
    ops.rt_init(x, src, tok, n, W, K, C, d, mode, w1 if mode else None, b1 if mode else None,
                h if mode else None, stats_out=stats)
    keep = torch.ones(x.shape[0], dtype=torch.bool, device=DEV)
    keep[::K + 1] = False
    assert torch.equal(x[keep], x0[keep]), 'hfl_rt_init wrote a token row'
    rt_r, rt_b, st_r, st_b, h_r, h_b = rt_ref(feat, lv, K, mode, w1, b1)
    out = [ratio((x[::K + 1].double() - rt_r).abs(), rt_b)]
    if mode:
        out += [ratio((stats[:, :mode].double() - st_r).abs(), st_b), ratio((h.double() - h_r).abs(), h_b)]
    else:
        assert bool((stats == 0).all()) and bool((h == 0).all())
    return out


@pytest.mark.parametrize('preset', list(PRESETS))
def test_rt_init_preset(preset):
    P = PRESETS[preset]
    for d in P['levels']:
        rs = _run_rt_init(P['depth'], d, P['K'], C1, P['mode'], P['mode'] == 0, 20 + d)
        _report(f'rt_init {preset} level {d} mode={MODE_NAMES[P["mode"]]} (rt, stats, h)', max(rs))


@pytest.mark.parametrize('K,C', [(48, 128), (64, 256), (48, 256), (64, 128)])
@pytest.mark.parametrize('src', ['src', 'no_src'])
@pytest.mark.parametrize('mode', [0, 3, 6, 9])
def test_rt_init_modes(mode, src, K, C):
    lv, _ = _level(7, 3, K)
    assert lv.n % K != 0
    rs = _run_rt_init(7, 3, K, C, mode, src == 'src', 30 + mode)
    _report(f'rt_init K={K} C={C} mode={MODE_NAMES[mode]} {src} (rt, stats, h)', max(rs))


# ---------------------------------------------------------------------------
# hfl_attn_pool: every level of a preset into one [B, ktot, C] buffer
# ---------------------------------------------------------------------------
SENTINEL = 7.25


def _pool_level(counts, K, kq, q_off, Tk, seed):
    """Runs hfl_attn_pool of one level (counts per submap) into Tk at q_off; returns max err/bound."""
    B = len(counts)
    n = int(sum(counts))
    W = max(1, -(-n // (K * DIL)) * DIL)
    rows = W * (K + 1)
    g = torch.Generator(device=DEV).manual_seed(seed)
    x = torch.randn(rows, C1, device=DEV, generator=g)
    x[hat_row(torch.arange(n, rows, device=DEV), K)[:max(0, W * K - n)]] = 0.0     # padding tokens
    xb = x.to(torch.bfloat16)
    npd = (kq + 63) // 64 * 64
    qp = torch.zeros(npd, C1, device=DEV, dtype=torch.bfloat16)
    qp[:kq] = torch.randn(kq, C1, device=DEV, generator=g).to(torch.bfloat16)
    logits = torch.empty(rows, npd, device=DEV)
    ops.gather_gemm(xb, qp, out_v_f32=logits)
    tok_off = torch.tensor([0] + list(np.cumsum(counts)), dtype=torch.int32, device=DEV)
    stat = torch.zeros(B, kq, 2, device=DEV)
    ops.attn_pool(logits, x, xb, tok_off, stat, Tk, B, kq, npd, K, C1, Tk.shape[1], q_off, C1 ** -0.5)
    r, bd = pool_ref(logits, xb, tok_off.cpu(), K, kq, C1 ** -0.5)
    return ratio((Tk[:, q_off:q_off + kq].double() - r).abs(), bd)


@pytest.mark.parametrize('preset', list(PRESETS))
def test_attn_pool_preset(preset):
    P = PRESETS[preset]
    o = _octree(P['depth'])
    ktot = sum(P['kq'])
    Tk = torch.full((o.batch_size, ktot, C1), SENTINEL, device=DEV)
    q_off = 0
    for j, (d, kq) in enumerate(zip(P['levels'], P['kq'])):
        counts = o.batch_nnum_nempty[d].numpy().astype(np.int64)
        r = _pool_level(counts, P['K'], kq, q_off, Tk, 40 + j)
        _report(f'attn_pool {preset} level {d} kq={kq} q_off={q_off}', r)
        q_off += kq
        assert bool((Tk[:, q_off:] == SENTINEL).all()), 'query slots of the other levels were written'


@pytest.mark.parametrize('kq', [148, 74, 72, 36, 18])
def test_attn_pool_segments(kq):
    """Segment lengths 0, 1, 63, 64, 65, 128, > 1000: tile edges, empty and one-token segments, segments that
    start mid-window; the query slots around this level's keep the sentinel."""
    counts = pool_segments()
    ktot, q_off = 300, 37
    Tk = torch.full((len(counts), ktot, C1), SENTINEL, device=DEV)
    r = _pool_level(counts, 48, kq, q_off, Tk, kq)
    _report(f'attn_pool segments kq={kq}', r)
    assert bool((Tk[:, :q_off] == SENTINEL).all()) and bool((Tk[:, q_off + kq:] == SENTINEL).all())


# ---------------------------------------------------------------------------
# Mixer tail, LayerNorm rows, GeM pooling and head
# ---------------------------------------------------------------------------
@pytest.mark.parametrize('preset', list(PRESETS))
def test_mixer_tail_and_ln_rows(preset):
    kin, kout, od = PRESETS[preset]['mixer']
    B = 5
    g = torch.Generator(device=DEV).manual_seed(50)
    x = torch.randn(B, kin, C1, device=DEV, generator=g) * 2 + 0.5
    wc, bc = torch.randn(kout, kin, device=DEV, generator=g) / kin ** 0.5, torch.randn(kout, device=DEV, generator=g) * 0.1
    wr, br = torch.randn(od, C1, device=DEV, generator=g) / C1 ** 0.5, torch.randn(od, device=DEV, generator=g) * 0.1
    for normalize in (True, False):
        out = torch.zeros(B, kout * od, device=DEV)
        ops.mixer_tail(x, wc, bc, wr, br, out, B, kin, kout, C1, od, normalize)
        r, bd = mixer_ref(x, wc, bc, wr, br, normalize)
        _report(f'mixer_tail {preset} {kin}->{kout} od={od} normalize={normalize}', ratio((out.double() - r).abs(), bd))
    lg, lb = torch.randn(C1, device=DEV, generator=g), torch.randn(C1, device=DEV, generator=g)
    y = torch.zeros(B * kin, C1, device=DEV, dtype=torch.bfloat16)
    ops.ln_rows(x.view(B * kin, C1), None, B * kin, C1, lg, lb, y)
    r, bd = ln_ref(x.view(B * kin, C1), lg, lb)
    _report(f'ln_rows {preset} rows={B * kin}', ratio((y.double() - r).abs(), bd))


@pytest.mark.parametrize('preset', ['oxford', 'cs-wild-places'])
def test_gem_pool_and_head(preset):
    P = PRESETS[preset]
    o, K = _octree(P['depth']), P['K']
    B, L = o.batch_size, len(P['levels'])
    pooled = torch.zeros(B, L * C1, device=DEV)
    g = torch.Generator(device=DEV).manual_seed(60)
    refs, bds = [], []
    for j, (d, pw) in enumerate(zip(P['levels'], (3.0, 2.5, 1.7))):
        counts = o.batch_nnum_nempty[d].numpy().astype(np.int64)
        n = int(counts.sum())
        W = -(-n // (K * DIL)) * DIL
        x = torch.zeros(W * (K + 1), C1, device=DEV)
        feat = torch.randn(n, C1, device=DEV, generator=g)
        x[hat_row(torch.arange(n, device=DEV), K)] = feat
        x[::K + 1] = 100.0                                # relay-token rows must not be pooled
        tok_off = torch.tensor([0] + list(np.cumsum(counts)), dtype=torch.int32, device=DEV)
        ops.gem_pool(x, tok_off, B, K, C1, pw, 1e-6, pooled, L * C1, j * C1)
        r, bd = gem_ref(feat, tok_off.cpu(), pw, 1e-6)
        refs.append(r)
        bds.append(bd)
    _report(f'gem_pool {preset}', ratio((pooled.double() - torch.cat(refs, 1)).abs(), torch.cat(bds, 1)))
    w = torch.randn(256, L * C1, device=DEV, generator=g) / (L * C1) ** 0.5
    bg, bb = torch.rand(256, device=DEV, generator=g) + 0.5, torch.randn(256, device=DEV, generator=g) * 0.1
    mu, var = torch.randn(256, device=DEV, generator=g) * 0.1, torch.rand(256, device=DEV, generator=g) + 0.5
    for normalize in (True, False):
        out = torch.zeros(B, 256, device=DEV)
        ops.gem_head(pooled, w, bg, bb, mu, var, 1e-5, normalize, out)
        r, bd = gem_head_ref(pooled, w, bg, bb, mu, var, 1e-5, normalize)
        _report(f'gem_head {preset} normalize={normalize}', ratio((out.double() - r).abs(), bd))


# ---------------------------------------------------------------------------
# empty problems at the ABI
# ---------------------------------------------------------------------------
def test_empty_problems_return_ok_and_write_nothing():
    """Every inference entry point of this stage returns HFL_OK and writes nothing when its problem is empty,
    and a normal call right after it still succeeds."""
    L = N.lib()
    s = N.stream()
    buf = torch.full((4096,), SENTINEL, device=DEV)
    bb = torch.zeros(4096, device=DEV, dtype=torch.bfloat16)
    ib = torch.full((4096,), -7, device=DEV, dtype=torch.int32)
    tok = torch.zeros(64 * 4, 4, device=DEV, dtype=torch.int16)
    off = torch.zeros(8, device=DEV, dtype=torch.int32)
    p, pb, pi, pt, po = N.ptr(buf), N.ptr(bb), N.ptr(ib), N.ptr(tok), N.ptr(off)
    calls = {
        'attn_pool B=0': lambda: L.hfl_attn_pool(p, p, pb, po, p, p, 0, 74, 128, 48, 256, 128, 0, 0.0625, s),
        'attn_pool kq=0': lambda: L.hfl_attn_pool(p, p, pb, po, p, p, 3, 0, 128, 48, 256, 128, 0, 0.0625, s),
        'mixer_tail B=0': lambda: L.hfl_mixer_tail(p, p, p, p, p, p, 0, 128, 32, 256, 8, 1, s),
        'gem_pool B=0': lambda: L.hfl_gem_pool(p, po, 0, 48, 256, 3.0, 1e-6, p, 768, 0, s),
        'gem_head B=0': lambda: L.hfl_gem_head(p, 0, 768, p, p, p, p, p, 1e-5, 256, 1, p, s),
        'window_attn n_win=0': lambda: L.hfl_window_attn(pb, pb, pt, p, 0, 16, 256, 64, 1, 1, 51, 0.25, s),
        'varlen_attn B=0': lambda: L.hfl_varlen_attn(pb, pb, po, pi, 0, 10, 16, 256, 0.25, s),
        'varlen_attn max_len=0': lambda: L.hfl_varlen_attn(pb, pb, po, pi, 3, 0, 16, 256, 0.25, s),
        'rt_init n_win=0': lambda: L.hfl_rt_init(p, None, pt, 0, 0, 48, 256, 5, 9, p, p, pb, p, s),
        'ln_rows m=0': lambda: L.hfl_ln_rows(p, None, 0, 256, p, p, pb, s),
        'cpe_ln rows=0': lambda: L.hfl_cpe_ln(p, pb, pi, pb, p, p, p, p, pb, None, 0, 0, 256, 48, s),
        'hat_rows n=0': lambda: L.hfl_hat_rows(pi, 0, 48, 0, s),
        'remap_hat n=0': lambda: L.hfl_remap_hat(pi, pi, 0, 48, s),
        'f32_to_bf16 n=0': lambda: L.hfl_f32_to_bf16(p, pb, 0, s),
    }
    x = torch.randn(2, 128, 256, device=DEV)
    wc, bc = torch.randn(32, 128, device=DEV) / 12, torch.zeros(32, device=DEV)
    wr, br = torch.randn(8, 256, device=DEV) / 16, torch.zeros(8, device=DEV)
    ref, bd = mixer_ref(x, wc, bc, wr, br, True)
    for name, call in calls.items():
        assert call() == 0, f'{name}: {N.lib().hfl_last_error_string()}'
        torch.cuda.synchronize()
        assert bool((buf == SENTINEL).all()) and bool((bb == 0).all()) and bool((ib == -7).all()), name
        out = torch.zeros(2, 256, device=DEV)
        ops.mixer_tail(x, wc, bc, wr, br, out, 2, 128, 32, 256, 8, True)
        assert ratio((out.double() - ref).abs(), bd) <= 1.0, f'call after {name}'
