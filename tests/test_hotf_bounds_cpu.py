"""Per-element error bounds of the HOTFormer-stage and pooling-head kernels, and the proof that they fit.

Each kernel of the embedding path after the OctFormer blocks (hfl_window_attn, hfl_varlen_attn, hfl_rt_init,
hfl_attn_pool, hfl_ln_rows, hfl_mixer_tail, hfl_gem_pool, hfl_gem_head) is compared in
tests/test_hotf_kernels_gpu.py with a float64 statement of its operation on the kernel's own operands, under a
bound per output element that names the rounding each term pays for.  This file holds those references and
bounds, and shows on the CPU that they are neither too loose nor too tight:

  * a small emulation of each kernel's arithmetic (bf16 P before P.V, fp16 RPE table entries and their fp16
    sum, bf16 outputs, fp32 statistics; ex2.approx taken as exact) stays within the bound;
  * each one-defect mutant of that emulation (a dropped key, a shifted RPE clamp, a query group read one
    column early, ...) breaks it.

Unit roundoffs: bf16 u = 2^-8 (8-bit significand), fp16 2^-11, fp32 2^-24.
"""
import math

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import model_ref as M

U = 2.0 ** -8          # bf16
U16 = 2.0 ** -11       # fp16
U32 = 2.0 ** -24       # fp32
SCALE = 0.25           # head_dim 16 ** -0.5
DIL = 4                # OctFormer dilation: every level is padded to a multiple of K * DIL tokens

# preset -> (depth, levels, K, ADaPE mode, pooling kq, mixer (kin, kout, od), uses hfl_window_attn)
PRESETS = {
    'oxford':         dict(depth=9, levels=(6, 5, 4), K=48, mode=9, kq=(74, 36, 18), mixer=(128, 32, 8), win=False),
    'cs-wild-places': dict(depth=7, levels=(4, 3, 2), K=64, mode=9, kq=(74, 36, 18), mixer=(128, 32, 8), win=True),
    'cs-campus3d':    dict(depth=7, levels=(4, 3, 2), K=64, mode=9, kq=(148, 72, 36), mixer=(256, 64, 4), win=True),
    'wild-places':    dict(depth=7, levels=(4, 3, 2), K=48, mode=0, kq=(148, 72, 36), mixer=(256, 64, 4), win=False),
}
MODE_NAMES = {0: 'none', 3: 'pos', 6: 'var', 9: 'cov'}


def bf16r(x):
    return x.to(torch.bfloat16).to(x.dtype)


def fp16r(x):
    return x.to(torch.float16).to(x.dtype)


def hat_row(t, K):
    return t + t // K + 1


def ratio(err, bound):
    """max err / bound (0 for empty tensors)."""
    return (err / bound).max().item() if err.numel() else 0.0


# ---------------------------------------------------------------------------
# batches: submaps shorter than a window, padding-only windows, a submap without relay tokens
# ---------------------------------------------------------------------------
def small_clouds(depth, seed=0):
    """Two big submaps around two tiny ones (a few nodes per level: they share windows with their neighbours,
    and at every preset's levels one of them owns no relay token)."""
    g = torch.Generator().manual_seed(seed)
    return [M.lidar_cloud(n, g) for n in (3000, 12, 40, 2500)]


def level_from_tokens(tok, n, depth, counts):
    """oracle Level of a padded (n_pad, 4) (x, y, z, submap) token table, on the table's device."""
    tok = tok.long()
    return M.Level(depth, n, tok.shape[0], tok[:, 3].clone(), tok[:, :3].clone(), np.asarray(counts, np.int64))


def ref_level(o, d, K):
    """(Level, token table) of depth d of an oracle octree, padded as the model pads (K * DIL)."""
    lv = M.make_level(o, d, K, DIL)
    tok = torch.cat([lv.xyz, lv.bid[:, None]], 1)
    return lv, tok


def window_ids(bid_w, hat):
    """(W, K + hat) attention ids: the relay token takes its window's first token's submap."""
    return torch.cat([bid_w[:, :1], bid_w], 1) if hat else bid_w


# ---------------------------------------------------------------------------
# attention: reference, bound
# ---------------------------------------------------------------------------
def _e1(P, v, r):
    """sum_j P_ij |v_j - r_i| over the last-but-one axis, in row chunks (P (..., L, Lk), v (..., Lk, D))."""
    L, Lk, D = P.shape[-2], P.shape[-1], v.shape[-1]
    lead = int(np.prod(P.shape[:-2])) if P.dim() > 2 else 1
    ch = max(1, (1 << 24) // max(1, lead * Lk * D))
    out = []
    for i0 in range(0, L, ch):
        i1 = min(L, i0 + ch)
        d = (v.unsqueeze(-3) - r[..., i0:i1, :].unsqueeze(-2)).abs()       # (..., c, Lk, D)
        out.append((P[..., i0:i1, :].unsqueeze(-1) * d).sum(-2))
    return torch.cat(out, -2)


def attn_bound(P, v, r, beta, centered):
    """Bound of |o - r| for o = bf16(softmax(s + e) v computed with bf16 P), with |e_ij| <= beta_i:
      u (1 + 2u) (|r| + A)    bf16 P (relative u per weight) and the bf16 output (u |o|); A = sum_j p_ij |v_j - r_i|
                              when the normaliser is the sum of the ROUNDED weights (the error is then centred on
                              r), else A = sum_j p_ij |v_j| (normaliser from the unrounded weights)
      expm1(2 beta) E1        score errors (fp16 RPE sum, fp32 q.k): softmax weights move by at most e^{+-2 beta}
      n 2^-24 sum p |v|       fp32 accumulation of the n-key products
      1e-6                    values next to zero"""
    E1 = _e1(P, v, r)
    Sv = P @ v.abs()
    lead = E1 if centered else Sv
    return U * (1 + 2 * U) * (r.abs() + lead) + torch.expm1(2 * beta) * E1 + P.shape[-1] * U32 * Sv + 1e-6


def rpe_pair(table, xyz, bnd, hat, clamp=None, relay_rpe=False):
    """(W, H, L, L) sum of the three table entries of each pair (tokens: clamp(dx, -bnd, bnd) + bnd + a num).
    hat: the relay token's row and column get nothing (relay_rpe: they get the first token's, a mutant)."""
    c = bnd if clamp is None else clamp
    num = 2 * bnd + 1
    if hat and relay_rpe:
        xyz = torch.cat([xyz[:, :1], xyz], 1)
    rel = (xyz.unsqueeze(2) - xyz.unsqueeze(1)).clamp(-c, c) + bnd
    parts = [table[rel[..., a] + a * num].permute(0, 3, 1, 2) for a in range(3)]    # (W, H, L', L')
    if hat and not relay_rpe:
        parts = [F.pad(p, (1, 0, 1, 0)) for p in parts]
    return parts


def window_ref(q, k, v, ids, xyz, table, K, hat):
    """float64 softmax(0.25 q k^T + same-submap mask + RPE) v per (window, head) and its bound.
    q, k, v (W, H, L, 16) f64; the RPE bias is oracle.model_ref._rpe_bias (relay row / column padded with 0).
    Returns r (W, H, L, 16), bound (same)."""
    s = (q @ k.transpose(-1, -2)) * SCALE
    beta = (q.abs() @ k.abs().transpose(-1, -2)) * SCALE * 2.0 ** -20          # fp32 q.k accumulation
    if table is not None:
        bias = M._rpe_bias({'t.rpe_table': table}, 't', xyz, K, 1)
        mag = M._rpe_bias({'t.rpe_table': table.abs()}, 't', xyz, K, 1)
        if hat:
            bias, mag = F.pad(bias, (1, 0, 1, 0)), F.pad(mag, (1, 0, 1, 0))
        s = s + bias
        # fp16 entries (3 roundings) + two fp16 adds, each relative 2^-11 of at most sum |entries|
        beta = beta + 5 * U16 * mag + 2.0 ** -20 * bias.abs()
    same = (ids.unsqueeze(2) == ids.unsqueeze(1)).unsqueeze(1)
    s = s.masked_fill(~same, float('-inf'))
    P = s.softmax(-1)
    r = P @ v
    beta = beta.masked_fill(~same, 0.0).amax(-1, keepdim=True)
    bound = attn_bound(P, v, r, beta, centered=True)
    return r, bound


def split_qkv(qkv, H):
    """(W, L, 3C) -> q, k, v (W, H, L, 16)."""
    W, L, C3 = qkv.shape
    return qkv.view(W, L, 3, H, 16).permute(2, 0, 3, 1, 4)


def window_check(out, qkv, ids, xyz, table, K, hat, H, chunk=16):
    """max |out - r| / bound over all windows; out (W, L, C), qkv (W, L, 3C) (kernel operands, any dtype)."""
    worst = 0.0
    W, L, C = out.shape
    for w0 in range(0, W, chunk):
        sl = slice(w0, w0 + chunk)
        q, k, v = split_qkv(qkv[sl].double(), H)
        r, bd = window_ref(q, k, v, ids[sl], xyz[sl], None if table is None else table.double(), K, hat)
        o = out[sl].double().view(-1, L, H, 16).transpose(1, 2)
        worst = max(worst, ratio((o - r).abs(), bd))
    return worst


WINDOW_MUTANTS = ['last_key_dropped', 'rpe_clamp_bnd_minus_1', 'rpe_on_relay_token', 'cross_submap_pair_unmasked']


def window_emulate(qkv, ids, xyz, table, K, hat, H, mutant=None):
    """hfl_window_attn's arithmetic: RPE entries as fp16 of entry / scale, summed (y + z) + x in fp16; scores
    q.k + bias / scale; token rows: P = 2^(...) rounded to bf16, normaliser = sum of the bf16 P; relay-token
    row: fp32 P; bf16 output."""
    W, L, _ = qkv.shape
    q, k, v = split_qkv(qkv.double(), H)
    s = q @ k.transpose(-1, -2)
    bnd = int(0.8 * K)
    if table is not None:
        t16 = fp16r(table.double() / SCALE)
        bx, by, bz = rpe_pair(t16, xyz, bnd, hat, clamp=bnd - 1 if mutant == 'rpe_clamp_bnd_minus_1' else None,
                              relay_rpe=mutant == 'rpe_on_relay_token')
        s = s + fp16r(fp16r(by + bz) + bx)
    s = s * SCALE
    same = (ids.unsqueeze(2) == ids.unsqueeze(1)).unsqueeze(1).expand(-1, H, -1, -1).clone()
    if mutant == 'last_key_dropped':
        same[..., L - 1] = False
    if mutant == 'cross_submap_pair_unmasked':
        w = int(torch.nonzero((ids != ids[:, :1]).any(1))[0])
        i = int(torch.nonzero(ids[w] != ids[w, -1])[-1])     # last token of the window's first-but-last submap
        same[w, :, L - 1, i] = True
    s = s.masked_fill(~same, float('-inf'))
    p = torch.exp(s - s.amax(-1, keepdim=True))
    pb = bf16r(p)
    if hat:
        pb[:, :, 0] = p[:, :, 0]                             # relay-token row: fp32 weights
    o = (pb @ v) / pb.sum(-1, keepdim=True)
    return bf16r(o).transpose(1, 2).reshape(W, L, H * 16)


# ---------------------------------------------------------------------------
# varlen (relay-token) attention
# ---------------------------------------------------------------------------
VA_KEYS = 80


def varlen_check(out, qkv, cu, ids, H):
    """max |out - r| / bound over the rows of every sequence [cu[b], cu[b+1])."""
    worst = 0.0
    cu = [int(c) for c in cu]
    for b in range(len(cu) - 1):
        s0, s1 = cu[b], cu[b + 1]
        if s1 <= s0:
            continue
        L = s1 - s0
        q, k, v = qkv[s0:s1].double().view(L, 3, H, 16).permute(1, 2, 0, 3)
        i = ids[s0:s1]
        s = (q @ k.transpose(-1, -2)) * SCALE
        same = (i[:, None] == i[None, :])[None]
        P = s.masked_fill(~same, float('-inf')).softmax(-1)
        r = P @ v
        beta = ((q.abs() @ k.abs().transpose(-1, -2)) * SCALE * 2.0 ** -20).masked_fill(~same, 0).amax(-1, True)
        bd = attn_bound(P, v, r, beta, centered=False)     # normaliser sums the unrounded fp32 weights
        o = out[s0:s1].double().view(L, H, 16).transpose(0, 1)
        worst = max(worst, ratio((o - r).abs(), bd))
    return worst


VARLEN_MUTANTS = ['cu_entry_moved_by_one', 'key_80_dropped']


def varlen_emulate(qkv, cu, ids, H, mutant=None):
    """hfl_varlen_attn's arithmetic: online softmax over blocks of 80 keys; per block P = 2^(s - running max)
    rounded to bf16 for P.V, the running sum l over the UNROUNDED P; out = bf16(o / l).  Rows in no
    sequence stay 0."""
    T = qkv.shape[0]
    out = torch.zeros(T, H * 16, dtype=torch.float64, device=qkv.device)
    cu = [int(c) for c in cu]
    if mutant == 'cu_entry_moved_by_one':
        cu[1] += 1
    for b in range(len(cu) - 1):
        s0, s1 = cu[b], cu[b + 1]
        L = s1 - s0
        if L <= 0:
            continue
        q, k, v = qkv[s0:s1].double().view(L, 3, H, 16).permute(1, 2, 0, 3)
        i = ids[s0:s1]
        m = torch.full((H, L, 1), float('-inf'), dtype=torch.float64, device=qkv.device)
        l = torch.zeros_like(m)
        o = torch.zeros(H, L, 16, dtype=torch.float64, device=qkv.device)
        for k0 in range(0, L, VA_KEYS):
            k1 = min(L, k0 + VA_KEYS)
            s = (q @ k[:, k0:k1].transpose(-1, -2)) * SCALE
            same = (i[:, None] == i[None, k0:k1])[None].expand(H, -1, -1).clone()
            if mutant == 'key_80_dropped' and k0 <= 80 < k1:
                same[..., 80 - k0] = False
            s = s.masked_fill(~same, float('-inf'))
            n = torch.maximum(m, s.amax(-1, keepdim=True))
            e = torch.where(n == float('-inf'), torch.zeros_like(n), n)
            c = torch.exp(m - e)
            p = torch.exp(s - e)
            l = l * c + p.sum(-1, keepdim=True)
            o = o * c + bf16r(p) @ v[:, k0:k1]
            m = n
        res = torch.where(l > 0, o / l, torch.zeros_like(o))
        out[s0:s1] = bf16r(res).transpose(0, 1).reshape(L, H * 16)
    return out


def varlen_layout(lens, pad_tail=0, device='cpu'):
    """cu / ids of sequences of the given lengths; the last pad_tail rows carry the padding id B."""
    cu = torch.tensor([0] + list(np.cumsum(lens)), dtype=torch.int32)
    ids = torch.cat([torch.full((l,), b, dtype=torch.int32) for b, l in enumerate(lens)]) if sum(lens) else \
        torch.zeros(0, dtype=torch.int32)
    if pad_tail:
        ids[-pad_tail:] = len(lens)
    return cu.to(device), ids.to(device)


# ---------------------------------------------------------------------------
# relay-token init + ADaPE statistics + fc1 / GELU
# ---------------------------------------------------------------------------
def window_stats64(lv, K, valid=None):
    """float64 form of oracle.model_ref.window_stats (cov layout: mean xyz, then xx xy xz yy yz zz) and its
    fp32 bound.  The points x 2^(1-d) - 1 are exact in fp32; the kernel pays for the sums only:
      mean  (K + 3) 2^-24 sum |p| / cnt                            K-term sum, division, reciprocal
      cov   (2K + 8) 2^-24 sum |d_a| |d_b| / (cnt - 1) + cnt dm_a dm_b / (cnt - 1)
            the rounded deviations d = p - mean, products, K-term sum, division; the mean's own error dm
            enters only at second order because the deviations sum to zero."""
    d = lv.depth
    pts = lv.xyz.double() * 2.0 ** (1 - d) - 1.0
    pts[lv.n:] = 0.0
    pts = pts.view(-1, K, 3)
    bid = lv.bid.view(-1, K)
    if valid is None:
        valid = bid == bid[:, :1]
    v = valid.unsqueeze(-1).double()
    cnt = valid.sum(1, keepdim=True).double()
    cc = cnt.clamp(min=1.0)
    mu = (pts * v).sum(1) / cc
    cen = (pts - mu.unsqueeze(1)) * v
    den = (cnt - 1).clamp(min=1.0)
    ok = (cnt >= 2).double()
    iu = torch.triu_indices(3, 3)
    cov = (cen.transpose(1, 2) @ cen)[:, iu[0], iu[1]] / den * ok
    mu_b = (K + 3) * U32 * (pts.abs() * v).sum(1) / cc
    acen = cen.abs()
    cov_b = ((2 * K + 8) * U32 * (acen.transpose(1, 2) @ acen)[:, iu[0], iu[1]]
             + cnt * (mu_b[:, iu[0]] * mu_b[:, iu[1]])) / den * ok
    return torch.cat([mu, cov], 1), torch.cat([mu_b, cov_b], 1) + 1e-12


def select_stats(st9, mode):
    """The mode's columns of the cov layout: pos = mean, var = mean + xx yy zz, cov = all nine."""
    cols = {3: [0, 1, 2], 6: [0, 1, 2, 3, 6, 8], 9: list(range(9))}[mode]
    return st9[:, cols]


def gelu64(a):
    return 0.5 * a * (1.0 + torch.erf(a / math.sqrt(2.0)))


def rt_ref(feat, lv, K, mode, w1, b1):
    """Reference relay-token rows (oracle rt_init on float64 token features), statistics of the mode and h,
    each with its bound:
      rt    (K + 3) 2^-24 sum |x| / cnt       fp32 K-term sum and the multiply by 1 / cnt
      h     u (1 + u) |h| + 1.13 da + |a| (2^-21 + |a| 2^-24) / 2 + 1e-7
            bf16 output; GELU slope <= 1.13 times the fc1 error da (statistics error through |w1| plus the
            fp32 dot product); erff (2 ulp) and the rounding of its argument."""
    rt = M.rt_init(feat.double(), lv, K)
    xp = torch.cat([feat.double(), feat.new_zeros(lv.n_pad - lv.n, feat.shape[1]).double()]).view(-1, K, feat.shape[1])
    bid = lv.bid.view(-1, K)
    v = (bid == bid[:, :1]).unsqueeze(-1).double()
    rt_b = (K + 3) * U32 * (xp.abs() * v).sum(1) / v.sum(1) + 1e-30
    if mode == 0:
        return rt, rt_b, None, None, None, None
    st9, st9_b = window_stats64(lv, K)
    st, st_b = select_stats(st9, mode), select_stats(st9_b, mode)
    w1, b1 = w1.double(), b1.double()
    a = st @ w1.t() + b1
    da = st_b @ w1.abs().t() + (mode + 2) * U32 * (st.abs() @ w1.abs().t() + b1.abs())
    h = gelu64(a)
    h_b = U * (1 + U) * h.abs() + 1.13 * da + 0.5 * a.abs() * (2.0 ** -21 + a.abs() * U32) + 1e-7
    return rt, rt_b, st, st_b, h, h_b


RT_MUTANTS = ['var_without_repack', 'cov_divided_by_cnt', 'padding_counted_in_real_window']


def rt_emulate(feat, lv, K, mode, w1, b1, mutant=None):
    """hfl_rt_init's arithmetic in fp32: masked sum then * (1 / cnt); statistics with fp32 sums; fc1 + GELU in
    fp32, bf16 h."""
    f32 = torch.float32
    C = feat.shape[1]
    xp = torch.cat([feat.to(f32), feat.new_zeros(lv.n_pad - lv.n, C).to(f32)]).view(-1, K, C)
    bid = lv.bid.view(-1, K)
    valid = bid == bid[:, :1]
    if mutant == 'padding_counted_in_real_window':
        valid = valid | (bid == int(lv.bid.max()))
    cnt = valid.sum(1, keepdim=True).to(f32)
    rt = (xp * valid.unsqueeze(-1)).sum(1) * (1.0 / cnt)
    if mode == 0:
        return rt, None, None
    pts = (lv.xyz.to(f32) * 2.0 ** (1 - lv.depth) - 1.0)
    pts[lv.n:] = 0.0
    pts = pts.view(-1, K, 3)
    v = valid.unsqueeze(-1).to(f32)
    mu = (pts * v).sum(1) / cnt.clamp(min=1.0)
    cen = (pts - mu.unsqueeze(1)) * v
    den = cnt if mutant == 'cov_divided_by_cnt' else (cnt - 1).clamp(min=1.0)
    ok = (cnt >= 2).to(f32)
    iu = torch.triu_indices(3, 3)
    cov = (cen.transpose(1, 2) @ cen)[:, iu[0], iu[1]] / den * ok
    st9 = torch.cat([mu, cov], 1)
    if mode == 6 and mutant == 'var_without_repack':
        st = st9[:, :6]
    else:
        st = select_stats(st9, mode)
    a = st @ w1.to(f32).t() + b1.to(f32)
    return rt, st, bf16r(F.gelu(a))


# ---------------------------------------------------------------------------
# attention pooling
# ---------------------------------------------------------------------------
PM_Q = 80


def pool_ref(logits, xb, tok_off, K, kq, scale):
    """float64 softmax_t(scale logits[t, q]) x[t] per segment over the hat rows of its tokens, and the bound
      u sum_t p_t |x_t|                     bf16 P (normalised before rounding; no re-normalisation)
      (n + 16) 2^-24 sum_t p_t |x_t|        fp32 sum of exp (per warp, then merged) and the fp32 P.X accumulation
      2^-22 (1 + 2 max |s|) sum_t p_t |x_t| fp32 rounding of the exponent argument s - max
      1e-6
    Returns r (B, kq, C), bound (B, kq, C)."""
    B = tok_off.numel() - 1
    C = xb.shape[1]
    r = torch.zeros(B, kq, C, dtype=torch.float64, device=xb.device)
    bd = torch.full_like(r, 1e-6)
    to = [int(t) for t in tok_off]
    for b in range(B):
        t0, t1 = to[b], to[b + 1]
        if t1 <= t0:
            continue
        rows = hat_row(torch.arange(t0, t1, device=xb.device), K)
        s = logits[rows, :kq].double().t() * scale                 # (kq, n)
        P = s.softmax(-1)
        x = xb[rows].double()
        r[b] = P @ x
        Sx = P @ x.abs()
        amax = s.abs().amax(-1, keepdim=True)
        bd[b] += (U + (t1 - t0 + 16) * U32 + 2.0 ** -22 * (1 + 2 * amax * 1.4426950408889634)) * Sx
    return r, bd


POOL_MUTANTS = ['second_query_group_at_qbase_minus_1', 'segment_last_token_dropped', 'rows_without_hat_offset']


def pool_emulate(logits, xb, tok_off, K, kq, scale, mutant=None):
    """hfl_attn_pool's arithmetic: (max, 1 / sum) per (segment, query), P = bf16(2^(s - max) / sum), out = P^T X."""
    B = tok_off.numel() - 1
    C = xb.shape[1]
    out = torch.zeros(B, kq, C, dtype=torch.float64, device=xb.device)
    to = [int(t) for t in tok_off]
    cols = torch.arange(kq, device=xb.device)
    if mutant == 'second_query_group_at_qbase_minus_1':
        cols = torch.where(cols >= PM_Q, cols - 1, cols)
    for b in range(B):
        t0, t1 = to[b], to[b + 1]
        if mutant == 'segment_last_token_dropped':
            t1 -= 1
        if t1 <= t0:
            continue
        t = torch.arange(t0, t1, device=xb.device)
        rows = t if mutant == 'rows_without_hat_offset' else hat_row(t, K)
        s = logits[rows][:, cols].double().t() * scale
        p = torch.exp(s - s.amax(-1, keepdim=True))
        P = bf16r(p / p.sum(-1, keepdim=True))
        out[b] = P @ xb[rows].double()
    return out


# ---------------------------------------------------------------------------
# LayerNorm rows, Mixer tail, GeM pooling and head (fp32 kernels)
# ---------------------------------------------------------------------------
def ln_ref(x, g, b):
    """LayerNorm (eps 1e-5) in float64 and the bound of the fp32 kernel with bf16 output:
    u (1 + u) |y| + (2C + 8) 2^-24 |g| (|xhat| + 1) + 2^-24 |b|   (mean / variance sums over C, rsqrt)."""
    x, g, b = x.double(), g.double(), b.double()
    C = x.shape[-1]
    mu = x.mean(-1, keepdim=True)
    var = ((x - mu) ** 2).mean(-1, keepdim=True)
    xh = (x - mu) / torch.sqrt(var + 1e-5)
    y = xh * g + b
    return y, U * (1 + U) * y.abs() + (2 * C + 8) * U32 * g.abs() * (xh.abs() + 1) + U32 * b.abs() + 1e-7


def mixer_ref(x, wc, bc, wr, br, normalize):
    """channel_proj over the token axis, row_proj, flatten, L2 normalise, float64, and the fp32 bound from the
    absolute-value chain: dy = (kin + 2) 2^-24 (|wc| |x| + |bc|), dd = (C + 2) 2^-24 (|wr| |y| + |br|) + |wr| dy,
    normalised: dd / |d| + |out| (|dd|_2 / |d| + (n + 4) 2^-24)."""
    x, wc, bc, wr, br = (t.double() for t in (x, wc, bc, wr, br))
    kin, C = x.shape[1], x.shape[2]
    y = torch.einsum('ok,bkc->boc', wc, x) + bc[None, :, None]
    dy = (kin + 2) * U32 * (torch.einsum('ok,bkc->boc', wc.abs(), x.abs()) + bc.abs()[None, :, None])
    d = y @ wr.t() + br
    dd = (C + 2) * U32 * (y.abs() @ wr.abs().t() + br.abs()) + dy @ wr.abs().t()
    d, dd = d.flatten(1), dd.flatten(1)
    if not normalize:
        return d, dd + 1e-7
    nrm = d.norm(dim=1, keepdim=True)
    out = d / nrm
    return out, dd / nrm + out.abs() * (dd.norm(dim=1, keepdim=True) / nrm + (d.shape[1] + 4) * U32) + 1e-7


def gem_ref(feat, tok_off, pw, eps):
    """(mean_t max(x, eps)^p)^(1/p) per segment, float64, and the fp32 bound: powf (4 ulp each), the n-term
    sum, the division and the final powf: |r| ((n + 8) 2^-24 / p + 8 2^-24 (1 + 1 / p))."""
    B = tok_off.numel() - 1
    C = feat.shape[1]
    r = torch.zeros(B, C, dtype=torch.float64, device=feat.device)
    bd = torch.zeros_like(r)
    to = [int(t) for t in tok_off]
    for b in range(B):
        t0, t1 = to[b], to[b + 1]
        n = max(t1 - t0, 0)
        a = feat[t0:t1].double().clamp(min=eps).pow(pw).sum(0) / max(n, 1)
        r[b] = a.pow(1.0 / pw)
        bd[b] = r[b].abs() * ((n + 8) * U32 / pw + 8 * U32 * (1 + 1 / pw))
    return r, bd + 1e-30


def gem_head_ref(pooled, w, g, b, mu, var, eps, normalize):
    """Linear (no bias) + eval BatchNorm1d (+ L2 normalise), float64, with the fp32 bound of the fmaf chain over
    in_dim, rsqrtf (2 ulp) and the normalisation."""
    pooled, w, g, b, mu, var = (t.double() for t in (pooled, w, g, b, mu, var))
    n = pooled.shape[1]
    a = pooled @ w.t()
    da = (n + 2) * U32 * (pooled.abs() @ w.abs().t())
    s = g / torch.sqrt(var + eps)
    y = (a - mu) * s + b
    dy = da * s.abs() + 8 * U32 * ((a - mu).abs() * s.abs() + b.abs())
    if not normalize:
        return y, dy + 1e-7
    nrm = y.norm(dim=1, keepdim=True)
    out = y / nrm
    return out, dy / nrm + out.abs() * (dy.norm(dim=1, keepdim=True) / nrm + (y.shape[1] + 4) * U32) + 1e-7


# ===========================================================================
# CPU proofs: every emulation within its bound, every mutant outside
# ===========================================================================
_BATCHES = {}


def _batch(depth):
    if depth not in _BATCHES:
        from oracle import octree_ref as R
        _BATCHES[depth] = R.build_batch(small_clouds(depth), depth)
    return _BATCHES[depth]


def wide_windows(W, K, B=3, seed=0):
    """Synthetic windows whose coordinates span 128 cells, so that offsets reach the RPE clamp (the coarse
    levels of a real batch are at most 16 cells wide); bid sorted, the last 37 tokens padding."""
    g = torch.Generator().manual_seed(seed)
    n_pad = W * K
    xyz = torch.randint(0, 128, (n_pad, 3), generator=g)
    bid = torch.sort(torch.randint(0, B, (n_pad,), generator=g)).values
    bid[n_pad - 37:] = B
    xyz[n_pad - 37:] = 0
    return xyz.view(W, K, 3), bid.view(W, K)


def _win_case(K, d, H, table_std, seed=0):
    """Windows of depth d of the CPU batch (d = None: wide synthetic windows), bf16 qkv, a table of std table_std."""
    if d is None:
        xyz, bid = wide_windows(12, K)
    else:
        lv, _ = ref_level(_batch(7), d, K)
        xyz, bid = lv.xyz.view(-1, K, 3), lv.bid.view(-1, K)
    ids = window_ids(bid, True)
    W, L = ids.shape
    g = torch.Generator().manual_seed(seed)
    qkv = bf16r(torch.randn(W, L, 3 * 16 * H, generator=g, dtype=torch.float64))
    bnd = int(0.8 * K)
    table = None if table_std is None else torch.randn(3 * (2 * bnd + 1), H, generator=g, dtype=torch.float64) * table_std
    return qkv, ids, xyz, table


def test_batches_have_the_edge_windows():
    """The CPU batches hold windows spanning several submaps, padding-only windows and a submap that owns no
    relay token at a coarse level."""
    o = _batch(7)
    for K in (48, 64):
        lvs = [ref_level(o, d, K)[0] for d in (4, 3, 2)]
        bids = [lv.bid.view(-1, K) for lv in lvs]
        assert any(bool((b != b[:, :1]).any(1).any()) for b in bids)
        assert any(bool((b == o.batch_size).all(1).any()) for b in bids)
        assert any(bool((lv.num_windows == 0).any()) for lv in lvs)


@pytest.mark.parametrize('K,d', [(64, 4), (64, 2), (64, None), (96, 3), (96, None)])
@pytest.mark.parametrize('table', ['rpe', 'no_rpe', 'rpe_large'])
def test_window_emulation_within_bound(K, d, table):
    std = {'rpe': 1.0, 'no_rpe': None, 'rpe_large': 16.0}[table]
    qkv, ids, xyz, tab = _win_case(K, d, 8, std)
    out = window_emulate(qkv, ids, xyz, tab, K, True, 8)
    r = window_check(out, qkv, ids, xyz, tab, K, True, 8)
    print(f'window_attn emulation K={K} d={d} {table}: max err/bound = {r:.3f}')
    assert r <= 1.0


@pytest.mark.parametrize('mutant', WINDOW_MUTANTS)
def test_window_mutant_rejected(mutant):
    qkv, ids, xyz, tab = _win_case(64, None if mutant == 'rpe_clamp_bnd_minus_1' else 3, 8, 1.0)
    out = window_emulate(qkv, ids, xyz, tab, 64, True, 8, mutant=mutant)
    r = window_check(out, qkv, ids, xyz, tab, 64, True, 8)
    print(f'window_attn mutant {mutant}: max err/bound = {r:.3f}')
    assert r > 1.0


def test_window_fp16_bias_is_what_the_bound_pays_for():
    """With a large table the fp16 bias sum is the dominant error: the bound without its beta term is broken
    by the emulation, so the beta term is needed (not slack)."""
    qkv, ids, xyz, tab = _win_case(64, 4, 8, 16.0)
    out = window_emulate(qkv, ids, xyz, tab, 64, True, 8)
    q, k, v = split_qkv(qkv, 8)
    s = (q @ k.transpose(-1, -2)) * SCALE + F.pad(M._rpe_bias({'t.rpe_table': tab}, 't', xyz, 64, 1), (1, 0, 1, 0))
    s = s.masked_fill(~(ids.unsqueeze(2) == ids.unsqueeze(1)).unsqueeze(1), float('-inf'))
    P = s.softmax(-1)
    r = P @ v
    bd = attn_bound(P, v, r, torch.zeros_like(r[..., :1]), centered=True)
    o = out.view(-1, 65, 8, 16).transpose(1, 2)
    assert ratio((o - r).abs(), bd) > 1.0


def _varlen_case(H, lens, pad_tail=3, seed=1):
    cu, ids = varlen_layout(lens, pad_tail)
    g = torch.Generator().manual_seed(seed)
    qkv = bf16r(torch.randn(int(cu[-1]), 3 * 16 * H, generator=g, dtype=torch.float64))
    return qkv, cu, ids


LENS = [0, 1, 79, 80, 81, 160, 255, 256, 257, 513]


@pytest.mark.parametrize('H', [16, 8])
def test_varlen_emulation_within_bound(H):
    qkv, cu, ids = _varlen_case(H, LENS)
    r = varlen_check(varlen_emulate(qkv, cu, ids, H), qkv, cu, ids, H)
    print(f'varlen_attn emulation H={H}: max err/bound = {r:.3f}')
    assert r <= 1.0


@pytest.mark.parametrize('mutant', VARLEN_MUTANTS)
def test_varlen_mutant_rejected(mutant):
    qkv, cu, ids = _varlen_case(8, [90, 160, 33])
    r = varlen_check(varlen_emulate(qkv, cu, ids, 8, mutant=mutant), qkv, cu, ids, 8)
    print(f'varlen_attn mutant {mutant}: max err/bound = {r:.3f}')
    assert r > 1.0


def _rt_case(K, C, mode, seed=2):
    o = _batch(7)
    lv, _ = ref_level(o, 3, K)
    g = torch.Generator().manual_seed(seed)
    feat = torch.randn(lv.n, C, generator=g)
    w1 = torch.randn(C, max(mode, 1), generator=g) * 0.5
    b1 = torch.randn(C, generator=g) * 0.1
    return lv, feat, w1, b1


def _rt_ratios(lv, feat, K, mode, w1, b1, rt, st, h):
    rt_r, rt_b, st_r, st_b, h_r, h_b = rt_ref(feat, lv, K, mode, w1, b1)
    out = [ratio((rt.double() - rt_r).abs(), rt_b)]
    if mode:
        out += [ratio((st.double() - st_r).abs(), st_b), ratio((h.double() - h_r).abs(), h_b)]
    return out


@pytest.mark.parametrize('K,C', [(48, 128), (64, 256)])
@pytest.mark.parametrize('mode', [0, 3, 6, 9])
def test_rt_init_emulation_within_bound(K, C, mode):
    lv, feat, w1, b1 = _rt_case(K, C, mode)
    assert lv.n % K != 0
    rs = _rt_ratios(lv, feat, K, mode, w1, b1, *rt_emulate(feat, lv, K, mode, w1, b1))
    print(f'rt_init emulation K={K} C={C} mode={MODE_NAMES[mode]}: max err/bound (rt, stats, h) = '
          + ', '.join(f'{r:.3f}' for r in rs))
    assert max(rs) <= 1.0


def test_window_stats_restatement_matches_the_oracle():
    """window_stats64 is oracle.model_ref.window_stats in float64: the oracle's fp32 values are within the fp32
    bound of it in every mode."""
    o = _batch(7)
    for K, d in ((48, 4), (64, 2)):
        lv, _ = ref_level(o, d, K)
        st9, b9 = window_stats64(lv, K)
        for mode, name in ((3, 'pos'), (6, 'var'), (9, 'cov')):
            ref = M.window_stats(lv, K, name).double()
            assert ratio((ref - select_stats(st9, mode)).abs(), select_stats(b9, mode)) <= 1.0, (K, d, name)


@pytest.mark.parametrize('mutant', RT_MUTANTS)
def test_rt_init_mutant_rejected(mutant):
    mode = 6 if mutant == 'var_without_repack' else (0 if mutant == 'padding_counted_in_real_window' else 9)
    lv, feat, w1, b1 = _rt_case(64, 128, mode)
    rs = _rt_ratios(lv, feat, 64, mode, w1, b1, *rt_emulate(feat, lv, 64, mode, w1, b1, mutant=mutant))
    print(f'rt_init mutant {mutant}: max err/bound = {max(rs):.3f}')
    assert max(rs) > 1.0


def pool_segments(total_long=1100):
    """Segment lengths of the synthetic pooling case: empty, 1, the 64-token tile edges and a long one."""
    return [0, 1, 63, 64, 65, 128, total_long, 5]


def _pool_case(kq, K=48, C=64, seed=3, counts=None):
    counts = counts or pool_segments()
    n = sum(counts)
    W = -(-n // K)
    rows = W * (K + 1)
    g = torch.Generator().manual_seed(seed)
    xb = bf16r(torch.randn(rows, C, generator=g))
    npd = (kq + 63) // 64 * 64
    qp = torch.zeros(npd, C)
    qp[:kq] = bf16r(torch.randn(kq, C, generator=g))
    logits = (xb.double() @ qp.double().t()).float()            # what the fp32 GEMM writes (to rounding)
    tok_off = torch.tensor([0] + list(np.cumsum(counts)), dtype=torch.int32)
    return logits, xb, tok_off, C ** -0.5


@pytest.mark.parametrize('kq', [148, 74, 18])
def test_pool_emulation_within_bound(kq):
    logits, xb, tok_off, sc = _pool_case(kq)
    r, bd = pool_ref(logits, xb, tok_off, 48, kq, sc)
    out = pool_emulate(logits, xb, tok_off, 48, kq, sc)
    rr = ratio((out - r).abs(), bd)
    print(f'attn_pool emulation kq={kq}: max err/bound = {rr:.3f}')
    assert rr <= 1.0


@pytest.mark.parametrize('mutant', POOL_MUTANTS)
def test_pool_mutant_rejected(mutant):
    logits, xb, tok_off, sc = _pool_case(148)
    r, bd = pool_ref(logits, xb, tok_off, 48, 148, sc)
    rr = ratio((pool_emulate(logits, xb, tok_off, 48, 148, sc, mutant=mutant) - r).abs(), bd)
    print(f'attn_pool mutant {mutant}: max err/bound = {rr:.3f}')
    assert rr > 1.0


@pytest.mark.parametrize('kin,kout,od', [(128, 32, 8), (256, 64, 4)])
def test_head_fp32_emulations_within_bound(kin, kout, od):
    """fp32 torch statements of ln_rows, mixer_tail and gem_pool stay within their bounds."""
    g = torch.Generator().manual_seed(4)
    B, C = 3, 256
    x = torch.randn(B * kin, C, generator=g) * 3 + 1
    lg, lb = torch.randn(C, generator=g), torch.randn(C, generator=g)
    y, yb = ln_ref(x, lg, lb)
    assert ratio((bf16r(F.layer_norm(x, (C,), lg, lb, 1e-5)).double() - y).abs(), yb) <= 1.0
    xm = x.view(B, kin, C)
    wc, bc = torch.randn(kout, kin, generator=g) / kin ** 0.5, torch.randn(kout, generator=g) * 0.1
    wr, br = torch.randn(od, C, generator=g) / C ** 0.5, torch.randn(od, generator=g) * 0.1
    for nz in (True, False):
        d = F.linear(F.linear(xm.transpose(1, 2), wc, bc).transpose(1, 2), wr, br).flatten(1)
        d = F.normalize(d, dim=1) if nz else d
        r, bd = mixer_ref(xm, wc, bc, wr, br, nz)
        assert ratio((d.double() - r).abs(), bd) <= 1.0
    counts = [300, 0, 1, 64]
    tok_off = torch.tensor([0] + list(np.cumsum(counts)))
    feat = torch.randn(sum(counts), C, generator=g)
    r, bd = gem_ref(feat, tok_off, 3.0, 1e-6)
    emu = torch.stack([(feat[a:b].clamp(min=1e-6).pow(3.0).sum(0) / max(b - a, 1)).pow(1 / 3.0)
                       for a, b in zip(tok_off[:-1].tolist(), tok_off[1:].tolist())])
    assert ratio((emu.double() - r).abs(), bd) <= 1.0
