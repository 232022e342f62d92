"""Timing and peak memory of the relay-token self-attention op (csrc/rt_attn_train.cu, through
hotformerloc_b200.relay_token_attention) at training sizes, against the padded fp32 torch statement of the
reference formulation on the same GPU (hotformerloc_backbone.py:83-119, 275-295; relay_token_utils.py:12-79;
models/octree.py:229-265), under autograd: the RTs padded to (B, Nmax, C), a (B, Nmax, Nmax) int64 mask, dense
attention with the -1000 bias, and the split back.

Two measurements per shape:
  core  : the attention core from qkv to before proj (relay_token_attention vs the padded statement)
  block : a whole RelayTokenTransformerBlock without drop path: pack, LayerNorm, qkv, core, proj, residual,
          LayerNorm, MLP, residual, unpack (torch layers around the native core vs the padded statement)
Shapes (128-submap training minibatches, C = 256, H = 16; RT counts from batch_nnum_nempty of the pyramid):
  oxford : 128 x 4096-point submaps, depth-9 octree, levels at depths 6 / 5 / 4, K = 48, dilation 4
  cswild : 128 aerial submaps of 30 k and 60 k points interleaved, depth-7 octree, levels 4 / 3 / 2, K = 64
Algorithmic work of the core, summed over the sequences: forward 4 n^2 C FLOPs, backward 10 n^2 C (the kernels
recompute the scores and dO.v once more: 14 n^2 C executed).  Bytes (each operand once): forward reads qkv and
writes o and lse; backward reads qkv, o, lse and dout and writes dqkv.

    python tools/rt_attn_train_bench.py [--iters 20] [--warmup 3] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
import torch.nn.functional as F

from hotformerloc_b200 import native as N
from hotformerloc_b200.models.hotformerloc import _RTSABlock
from hotformerloc_b200.octree import build_batch
from hotformerloc_b200.relay_token_attention import RTAttention, relay_token_attention, rt_layout
from oracle import model_ref as M

HBM_GBPS = 7700.0


def device_info():
    idx = torch.cuda.current_device()
    info = {'name': torch.cuda.get_device_name(idx)}
    try:
        r = subprocess.run(['nvidia-smi', '-i', str(idx), '--query-gpu=power.limit,clocks.max.sm',
                            '--format=csv,noheader,nounits'], capture_output=True, text=True, timeout=30)
        pl, mhz = [x.strip() for x in r.stdout.strip().split(',')]
        info.update(power_limit_w=float(pl), sm_max_mhz=float(mhz))
    except Exception as e:                     # report, do not guess
        info.update(power_limit_w=None, sm_max_mhz=None, query_error=str(e))
    return info


def time_ms(fn, iters, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(iters):
        fn()
    e.record()
    torch.cuda.synchronize()
    return s.elapsed_time(e) / iters


def peak_mb(fn):
    """Peak of the bytes tensors request during fn (without the caching allocator's block rounding)."""
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    base = torch.cuda.memory_stats()['requested_bytes.all.current']
    torch.cuda.reset_peak_memory_stats()
    fn()
    torch.cuda.synchronize()
    return round((torch.cuda.memory_stats()['requested_bytes.all.peak'] - base) / 2 ** 20, 1)


def padded_plan(layout):
    """concat_and_pad_rt's (B, Nmax) gather (-1 = padding slot) of the packed rows and of the rows of the
    level concatenation, and its ids (padding slots: an id no RT has), from the layout's host counts."""
    lens = np.sum(layout.num_windows, axis=0)
    B, nmax = len(lens), int(lens.max())
    cu = np.concatenate([[0], np.cumsum(lens)])
    t = np.arange(nmax)[None]
    index = np.where(t < lens[:, None], cu[:-1, None] + t, -1)
    index = torch.from_numpy(index).cuda()
    ids = torch.where(index >= 0, layout.ids.long()[index.clamp(min=0)], torch.full_like(index, 10000))
    index_cat = torch.where(index >= 0, layout.index.long()[index.clamp(min=0)], index)
    return index, index_cat, ids


def torch_core(qkv, index, ids, H):
    """fp32 reference formulation: pad to (B, Nmax, 3C), (B, Nmax, Nmax) int64 mask, dense attention, unpad."""
    real = index >= 0
    xp = qkv[index.clamp(min=0)] * real.unsqueeze(-1)
    B, L, C3 = xp.shape
    C = C3 // 3
    mask = (ids.unsqueeze(2) != ids.unsqueeze(1)).to(torch.int64)                          # (B, Nmax, Nmax)
    q, k, v = xp.view(B, L, 3, H, C // H).permute(2, 0, 3, 1, 4)
    att = (q @ k.transpose(-1, -2)) * (C // H) ** -0.5 + mask.unsqueeze(1).float() * -1000.0
    op = (att.softmax(-1) @ v).transpose(1, 2).reshape(B, L, C)
    return op[real]


def torch_block(blk, rts, index, ids, H):
    """RelayTokenTransformerBlock in the reference formulation (padded), fp32."""
    cat = torch.cat(rts)
    real = index >= 0
    x = cat[index.clamp(min=0)] * real.unsqueeze(-1)
    B, L, C = x.shape
    a = blk.rt_attention
    qkv = F.linear(blk.norm1(x), a.qkv.weight, a.qkv.bias)
    mask = (ids.unsqueeze(2) != ids.unsqueeze(1)).to(torch.int64)
    q, k, v = qkv.view(B, L, 3, H, C // H).permute(2, 0, 3, 1, 4)
    att = (q @ k.transpose(-1, -2)) * (C // H) ** -0.5 + mask.unsqueeze(1).float() * -1000.0
    x = x + F.linear((att.softmax(-1) @ v).transpose(1, 2).reshape(B, L, C), a.proj.weight, a.proj.bias)
    x = x + blk.mlp.fc2(F.gelu(blk.mlp.fc1(blk.norm2(x))))
    out = torch.empty_like(cat)
    out[index[real]] = x[real]
    return list(out.split([r.shape[0] for r in rts]))


def native_block(blk, rts, layout):
    x = layout.pack(rts)
    x = x + blk.rt_attention(blk.norm1(x), layout)
    x = x + blk.mlp.fc2(F.gelu(blk.mlp.fc1(blk.norm2(x))))
    return layout.unpack(x)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--iters', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--out', default=None, help='also write the JSON here')
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('rt_attn_train_bench needs a CUDA device')
    torch.cuda.set_device(0)
    torch.backends.cuda.matmul.allow_tf32 = False
    g = torch.Generator().manual_seed(7)
    oxford = build_batch([M.lidar_cloud(4096, g) for _ in range(128)], 9).finalize()
    cswild = build_batch([M.lidar_cloud(30000 if i % 2 == 0 else 60000, g, aerial=True) for i in range(128)],
                         7).finalize()
    shapes = {'oxford': (oxford, (6, 5, 4), 48), 'cswild': (cswild, (4, 3, 2), 64)}
    C, H = 256, 16
    L = N.lib()
    result = {'device': device_info(), 'iters': args.iters, 'warmup': args.warmup,
              'hbm_datasheet_gbps': HBM_GBPS, 'rows': []}
    for name, (o, depths, K) in shapes.items():
        layout = rt_layout([o.batch_nnum_nempty[d] for d in depths], K, 4, 'cuda')
        index, index_cat, ids = padded_plan(layout)
        lens = np.sum(layout.num_windows, axis=0).astype(np.int64)
        T, B, nmax = layout.total, len(lens), int(lens.max())
        sq = int((lens ** 2).sum())
        row = {'shape': name, 'T': T, 'B': B, 'Nmax': nmax, 'min_len': int(lens.min()), 'C': C, 'H': H,
               'flops_fwd': 4 * sq * C, 'flops_bwd': 10 * sq * C,
               'bytes_fwd': (T * 3 * C + T * C + T * H) * 4, 'bytes_bwd': (2 * T * 3 * C + 2 * T * C + T * H) * 4,
               'ws_mb': round(int(L.hfl_rt_attn_train_workspace_bytes(T, B, H)) / 2 ** 20, 2),
               'ref_mask_int64_mb': round(B * nmax * nmax * 8 / 2 ** 20, 1),
               'ref_probs_fp32_mb': round(B * H * nmax * nmax * 4 / 2 ** 20, 1)}
        torch.manual_seed(0)
        qkv = torch.randn(T, 3 * C, device='cuda', requires_grad=True)
        dout = torch.randn(T, C, device='cuda')
        for arm, fn in (('native', lambda: relay_token_attention(qkv, layout, H)),
                        ('torch_fp32', lambda: torch_core(qkv, index, ids, H))):
            out = fn()
            row[f'core_{arm}_fwd_ms'] = round(time_ms(lambda: fn().detach(), args.iters, args.warmup), 4)
            row[f'core_{arm}_bwd_ms'] = round(time_ms(
                lambda: torch.autograd.grad(out, [qkv], dout, retain_graph=True), args.iters, args.warmup), 4)
            row[f'core_{arm}_fwd+bwd_ms'] = round(time_ms(
                lambda: torch.autograd.grad(fn(), [qkv], dout), args.iters, args.warmup), 4)
            del out
            row[f'core_{arm}_peak_mb'] = peak_mb(lambda: torch.autograd.grad(fn(), [qkv], dout))
        for ph in ('fwd', 'bwd'):
            ms = row[f'core_native_{ph}_ms']
            row[f'core_native_{ph}_tflops'] = round(row[f'flops_{ph}'] / (ms * 1e-3) / 1e12, 2)
            row[f'core_native_{ph}_gbps'] = round(row[f'bytes_{ph}'] / (ms * 1e-3) / 1e9, 1)
        row['core_speedup_fwd+bwd_vs_torch'] = round(row['core_torch_fp32_fwd+bwd_ms'] /
                                                     row['core_native_fwd+bwd_ms'], 2)
        del qkv, dout

        blk = _RTSABlock(C)
        blk.rt_attention = RTAttention(C, H)
        blk = blk.cuda()
        rts = [torch.randn(n, C, device='cuda', requires_grad=True) for n in layout.windows]
        w = [torch.randn(n, C, device='cuda') for n in layout.windows]
        params = list(blk.parameters()) + rts
        for arm, fn in (('native', lambda: native_block(blk, rts, layout)),
                        ('torch_fp32', lambda: torch_block(blk, rts, index_cat, ids, H))):
            step = lambda: torch.autograd.grad(fn(), params, w)
            row[f'block_{arm}_fwd_ms'] = round(time_ms(lambda: [x.detach() for x in fn()], args.iters,
                                                       args.warmup), 4)
            row[f'block_{arm}_fwd+bwd_ms'] = round(time_ms(step, args.iters, args.warmup), 4)
            row[f'block_{arm}_peak_mb'] = peak_mb(step)
        row['block_speedup_fwd+bwd_vs_torch'] = round(row['block_torch_fp32_fwd+bwd_ms'] /
                                                      row['block_native_fwd+bwd_ms'], 2)
        result['rows'].append(row)
        print(json.dumps(row), file=sys.stderr)
        del blk, rts, w, params
        torch.cuda.empty_cache()
    line = json.dumps(result)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            f.write(line + '\n')


if __name__ == '__main__':
    main()
