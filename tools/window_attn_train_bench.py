"""Timing and peak memory of the window attention core (csrc/window_attn_train.cu, through
hotformerloc_b200.window_attention) at training sizes, against the fp32 torch statement of the
reference formulation on the same GPU: int64 rel_pos (N_win, K, K, 3), one table gather per axis,
a dense (N_win, 1, L, L) mask and autograd over softmax (oracle.model_ref._rpe_bias + the core of
_attention).

Shapes (windows cut from real batches as oracle.model_ref.make_level / window_rows do):
  oxford_l7_dil1 / _dil4 : 128 x 4096-point submaps (batch_split_size), depth 7 of a depth-9 octree,
                           K = 48, H = 8, dilation 1 and 4 (padding to a multiple of K dil)
  oxford_l6_hosa         : same batch, depth 6, K = 48 + relay token, H = 16 (padding to 4 K)
  cswild_l4_hosa         : 64 x 30 k-point aerial submaps, depth 4 of a depth-7 octree, K = 64 + relay, H = 16
Inputs are > 126 MB (the L2) for the Oxford shapes; the CS-Wild-Places level is small and L2-resident.

Algorithmic work per (window, head, query, key): forward 64 FLOPs (q.k and p v, 16 FMAs each),
backward 160 (q.k recomputed, dO.v, dq, dk, dv).  Bytes (each operand once): forward reads qkv, ids,
xyz and writes o and lse; backward reads qkv, ids, xyz, o, lse, dO and writes dqkv.

    python tools/window_attn_train_bench.py [--iters 20] [--warmup 3] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import torch.nn.functional as F

from hotformerloc_b200.octree import build_batch
from hotformerloc_b200.window_attention import window_attention
from oracle import model_ref as M

HBM_GBPS = 7700.0
HD = 16


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


def windows(o, d, K, dil, pad_dil, hat):
    n = o.n(d)
    n_pad = -(-n // (K * pad_dil)) * (K * pad_dil)
    tok = o.tokens(d, n_pad).long()
    rows = M.window_rows(n_pad, K, dil).cuda()
    xyz, ids = tok[rows, :3].contiguous(), tok[rows, 3].contiguous()
    if hat:
        ids = torch.cat([ids[:, :1], ids], 1).contiguous()
    return xyz, ids


def torch_statement(qkv, xyz, ids, table, K, dil, hat, H):
    """fp32 reference formulation: rel_pos, per-axis table gathers, dense mask, softmax."""
    N, L, C3 = qkv.shape
    C = C3 // 3
    q, k, v = qkv.view(N, L, 3, H, C // H).permute(2, 0, 3, 1, 4)
    bias = torch.zeros(N, 1, L, L, dtype=qkv.dtype, device=qkv.device)
    bias = bias.masked_fill((ids.unsqueeze(2) != ids.unsqueeze(1)).unsqueeze(1), -1000.0)
    rpe = M._rpe_bias({'t.rpe_table': table}, 't', xyz, K, dil)
    if hat:
        rpe = F.pad(rpe, (1, 0, 1, 0))
    att = (q @ k.transpose(-1, -2)) * ((C // H) ** -0.5) + (bias + rpe)
    return (att.softmax(-1) @ v).transpose(1, 2).reshape(N, L, C)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--iters', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--out', default=None, help='also write the JSON here')
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('window_attn_train_bench needs a CUDA device')
    torch.cuda.set_device(0)
    torch.backends.cuda.matmul.allow_tf32 = False
    g = torch.Generator().manual_seed(7)
    oxford = build_batch([M.lidar_cloud(4096, g) for _ in range(128)], 9).finalize()
    cswild = build_batch([M.lidar_cloud(30000, g, aerial=True) for _ in range(64)], 7).finalize()
    shapes = {  # name: octree, depth, K, H, dil, padding multiple of K, hat
        'oxford_l7_dil1': (oxford, 7, 48, 8, 1, 1, False),
        'oxford_l7_dil4': (oxford, 7, 48, 8, 4, 4, False),
        'oxford_l6_hosa': (oxford, 6, 48, 16, 1, 4, True),
        'cswild_l4_hosa': (cswild, 4, 64, 16, 1, 4, True),
    }
    result = {'device': device_info(), 'iters': args.iters, 'warmup': args.warmup,
              'hbm_datasheet_gbps': HBM_GBPS, 'rows': []}
    for name, (o, d, K, H, dil, pad_dil, hat) in shapes.items():
        xyz, ids = windows(o, d, K, dil, pad_dil, hat)
        n_win, L, C = ids.shape[0], K + int(hat), HD * H
        bnd = int(0.8 * K * dil ** 0.5)
        torch.manual_seed(0)
        qkv = torch.randn(n_win, L, 3 * C, device='cuda', requires_grad=True)
        table = (torch.randn(3 * (2 * bnd + 1), H, device='cuda') * 0.5).requires_grad_()
        dout = torch.randn(n_win, L, C, device='cuda')
        pairs = n_win * H * L * L
        idx_b = xyz.numel() * 8 + ids.numel() * 8
        b_fwd = qkv.numel() * 4 + idx_b + dout.numel() * 4 + n_win * H * L * 4
        b_bwd = 2 * qkv.numel() * 4 + idx_b + 2 * dout.numel() * 4 + n_win * H * L * 4
        row = {'shape': name, 'depth': d, 'n_win': n_win, 'K': K, 'hat': int(hat), 'L': L, 'H': H, 'dil': dil,
               'bnd': bnd, 'flops_fwd': 64 * pairs, 'flops_bwd': 160 * pairs, 'bytes_fwd': b_fwd,
               'bytes_bwd': b_bwd, 'dense_nhll_fp32_mb': round(pairs * 4 / 2 ** 20, 1)}
        for arm, fn in (('native', lambda: window_attention(qkv, xyz, ids, table, bnd, hat, H)),
                        ('torch_fp32', lambda: torch_statement(qkv, xyz, ids, table, K, dil, hat, H))):
            out = fn()
            row[f'{arm}_fwd_ms'] = round(time_ms(lambda: fn().detach(), args.iters, args.warmup), 4)
            row[f'{arm}_bwd_ms'] = round(time_ms(
                lambda: torch.autograd.grad(out, [qkv, table], dout, retain_graph=True), args.iters, args.warmup), 4)
            row[f'{arm}_fwd+bwd_ms'] = round(time_ms(
                lambda: torch.autograd.grad(fn(), [qkv, table], dout), args.iters, args.warmup), 4)
            del out
            row[f'{arm}_peak_mb'] = peak_mb(lambda: torch.autograd.grad(fn(), [qkv, table], dout))
        for ph, fl, by in (('fwd', row['flops_fwd'], b_fwd), ('bwd', row['flops_bwd'], b_bwd)):
            ms = row[f'native_{ph}_ms']
            row[f'native_{ph}_tflops'] = round(fl / (ms * 1e-3) / 1e12, 2)
            row[f'native_{ph}_gbps'] = round(by / (ms * 1e-3) / 1e9, 1)
            row[f'native_{ph}_hbm_fraction'] = round(by / (ms * 1e-3) / 1e9 / HBM_GBPS, 4)
        row['speedup_fwd+bwd_vs_torch'] = round(row['torch_fp32_fwd+bwd_ms'] / row['native_fwd+bwd_ms'], 2)
        result['rows'].append(row)
        print(json.dumps(row), file=sys.stderr)
        del qkv, table, dout
        torch.cuda.empty_cache()
    line = json.dumps(result)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            f.write(line + '\n')


if __name__ == '__main__':
    main()
