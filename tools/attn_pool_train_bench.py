"""Timing and peak memory of the attention-pooling head's pooling op (csrc/attn_pool_train.cu, through
hotformerloc_b200.attention_pool.attention_pool) at training sizes, against the fp32 torch statement of the
reference formulation on the same GPU (pooling.py:209-232, salsa.py:25-55): the level's tokens split and padded
to (B, Nmax, C), a (B, Nmax, Nmax) int64 mask of which row 0 is kept, and single-head
F.scaled_dot_product_attention of the learned queries, under autograd.

Shapes (128-submap training minibatches, batch_split_size; counts = batch_nnum_nempty of the pyramid levels):
  oxford : 128 x 4096-point submaps, depth-9 octree, levels at depths 6 / 5 / 4, C = 256, with the k set
           74 / 36 / 18 (Oxford and CS-Wild-Places cfgs) and 148 / 72 / 36 (Wild-Places and CS-Campus3D cfgs)
  cswild : 128 x 30 k-point aerial submaps, depth-7 octree, levels at depths 4 / 3 / 2, k = 74 / 36 / 18
Level 0 of the Oxford minibatch (x about 200 MB) is larger than the 126 MB L2; the deeper levels are L2-resident.

Algorithmic work per token: forward 4 k C FLOPs (scores and P.x), backward 10 k C (scores, dO.x, dx and dQ;
the kernels recompute the scores and dO.x once more for dQ: 14 k C executed).  Bytes (each operand once):
forward reads x and Q and writes out and lse; backward reads x, Q, out, lse and dout and writes dx and dQ.

    python tools/attn_pool_train_bench.py [--iters 20] [--warmup 3] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import torch.nn.functional as F

from hotformerloc_b200 import native as N
from hotformerloc_b200.attention_pool import attention_pool
from hotformerloc_b200.octree import build_batch
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


def torch_statement(x, counts, query):
    """fp32 reference formulation: pad to (B, Nmax, C), (B, Nmax, Nmax) int64 mask, row 0, SDPA."""
    B, nmax, k = len(counts), max(counts), query.shape[0]
    xp = torch.nn.utils.rnn.pad_sequence(list(x.split(counts)), batch_first=True)          # (B, Nmax, C)
    lens = torch.tensor(counts, device=x.device)
    valid = torch.arange(nmax, device=x.device)[None] < lens[:, None]
    mask = (valid[:, :, None] & valid[:, None, :]).to(torch.int64)                         # (B, Nmax, Nmax)
    keep = mask[:, 0].bool()[:, None, :]                                                  # (B, 1, Nmax)
    q = query.unsqueeze(0).expand(B, k, query.shape[1])
    return F.scaled_dot_product_attention(q, xp, xp, attn_mask=keep)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--iters', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--out', default=None, help='also write the JSON here')
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('attn_pool_train_bench needs a CUDA device')
    torch.cuda.set_device(0)
    torch.backends.cuda.matmul.allow_tf32 = False
    g = torch.Generator().manual_seed(7)
    oxford = build_batch([M.lidar_cloud(4096, g) for _ in range(128)], 9).finalize()
    cswild = build_batch([M.lidar_cloud(30000, g, aerial=True) for _ in range(128)], 7).finalize()
    shapes = {  # name: octree, level depths, k per level
        'oxford_k74': (oxford, (6, 5, 4), (74, 36, 18)),
        'oxford_k148': (oxford, (6, 5, 4), (148, 72, 36)),
        'cswild_k74': (cswild, (4, 3, 2), (74, 36, 18)),
    }
    C = 256
    L = N.lib()
    result = {'device': device_info(), 'iters': args.iters, 'warmup': args.warmup,
              'hbm_datasheet_gbps': HBM_GBPS, 'rows': []}
    for name, (o, depths, ks) in shapes.items():
        for j, (d, k) in enumerate(zip(depths, ks)):
            counts = [int(c) for c in o.batch_nnum_nempty[d]]
            n, B, nmax = sum(counts), len(counts), max(counts)
            torch.manual_seed(0)
            x = torch.randn(n, C, device='cuda', requires_grad=True)
            query = torch.randn(k, C, device='cuda', requires_grad=True)
            dout = torch.randn(B, k, C, device='cuda')
            b_fwd = (n * C + k * C + B * k * C + B * k) * 4
            b_bwd = (2 * n * C + 2 * k * C + 2 * B * k * C + B * k) * 4
            row = {'shape': name, 'level': j, 'depth': d, 'n': n, 'B': B, 'Nmax': nmax, 'k': k, 'C': C,
                   'flops_fwd': 4 * k * C * n, 'flops_bwd': 10 * k * C * n, 'bytes_fwd': b_fwd, 'bytes_bwd': b_bwd,
                   'ws_fwd_mb': round(int(L.hfl_attn_pool_train_fwd_workspace_bytes(n, B, k, C)) / 2 ** 20, 1),
                   'ws_bwd_mb': round(int(L.hfl_attn_pool_train_bwd_workspace_bytes(n, B, k, C)) / 2 ** 20, 1),
                   'ref_mask_int64_mb': round(B * nmax * nmax * 8 / 2 ** 20, 1),
                   'ref_padded_fp32_mb': round(B * nmax * C * 4 / 2 ** 20, 1)}
            for arm, fn in (('native', lambda: attention_pool(x, counts, query)),
                            ('torch_fp32', lambda: torch_statement(x, counts, query))):
                out = fn()
                row[f'{arm}_fwd_ms'] = round(time_ms(lambda: fn().detach(), args.iters, args.warmup), 4)
                row[f'{arm}_bwd_ms'] = round(time_ms(
                    lambda: torch.autograd.grad(out, [x, query], dout, retain_graph=True), args.iters,
                    args.warmup), 4)
                row[f'{arm}_fwd+bwd_ms'] = round(time_ms(
                    lambda: torch.autograd.grad(fn(), [x, query], dout), args.iters, args.warmup), 4)
                del out
                row[f'{arm}_peak_mb'] = peak_mb(lambda: torch.autograd.grad(fn(), [x, query], dout))
            for ph in ('fwd', 'bwd'):
                ms = row[f'native_{ph}_ms']
                row[f'native_{ph}_tflops'] = round(row[f'flops_{ph}'] / (ms * 1e-3) / 1e12, 2)
                row[f'native_{ph}_gbps'] = round(row[f'bytes_{ph}'] / (ms * 1e-3) / 1e9, 1)
            row['speedup_fwd+bwd_vs_torch'] = round(row['torch_fp32_fwd+bwd_ms'] / row['native_fwd+bwd_ms'], 2)
            result['rows'].append(row)
            print(json.dumps(row), file=sys.stderr)
            del x, query, dout
            torch.cuda.empty_cache()
    line = json.dumps(result)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            f.write(line + '\n')


if __name__ == '__main__':
    main()
