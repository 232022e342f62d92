"""Timing of the dwconv drop-in (csrc/dwconv.cu) at training sizes, against the pure-torch
formulation of ocnn.nn.OctreeDWConv (gather into an (n, K, C) buffer + einsum, oracle.ocnn_standin)
on the same GPU.

Tables: the 27-neighbour non-empty tables of a batch of `--clouds` lidar-ish submaps (4096 points,
Oxford cfg depth 9; the training cfg's batch_split_size is 128 submaps per forward): depth 7 at
C = 128 (~4029 rows per submap) and depth 6 at C = 256, each as int64 (the reference layout) and
int32.  Data and output gradient (>= 240 MB each at these sizes) exceed the 126 MB L2.

Algorithmic bytes (each unique operand once): forward / input gradient and weight gradient
2 n C 4 + n K idx_bytes, inverse n K idx_bytes read + n K idx_bytes written; "fwd+bwd" is the sum
of forward, inverse, input gradient and weight gradient.  Achieved GB/s = bytes / time, and its
fraction of the data-sheet 7.7 TB/s HBM3e bandwidth.

    python tools/dwconv_bench.py [--iters 20] [--warmup 3] [--clouds 128] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from hotformerloc_b200 import dwconv as D
from hotformerloc_b200.octree import build_batch
from oracle import model_ref as M
from oracle import ocnn_standin as S

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


def standin_fwd_bwd(data, w, t, grad):
    d = data.detach().requires_grad_()
    ww = w.detach().requires_grad_()
    y = torch.einsum('ikc,kc->ic', S._gather(d, t), ww[:, 0, :])
    y.backward(grad)


def native_fwd_bwd(data, w, t, grad):
    d = data.detach().requires_grad_()
    ww = w.detach().requires_grad_()
    D.octree_dwconv(d, ww, t).backward(grad)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--iters', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--clouds', type=int, default=128)
    ap.add_argument('--out', default=None, help='also write the JSON here')
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('dwconv_bench needs a CUDA device')
    torch.cuda.set_device(0)
    g = torch.Generator().manual_seed(7)
    octree = build_batch([M.lidar_cloud(4096, g) for _ in range(args.clouds)], 9).finalize()
    result = {'device': device_info(), 'clouds': args.clouds, 'iters': args.iters, 'warmup': args.warmup,
              'hbm_datasheet_gbps': HBM_GBPS, 'rows': []}
    for depth, C in ((7, 128), (6, 256)):
        t32 = octree.ne_table(depth).contiguous()
        n, K = t32.shape
        torch.manual_seed(0)
        data = torch.randn(n, C, device='cuda')
        grad = torch.randn(n, C, device='cuda')
        w = torch.randn(K, 1, C, device='cuda')
        for t in (t32.long(), t32):
            ib = t.element_size()
            b_conv = 2 * n * C * 4 + n * K * ib
            b_inv = 2 * n * K * ib
            ops = {
                'forward': (lambda: D.dwconv_forward_backward(data, w, t), b_conv),
                'inverse': (lambda: D.inverse_neigh(t), b_inv),
                'inverse+input_grad': (lambda: D.dwconv_forward_backward(grad, w, D.inverse_neigh(t)),
                                       b_inv + b_conv),
                'weight_grad': (lambda: D.dwconv_weight_backward(grad, data, t), b_conv),
                'autograd_fwd+bwd': (lambda: native_fwd_bwd(data, w, t, grad), 3 * b_conv + b_inv),
                'standin_fwd+bwd': (lambda: standin_fwd_bwd(data, w, t, grad), 3 * b_conv + b_inv),
            }
            for name, (fn, nbytes) in ops.items():
                ms = time_ms(fn, args.iters, args.warmup)
                gbps = nbytes / (ms * 1e-3) / 1e9
                row = {'depth': depth, 'n': n, 'C': C, 'K': K, 'idx': str(t.dtype).replace('torch.', ''),
                       'op': name, 'ms': round(ms, 4), 'alg_bytes': nbytes, 'gbps': round(gbps, 1),
                       'hbm_fraction': round(gbps / HBM_GBPS, 4)}
                result['rows'].append(row)
                print(json.dumps(row), file=sys.stderr)
            torch.cuda.empty_cache()
    for depth, C in ((7, 128), (6, 256)):
        for idx in ('int64', 'int32'):
            sel = {r['op']: r['ms'] for r in result['rows'] if (r['depth'], r['C'], r['idx']) == (depth, C, idx)}
            result.setdefault('speedup_fwd+bwd_vs_standin', {})[f'd{depth}_C{C}_{idx}'] = \
                round(sel['standin_fwd+bwd'] / sel['autograd_fwd+bwd'], 2)
    line = json.dumps(result)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            f.write(line + '\n')


if __name__ == '__main__':
    main()
