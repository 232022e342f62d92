"""Training octree convolution (hotformerloc_b200.octree_conv) against the torch stand-in statement
(gather into (n, K, Cin), then matmul; oracle.ocnn_standin.OctreeConv) on every OctreeConv layer of the
model at the training minibatch (batch_split_size = 128): Oxford 128 x 4096 points (depth 9) and
CS-Wild-Places 128 x 30 k points (depth 7), synthetic lidar_cloud submaps.

Per layer: forward, backward and forward + backward times (CUDA events, after warm-up), peak memory, the
occupied (row, tap) pairs and algorithmic FLOPs read from the tables, the executed FLOPs of each kernel
from its compaction rule (csrc/octree_conv_train.cu) on the same tables, achieved algorithmic TFLOP/s, and
the card's name and power limit read in the same run.  Writes one JSON file (--out)."""
import argparse
import json
import math
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from oracle import model_ref as M  # noqa: E402

PRESETS = {'oxford': (4096, 9), 'cs-wild-places': (30000, 7)}
LAYERS = [('convs.0', 0, 1, 3, 32), ('downsamples.0', 0, 2, 32, 64), ('convs.1', 1, 1, 64, 64),
          ('downsamples.1', 1, 2, 64, 128), ('proj', 2, 1, 128, 128), ('downsample.0', 2, 2, 128, 256),
          ('hotf_stage.downsamples.0', 3, 2, 256, 256), ('hotf_stage.downsamples.1', 4, 2, 256, 256)]


def card():
    r = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'],
                       capture_output=True, text=True)
    name, power = (r.stdout.strip().splitlines() or ['?, ?'])[torch.cuda.current_device()].split(', ')
    return {'name': name, 'power_limit': power}


def fwd_executed_fmas(neigh, n_in, cin, cout):
    """k_oconv_fwd's rule: per 128-row tile and tap, ceil(m / LR) LR rows x Cin x the padded columns."""
    lc = 2 if cout <= 32 else 4 if cout <= 64 else 8
    lr, tn = 32 // lc, 16 * lc
    occ = ((neigh >= 0) & (neigh < n_in)).to(torch.int64)
    n, K = occ.shape
    pad = -n % 128
    occ = torch.cat([occ, occ.new_zeros(pad, K)]).view(-1, 128, K).sum(1)
    rows = ((occ + lr - 1) // lr * lr).sum().item()
    return rows * cin * math.ceil(cout / tn) * tn


def wgrad_executed_fmas(pairs, cin, cout):
    ti = 4 if cin <= 4 else 32 if cin <= 32 else 64
    to = 32 if cout <= 32 else 64
    return pairs * math.ceil(cin / ti) * ti * math.ceil(cout / to) * to


def timed(fn, warmup, reps):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / reps, torch.cuda.max_memory_allocated() - base


def standin(data, w, neigh):
    buf = data.new_zeros(neigh.shape[0], neigh.shape[1], data.shape[1])
    valid = neigh >= 0
    buf[valid] = data[neigh[valid]]
    return buf.flatten(1) @ w.flatten(0, 1)


def bench_layer(o, depth, stride, cin, cout, warmup, reps):
    from hotformerloc_b200.dwconv import _inverse
    from hotformerloc_b200.octree_conv import octree_conv
    neigh = o.ne_table(depth) if stride == 1 else o.child_table(depth)
    n_out, K = neigh.shape
    n_in = o.n(depth)
    g = torch.Generator(device='cuda').manual_seed(0)
    data = torch.randn(n_in, cin, device='cuda', generator=g, requires_grad=True)
    w = (torch.randn(K, cin, cout, device='cuda', generator=g) / math.sqrt(cin)).requires_grad_()
    dout = torch.randn(n_out, cout, device='cuda', generator=g)
    pairs = int(((neigh >= 0) & (neigh < n_in)).sum())
    inv = _inverse(neigh, n_in, 0)
    alg = 2 * pairs * cin * cout
    ex = {'forward': 2 * fwd_executed_fmas(neigh, n_in, cin, cout),
          'input_grad': 2 * fwd_executed_fmas(inv, n_out, cout, cin),
          'weight_grad': 2 * wgrad_executed_fmas(pairs, cin, cout)}
    rec = {'n_out': n_out, 'n_in': n_in, 'K': K, 'Cin': cin, 'Cout': cout, 'pairs': pairs,
           'pairs_per_row': pairs / max(n_out, 1), 'algorithmic_flop_per_kernel': alg,
           'executed_flop': ex, 'executed_over_algorithmic': {k: v / max(alg, 1) for k, v in ex.items()}}
    neigh64 = neigh.long()
    for impl, f in (('native', lambda x, ww: octree_conv(x, ww, neigh)),
                    ('torch_standin', lambda x, ww: standin(x, ww, neigh64))):
        def fwd():
            with torch.no_grad():
                f(data, w)

        def both():
            data.grad = w.grad = None
            f(data, w).backward(dout)
        t_f, m_f = timed(fwd, warmup, reps)
        t_fb, m_fb = timed(both, warmup, reps)
        r = {'fwd_ms': t_f, 'fwd_bwd_ms': t_fb, 'bwd_ms': t_fb - t_f, 'peak_fwd_MiB': m_f / 2 ** 20,
             'peak_fwd_bwd_MiB': m_fb / 2 ** 20}
        r['alg_TFLOPs_fwd_bwd'] = 3 * alg / (t_fb * 1e-3) / 1e12
        rec[impl] = r
        torch.cuda.empty_cache()
    return rec


def main():
    ap = argparse.ArgumentParser(description=__doc__.split('\n')[0])
    ap.add_argument('--out', default='profiles/r06_octree_conv_train_bench.json')
    ap.add_argument('--batch', type=int, default=128)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--reps', type=int, default=10)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('this benchmark needs a CUDA device')
    from hotformerloc_b200.octree import build_batch
    res = {'card': card(), 'batch': args.batch, 'layers': {}}
    for preset, (pts, depth) in PRESETS.items():
        g = torch.Generator().manual_seed(7)
        o = build_batch([M.lidar_cloud(pts, g) for _ in range(args.batch)], depth).finalize()
        for name, dd, stride, cin, cout in LAYERS:
            rec = bench_layer(o, depth - dd, stride, cin, cout, args.warmup, args.reps)
            rec['input_depth'] = depth - dd
            res['layers'][f'{preset}/{name}'] = rec
            nv, st = rec['native'], rec['torch_standin']
            print(f"{preset:15s} {name:26s} n {rec['n_out']:8d} pairs/row {rec['pairs_per_row']:5.2f} "
                  f"exec/alg fwd {rec['executed_over_algorithmic']['forward']:.2f} "
                  f"dgrad {rec['executed_over_algorithmic']['input_grad']:.2f} "
                  f"wgrad {rec['executed_over_algorithmic']['weight_grad']:.2f} | "
                  f"fwd+bwd {nv['fwd_bwd_ms']:.3f} ms ({nv['alg_TFLOPs_fwd_bwd']:.1f} TFLOP/s, "
                  f"{nv['peak_fwd_bwd_MiB']:.0f} MiB) vs stand-in {st['fwd_bwd_ms']:.3f} ms "
                  f"({st['peak_fwd_bwd_MiB']:.0f} MiB)", flush=True)
        del o
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, 'w') as f:
        json.dump(res, f)
    print(f"card {res['card']}; wrote {args.out}")


if __name__ == '__main__':
    main()
