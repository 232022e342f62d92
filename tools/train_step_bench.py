"""Training step of the whole model through the differentiable forward (hotformerloc_b200/models/differentiable.py):
forward + backward per minibatch, timed with CUDA events after warm-up, with gradient checkpointing on and off,
next to the bf16 inference forward of the same batch.

Workloads (128-submap training minibatches, the presets' batch_split_size, shipped block counts):
  oxford  : the Oxford preset, 128 x 4096-point submaps, depth-9 octree
  cswild  : the CS-Wild-Places preset, 128 synthetic submaps alternating ground (30 k points) and aerial (60 k),
            depth-7 octree (datasets/synthetic.py)
The loss is a fixed linear functional of the descriptors, sum(descriptor * R) for a seeded R: losses and the
trainer are not measured.  Weights are the model's own seeded initialisation; the model is in eval mode
(OctreeDropPath is not implemented, so drop_path has no effect on what is timed).

Per workload and checkpointing setting: mean and min step time over the repetitions, submaps/s from the mean,
and torch.cuda.max_memory_allocated over the timed steps; an out-of-memory is reported as such.  The GPU name
and power limit are read in the same run (nvidia-smi query only).

    python tools/train_step_bench.py [--reps 5] [--warmup 2] [--out FILE]
    python tools/train_step_bench.py --profile DIR      # torch.profiler CUDA time by op family, one step each
"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from hotformerloc_b200.config.presets import write_configs
from hotformerloc_b200.datasets.synthetic import lidar_cloud
from hotformerloc_b200.misc.utils import ModelParams
from hotformerloc_b200.models.model_factory import model_factory
from hotformerloc_b200.octree import build_batch


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


def workloads(B):
    g = torch.Generator().manual_seed(7)
    yield 'oxford', 'oxford', lambda: build_batch([lidar_cloud(4096, g) for _ in range(B)], 9).finalize()
    yield 'cswild', 'cs-wild-places', lambda: build_batch(
        [lidar_cloud(30000 if i % 2 == 0 else 60000, g, aerial=i % 2 == 1) for i in range(B)], 7).finalize()


def make_model(preset, tmp):
    torch.manual_seed(0)
    paths = write_configs(tmp, preset)
    return model_factory(ModelParams(paths['model_config'])).cuda().eval()


def step(model, o, R):
    model.zero_grad(set_to_none=True)
    y = model({'octree': o})['global']
    (y * R).sum().backward()


def time_steps(fn, reps, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    ts = []
    for _ in range(reps):
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        fn()
        e.record()
        e.synchronize()
        ts.append(s.elapsed_time(e))
    return ts, torch.cuda.max_memory_allocated()


def family(name: str) -> str:
    n = name.lower()
    if n.startswith('void hfl::') or 'hfl::' in n or n.startswith('k_'):
        return 'project kernels (octree conv, dwconv, attention, RT init, pooling)'
    if 'gemm' in n or 'cutlass' in n or 'cublas' in n or 'nvjet' in n:
        return 'GEMM (torch Linear, fp32)'
    if 'layer_norm' in n or 'layernorm' in n:
        return 'LayerNorm'
    if 'memcpy' in n or 'memset' in n:
        return 'copies / memsets'
    if 'index' in n or 'gather' in n or 'scatter' in n or 'cat' in n:
        return 'gathers / cat / index'
    if 'reduce' in n:
        return 'reductions (bias grads)'
    return 'elementwise and other'


def profile(model, o, R, out_dir, name):
    from torch.profiler import ProfilerActivity, profile as prof
    step(model, o, R)
    torch.cuda.synchronize()
    with prof(activities=[ProfilerActivity.CUDA]) as p:
        step(model, o, R)
        torch.cuda.synchronize()
    fam = {}
    for ev in p.key_averages():
        t = getattr(ev, 'device_time_total', None)
        if t is None:
            t = ev.cuda_time_total
        if t <= 0:
            continue
        f = family(ev.key)
        fam[f] = fam.get(f, 0.0) + t / 1e3
    table = p.key_averages().table(sort_by='device_time_total', row_limit=40)
    with open(os.path.join(out_dir, f'train_step_profile_{name}.txt'), 'w') as f:
        f.write(table)
    return {k: round(v, 2) for k, v in sorted(fam.items(), key=lambda kv: -kv[1])}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--reps', type=int, default=5)
    ap.add_argument('--warmup', type=int, default=2)
    ap.add_argument('--batch', type=int, default=128)
    ap.add_argument('--out', default=None, help='also write the JSON here')
    ap.add_argument('--profile', default=None, metavar='DIR', help='profile one step per workload instead')
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('train_step_bench needs a CUDA device')
    torch.cuda.set_device(0)
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    import tempfile
    tmp = tempfile.mkdtemp(prefix='hfl_train_bench_')
    result = {'device': device_info(), 'batch': args.batch, 'reps': args.reps, 'warmup': args.warmup,
              'loss': 'sum(descriptor * R), R seeded', 'rows': []}
    for name, preset, build in workloads(args.batch):
        o = build()
        model = make_model(preset, tmp)
        R = torch.randn(o.batch_size, model.pooling.output_dim, generator=torch.Generator().manual_seed(1)).cuda()
        if args.profile:
            os.makedirs(args.profile, exist_ok=True)
            model.differentiable = True
            result['rows'].append({'workload': name, 'grad_checkpoint': True,
                                   'cuda_ms_by_family': profile(model, o, R, args.profile, name)})
            continue
        model.differentiable = False

        def infer():
            with torch.no_grad():
                model({'octree': o})
        ts, mem = time_steps(infer, args.reps, args.warmup)
        result['rows'].append({'workload': name, 'path': 'bf16 inference forward', 'mean_ms': sum(ts) / len(ts),
                               'min_ms': min(ts), 'submaps_per_s': o.batch_size * 1e3 * len(ts) / sum(ts),
                               'max_memory_allocated_mib': round(mem / 2 ** 20, 1)})
        model.differentiable = True
        for ckpt in (True, False):
            model.backbone.grad_checkpoint = ckpt
            row = {'workload': name, 'path': 'fp32 differentiable forward + backward', 'grad_checkpoint': ckpt}
            try:
                ts, mem = time_steps(lambda: step(model, o, R), args.reps, args.warmup)
                row.update(mean_ms=sum(ts) / len(ts), min_ms=min(ts), times_ms=ts,
                           submaps_per_s=o.batch_size * 1e3 * len(ts) / sum(ts),
                           max_memory_allocated_mib=round(mem / 2 ** 20, 1))
            except torch.OutOfMemoryError as e:
                row.update(out_of_memory=True, error=str(e).splitlines()[0])
            model.zero_grad(set_to_none=True)
            torch.cuda.empty_cache()
            result['rows'].append(row)
            print(json.dumps(row), flush=True)
        del model, o
        torch.cuda.empty_cache()
    line = json.dumps(result)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            f.write(line + '\n')


if __name__ == '__main__':
    main()
