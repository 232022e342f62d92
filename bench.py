#!/usr/bin/env python
"""bench.py -- headline benchmark of the HOTFormerLoc embedding hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl native|reference] [--dump-outputs DIR]

One "step" = one pass of the hot path over one batch of synthetic submaps:
raw points -> batched octree build -> hierarchical octree transformer -> (B,256)
descriptors.  Default workload = BASELINE.json configs[1]: Oxford cfg, 256
synthetic 4096-point submaps, bf16 tensor-core compute with fp32 accumulation,
random-init weights.  Prints ONE JSON line (see the driver contract).

  value        submaps/s with the packed points already resident in HBM
  e2e          same metric through the reference-facing API with HOST buffers
               (pinned H2D of the points inside the timed region, D2H of descriptors)
  roofline     dominant kernel family (time share measured live with CUDA events)
  cpu_baseline the oracle (CPU port of the reference path) on a bounded sample

--dump-outputs DIR writes the descriptors of the last timed step of each path as DIR/global.npy
(resident path; all ranks' rows when sharded) and DIR/e2e_global.npy (end-to-end path, rank 0's host copy),
float32.  The inputs and weights are seeded, so two builds run with the same arguments can be compared
output for output.

Multi-GPU (torchrun, one rank per GPU): evaluation batches are sharded across
ranks (batch t -> rank t mod W, SURVEY.md section 8e), no data-path collective
except the descriptor all-gather; weak scaling; time = max over ranks.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np
import torch

METRIC = 'submaps_per_sec_octree_build_plus_embed'
UNIT = 'submaps/s'


def synthetic_batches(n_batches, B, P, seed0=1000):
    from hotformerloc_b200.datasets.synthetic import lidar_cloud
    out = []
    for i in range(n_batches):
        g = torch.Generator().manual_seed(seed0 + i)
        out.append([lidar_cloud(P, g) for _ in range(B)])
    return out


def make_model(cfg_name, device):
    from hotformerloc_b200.config.presets import write_configs, TRAIN_PRESETS
    from hotformerloc_b200.misc.utils import ModelParams
    from hotformerloc_b200.models.model_factory import model_factory
    d = tempfile.mkdtemp(prefix='hfl_cfg_')
    paths = write_configs(d, cfg_name, dataset_folder=d)
    torch.manual_seed(0)
    model = model_factory(ModelParams(paths['model_config']))
    return model.to(device).eval(), paths, TRAIN_PRESETS[cfg_name]['octree_depth']


class ClockSampler(threading.Thread):
    """Samples SM clock / throttle reasons during the timed region (NVML)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.stop_flag = index, [], set(), False
        self.max_mhz = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {nv.nvmlClocksThrottleReasonHwSlowdown: 'hw_slowdown',
                 nv.nvmlClocksThrottleReasonHwThermalSlowdown: 'hw_thermal_slowdown',
                 nv.nvmlClocksThrottleReasonSwThermalSlowdown: 'sw_thermal_slowdown',
                 nv.nvmlClocksThrottleReasonSwPowerCap: 'sw_power_cap'}
        while not self.stop_flag:
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.05)

    def summary(self):
        return {'sm_mhz': float(np.median(self.samples)) if self.samples else None,
                'sm_max_mhz': self.max_mhz, 'reasons': sorted(self.reasons)}


def kernel_profile(model, octree_fn):
    """Per kernel-family device time + algorithmic work for one step, using CUDA
    events on the launching stream (an instrumented extra step, not the timed one)."""
    from hotformerloc_b200 import ops, octree as oct_mod
    rec = []

    def wrap(name, fn, work):
        def inner(*a, **k):
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            r = fn(*a, **k)
            e.record()
            rec.append((name, s, e, work(*a, **k)))
            return r
        return inner

    # Algorithmic work per launch (DESIGN.md section 5): flops of the dense math and the bytes
    # that MUST cross HBM once (unique inputs + outputs; gathers that re-read rows count once).
    def gemm_work(A, W, **k):
        M = k.get('M') or (k['idx'].shape[0] if k.get('idx') is not None else A.shape[0])
        N, Kt = W.shape
        out_b = sum(N * b for key, b in (('out_v_f32', 4), ('out_v_bf16', 2), ('out_y_f32', 4), ('out_y_bf16', 2))
                    if k.get(key) is not None)
        rows_in = min(A.shape[0], M * k.get('KD', 1))
        byte = rows_in * A.shape[1] * 2 + M * out_b + (M * N * 4 if k.get('res') is not None else 0) + N * Kt * 2
        if k.get('idx') is not None:
            byte += k['idx'].numel() * 4
        return {'flop': 2.0 * M * N * Kt, 'byte': float(byte)}

    def attn_work(qkv, out, xyzb, rpe, n_win, H, C, K, dil, hat, bnd, scale):
        L = K + (1 if hat else 0)
        rows = n_win * L
        return {'flop': 4.0 * n_win * L * L * C, 'byte': float(rows * (3 * C * 2 + C * 2) + n_win * K * 16)}

    def cpe_work(x, xb, ne, w, g, b, g1, b1, y1, cpe_out, n, rows, C, K):
        return {'flop': 0.0, 'byte': float(rows * C * (4 + 4 + 2) + n * (27 * 4 + 2 * C))}

    saved = {}
    def mlp_work(A, W1, b1, W2, b2, **k):
        M = k.get('M') or A.shape[0]
        C = A.shape[1]
        return {'flop': 4.0 * M * W1.shape[0] * W1.shape[1],
                'byte': float(M * C * (2 + 4 + 4 + (2 if k.get('out_bf16') is not None else 0)))}

    def proj_mlp_work(O, Wp, bp, g, b, W1, b1, W2, b2, **k):
        M = k.get('M') or O.shape[0]
        C = O.shape[1]
        return {'flop': 2.0 * M * C * C + 4.0 * M * W1.shape[0] * W1.shape[1],
                'byte': float(M * C * (2 + 4 + 4 + (2 if k.get('out_bf16') is not None else 0)))}

    def qkv_attn_work(y, Wg, bg, out, xyzb, rpe, n_win, H, C, K, dil, hat, bnd, scale, codes=None):
        L = K + (1 if hat else 0)
        rows = n_win * L
        return {'flop': 2.0 * rows * C * 3 * C + 4.0 * n_win * L * L * C,
                'byte': float(rows * (C * 2 + C * 2) + n_win * K * 8 + 3 * C * C * 2)}

    patches = {'qkv_attn': qkv_attn_work, 'gather_gemm': gemm_work, 'window_attn': attn_work, 'cpe_ln': cpe_work,
               'mlp_fused': mlp_work, 'proj_mlp_fused': proj_mlp_work}
    for name, work in patches.items():
        saved[name] = getattr(ops, name)
        setattr(ops, name, wrap(name, saved[name], work))
    others = ['varlen_attn', 'stem_conv', 'ln_rows', 'rt_init', 'attn_pool', 'mixer_tail', 'qkv_attn_codes',
              'hat_rows', 'remap_hat']
    for name in others:
        saved[name] = getattr(ops, name)
        setattr(ops, name, wrap(name, saved[name], lambda *a, **k: {}))
    s0, e0 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    try:
        s0.record()
        o = octree_fn()
        e0.record()
        model({'octree': o})
        torch.cuda.synchronize()
    finally:
        for name, fn in saved.items():
            setattr(ops, name, fn)
    fam = {'octree_build': {'ms': s0.elapsed_time(e0), 'launches': 0, 'flop': 0.0, 'byte': 0.0}}
    for name, s, e, work in rec:
        f = fam.setdefault(name, {'ms': 0.0, 'launches': 0, 'flop': 0.0, 'byte': 0.0})
        f['ms'] += s.elapsed_time(e)
        f['launches'] += 1
        for kind, amount in work.items():
            f[kind] += amount
    return fam


def run_native(args, rank, world, device):
    from hotformerloc_b200 import native
    from hotformerloc_b200.octree import build_batch, build_batch_device
    import torch.distributed as dist
    model, paths, depth = make_model(args.config, device)
    B, P = args.batch, args.points
    n_pool = 3
    batches = synthetic_batches(n_pool, B, P, seed0=1000 + 17 * rank)
    dev_batches = []
    for clouds in batches:
        pts = torch.from_numpy(np.concatenate(clouds)).to(device)
        off = torch.tensor(np.concatenate([[0], np.cumsum([len(c) for c in clouds])]),
                           dtype=torch.int32, device=device)
        dev_batches.append((pts, off))

    # Each step = one octree build + one forward.  The build of batch i+1 is enqueued ahead of
    # the forward of batch i (same stream), so the host's wait for the node counts of batch i+1
    # overlaps GPU work instead of draining the queue; K timed steps contain K builds + K forwards.
    ahead = {}

    def step_resident(i):
        o = ahead.pop(('r', i), None) or build_batch_device(*dev_batches[i % n_pool], depth, 2)
        ahead[('r', i + 1)] = build_batch_device(*dev_batches[(i + 1) % n_pool], depth, 2)
        return model({'octree': o})['global']

    # End to end: host point clouds in, host descriptors out, every step.  The descriptor read-back
    # is a non-blocking copy into pinned memory that the host consumes two steps later (after the
    # next steps are enqueued), so the GPU queue never drains; all K results are read inside the
    # timed region (drain_e2e runs before the closing event).
    res_pin = [torch.empty((B, 256), dtype=torch.float32).pin_memory() for _ in range(2)]
    res_evt = [None, None]
    consumed = []

    def consume(k):
        if res_evt[k] is not None:
            res_evt[k].synchronize()
            consumed.append(float(res_pin[k][0, 0]) + float(res_pin[k][-1, -1]))
            res_evt[k] = None

    def step_e2e(i):
        o = ahead.pop(('e', i), None) or build_batch(batches[i % n_pool], depth, 2, device)
        ahead[('e', i + 1)] = build_batch(batches[(i + 1) % n_pool], depth, 2, device)
        d = model({'octree': o})['global']
        if world > 1:
            d = gather(d)[rank]                      # the descriptor all-gather is part of the end-to-end step
        k = i & 1
        consume(k)                                   # result of step i - 2
        res_pin[k].copy_(d, non_blocking=True)
        res_evt[k] = torch.cuda.Event()
        res_evt[k].record()
        return None

    def drain_e2e():
        consume(0)
        consume(1)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def gather(desc):
        if world > 1:
            out = torch.empty((world,) + tuple(desc.shape), dtype=desc.dtype, device=desc.device)
            dist.all_gather_into_tensor(out, desc)
            return out
        return desc

    def timed(fn, steps, warmup, drain=None):
        for i in range(warmup):
            fn(i)
        if drain:
            drain()
        barrier()
        l0 = native.launch_count()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        for i in range(steps):
            d = fn(warmup + i)
            if torch.is_tensor(d) and d.is_cuda:
                d = gather(d)
        if drain:
            drain()
        e.record()
        barrier()
        ms = torch.tensor([s.elapsed_time(e)], device=device)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()), native.launch_count() - l0, d

    sampler = ClockSampler(torch.cuda.current_device())
    sampler.start()
    if args.ncu_step:
        for i in range(args.warmup):
            step_resident(i)
        barrier()
        torch.cuda.profiler.start()
        step_resident(args.warmup)
        barrier()
        torch.cuda.profiler.stop()
        return
    ms, launches, last = timed(step_resident, args.steps, args.warmup)
    sampler.stop_flag = True
    outputs = {}
    if args.dump_outputs:     # copied now: the next forward may reuse the buffers behind `last`
        outputs['global'] = last.float().reshape(-1, last.shape[-1]).cpu().numpy()
    e2e_steps = args.steps
    e2e_warmup = max(3, args.warmup)
    ms_e2e, _, _ = timed(step_e2e, e2e_steps, e2e_warmup, drain=drain_e2e)
    if rank != 0:
        return
    if args.dump_outputs:
        outputs['e2e_global'] = res_pin[(e2e_warmup + e2e_steps - 1) & 1].numpy().copy()
        dump_outputs(args.dump_outputs, outputs)
    value = world * B * args.steps / (ms / 1e3)
    e2e_value = world * B * e2e_steps / (ms_e2e / 1e3)
    # ---- roofline of the dominant kernel family (rank 0, one instrumented step) ----
    fam = kernel_profile(model, lambda: build_batch_device(*dev_batches[0], depth, 2))
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
    except Exception:
        pass
    tf_peak = peaks.get('bf16_tflops_sustained', 1400.0)
    hbm_peak = peaks.get('hbm_gbs', 6650.0)
    peak_src = 'measured' if peaks else 'fallback'
    # every family is placed against BOTH roofs; the one it sits closer to is the binding bound
    def roof_of(name):
        f = fam[name]
        tf = f['flop'] / (f['ms'] / 1e3) / 1e12
        gb = f['byte'] / (f['ms'] / 1e3) / 1e9
        if tf / tf_peak >= gb / hbm_peak:
            r = {'kernel': name, 'bound': 'tensor', 'achieved': tf, 'peak': tf_peak, 'unit': 'TFLOP/s',
                 'frac': tf / tf_peak}
        else:
            r = {'kernel': name, 'bound': 'hbm', 'achieved': gb, 'peak': hbm_peak, 'unit': 'GB/s',
                 'frac': gb / hbm_peak}
        r.update({'traffic': None, 'peak_source': peak_src, 'launches_per_step': f['launches'],
                  'ms_per_step': f['ms'], 'tflops': tf, 'gbs': gb})
        return r
    dom = max((k for k in fam if k != 'octree_build'), key=lambda k: fam[k]['ms'])
    roof = roof_of(dom)
    try:        # DRAM bytes of this family's largest launch from the committed ncu --set full capture
        cap = json.load(open(os.path.join(ROOT, 'profiles', 'r02_traffic.json'))).get(dom)
        if cap:
            roof['traffic'] = cap['dram_bytes']
            roof['traffic_source'] = (f"profiles/r02_traffic.json: {cap['kernel']}, the family's largest launch "
                                      f"({cap['ms']:.3f} ms) under ncu --set full")
    except Exception:
        pass
    roof_all = {k: {kk: (round(v, 4) if isinstance(v, float) else v) for kk, v in roof_of(k).items()
                    if kk in ('bound', 'frac', 'tflops', 'gbs', 'ms_per_step', 'launches_per_step')}
                for k in fam if k != 'octree_build' and (fam[k]['flop'] > 0 or fam[k]['byte'] > 0)}
    tot = sum(v['ms'] for v in fam.values())
    shares = {k: round(v['ms'] / tot, 4) for k, v in sorted(fam.items(), key=lambda kv: -kv[1]['ms'])}
    cpu = cpu_baseline(args, sample=args.cpu_sample) if not args.no_cpu else None
    h2d = sum(c.nbytes for c in batches[0]) + 4 * (B + 1)
    out = {
        'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': world, 'steps': args.steps,
        'warmup': args.warmup, 'ms_per_step': ms / args.steps, 'higher_is_better': True,
        'scaling': 'weak', 'vs_baseline': None, 'dtype': 'bf16', 'data': 'synthetic',
        'config': {'workload': f'{args.config} cfg, {B} synthetic {P}-point submaps per step per GPU, '
                               f'random-init weights (BASELINE.json configs[1])',
                   'octree_depth': depth, 'l2': 'per-step working set (GBs of activations) >> 126 MB L2; '
                                                'inputs cycle over 3 distinct batches',
                   'parallelism': f'batch-sharded x{world}'},
        'e2e': {'value': e2e_value, 'unit': UNIT, 'h2d_bytes_per_step': int(h2d),
                'd2h_bytes_per_step': int(B * 256 * 4), 'steps': e2e_steps},
        'gpu_launches': int(launches), 'clocks': sampler.summary(), 'roofline': roof, 'roofline_by_kernel': roof_all,
        'kernel_time_shares': shares, 'cpu_baseline': cpu,
    }
    emit(out)


_REAL_STDOUT = None


def emit(obj):
    line = (json.dumps(obj) + '\n').encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(line.decode())
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, line)


DUMP_BYTES = 64 << 20


def dump_outputs(out_dir, arrays):
    """Writes every array as out_dir/<name>.npy in float32.  All of them together stay within DUMP_BYTES: an
    array over its share keeps a seeded, sorted sample of its rows, the same sample for the same shape."""
    os.makedirs(out_dir, exist_ok=True)
    share = DUMP_BYTES // len(arrays)
    for name, a in arrays.items():
        a = np.ascontiguousarray(a, dtype=np.float32)
        if a.nbytes > share:
            keep = np.random.default_rng(0).choice(len(a), share // a[0].nbytes, replace=False)
            a = a[np.sort(keep)]
        np.save(os.path.join(out_dir, f'{name}.npy'), a)


def cpu_baseline(args, sample=4, steps=1, warmup=0):
    """The reference's CPU implementation of the path on a bounded sample of the same workload, in the three
    phases of BASELINE.md section 3: per-submap octree build loop, merge_octrees + construct_all_neigh, model
    forward.  kind = "reference": the reference's OWN, unmodified models/*.py + model_factory staged under
    oracle/_ref (oracle/build_ref.py), run over the ocnn stand-ins of oracle/ocnn_standin.py (ocnn 2.2.2 and the
    CUDA-only dwconv extension cannot be installed offline).  kind = "port" (oracle/model_ref.py) only when
    oracle/_ref has not been staged."""
    from oracle import build_ref
    from hotformerloc_b200.config.presets import write_configs, TRAIN_PRESETS
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    depth = TRAIN_PRESETS[args.config]['octree_depth']
    d = tempfile.mkdtemp(prefix='hfl_cfg_')
    paths = write_configs(d, args.config, dataset_folder=d)
    phases = {'octree_build_loop': [], 'merge_and_neigh': [], 'forward': []}
    if build_ref.available():
        from oracle import ocnn_standin as S
        S.install(build_ref.DST)
        torch.manual_seed(0)
        model = S.reference_model(paths['model_config'])
        kind = 'reference'

        def one(clouds):
            t0 = time.perf_counter()
            octs = []
            for c in clouds:                                   # eval/pnv_evaluate.py:173-176
                o = S.Octree(depth, 2)
                o.build_octree(S.Points(torch.as_tensor(c)))
                octs.append(o)
            t1 = time.perf_counter()
            mo = S.merge_octrees(octs)                         # eval/pnv_evaluate.py:122-126
            mo.construct_all_neigh()
            t2 = time.perf_counter()
            with torch.inference_mode():
                model({'octree': mo})['global']
            t3 = time.perf_counter()
            return t1 - t0, t2 - t1, t3 - t2
    else:
        from oracle import model_ref as M, octree_ref as R
        hp = M.HParams.from_cfg(paths['model_config'])
        shapes = json.load(open(os.path.join(ROOT, 'tests', 'golden', f'state_shapes_{args.config}.json')))
        sd = M.synthetic_state_dict(shapes, mode='init')
        kind = 'port'

        def one(clouds):
            t0 = time.perf_counter()
            o = R.build_batch(clouds, depth)                   # build + merge + neighbours in one call
            t1 = time.perf_counter()
            M.forward(sd, o, hp)
            t2 = time.perf_counter()
            return t1 - t0, 0.0, t2 - t1
    times = []
    for i in range(warmup + steps):
        clouds = synthetic_batches(1, sample, args.points, seed0=5000 + i)[0]
        ph = one(clouds)
        if i >= warmup:
            times.append(sum(ph))
            for k, v in zip(phases, ph):
                phases[k].append(v)
    sec = float(np.mean(times))
    return {'value': sample / sec, 'unit': UNIT, 'cores': cores, 'kind': kind,
            'sample': f'{sample} submaps of {args.points} points per step, {steps} step(s), '
                      f'fp32, torch threads = {cores}', 'seconds_per_step': sec,
            'phase_seconds_per_step': {k: float(np.mean(v)) for k, v in phases.items()}}


def run_reference(args, rank, world):
    if rank != 0:
        return
    sample = args.cpu_sample
    cpu = cpu_baseline(args, sample=sample, steps=args.steps, warmup=min(args.warmup, 1))
    out = {'impl': 'reference', 'metric': METRIC, 'value': cpu['value'], 'unit': UNIT,
           'n_gpus': world, 'steps': args.steps, 'warmup': min(args.warmup, 1),
           'ms_per_step': cpu['seconds_per_step'] * 1e3, 'higher_is_better': True,
           'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
           'config': {'workload': f'{args.config} cfg, {args.batch} synthetic {args.points}-point submaps per step per GPU, '
                                  f'random-init weights (BASELINE.json configs[1])',
                      'sample': f'each step = {sample} submaps of that workload on the host cores ({cpu["kind"]}: see cpu_baseline)'},
           'cpu_baseline': cpu,
           'e2e': {'value': cpu['value'], 'unit': UNIT, 'h2d_bytes_per_step': 0,
                   'd2h_bytes_per_step': 0}}
    emit(out)


def run_eval_workload(args, rank, world):
    """BASELINE.json configs[3] as a bench line: Wild-Places cfg, `--eval-runs` traversals x `--eval-per-run`
    submaps of ~30 k points in the reference's on-disk format -> loaders -> Normalize / cylindrical -> device
    octrees -> descriptors (batches sharded over the ranks) -> all-gather -> database-sharded top-25 -> merge ->
    recall.  One step = the whole evaluation (files already written); time = wall clock around embed + search,
    max over ranks through the barriers inside (tools/config4_eval.py)."""
    sys.path.insert(0, os.path.join(ROOT, 'tools'))
    import config4_eval
    # the bench writes nothing into the tree: config4_eval's own JSON record goes to a temporary directory
    out = os.path.join(tempfile.mkdtemp(prefix='hfl_config4_out_'), f'config4_{world}gpu.json')
    r = config4_eval.main(['--runs', str(args.eval_runs), '--per-run', str(args.eval_per_run), '--points', '30000',
                           '--out', out], emit=False)
    if rank != 0:
        return
    sec = r['embed_seconds_incl_file_io_and_host_prep'] + r['search_seconds']
    emit({'metric': 'submaps_per_sec_eval_files_to_recall', 'value': r['submaps'] / sec, 'unit': UNIT, 'n_gpus': world,
          'steps': 1, 'warmup': 1, 'ms_per_step': sec * 1e3, 'higher_is_better': True, 'scaling': 'strong',
          'vs_baseline': None, 'dtype': 'bf16', 'data': 'synthetic',
          'config': {'workload': r['config'] + ' (BASELINE.json configs[3])', 'parallelism': f'batch-sharded x{world}, '
                     'database-sharded top-k'},
          'recall': {k: r[k] for k in ('recall_at_1', 'recall_at_5', 'recall_at_1pct', 'mrr')},
          'embed_seconds': r['embed_seconds_incl_file_io_and_host_prep'], 'search_seconds': r['search_seconds'],
          'checks': r['checks']})


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=10)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='native', choices=['native', 'reference'])
    ap.add_argument('--config', default='oxford')
    ap.add_argument('--batch', type=int, default=256)
    ap.add_argument('--points', type=int, default=4096)
    ap.add_argument('--cpu-sample', type=int, default=4)
    ap.add_argument('--no-cpu', action='store_true')
    ap.add_argument('--workload', default='embed', choices=['embed', 'eval'],
                    help='embed = the headline step (default); eval = BASELINE.json configs[3], files -> recall')
    ap.add_argument('--eval-runs', type=int, default=4)
    ap.add_argument('--eval-per-run', type=int, default=8192)
    ap.add_argument('--ncu-step', action='store_true',
                    help='profiling aid: warm up, then run ONE step between cudaProfilerStart/Stop and exit '
                         '(use with ncu --profile-from-start off); prints no bench line')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='after the timed steps, write the descriptors of the last timed step as DIR/<name>.npy '
                         '(float32, at most 64 MB in all)')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and (args.impl != 'native' or args.workload != 'embed' or args.ncu_step):
        ap.error('--dump-outputs needs the native embed workload (--impl native --workload embed, no --ncu-step)')
    # stdout carries exactly ONE JSON line: anything a library prints there (NCCL's version banner
    # at NCCL_DEBUG=VERSION, for one) is sent to stderr; emit() writes to the saved descriptor
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    rank = int(os.environ.get('RANK', 0))
    world = int(os.environ.get('WORLD_SIZE', 1))
    local = int(os.environ.get('LOCAL_RANK', 0))
    if args.impl == 'reference':
        run_reference(args, rank, world)
        return
    args.warmup = max(args.warmup, 3)
    assert torch.cuda.is_available(), 'bench.py needs a GPU (there is no CPU fallback)'
    torch.cuda.set_device(local)
    device = torch.device('cuda', local)
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        dist.init_process_group('nccl', device_id=device)
    try:
        if args.workload == 'eval':
            run_eval_workload(args, rank, world)
        else:
            run_native(args, rank, world, device)
    finally:
        if world > 1:
            import torch.distributed as dist
            dist.destroy_process_group()


if __name__ == '__main__':
    main()
