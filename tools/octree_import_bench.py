"""Timing of the ocnn octree import (hotformerloc_b200.octree.from_ocnn, csrc/octree.cu
hfl_octree_import) at the evaluation batch sizes of two configs, next to the native build from the
same clouds and one model forward:

    oxford          256 submaps x 4096 points, depth 9 (val_batch_size 256)
    cs-wild-places  128 submaps x 30000 points, depth 7 (val_batch_size 128)

The ocnn-layout input is the native build's own keys / children / points / nnum* views, which are
that layout; the CPU-resident variant is the same tensors copied to the host, as an ocnn octree is
before to_device.  Rows:
    import_kernels   hfl_octree_import alone on GPU-resident input (CUDA events)
    from_ocnn_gpu    from_ocnn(...).finalize() on GPU-resident input: import, neighbour tables, read-back
    from_ocnn_cpu    the same from CPU-resident tensors: adds the pinned host copy and the H2D upload
    build_batch      build_batch(clouds).finalize() from the host clouds
    model_forward    model({'octree': native})['global'] at the config's preset, random weights
Algorithmic bytes of the import (each unique operand once): per depth, keys 8 + children 4 read
and children 4 written per node, nidx 4 + nkey 8 written per non-empty node; leaf points 12 B read
and written per leaf.  The kernels also re-read children once (the rank count) and each node reads
its parent's key; those are not counted.  The inputs (about 0.4 GB at both sizes) exceed the 126 MB L2.

    python tools/octree_import_bench.py [--iters 10] [--warmup 4] [--out FILE]
"""
import argparse
import ctypes as C
import json
import os
import sys
import tempfile
import types

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from dwconv_bench import HBM_GBPS, device_info, time_ms
from hotformerloc_b200 import native as N
from hotformerloc_b200.octree import Octree, build_batch, from_ocnn
from oracle import model_ref as M

CONFIGS = (('oxford', 256, 4096, 9), ('cs-wild-places', 128, 30000, 7))


def ocnn_views(o: Octree, device):
    """The ocnn attributes of a native octree, as tensors on `device`."""
    D = o.depth
    v = types.SimpleNamespace(depth=D, full_depth=o.full_depth, batch_size=o.batch_size, nnum=o.nnum,
                              nnum_nempty=o.nnum_nempty, batch_nnum_nempty=o.batch_nnum_nempty)
    v.keys = [k.to(device) for k in o.keys]
    v.children = [c.to(device) for c in o.children]
    v.points = [None] * D + [o.points[D].to(device)]
    return v


def import_kernels(v):
    """hfl_octree_import on GPU-resident views, into an output allocated once."""
    L = N.lib()
    D, F, B = v.depth, v.full_depth, v.batch_size
    desc = N.hfl_ocnn_octree()
    desc.depth, desc.full_depth, desc.batch = D, F, B
    for d in range(D + 1):
        desc.nnum[d], desc.nnum_nempty[d] = int(v.nnum[d]), int(v.nnum_nempty[d])
        desc.keys[d], desc.children[d] = v.keys[d].data_ptr(), v.children[d].data_ptr()
    desc.points = v.points[D].data_ptr()
    out = Octree(D, F, B, 'cuda')
    out._carve([B * 8 ** d if d <= F else int(v.nnum_nempty[d]) for d in range(D + 1)], 0, n_status=2)
    status = out._counts_dev[(D + 1) * (B + 2):]
    ws_bytes = int(L.hfl_octree_import_workspace_bytes(C.byref(desc)))
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device='cuda')

    def run():
        N.check(L.hfl_octree_import(C.byref(desc), C.byref(out._desc), N.ptr(status), N.ptr(ws), ws_bytes,
                                    N.stream()))
    return run, status


def alg_bytes(v):
    nn = [int(x) for x in v.nnum]
    ne = [int(x) for x in v.nnum_nempty]
    return sum(16 * nn[d] + 12 * ne[d] for d in range(v.depth + 1)) + 24 * ne[v.depth]


def model_for(cfg):
    from hotformerloc_b200.config.presets import write_configs
    from hotformerloc_b200.misc.utils import ModelParams
    from hotformerloc_b200.models.model_factory import model_factory
    d = tempfile.mkdtemp(prefix='hfl_import_bench_')
    torch.manual_seed(0)
    return model_factory(ModelParams(write_configs(d, cfg, dataset_folder=d)['model_config'])).cuda().eval()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--iters', type=int, default=10)
    ap.add_argument('--warmup', type=int, default=4)   # >= the pinned pool's slots: first uses allocate them
    ap.add_argument('--out', default=None, help='also write the JSON here')
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('octree_import_bench needs a CUDA device')
    torch.cuda.set_device(0)
    result = {'device': device_info(), 'iters': args.iters, 'warmup': args.warmup,
              'hbm_datasheet_gbps': HBM_GBPS, 'rows': []}
    for cfg, B, P, D in CONFIGS:
        g = torch.Generator().manual_seed(5)
        clouds = [M.lidar_cloud(P, g) for _ in range(B)]
        native = build_batch(clouds, D, 2, 'cuda').finalize()
        gpu, cpu = ocnn_views(native, 'cuda'), ocnn_views(native, 'cpu')
        nbytes = alg_bytes(gpu)
        head = {'config': cfg, 'batch': B, 'points': P, 'depth': D,
                'nodes': int(native.nnum.sum()), 'nonempty_nodes': int(native.nnum_nempty.sum())}
        # every path must give the native octree back
        for v in (gpu, cpu):
            o = from_ocnn(v).finalize()
            assert all(torch.equal(o.children[d], native.children[d]) for d in range(D + 1))
            assert torch.equal(o.ne_table(D), native.ne_table(D))
        run, status = import_kernels(gpu)
        l0 = N.launch_count()
        run()
        launches = N.launch_count() - l0
        torch.cuda.synchronize()
        assert int(status[0]) == 0
        model = model_for(cfg)
        ops = {
            'import_kernels': run,
            'from_ocnn_gpu': lambda: from_ocnn(gpu).finalize(),
            'from_ocnn_cpu': lambda: from_ocnn(cpu).finalize(),
            'build_batch': lambda: build_batch(clouds, D, 2, 'cuda').finalize(),
            'model_forward': lambda: model({'octree': native})['global'],
        }
        for name, fn in ops.items():
            ms = time_ms(fn, args.iters, args.warmup)
            row = dict(head, op=name, ms=round(ms, 4))
            if name == 'import_kernels':
                gbps = nbytes / (ms * 1e-3) / 1e9
                row.update(alg_bytes=nbytes, gbps=round(gbps, 1), hbm_fraction=round(gbps / HBM_GBPS, 4),
                           launches=launches)
            result['rows'].append(row)
            print(json.dumps(row), file=sys.stderr)
        del model, native, gpu, cpu, run, status
        torch.cuda.empty_cache()
    line = json.dumps(result)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            f.write(line + '\n')


if __name__ == '__main__':
    main()
