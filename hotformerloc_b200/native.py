"""ctypes binding of libhfl_b200.so (the C ABI declared in include/hfl.h).

The product path has no CPU or library fallback: if the shared library is
missing or a call fails, this module raises.  PyTorch only supplies device
memory (tensors' data_ptr) and the current CUDA stream.
"""
from __future__ import annotations

import ctypes as C
import glob
import os
import subprocess
from typing import Optional

import torch

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(PKG_DIR)
CSRC = os.path.join(PKG_DIR, 'csrc')
LIB_PATH = os.path.join(PKG_DIR, 'libhfl_b200.so')
HFL_MAX_DEPTH = 15

NVCC_FLAGS = ['-gencode', 'arch=compute_100a,code=sm_100a', '-lineinfo', '-O3',
              '-std=c++17', '-Xcompiler', '-fPIC',
              '-Xcompiler', '-O3', '--expt-relaxed-constexpr']


class HflError(RuntimeError):
    pass


class hfl_octree(C.Structure):
    _fields_ = [
        ('depth', C.c_int32), ('full_depth', C.c_int32), ('batch', C.c_int32), ('_pad', C.c_int32),
        ('n_points', C.c_int64),
        ('cap', C.c_int64 * (HFL_MAX_DEPTH + 1)),
        ('nkey', C.c_void_p * (HFL_MAX_DEPTH + 1)),
        ('children', C.c_void_p * (HFL_MAX_DEPTH + 1)),
        ('nidx', C.c_void_p * (HFL_MAX_DEPTH + 1)),
        ('leaf_points', C.c_void_p),
        ('point_leaf', C.c_void_p),
        ('counts', C.c_void_p),
    ]


class hfl_ocnn_octree(C.Structure):
    _fields_ = [
        ('depth', C.c_int32), ('full_depth', C.c_int32), ('batch', C.c_int32), ('_pad', C.c_int32),
        ('nnum', C.c_int64 * (HFL_MAX_DEPTH + 1)),
        ('nnum_nempty', C.c_int64 * (HFL_MAX_DEPTH + 1)),
        ('keys', C.c_void_p * (HFL_MAX_DEPTH + 1)),
        ('children', C.c_void_p * (HFL_MAX_DEPTH + 1)),
        ('points', C.c_void_p),
    ]


HFL_IMPORT_BAD_CHILDREN = 1
HFL_IMPORT_BAD_KEYS = 2


def sources():
    return sorted(glob.glob(os.path.join(CSRC, '*.cu')))


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile every CUDA source for sm_100a into one in-tree shared library."""
    srcs = sources()
    deps = srcs + glob.glob(os.path.join(CSRC, '*.cuh')) + [os.path.join(ROOT, 'include', 'hfl.h')]
    if (not force and os.path.exists(LIB_PATH)
            and os.path.getmtime(LIB_PATH) >= max(os.path.getmtime(p) for p in deps)):
        return LIB_PATH
    nvcc = os.environ.get('NVCC', '/usr/local/cuda/bin/nvcc')
    objs = []
    os.makedirs(os.path.join(PKG_DIR, 'build'), exist_ok=True)
    procs = []
    for s in srcs:
        o = os.path.join(PKG_DIR, 'build', os.path.basename(s)[:-3] + '.o')
        objs.append(o)
        if (not force and os.path.exists(o)
                and os.path.getmtime(o) >= max(os.path.getmtime(p) for p in
                                               [s] + deps[len(srcs):])):
            continue
        cmd = [nvcc] + NVCC_FLAGS + ['-c', s, '-o', o]
        if verbose:
            cmd.insert(1, '-Xptxas=-v')
        procs.append((s, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT)))
    for s, p in procs:
        out, _ = p.communicate()
        if verbose and out:
            print(out.decode())
        if p.returncode != 0:
            raise HflError(f'nvcc failed on {s}:\n{out.decode()}')
    cmd = [nvcc, '-shared', '-o', LIB_PATH] + objs + ['-lcudart']
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT)
    if r.returncode != 0:
        raise HflError(f'link failed:\n{r.stdout.decode()}')
    return LIB_PATH


_lib: Optional[C.CDLL] = None
_p, _i32, _i64, _f32, _sz = C.c_void_p, C.c_int32, C.c_int64, C.c_float, C.c_size_t

# name -> (restype, argtypes); mirrors include/hfl.h one to one
SIGNATURES = {
    'hfl_last_error_string': (C.c_char_p, []),
    'hfl_version': (C.c_int, []),
    'hfl_launch_count': (_i64, []),
    'hfl_octree_build_workspace_bytes': (_sz, [_i64, _i32, _i32]),
    'hfl_octree_build': (C.c_int, [_p, _p, C.POINTER(hfl_octree), _p, _sz, _p]),
    'hfl_octree_import_check': (C.c_int, [C.POINTER(hfl_ocnn_octree)]),
    'hfl_octree_import_workspace_bytes':(_sz, [C.POINTER(hfl_ocnn_octree)]),
    'hfl_octree_import': (C.c_int, [C.POINTER(hfl_ocnn_octree), C.POINTER(hfl_octree), _p, _p, _sz, _p]),
    'hfl_octree_neigh': (C.c_int, [C.POINTER(hfl_octree), _i32, _p, _p, _p, _p, _p]),
    'hfl_octree_neigh_full': (C.c_int, [C.POINTER(hfl_octree), _i32, _p, _p, _p]),
    'hfl_octree_full_keys': (C.c_int, [C.POINTER(hfl_octree), _i32, _p, _p]),
    'hfl_octree_tokens': (C.c_int, [C.POINTER(hfl_octree), _i32, _i64, _p, _p]),
    'hfl_gather_gemm': (C.c_int, [_p, _p, _p, _i64, _i32, _i32, _i32, _p, _p, _i32, _p, _p, _p, _p,
                                  _i32, _i32, _p, _p, _p, _p]),
    'hfl_mlp_fused': (C.c_int, [_p, _p, _p, _p, _p, _i64, _i32, _p, _p, _p, _p, _p]),
    'hfl_proj_mlp_fused': (C.c_int, [_p, _p, _p, _p, _p, _p, _p, _p, _p, _i64, _i32, _p, _p, _p, _p, _p]),
    'hfl_window_attn': (C.c_int, [_p, _p, _p, _p, _i64, _i32, _i32, _i32, _i32, _i32, _i32, _f32, _p]),
    'hfl_qkv_attn_supported': (C.c_int, [_i32, _i32, _i32, _i32, _i32, _i32]),
    'hfl_qkv_attn': (C.c_int, [_p, _p, _p, _p, _p, _p, _i64, _i64, _i32, _i32, _i32, _i32, _i32, _i32, _f32, _p, _p]),
    'hfl_qkv_attn_codes_bytes': (C.c_int64, [_i64, _i32, _i32]),
    'hfl_qkv_attn_codes': (C.c_int, [_p, _i64, _i32, _i32, _i32, _i32, _i32, _p, _p]),
    'hfl_varlen_attn': (C.c_int, [_p, _p, _p, _p, _i32, _i32, _i32, _i32, _f32, _p]),
    'hfl_stem_conv': (C.c_int, [_p, _p, _i64, _i32, _p, _p, _p, _p, _p]),
    'hfl_cpe_ln': (C.c_int, [_p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _i64, _i64, _i32, _i32, _p]),
    'hfl_ln_rows': (C.c_int, [_p, _p, _i64, _i32, _p, _p, _p, _p]),
    'hfl_rt_init': (C.c_int, [_p, _p, _p, _i64, _i64, _i32, _i32, _i32, _i32, _p, _p, _p, _p, _p]),
    'hfl_hat_rows': (C.c_int, [_p, _i64, _i32, _i32, _p]),
    'hfl_remap_hat': (C.c_int, [_p, _p, _i64, _i32, _p]),
    'hfl_f32_to_bf16': (C.c_int, [_p, _p, _i64, _p]),
    'hfl_attn_pool': (C.c_int, [_p, _p, _p, _p, _p, _p, _i32, _i32, _i32, _i32, _i32, _i32, _i32, _f32, _p]),
    'hfl_mixer_tail': (C.c_int, [_p, _p, _p, _p, _p, _p, _i32, _i32, _i32, _i32, _i32, _i32, _p]),
    'hfl_gem_pool': (C.c_int, [_p, _p, _i32, _i32, _i32, _f32, _f32, _p, _i32, _i32, _p]),
    'hfl_gem_head': (C.c_int, [_p, _i32, _i32, _p, _p, _p, _p, _p, _f32, _i32, _i32, _p, _p]),
    'hfl_knn_topk': (C.c_int, [_p, _i32, _p, _i32, _i32, _i32, _i32, _p, _p, _p]),
    'hfl_prepare_clouds': (C.c_int, [_p, _p, _i32, _i64, _i32, _i32, _f32, _f32, _i32, _p, _p, _p, _p, _p, _p]),
    'hfl_knn_workspace_bytes': (C.c_int64, [_i32, _i32, _i32]),
    'hfl_knn_topk_ws': (C.c_int, [_p, _i32, _p, _i32, _i32, _i32, _i32, _p, _p, _p, _i64, _p]),
    'hfl_topk_merge': (C.c_int, [_p, _p, _i32, _i32, _i32, _p, _p, _p]),
    'hfl_dwconv': (C.c_int, [_p, _p, _i32, _p, _i64, _i64, _i32, _i32, _p, _p]),
    'hfl_dwconv_inverse': (C.c_int, [_p, _i32, _i64, _i64, _i32, _p, _p]),
    'hfl_dwconv_wgrad_workspace_bytes': (C.c_int64, [_i64, _i32, _i32]),
    'hfl_dwconv_wgrad': (C.c_int, [_p, _p, _p, _i32, _i64, _i64, _i32, _i32, _p, _p, _i64, _p]),
    'hfl_window_attn_train_fwd': (C.c_int, [_p, _p, _i32, _p, _i32, _p, _i64, _i32, _i32, _i32, _i32, _p, _p, _p]),
    'hfl_window_attn_train_bwd_workspace_bytes': (C.c_int64, [_i32, _i32, _i32]),
    'hfl_window_attn_train_bwd': (C.c_int, [_p, _p, _i32, _p, _i32, _p, _p, _p, _p, _i64, _i32, _i32, _i32, _i32,
                                            _p, _p, _p, _i64, _p]),
    'hfl_attn_pool_train_fwd_workspace_bytes': (C.c_int64, [_i64, _i32, _i32, _i32]),
    'hfl_attn_pool_train_bwd_workspace_bytes': (C.c_int64, [_i64, _i32, _i32, _i32]),
    'hfl_attn_pool_train_fwd': (C.c_int, [_p, _p, _p, _i64, _i32, _i32, _i32, _p, _p, _p, _i64, _p]),
    'hfl_attn_pool_train_bwd': (C.c_int, [_p, _p, _p, _p, _p, _p, _i64, _i32, _i32, _i32, _p, _p, _p, _i64, _p]),
    'hfl_rt_attn_train_workspace_bytes': (C.c_int64, [_i64, _i32, _i32]),
    'hfl_rt_attn_train_fwd': (C.c_int, [_p, _p, _p, _i32, _i32, _i64, _i32, _p, _p, _p, _i64, _p]),
    'hfl_rt_attn_train_bwd': (C.c_int, [_p, _p, _p, _i32, _p, _p, _p, _i32, _i64, _i32, _p, _p, _i64, _p]),
    'hfl_octree_conv_train_fwd': (C.c_int, [_p, _p, _i32, _p, _i64, _i64, _i32, _i32, _i32, _p, _p]),
    'hfl_octree_conv_train_wgrad_workspace_bytes': (C.c_int64, [_i64, _i32, _i32, _i32]),
    'hfl_octree_conv_train_wgrad': (C.c_int, [_p, _p, _i32, _p, _i64, _i64, _i32, _i32, _i32, _p, _p, _i64, _p]),
}


def register(sigs):
    SIGNATURES.update(sigs)
    if _lib is not None:
        _bind(_lib, sigs)


def _bind(lib, sigs):
    for name, (res, args) in sigs.items():
        fn = getattr(lib, name)          # AttributeError if the symbol is missing
        fn.restype = res
        fn.argtypes = args


def lib() -> C.CDLL:
    """Load the shared library (never builds implicitly on a GPU box: the .so
    travels in-tree; use __graft_entry__.build() / native.build() to compile)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise HflError(f'{LIB_PATH} is missing: run `python -c "import __graft_entry__ as g; '
                           f'g.build()"` (there is no CPU fallback)')
        l = C.CDLL(LIB_PATH)
        _bind(l, SIGNATURES)
        _lib = l
    return _lib


def check(status: int):
    if status != 0:
        raise HflError(f'hfl status {status}: {lib().hfl_last_error_string().decode()}')


def ptr(t: Optional[torch.Tensor]):
    if t is None:
        return None
    assert t.is_cuda and t.is_contiguous(), 'device-resident contiguous tensor required'
    return C.c_void_p(t.data_ptr())


def stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def launch_count() -> int:
    return int(lib().hfl_launch_count())


class PinnedPool:
    """Rotating pinned staging buffers: cudaHostAlloc is far too slow to pay per
    batch.  A buffer is reused only after the H2D copy that read it has completed."""

    def __init__(self, slots: int = 4):
        self.slots = [None] * slots
        self.i = 0
        self.gen = [0] * slots            # how often each slot has been handed out

    def take(self, nbytes: int) -> torch.Tensor:
        self.i = (self.i + 1) % len(self.slots)
        self.gen[self.i] += 1
        slot = self.slots[self.i]
        if slot is not None:
            slot[1].synchronize()
        if slot is None or slot[0].numel() < nbytes:
            cap = max(1 << 16, 1 << (int(nbytes) - 1).bit_length())
            slot = [torch.empty(cap, dtype=torch.uint8, pin_memory=True), torch.cuda.Event()]
            self.slots[self.i] = slot
        return slot[0][:nbytes]

    def ticket(self):
        """Identifies the buffer last taken; valid(ticket) tells whether it is still that hand-out."""
        return (self.i, self.gen[self.i])

    def valid(self, ticket) -> bool:
        return self.gen[ticket[0]] == ticket[1]

    def mark(self):
        """Call after enqueuing the H2D copy that reads the buffer last taken."""
        self.slots[self.i][1].record()


pinned = PinnedPool()
pinned_d2h = PinnedPool(slots=8)      # node-count read-backs (one per built octree)
