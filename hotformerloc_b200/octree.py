"""Device-resident batched octree -- the host-side mirror of the third-party
``ocnn.octree.Octree`` interface that the reference model reads
(``depth, full_depth, batch_size, device, keys, children, neighs, points,
nnum, nnum_nempty, batch_nnum_nempty`` and ``key / xyzb / batch_id /
get_neigh / nempty_mask``; SURVEY.md section 7 step 1, Appendix A).

The whole batch is built by one call into libhfl_b200.so
(``hfl_octree_build``): there is no per-submap host loop, no ``merge_octrees``
and no CPU implementation.  Replaces eval/pnv_evaluate.py:173-175 + :122-126
and misc/torch_utils.py:48-51 of the reference.
"""
from __future__ import annotations

import ctypes as C
from typing import List, Optional, Sequence, Union

import numpy as np
import torch

from . import native as N

BATCH_SHIFT = 48
LUT_KERNEL = {                       # ocnn's kernel shapes -> columns of the 27-neighbour table
    '222': [13, 14, 16, 17, 22, 23, 25, 26],
    '311': [4, 13, 22], '131': [10, 13, 16], '113': [12, 13, 14],
    '331': [1, 4, 7, 10, 13, 16, 19, 22, 25],
    '313': [3, 4, 5, 12, 13, 14, 21, 22, 23],
    '133': [9, 10, 11, 12, 13, 14, 15, 16, 17],
    '333': list(range(27)),
}


class Points:
    """Mirror of ``ocnn.octree.Points`` as used at eval/pnv_evaluate.py:173."""

    def __init__(self, points, normals=None, features=None, labels=None,
                 batch_id=None, batch_size: int = 1):
        self.points = torch.as_tensor(points, dtype=torch.float32)
        self.batch_size = batch_size


def _arena(total: int, device) -> torch.Tensor:
    return torch.empty(total, dtype=torch.uint8, device=device)


class Octree:
    def __init__(self, depth: int, full_depth: int = 2, batch_size: int = 1,
                 device: Union[str, torch.device] = 'cuda'):
        assert 1 <= full_depth < depth <= N.HFL_MAX_DEPTH
        self.depth, self.full_depth, self.batch_size = int(depth), int(full_depth), int(batch_size)
        self.device = torch.device(device)
        self._pending: List[np.ndarray] = []
        self._built = False
        self._keys = {}
        self._neighs = {}
        self._ne = {}                # depth -> (n_d,27) int32 non-empty neighbour table
        self._tok = {}
        self._src = None             # the input clouds, kept so that merge_octrees can rebuild the batch

    # ------------------------------------------------------------------ build
    def build_octree(self, point_cloud: Points):
        """ocnn Octree.build_octree for ONE submap (kept for API parity; the
        batched path is :func:`build_batch`).  Returns the leaf index of every
        point (ocnn's return value)."""
        pts = point_cloud.points if isinstance(point_cloud, Points) else torch.as_tensor(point_cloud)
        o = build_batch([pts], self.depth, self.full_depth, self.device, want_point_leaf=True)
        self.__dict__.update(o.__dict__)
        return self._point_leaf.long()

    def _build(self, clouds: Sequence, want_point_leaf: bool = False, neigh: bool = True):
        L = N.lib()
        if self.device.type != 'cuda':
            raise N.HflError('the octree is built on the GPU only (no CPU fallback)')
        B, D, F = len(clouds), self.depth, self.full_depth
        self.batch_size = B
        self._src = ('host', list(clouds))
        sizes = [int(c.shape[0]) for c in clouds]
        if min(sizes) < 1:
            raise ValueError('every submap needs at least one point')
        n = int(sum(sizes))
        # one pinned staging buffer: [points fp32 (n,3) | offsets int32 (B+1)] -> one H2D copy
        nb_pts = 12 * n
        stage = N.pinned.take(nb_pts + 4 * (B + 1))
        host = stage[:nb_pts].view(torch.float32).view(n, 3)
        off = stage[nb_pts:].view(torch.int32)
        o = 0
        off[0] = 0
        for i, c in enumerate(clouds):
            host[o:o + sizes[i]] = torch.as_tensor(c, dtype=torch.float32)
            o += sizes[i]
            off[i + 1] = o
        self._h2d_bytes = stage.numel()
        devbuf = stage.to(self.device, non_blocking=True)
        N.pinned.mark()
        pts = devbuf[:nb_pts].view(torch.float32).view(n, 3)
        offs = devbuf[nb_pts:].view(torch.int32)
        self._build_device(pts, offs, n, want_point_leaf, neigh)

    def _build_device(self, pts: torch.Tensor, offs: torch.Tensor, n: int,
                      want_point_leaf: bool = False, neigh: bool = True):
        L = N.lib()
        B, D, F, dev = self.batch_size, self.depth, self.full_depth, self.device
        cap = []
        for d in range(D + 1):
            full = B * 8 ** d
            cap.append(full if d <= F else min(full, n))
        al = lambda x: (x + 255) // 256 * 256
        sz_key = [al(8 * cap[d]) for d in range(D + 1)]
        sz_idx = [al(4 * cap[d]) for d in range(D + 1)]
        sz_chl = [al(4 * (cap[d] if d <= F else 8 * cap[d - 1])) for d in range(D + 1)]
        ws_bytes = int(L.hfl_octree_build_workspace_bytes(n, B, D))
        total = sum(sz_key) + sum(sz_idx) + sum(sz_chl) + al(12 * cap[D]) + al(4 * n) \
            + al(4 * (D + 1) * (B + 2))
        arena = _arena(total, dev)
        ws = _arena(ws_bytes, dev)
        self._arena = arena
        base = arena.data_ptr()
        pos = 0
        desc = N.hfl_octree()
        desc.depth, desc.full_depth, desc.batch, desc.n_points = D, F, B, n

        def take(nbytes, dtype, count):
            nonlocal pos
            t = arena[pos:pos + nbytes].view(dtype)[:count]
            pos += nbytes
            return t
        self._nkey, self._nidx, self._children_buf = [], [], []
        for d in range(D + 1):
            desc.cap[d] = cap[d]
            k = take(sz_key[d], torch.int64, cap[d])
            i = take(sz_idx[d], torch.int32, cap[d])
            c = take(sz_chl[d], torch.int32, cap[d] if d <= F else 8 * cap[d - 1])
            self._nkey.append(k); self._nidx.append(i); self._children_buf.append(c)
            desc.nkey[d], desc.nidx[d], desc.children[d] = k.data_ptr(), i.data_ptr(), c.data_ptr()
        self._leaf_points = take(al(12 * cap[D]), torch.float32, 3 * cap[D])
        self._point_leaf = take(al(4 * n), torch.int32, n)
        self._counts_dev = take(al(4 * (D + 1) * (B + 2)), torch.int32, (D + 1) * (B + 2))
        desc.leaf_points = self._leaf_points.data_ptr()
        desc.point_leaf = self._point_leaf.data_ptr() if want_point_leaf else None
        desc.counts = self._counts_dev.data_ptr()
        self._desc, self._cap, self._n_points = desc, cap, n
        N.check(L.hfl_octree_build(N.ptr(pts), N.ptr(offs), C.byref(desc), N.ptr(ws), ws_bytes,
                                   N.stream()))
        # counts -> host (the only D2H of the build; shapes of every later tensor).  The pinned slot is
        # shared and rotates: finalize() re-reads from the device if it was handed out again meanwhile.
        self._counts_host = N.pinned_d2h.take(4 * (D + 1) * (B + 2)).view(torch.int32).view(D + 1, B + 2)
        self._counts_slot = N.pinned_d2h.ticket()
        self._counts_host.copy_(self._counts_dev.view(D + 1, B + 2), non_blocking=True)
        N.pinned_d2h.mark()
        self._ready = torch.cuda.Event()
        self._ready.record()
        self._pts_keepalive = (pts, offs, ws)
        self._built = True
        self._finalized = False
        if neigh:
            self._construct_ne_all()

    def _construct_ne_all(self):
        """Non-empty 27-neighbour tables for every depth >= full_depth, capacity
        sized, no host sync (misc/torch_utils.py:49-51 + ocnn get_neigh)."""
        L = N.lib()
        B, D, F, dev = self.batch_size, self.depth, self.full_depth, self.device
        cap = self._cap
        grid = torch.empty(B * 8 ** F * 27, dtype=torch.int32, device=dev)
        na_prev = torch.empty(cap[F] * 27, dtype=torch.int32, device=dev)
        ne = torch.empty(cap[F] * 27, dtype=torch.int32, device=dev)
        N.check(L.hfl_octree_neigh(C.byref(self._desc), F, None, N.ptr(grid), N.ptr(na_prev),
                                   N.ptr(ne), N.stream()))
        self._ne_buf = {F: ne}
        self._na_full_depth = na_prev
        for d in range(F + 1, D + 1):
            na = torch.empty(cap[d] * 27, dtype=torch.int32, device=dev)
            ne = torch.empty(cap[d] * 27, dtype=torch.int32, device=dev)
            N.check(L.hfl_octree_neigh(C.byref(self._desc), d, N.ptr(na_prev), None, N.ptr(na),
                                       N.ptr(ne), N.stream()))
            self._ne_buf[d] = ne
            na_prev = na
        self._na_last = na_prev

    def finalize(self):
        """Wait for the node counts (one event sync) and publish the host-side
        shape tables the reference keeps on the CPU (ocnn Octree.nnum*,
        batch_nnum*; SURVEY Appendix A)."""
        if self._finalized:
            return self
        self._ready.synchronize()
        B = self.batch_size
        if N.pinned_d2h.valid(self._counts_slot):
            c = self._counts_host.to(torch.int64)    # copies out of the pinned staging slot
        else:                                        # the slot served a later build: read the device copy
            c = self._counts_dev.view(self.depth + 1, B + 2).cpu().to(torch.int64)
        self.batch_nnum_nempty = c[:, :B].clone()
        self.nnum_nempty = c[:, B].clone()
        self.nnum = c[:, B + 1].clone()
        bn = self.batch_nnum_nempty.clone()
        for d in range(self.depth + 1):
            bn[d] = 8 * self.batch_nnum_nempty[d - 1] if d > self.full_depth else 8 ** d
        self.batch_nnum = bn
        self._finalized = True
        return self

    # ------------------------------------------------ reference-layout views
    def n(self, d: int) -> int:
        return int(self.finalize().nnum_nempty[d])

    @property
    def children(self):
        self.finalize()
        return [self._children_buf[d][:int(self.nnum[d])] for d in range(self.depth + 1)]

    @property
    def keys(self):
        """ocnn Octree.keys: int64 (submap<<48 | morton) for ALL nodes per depth."""
        self.finalize()
        L = N.lib()
        out = []
        for d in range(self.depth + 1):
            if d not in self._keys:
                k = torch.empty(int(self.nnum[d]), dtype=torch.int64, device=self.device)
                N.check(L.hfl_octree_full_keys(C.byref(self._desc), d, N.ptr(k), N.stream()))
                self._keys[d] = k
            out.append(self._keys[d])
        return out

    @property
    def points(self):
        self.finalize()
        pts = [None] * (self.depth + 1)
        pts[self.depth] = self._leaf_points.view(-1, 3)[:self.n(self.depth)]
        return pts

    @property
    def neighs(self):
        """ocnn Octree.neighs: (nnum[d],27) int64 tables over ALL nodes."""
        self.finalize()
        L = N.lib()
        D, F = self.depth, self.full_depth
        if not self._neighs:
            prev = None                       # NA[d-1]: rows = non-empty nodes of depth d-1
            for d in range(1, D + 1):
                full = torch.empty(int(self.nnum[d]) * 27, dtype=torch.int32, device=self.device)
                N.check(L.hfl_octree_neigh_full(C.byref(self._desc), d,
                                                N.ptr(prev) if d > F else None, N.ptr(full),
                                                N.stream()))
                self._neighs[d] = full.view(-1, 27).long()
                if d == F:
                    prev = self._na_full_depth
                elif F < d < D:               # NA of intermediate depths is transient: rebuild
                    nxt = torch.empty(self._cap[d] * 27, dtype=torch.int32, device=self.device)
                    N.check(L.hfl_octree_neigh(C.byref(self._desc), d, N.ptr(prev), None,
                                               N.ptr(nxt), None, N.stream()))
                    prev = nxt
        return [None] + [self._neighs[d] for d in range(1, D + 1)]

    def nempty_mask(self, depth: int):
        return self.children[depth] >= 0

    def key(self, depth: int, nempty: bool = False):
        key = self.keys[depth]
        return key[self.nempty_mask(depth)] if nempty else key

    def batch_id(self, depth: int, nempty: bool = False):
        return self.key(depth, nempty) >> BATCH_SHIFT

    def xyzb(self, depth: int, nempty: bool = False):
        t = self.tokens(depth, self.n(depth)) if nempty else None
        if t is not None:
            t = t.long()
            return t[:, 0], t[:, 1], t[:, 2], t[:, 3]
        raise NotImplementedError('xyzb(nempty=False) is not on the hot path')

    def ne_table(self, depth: int) -> torch.Tensor:
        """(n_d,27) int32: get_neigh(depth,'333',1,nempty=True) without the int64 blow-up."""
        return self._ne_buf[depth].view(-1, 27)[:self.n(depth)]

    def child_table(self, depth: int) -> torch.Tensor:
        """(n_{d-1},8) int32: get_neigh(depth,'222',stride=2,nempty=True)."""
        return self.children[depth].view(-1, 8)

    def get_neigh(self, depth: int, kernel: str = '333', stride: int = 1, nempty: bool = False):
        """ocnn Octree.get_neigh (reference layout, int64)."""
        if isinstance(kernel, (list, tuple)):
            kernel = ''.join(str(k) for k in kernel)
        if nempty and stride == 1:
            t = self.ne_table(depth).long()
        elif nempty and stride == 2:
            full = self.neighs[depth][::8]
            child = self.children[depth].long()
            t = torch.where(full >= 0, child[full.clamp(min=0)], full)
        else:
            t = self.neighs[depth]
            if stride == 2:
                t = t[::8].clone()
        if kernel != '333':
            t = t[:, LUT_KERNEL[kernel]]
        return t

    def tokens(self, depth: int, n_pad: int) -> torch.Tensor:
        """(n_pad,4) int16 (x,y,z,submap); padding rows are (0,0,0,batch)."""
        key = (depth, n_pad)
        if key not in self._tok:
            out = torch.empty((n_pad, 4), dtype=torch.int16, device=self.device)
            N.check(N.lib().hfl_octree_tokens(C.byref(self._desc), depth, n_pad, N.ptr(out),
                                              N.stream()))
            self._tok[key] = out
        return self._tok[key]

    def to(self, device, non_blocking: bool = False):
        if torch.device(device).type != 'cuda':
            raise N.HflError('the native octree lives on the GPU (no CPU fallback)')
        return self

    def cuda(self):
        return self

    def construct_all_neigh(self):
        if not hasattr(self, '_ne_buf'):
            self._construct_ne_all()


def build_batch(clouds: Sequence, depth: int, full_depth: int = 2,
                device: Union[str, torch.device] = 'cuda', want_point_leaf: bool = False,
                neigh: bool = True) -> Octree:
    """Build ONE merged octree for a list of (P_i,3) fp32 clouds in [-1,1]:
    the per-batch host path of eval/pnv_evaluate.py:155-185 in one device pass."""
    o = Octree(depth, full_depth, len(clouds), device)
    o._build(clouds, want_point_leaf, neigh)
    return o


def build_batch_device(points: torch.Tensor, offsets: torch.Tensor, depth: int,
                       full_depth: int = 2, neigh: bool = True) -> Octree:
    """Same, for points already resident in HBM: (P,3) fp32 + (B+1,) int32 offsets."""
    B = offsets.numel() - 1
    o = Octree(depth, full_depth, B, points.device)
    points, offsets = points.contiguous(), offsets.contiguous().to(torch.int32)
    o._src = ('device', points, offsets)
    o._build_device(points, offsets, int(points.shape[0]), False, neigh)
    return o


def merge_octrees(octrees: Sequence[Octree]) -> Octree:
    """ocnn.octree.merge_octrees (eval/pnv_evaluate.py:123): one batch octree from per-submap (or already
    batched) octrees, submap order = list order.  The merged structure is produced by ONE batched device
    build over the retained input clouds -- identical, node for node, to concatenating the per-submap
    octrees with submap ids in the key bits >= 48 and children offset by the running non-empty counts
    (SURVEY.md Appendix A; pinned by the reference's batch_45 fixture), without the O(depth x B) host loop."""
    octrees = list(octrees)
    if not octrees:
        raise ValueError('merge_octrees needs at least one octree')
    if len(octrees) == 1:
        return octrees[0]
    first = octrees[0]
    for o in octrees:
        if not isinstance(o, Octree) or o._src is None:
            raise N.HflError('merge_octrees: every octree must have been built by Octree.build_octree / build_batch')
        if (o.depth, o.full_depth) != (first.depth, first.full_depth):
            raise ValueError('merge_octrees: depth / full_depth differ')
    if all(o._src[0] == 'host' for o in octrees):
        clouds = [c for o in octrees for c in o._src[1]]
        return build_batch(clouds, first.depth, first.full_depth, first.device)
    pts, offs, base = [], [torch.zeros(1, dtype=torch.int32, device=first.device)], 0
    for o in octrees:
        if o._src[0] == 'host':
            for c in o._src[1]:
                t = torch.as_tensor(c, dtype=torch.float32).to(first.device)
                pts.append(t)
                base += t.shape[0]
                offs.append(torch.tensor([base], dtype=torch.int32, device=first.device))
        else:
            pts.append(o._src[1])
            offs.append(o._src[2][1:] + base)
            base += int(o._src[1].shape[0])
    return build_batch_device(torch.cat(pts), torch.cat(offs), first.depth, first.full_depth)
