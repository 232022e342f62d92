"""hotformerloc_b200.octree.from_ocnn and the model's ocnn-octree entry points on the GPU.

The ocnn octrees come from the pure-torch ocnn stand-in (oracle/ocnn_standin.py), built with the
reference's own call flow: one Octree(depth, full_depth).build_octree(Points(x)) per submap,
merge_octrees, construct_all_neigh.  Every case runs once with the ocnn tensors left on the CPU and
once moved to CUDA.  The imported octree must equal build_batch on the same clouds bit for bit, and
so must the model's outputs; a malformed octree must raise HflError naming the violated invariant."""
import copy
import os

import numpy as np
import pytest
import torch

from oracle import model_ref as M
from oracle import ocnn_standin as S
from oracle.make_golden import CASES
from tests.common import case_clouds, case_state_dict, native_model

pytestmark = pytest.mark.gpu

WHERE = ['cpu', 'cuda']


def _ocnn(clouds, depth, full_depth=2, where='cpu'):
    octs = []
    for c in clouds:
        o = S.Octree(depth, full_depth)
        o.build_octree(S.Points(torch.as_tensor(c)))
        octs.append(o)
    m = S.merge_octrees(octs)
    m.construct_all_neigh()
    if where == 'cuda':                 # what to_device does to the tensors of an ocnn octree
        m = copy.copy(m)
        m.keys = [k.cuda() for k in m.keys]
        m.children = [c.cuda() for c in m.children]
        m.points = [None if p is None else p.cuda() for p in m.points]
    return m


def _import(ocnn):
    from hotformerloc_b200.octree import from_ocnn
    return from_ocnn(ocnn).finalize()


def _assert_same(o, ref, full_neigh=True, ocnn=None):
    """o (imported) against ref (build_batch), table by table."""
    D, F = ref.depth, ref.full_depth
    assert (o.depth, o.full_depth, o.batch_size) == (D, F, ref.batch_size)
    for name in ('nnum', 'nnum_nempty', 'batch_nnum', 'batch_nnum_nempty'):
        assert torch.equal(getattr(o, name), getattr(ref, name)), name
    for d in range(D + 1):
        assert torch.equal(o.keys[d], ref.keys[d]), f'keys[{d}]'
        assert torch.equal(o.children[d], ref.children[d]), f'children[{d}]'
    assert torch.equal(o.points[D], ref.points[D])
    for d in range(F, D + 1):
        assert torch.equal(o.ne_table(d), ref.ne_table(d)), f'ne_table({d})'
        assert torch.equal(o.child_table(d), ref.child_table(d)), f'child_table({d})'
        assert torch.equal(o.get_neigh(d, '333', 1, True), ref.get_neigh(d, '333', 1, True))
        n = o.n(d)
        n_pad = -(-n // 192) * 192
        assert torch.equal(o.tokens(d, n_pad), ref.tokens(d, n_pad)), f'tokens({d})'
    if full_neigh:
        for d in range(1, D + 1):
            assert torch.equal(o.neighs[d], ref.neighs[d]), f'neighs[{d}]'
            if ocnn is not None:         # and ocnn's own (discarded) tables
                assert torch.equal(o.neighs[d].cpu(), ocnn.neighs[d].cpu()), f'ocnn neighs[{d}]'
        assert torch.equal(o.get_neigh(D, '222', 2, True), ref.get_neigh(D, '222', 2, True))
        assert torch.equal(o.get_neigh(D - 1, '333', 1, False), ref.get_neigh(D - 1, '333', 1, False))
        assert torch.equal(o.get_neigh(D, '311', 1, True), ref.get_neigh(D, '311', 1, True))


def _check(clouds, depth, full_depth=2, where='cpu', full_neigh=True):
    from hotformerloc_b200.octree import build_batch
    ocnn = _ocnn(clouds, depth, full_depth, where)
    o = _import(ocnn)
    ref = build_batch(clouds, depth, full_depth, 'cuda').finalize()
    _assert_same(o, ref, full_neigh, ocnn)
    return o


# ---------------------------------------------------------------------------------------------------
# 1. structure
# ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('where', WHERE)
def test_reference_fixtures(golden_dir, where):
    fx = np.load(os.path.join(golden_dir, 'octree_fixtures.npz'))
    for i in range(1, 6):
        D, F = int(fx[f't{i}_depth']), int(fx[f't{i}_full_depth'])
        o = _check([fx[f't{i}_points']], D, F, where)
        assert np.array_equal(torch.cat(o.keys).cpu().numpy(), fx[f't{i}_key'])
        assert np.array_equal(torch.cat(o.children).cpu().numpy(), fx[f't{i}_child'])
        assert np.array_equal(o.nnum.numpy(), fx[f't{i}_nnum'])
        assert np.array_equal(o.nnum_nempty.numpy(), fx[f't{i}_nnum_nempty'])
    o = _check([fx['t4_points'], fx['t5_points']], 6, 3, where)
    assert np.array_equal(torch.cat(o.keys).cpu().numpy(), fx['b45_key'])
    assert np.array_equal(torch.cat(o.children).cpu().numpy(), fx['b45_child'])
    assert np.array_equal(torch.cat(o.neighs[1:]).cpu().numpy(), fx['b45_neigh'])


@pytest.mark.parametrize('where', WHERE)
@pytest.mark.parametrize('depth,n,B', [(9, 4096, 5), (7, 30000, 3)])
def test_lidar_clouds(depth, n, B, where):
    g = torch.Generator().manual_seed(11)
    _check([M.lidar_cloud(n, g) for _ in range(B)], depth, where=where)


@pytest.mark.parametrize('where', WHERE)
def test_ragged_and_edge_clouds(where):
    rng = np.random.default_rng(3)
    clouds = [
        np.array([[1.0, 1.0, 1.0], [-1.0, -1.0, -1.0], [-0.0, 0.0, 0.0], [1.0, -1.0, 0.5]], np.float32),
        np.zeros((1, 3), np.float32),                                  # P = 1
        np.full((100, 3), 0.123, np.float32),                          # one leaf
        rng.uniform(-1, 1, size=(5000, 3)).astype(np.float32),         # uniform cube
        np.repeat(rng.uniform(-1, 1, size=(50, 3)).astype(np.float32), 7, 0),   # duplicates
    ]
    _check(clouds, 9, where=where)
    _check(clouds[::-1], 5, where=where)
    _check(clouds[3:4], 3, full_depth=2, where=where)
    _check(clouds[1:3], 4, full_depth=1, where=where)


def test_round_trip_of_a_full_size_native_build():
    """256 x 4096 points at depth 9 (Oxford's evaluation batch): the native octree's own ocnn-layout
    views (keys, children, points, nnum*) imported back give the same octree."""
    from hotformerloc_b200.octree import build_batch, from_ocnn
    g = torch.Generator().manual_seed(21)
    clouds = [M.lidar_cloud(4096, g) for _ in range(256)]
    ref = build_batch(clouds, 9, 2, 'cuda').finalize()
    o = from_ocnn(ref).finalize()
    _assert_same(o, ref, full_neigh=False)


# ---------------------------------------------------------------------------------------------------
# 2. descriptors
# ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('where', WHERE)
@pytest.mark.parametrize('name', ['oxford_b4_stress', 'cswp_b6_stress', 'wp_b3_stress'])
def test_model_outputs_equal_the_native_octree(name, where, tmp_path):
    from hotformerloc_b200.octree import Octree, build_batch
    cfg, depth, spec, seed, mode = CASES[name]
    model, _ = native_model(cfg, case_state_dict(name), tmp_path)
    clouds = case_clouds(name)
    native = build_batch(clouds, depth, 2, 'cuda')
    ocnn = _ocnn(clouds, depth, 2, where)
    y = model({'octree': native})['global']
    assert torch.equal(model({'octree': ocnn})['global'], y)
    y_dbg, inter = model.forward_debug({'octree': ocnn})
    assert torch.equal(y_dbg, y)
    feat = model.get_input_feature(ocnn)
    assert torch.equal(feat.cuda(), model.get_input_feature(native))
    local, relay, oct_n = model.backbone(model.get_input_feature(native), native, depth)
    local_o, relay_o, oct_o = model.backbone(feat, ocnn, depth)
    assert oct_n is native and isinstance(oct_o, Octree) and oct_o is not ocnn
    assert sorted(local_o) == sorted(local) and sorted(relay_o) == sorted(relay)
    for d in local:
        assert torch.equal(local_o[d], local[d]), d
        assert torch.equal(relay_o[d], relay[d]), d
    # the returned octree carries the window tables the backbone used
    assert torch.equal(oct_o.tokens(depth - 3, 192), native.tokens(depth - 3, 192))


# ---------------------------------------------------------------------------------------------------
# 3. malformed input
# ---------------------------------------------------------------------------------------------------
DEPTH = 7


@pytest.fixture(scope='module')
def small():
    g = torch.Generator().manual_seed(43)
    clouds = [M.lidar_cloud(n, g) for n in (3000, 1200, 400)]
    return clouds, _ocnn(clouds, DEPTH)


def _copy(o):
    c = copy.copy(o)
    c.keys = [k.clone() for k in o.keys]
    c.children = [x.clone() for x in o.children]
    c.batch_nnum_nempty = o.batch_nnum_nempty.clone()
    return c


def _nonneg(c):
    return (c >= 0).nonzero().flatten()


def _children_duplicate(o):
    c, j = o.children[5], _nonneg(o.children[5])
    c[j[10]] = c[j[9]]


def _children_out_of_order(o):
    c, j = o.children[DEPTH], _nonneg(o.children[DEPTH])
    c[j[3]], c[j[4]] = int(c[j[4]]), int(c[j[3]])


def _children_below_minus_one(o):
    c = o.children[6]
    c[(c < 0).nonzero().flatten()[0]] = -2


def _children_too_large(o):
    c, j = o.children[4], _nonneg(o.children[4])
    c[j[-1]] = int(o.nnum_nempty[4])


def _children_missing(o):           # one non-empty node fewer than nnum_nempty says
    c, j = o.children[DEPTH], _nonneg(o.children[DEPTH])
    c[j[-1]] = -1


def _children_grid(o):              # d < full_depth: children[d][i] == i
    c = o.children[1]
    c[2], c[3] = 3, 2


def _key_morton_vs_parent(o):
    k = o.keys[6]
    k[1000] = k[1000] ^ (1 << 3)    # a parent bit of the Morton code


def _key_child_position(o):
    k = o.keys[DEPTH]
    k[17] = k[17] ^ 1


def _key_batch_id(o):
    k = o.keys[5]
    k[-1] = (k[-1] & ((1 << 48) - 1)) | (o.batch_size << 48)


def _key_batch_id_full_depth(o):
    k = o.keys[2]
    k[5] = k[5] | (o.batch_size << 48)


def _key_stray_bits(o):
    k = o.keys[DEPTH]
    k[123] = k[123] | (1 << 40)     # between bit 3 * depth and the batch id at bit 48


def _counts_per_submap(o):
    bn = o.batch_nnum_nempty
    bn[5, 0] += 1
    bn[5, 1] -= 1


@pytest.mark.parametrize('breaks, match', [
    (_children_duplicate, 'invariant C .* depth 5'),
    (_children_out_of_order, f'invariant C .* depth {DEPTH}'),
    (_children_below_minus_one, 'invariant C .* depth 6'),
    (_children_too_large, 'invariant C .* depth 4'),
    (_children_missing, f'invariant C .* depth {DEPTH}'),
    (_children_grid, 'invariant C .* depth 1'),
    (_key_morton_vs_parent, 'invariant K .* depth 6'),
    (_key_child_position, f'invariant K .* depth {DEPTH}'),
    (_key_batch_id, 'invariant K .* depth 5'),
    (_key_batch_id_full_depth, 'invariant K .* depth 2'),
    (_key_stray_bits, f'invariant K .* depth {DEPTH}'),
    (_counts_per_submap, r'batch_nnum_nempty\[5\]'),
])
def test_malformed_octree_is_rejected(small, breaks, match):
    from hotformerloc_b200.native import HflError
    from hotformerloc_b200.octree import build_batch, from_ocnn
    clouds, ocnn = small
    bad = _copy(ocnn)
    breaks(bad)
    o = from_ocnn(bad)
    with pytest.raises(HflError, match=match):
        o.finalize()
    with pytest.raises(HflError, match=match):          # and so does every consumer
        o.keys
    # no CUDA error was left behind: a valid import right afterwards is exact
    good = _import(ocnn)
    torch.cuda.synchronize()
    assert torch.equal(torch.cat(good.keys).cpu(), torch.cat(ocnn.keys))
    assert torch.equal(good.ne_table(DEPTH), build_batch(clouds, DEPTH, 2, 'cuda').ne_table(DEPTH))


def test_malformed_octree_is_rejected_by_the_model(small, tmp_path):
    from hotformerloc_b200.native import HflError
    name = 'cswp_b6_stress'
    model, _ = native_model(CASES[name][0], case_state_dict(name), tmp_path)
    bad = _copy(small[1])
    _key_stray_bits(bad)
    with pytest.raises(HflError, match='invariant K'):
        model({'octree': bad})
