"""Host-side checks of hotformerloc_b200.octree.from_ocnn: a malformed ocnn octree (count relations,
lengths, dtypes, points rows) is rejected before anything touches the device, and an object that is
not an octree is a TypeError naming what it lacks."""
import copy

import numpy as np
import pytest
import torch

from oracle import model_ref as M
from oracle import ocnn_standin as S

DEPTH, FULL = 6, 2


@pytest.fixture(scope='module')
def ocnn_octree():
    g = torch.Generator().manual_seed(41)
    octs = []
    for n in (1500, 700, 40):
        o = S.Octree(DEPTH, FULL)
        o.build_octree(S.Points(torch.from_numpy(M.lidar_cloud(n, g))))
        octs.append(o)
    return S.merge_octrees(octs)


def _copy(o):
    c = copy.copy(o)
    c.keys, c.children, c.points = list(o.keys), list(o.children), list(o.points)
    c.nnum, c.nnum_nempty = o.nnum.clone(), o.nnum_nempty.clone()
    c.batch_nnum_nempty = o.batch_nnum_nempty.clone()
    return c


@pytest.fixture
def no_device(monkeypatch):
    """Any query of the CUDA runtime fails the test: the checks must come first."""
    def touched(*a, **k):
        raise AssertionError('the device was touched before the host-side checks')
    monkeypatch.setattr(torch.cuda, 'is_available', touched)
    monkeypatch.setattr(torch.cuda, 'current_device', touched)
    from hotformerloc_b200 import native as N
    monkeypatch.setattr(N.pinned, 'take', touched)


def _nnum_relation(o):
    o.nnum[DEPTH] += 8                  # d > full_depth: nnum[d] != 8 * nnum_nempty[d-1]


def _nnum_full(o):
    o.nnum[FULL] -= 1                   # nnum[full_depth] != batch * 8^full_depth


def _nempty_below_full(o):
    o.nnum_nempty[1] -= 1               # d < full_depth: every node is non-empty


def _nempty_above_nnum(o):
    o.nnum_nempty[DEPTH] = o.nnum[DEPTH] + 1


def _keys_length(o):
    o.keys[4] = o.keys[4][:-1]


def _children_length(o):
    o.children[DEPTH] = torch.cat([o.children[DEPTH], o.children[DEPTH][:1]])


def _keys_dtype(o):
    o.keys[3] = o.keys[3].to(torch.int32)


def _children_dtype(o):
    o.children[5] = o.children[5].to(torch.int64)


def _points_rows(o):
    o.points[DEPTH] = o.points[DEPTH][:-1]


def _points_dtype(o):
    o.points[DEPTH] = o.points[DEPTH].double()


def _batch_counts_shape(o):
    o.batch_nnum_nempty = o.batch_nnum_nempty[:, :-1]


def _depth_range(o):
    o.depth = 16


def _full_depth_range(o):
    o.full_depth = o.depth


def _batch_size(o):
    o.batch_size = 0


@pytest.mark.parametrize('breaks, match', [
    (_nnum_relation, r'nnum\[d\] == 8 \* nnum_nempty'),
    (_nnum_full, r'batch \* 8\^d'),
    (_nempty_below_full, r'nnum_nempty\[d\] == nnum\[d\]'),
    (_nempty_above_nnum, r'nnum_nempty\[d\] <= nnum\[d\]'),
    (_keys_length, r'keys\[4\]'),
    (_children_length, r'children\[6\]'),
    (_keys_dtype, r'keys\[3\]'),
    (_children_dtype, r'children\[5\]'),
    (_points_rows, r'points\[6\]'),
    (_points_dtype, r'points\[6\]'),
    (_batch_counts_shape, r'batch_nnum_nempty'),
    (_depth_range, r'depth'),
    (_full_depth_range, r'full_depth < depth'),
    (_batch_size, r'batch must be'),
])
def test_host_checks_raise_before_the_device(ocnn_octree, no_device, breaks, match):
    from hotformerloc_b200.native import HflError
    from hotformerloc_b200.octree import from_ocnn
    bad = _copy(ocnn_octree)
    breaks(bad)
    with pytest.raises(HflError, match=match):
        from_ocnn(bad)


def test_not_an_octree_is_a_type_error_naming_what_is_missing(ocnn_octree, tmp_path):
    from hotformerloc_b200.octree import from_ocnn
    bad = _copy(ocnn_octree)
    del bad.children
    del bad.batch_nnum_nempty
    with pytest.raises(TypeError, match='has no children, batch_nnum_nempty'):
        from_ocnn(bad)
    with pytest.raises(TypeError, match='has no depth'):
        from_ocnn(np.zeros(3))
    # the model's public entry points take the same path
    from hotformerloc_b200.config.presets import write_configs
    from hotformerloc_b200.misc.utils import ModelParams
    from hotformerloc_b200.models.model_factory import model_factory
    model = model_factory(ModelParams(write_configs(str(tmp_path), 'oxford')['model_config']))
    with pytest.raises(TypeError, match='has no'):
        model({'octree': object()})
    with pytest.raises(TypeError, match='has no'):
        model.backbone(None, object(), 9)


@pytest.mark.skipif(torch.cuda.is_available(), reason='checks the behaviour without a GPU')
def test_valid_octree_without_cuda_fails_loudly(ocnn_octree):
    from hotformerloc_b200.native import HflError
    from hotformerloc_b200.octree import from_ocnn
    with pytest.raises(HflError, match='GPU only'):
        from_ocnn(ocnn_octree)
