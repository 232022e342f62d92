"""CPU tests of the differentiable forward's interface and of the oracle's autograd entry
(tests/oracle_autograd.py: oracle.model_ref.forward with autograd): the entry's fp32 result equals
oracle.model_ref.forward bit for bit and its float64 result reproduces the reference goldens; the ``differentiable`` flag defaults to False and leaves the state_dict
alone; the unimplemented cases raise NotImplementedError naming the config key; a CPU model has no
differentiable path."""
import json
import os
import re

import numpy as np
import pytest
import torch

from oracle import model_ref as M
from oracle import octree_ref as R
from oracle.make_golden import CASES
from tests import oracle_autograd as A
from tests.common import case_clouds, case_state_dict


def _model(cfg, tmp_path, **overrides):
    from hotformerloc_b200.config.presets import write_configs
    from hotformerloc_b200.misc.utils import ModelParams
    from hotformerloc_b200.models.model_factory import model_factory
    paths = write_configs(str(tmp_path), cfg)
    text = open(paths['model_config']).read()
    for k, v in overrides.items():
        text = re.sub(rf'{k}=.*', f'{k}={v}', text) if f'{k}=' in text else text + f'{k}={v}\n'
    open(paths['model_config'], 'w').write(text)
    return model_factory(ModelParams(paths['model_config'])), paths


@pytest.mark.parametrize('cfg', ['oxford', 'wild-places'])
def test_autograd_entry_fp32_equals_forward_bitwise(cfg, tmp_path):
    model, paths = _model(cfg, tmp_path, num_blocks='2,2')
    shapes = {k: tuple(v.shape) for k, v in model.state_dict().items()}
    sd = M.synthetic_state_dict(shapes, mode='stress')
    hp = M.HParams.from_cfg(paths['model_config'])
    g = torch.Generator().manual_seed(3)
    clouds = [M.lidar_cloud(2000, g) for _ in range(2)]
    if cfg == 'wild-places':
        from hotformerloc_b200.datasets.coordinate_utils import cylindrical_for_octree
        clouds = [cylindrical_for_octree(c) for c in clouds]
    o = R.build_batch(clouds, 9 if cfg == 'oxford' else 7)
    y = M.forward(sd, o, hp)
    z = A.forward_autograd(sd, o, hp)
    assert z.dtype == torch.float32 and torch.equal(y, z.detach())


def test_autograd_entry_float64_reproduces_reference_golden(golden_dir, tmp_path):
    name = 'oxford_b1_init'
    cfg, depth, *_ = CASES[name]
    from hotformerloc_b200.config.presets import write_configs
    hp = M.HParams.from_cfg(write_configs(str(tmp_path), cfg)['model_config'])
    sd = {k: v.double().requires_grad_(v.is_floating_point()) for k, v in case_state_dict(name).items()}
    y = A.forward_autograd(sd, R.build_batch(case_clouds(name), depth), hp)
    assert y.dtype == torch.float64 and y.grad_fn is not None
    ref = np.load(os.path.join(golden_dir, 'descriptors.npz'))[name + '_reference']
    assert np.abs(y.detach().numpy() - ref).max() < 1e-5


def test_flag_defaults_off_and_keeps_state_dict(tmp_path):
    model, _ = _model('oxford', tmp_path)
    keys = list(model.state_dict())
    assert model.differentiable is False and model.backbone.differentiable is False
    model.differentiable = True
    assert model.backbone.differentiable is True                     # one source of truth
    assert list(model.state_dict()) == keys
    model.backbone.differentiable = False
    assert model.differentiable is False
    shapes = json.load(open(os.path.join(os.path.dirname(__file__), 'golden', 'state_shapes_oxford.json')))
    assert set(keys) == set(shapes)


def test_pyramid_gem_is_refused(tmp_path):
    model, _ = _model('oxford', tmp_path, pooling='PyramidOctGeM')
    model.eval().differentiable = True
    with pytest.raises(NotImplementedError, match='pooling'):
        model({'octree': None})


def test_training_with_drop_path_is_refused(tmp_path):
    model, _ = _model('oxford', tmp_path)
    assert model.backbone.drop_path > 0                              # the default of the [MODEL] section
    model.train().differentiable = True
    with pytest.raises(NotImplementedError, match='drop_path'):
        model({'octree': None})
    with pytest.raises(NotImplementedError, match='drop_path'):
        model.backbone(None, None, 9)


def test_cpu_model_has_no_differentiable_path(tmp_path):
    from hotformerloc_b200.native import HflError
    model, _ = _model('oxford', tmp_path, drop_path=0)
    model.train().differentiable = True                              # drop_path = 0 may train
    with pytest.raises(HflError, match='GPU'):
        model({'octree': None})
    with pytest.raises(HflError, match='GPU'):
        model.backbone(None, None, 9)
