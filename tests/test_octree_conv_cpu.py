"""Device-free checks of the octree convolution module (hotformerloc_b200.octree_conv): ocnn's constructor,
the parameter names and shapes a checkpoint's ``*.conv.*`` tensors load into, and the shapes it refuses."""
import pytest
import torch

from hotformerloc_b200.octree_conv import OctreeConv

BB = 'backbone.backbone'
# preset -> (module prefix, OctreeConv arguments)
LAYERS = [
    (f'{BB}.patch_embed.convs.0', dict(kernel_size=[3], stride=1, use_bias=False)),
    (f'{BB}.patch_embed.downsamples.1', dict(kernel_size=[2], stride=2, use_bias=False)),
    (f'{BB}.patch_embed.proj', dict(kernel_size=[3], stride=1, use_bias=False)),
    (f'{BB}.downsample.0', dict(kernel_size=[2], stride=2, use_bias=True)),
    (f'{BB}.hotf_stage.downsamples.0', dict(kernel_size=[2], stride=2, use_bias=True)),
]


@pytest.fixture(scope='module', params=['oxford', 'cs-wild-places'])
def preset_state(request, tmp_path_factory):
    from hotformerloc_b200.config.presets import write_configs
    from hotformerloc_b200.misc.utils import ModelParams
    from hotformerloc_b200.models.model_factory import model_factory
    paths = write_configs(str(tmp_path_factory.mktemp(request.param)), request.param)
    torch.manual_seed(0)
    return model_factory(ModelParams(paths['model_config'])).state_dict()


@pytest.mark.parametrize('prefix,kw', LAYERS, ids=[p.split('.', 2)[2] for p, _ in LAYERS])
def test_checkpoint_tensors_load(preset_state, prefix, kw):
    w = preset_state[prefix + '.conv.weights']
    kdim, cin, cout = w.shape
    conv = OctreeConv(cin, cout, nempty=True, **kw)
    assert conv.kdim == kdim == (27 if kw['stride'] == 1 else 8)
    sub = {k[len(prefix) + 6:]: v for k, v in preset_state.items() if k.startswith(prefix + '.conv.')}
    assert set(sub) == set(conv.state_dict())
    conv.load_state_dict(sub)
    assert torch.equal(conv.weights, w)
    if kw['use_bias']:
        assert torch.equal(conv.bias, preset_state[prefix + '.conv.bias'])


def test_ocnn_constructor_and_defaults():
    conv = OctreeConv(3, 32, [3], 1, True, direct_method=True, use_bias=False, max_buffer=1)
    assert conv.weights.shape == (27, 3, 32) and not hasattr(conv, 'bias')
    assert conv.weights.abs().max() > 0                       # xavier-uniform, not zeros
    down = OctreeConv(256, 256, kernel_size=[2], stride=2, nempty=True, use_bias=True)
    assert down.weights.shape == (8, 256, 256) and down.bias.shape == (256,)
    assert [n for n, _ in down.named_parameters()] == ['weights', 'bias']
    assert 'stride=2' in repr(down)


@pytest.mark.parametrize('kw', [
    dict(kernel_size=[3], stride=1, nempty=False),            # ocnn's default nempty
    dict(kernel_size=[2], stride=2, nempty=False),
    dict(kernel_size=[3], stride=2, nempty=True),
    dict(kernel_size=[2], stride=1, nempty=True),
    dict(kernel_size=[3, 3, 1], stride=1, nempty=True),
    dict(kernel_size=[1], stride=1, nempty=True),
    dict(kernel_size=[5], stride=1, nempty=True),
])
def test_unsupported_shapes_raise(kw):
    with pytest.raises(ValueError):
        OctreeConv(32, 32, **kw)


@pytest.mark.parametrize('cin,cout', [(0, 32), (32, 0), (257, 32), (32, 512)])
def test_unsupported_widths_raise(cin, cout):
    with pytest.raises(ValueError):
        OctreeConv(cin, cout, [3], 1, nempty=True)
