"""Device-free checks of the window attention module (hotformerloc_b200.window_attention)."""
import pytest


@pytest.mark.parametrize('dim,patch,heads,dil,use_rpe,hat', [
    (128, 48, 8, 1, True, False),
    (128, 48, 8, 4, True, False),
    (256, 48, 16, 1, True, True),
    (256, 64, 16, 1, True, True),
    (64, 48, 4, 1, False, False),
])
def test_module_builds_without_device_with_reference_parameters(dim, patch, heads, dil, use_rpe, hat):
    from hotformerloc_b200.models.hotformerloc import _Attention
    from hotformerloc_b200.window_attention import OctreeAttention
    m = OctreeAttention(dim, patch, heads, dilation=dil, use_rpe=use_rpe, hat=hat)
    ref = _Attention(dim, patch, heads, dil, use_rpe)
    shapes = {k: tuple(v.shape) for k, v in m.state_dict().items()}
    assert shapes == {k: tuple(v.shape) for k, v in ref.state_dict().items()}
    if use_rpe:
        bnd = int(0.8 * patch * dil ** 0.5)
        assert m.rpe.pos_bnd == bnd and shapes['rpe.rpe_table'] == (3 * (2 * bnd + 1), heads)
    m.load_state_dict(ref.state_dict())


def test_dim_must_be_sixteen_per_head():
    from hotformerloc_b200.window_attention import OctreeAttention
    with pytest.raises(ValueError):
        OctreeAttention(96, 48, 8)


def test_bad_arguments_raise_before_the_device_is_queried():
    import torch
    from hotformerloc_b200.native import HflError
    from hotformerloc_b200.window_attention import window_attention
    qkv = torch.zeros(2, 8, 96)
    xyz = torch.zeros(2, 8, 3, dtype=torch.int64)
    ids = torch.zeros(2, 8, dtype=torch.int64)
    with pytest.raises(HflError):
        window_attention(qkv, xyz, ids, None, 0, False, 2)          # CPU tensors
    with pytest.raises(HflError):
        window_attention(torch.zeros(2, 8, 90), xyz, ids, None, 0, False, 2)   # C != 16 H
