"""Device-free checks of the dwconv drop-in (hotformerloc_b200.dwconv)."""
from oracle import octree_ref as R


def test_lut_kernel_matches_ocnn():
    from hotformerloc_b200.octree import LUT_KERNEL
    assert LUT_KERNEL == R.LUT_KERNEL


def test_dwconv_module_imports_without_device():
    from hotformerloc_b200 import dwconv
    m = dwconv.OctreeDWConv(8, [3, 1, 3], nempty=True, use_bias=True)
    assert m.kernel == '313' and m.kdim == 9
    assert {k: tuple(v.shape) for k, v in m.state_dict().items()} == {'weights': (9, 1, 8), 'bias': (8,)}
