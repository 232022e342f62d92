"""GPU parity of the dwconv drop-in (hotformerloc_b200.dwconv, csrc/dwconv.cu) against the pure-torch
statement of ocnn.nn.OctreeDWConv (oracle.ocnn_standin), following the reference's own test recipe
(libs/dwconv/test/test_octree_dwconv.py: 8 kernel shapes x nempty, depth 4, C = 256, batch octree of
fixtures 4 and 5) plus edge shapes, int32 / int64 tables and a training-sized batch."""
import os

import numpy as np
import pytest
import torch

from oracle import model_ref as M
from oracle import ocnn_standin as S

pytestmark = pytest.mark.gpu

KERNELS = ['333', '222', '311', '131', '113', '331', '313', '133']


@pytest.fixture(scope='module')
def fixture_octree(golden_dir):
    from hotformerloc_b200.octree import build_batch
    fx = np.load(os.path.join(golden_dir, 'octree_fixtures.npz'))
    return build_batch([fx['t4_points'], fx['t5_points']], 6, 3, 'cuda').finalize()


def np_inverse(t: np.ndarray, n_data: int) -> np.ndarray:
    """ineigh[t[i,k], k] = i (largest i where several rows hit), -1 elsewhere."""
    out = np.full((n_data, t.shape[1]), -1, t.dtype)
    i, k = np.nonzero((t >= 0) & (t < n_data))
    np.maximum.at(out, (t[i, k], k), i.astype(t.dtype))
    return out


def random_table(n_out, n_in, K, g, empty=0.4, dtype=torch.int64):
    """Each column hits a data row at most once, as in an octree table (n_out <= n_in)."""
    t = torch.stack([torch.randperm(n_in, generator=g)[:n_out] for _ in range(K)], 1)
    t[torch.rand(n_out, K, generator=g) < empty] = -1
    return t.to(dtype).cuda()


def ref64(data, w, neigh):
    """fp64 forward and the per-element scale sum_k |w data|."""
    d, wk = data.double(), w.double()[:, 0, :]
    out = torch.zeros(neigh.shape[0], data.shape[1], dtype=torch.float64, device=data.device)
    scale = torch.zeros_like(out)
    for k in range(neigh.shape[1]):
        e = neigh[:, k].long()
        m = e >= 0
        p = d[e.clamp(min=0)] * wk[k] * m[:, None]
        out += p
        scale += p.abs()
    return out, scale


def wgrad64(grad, data, neigh):
    g, d = grad.double(), data.double()
    dw, scale = [], []
    for k in range(neigh.shape[1]):
        e = neigh[:, k].long()
        p = g * d[e.clamp(min=0)] * (e >= 0)[:, None]
        dw.append(p.sum(0))
        scale.append(p.abs().sum(0))
    return torch.stack(dw)[:, None, :], torch.stack(scale)[:, None, :]


# --------------------------------------------------------------------------- reference recipe
@pytest.mark.parametrize('nempty', [True, False])
@pytest.mark.parametrize('kernel', KERNELS)
def test_reference_recipe(fixture_octree, kernel, nempty):
    from hotformerloc_b200 import dwconv as D
    octree, depth, C = fixture_octree, 4, 256
    torch.manual_seed(0)
    nnum = int(octree.nnum_nempty[depth] if nempty else octree.nnum[depth])
    kernel_size = [int(c) for c in kernel]
    ref = S.OctreeDWConv(C, kernel_size, 1, nempty).cuda()
    mod = D.OctreeDWConv(C, kernel_size, nempty).cuda()
    mod.load_state_dict(ref.state_dict())
    data = torch.rand(nnum, C, device='cuda')
    grad = torch.rand(nnum, C, device='cuda')
    neigh = octree.get_neigh(depth, kernel, 1, nempty)
    assert neigh.dtype == torch.int64 and neigh.shape == (nnum, ref.kdim)

    data_ref = data.clone().requires_grad_()
    out_ref = ref(data_ref, octree, depth)
    out_ref.backward(grad)

    w = mod.weights.detach()
    out = D.dwconv_forward_backward(data, w, neigh)
    assert torch.allclose(out, out_ref.detach(), atol=1e-6)
    ineigh = D.inverse_neigh(neigh)
    assert np.array_equal(ineigh.cpu().numpy(), np_inverse(neigh.cpu().numpy(), nnum))
    grad_d = D.dwconv_forward_backward(grad, w, ineigh)
    assert torch.allclose(grad_d, data_ref.grad, atol=1e-6)
    grad_w = D.dwconv_weight_backward(grad, data, neigh)
    assert grad_w.shape == ref.weights.shape
    assert torch.allclose(grad_w, ref.weights.grad, atol=5e-5)

    # the autograd function
    d1 = data.clone().requires_grad_()
    w1 = w.clone().requires_grad_()
    out1 = D.octree_dwconv(d1, w1, neigh)
    out1.backward(grad)
    assert torch.equal(out1.detach(), out)
    assert torch.equal(d1.grad, grad_d) and torch.equal(w1.grad, grad_w)

    # the module
    d2 = data.clone().requires_grad_()
    out2 = mod(d2, octree, depth)
    out2.backward(grad)
    assert torch.allclose(out2.detach(), out_ref.detach(), atol=1e-6)
    assert torch.allclose(d2.grad, data_ref.grad, atol=1e-6)
    assert torch.allclose(mod.weights.grad, ref.weights.grad, atol=5e-5)


# --------------------------------------------------------------------------- inverse table
def test_inverse_is_the_mirror_of_real_333_tables(fixture_octree):
    from hotformerloc_b200 import dwconv as D
    o = fixture_octree
    tables = [o.ne_table(d) for d in range(o.full_depth, o.depth + 1)]
    tables += [o.neighs[d] for d in range(1, o.depth + 1)]
    for t in tables:
        inv = D.inverse_neigh(t)
        assert inv.dtype == t.dtype and inv.shape == t.shape
        assert np.array_equal(inv.cpu().numpy(), np_inverse(t.cpu().numpy(), t.shape[0]))
        # the neighbour at offset d sees this node at offset -d
        assert torch.equal(inv, t.flip(1))


@pytest.mark.parametrize('dtype', [torch.int32, torch.int64])
def test_inverse_of_malformed_table_keeps_largest_row(dtype):
    from hotformerloc_b200 import dwconv as D
    g = torch.Generator().manual_seed(4)
    t = random_table(5000, 5000, 27, g, empty=0.2, dtype=dtype)
    t[:, 3] = 7                                  # every row hits (7, 3)
    inv = D.inverse_neigh(t)
    assert np.array_equal(inv.cpu().numpy(), np_inverse(t.cpu().numpy(), 5000))
    assert int(inv[7, 3]) == 4999


# --------------------------------------------------------------------------- dtype independence
def test_int32_and_int64_tables_bitwise_equal(fixture_octree):
    from hotformerloc_b200 import dwconv as D
    o = fixture_octree
    t32 = o.ne_table(o.depth)
    t64 = t32.long()
    n, C = t32.shape[0], 96
    torch.manual_seed(1)
    data, grad = torch.randn(n, C, device='cuda'), torch.randn(n, C, device='cuda')
    w = torch.randn(27, 1, C, device='cuda')
    outs = []
    for t in (t32, t64):
        d = data.clone().requires_grad_()
        ww = w.clone().requires_grad_()
        y = D.octree_dwconv(d, ww, t)
        y.backward(grad)
        outs.append((y.detach(), d.grad, ww.grad, D.inverse_neigh(t).long()))
    for a, b in zip(*outs):
        assert torch.equal(a, b)


# --------------------------------------------------------------------------- edge shapes
@pytest.mark.parametrize('C', [1, 3, 32, 96, 128, 256])
@pytest.mark.parametrize('K', [1, 3, 8, 9, 27])
def test_edge_shapes(C, K):
    from hotformerloc_b200 import dwconv as D
    g = torch.Generator().manual_seed(100 * K + C)
    n_in, n_out = 1000, 777
    t = random_table(n_out, n_in, K, g)
    t[5] = -1                                    # a row without neighbours
    data = torch.randn(n_in, C, generator=g).cuda()
    grad = torch.randn(n_out, C, generator=g).cuda()
    w = torch.randn(K, 1, C, generator=g).cuda()
    out = D.dwconv_forward_backward(data, w, t)
    ref, scale = ref64(data, w, t)
    assert (out[5] == 0).all()
    assert ((out.double() - ref).abs() <= 1e-5 * scale + 1e-30).all()
    # a 4-byte misaligned copy of the operands takes the scalar path: same order, same bits
    buf = torch.empty(n_in * C + 1, device='cuda')
    data_u = buf[1:].view(n_in, C)
    data_u.copy_(data)
    assert torch.equal(D.dwconv_forward_backward(data_u, w, t), out)
    dw = D.dwconv_weight_backward(grad, data, t)
    ref_w, scale_w = wgrad64(grad, data, t)
    assert ((dw.double() - ref_w).abs() <= 1e-5 * scale_w + 1e-30).all()
    assert torch.allclose(D.dwconv_weight_backward(grad, data_u, t), dw, rtol=1e-6, atol=1e-6)
    # input gradient with n_out != n_in through the autograd function
    d = data.clone().requires_grad_()
    D.octree_dwconv(d, w, t).backward(grad)
    gi = torch.zeros(n_in, C, dtype=torch.float64, device='cuda')
    gs = torch.zeros_like(gi)
    for k in range(K):
        m = t[:, k] >= 0
        p = grad.double()[m] * w.double()[k, 0]
        gi.index_add_(0, t[m, k].long(), p)
        gs.index_add_(0, t[m, k].long(), p.abs())
    assert ((d.grad.double() - gi).abs() <= 1e-5 * gs + 1e-30).all()


def test_empty_and_all_empty_rows():
    from hotformerloc_b200 import dwconv as D
    C, K = 64, 27
    data = torch.randn(10, C, device='cuda')
    w = torch.randn(K, 1, C, device='cuda')
    t0 = torch.empty(0, K, dtype=torch.int64, device='cuda')
    assert D.dwconv_forward_backward(data, w, t0).shape == (0, C)
    assert D.inverse_neigh(t0).shape == (0, K)
    assert torch.equal(D.dwconv_weight_backward(torch.empty(0, C, device='cuda'), data, t0),
                       torch.zeros(K, 1, C, device='cuda'))
    tm = torch.full((50, K), -1, dtype=torch.int32, device='cuda')
    assert torch.equal(D.dwconv_forward_backward(data, w, tm), torch.zeros(50, C, device='cuda'))
    assert torch.equal(D.inverse_neigh(tm), tm)
    assert torch.equal(D.dwconv_weight_backward(torch.randn(50, C, device='cuda'), data, tm),
                       torch.zeros(K, 1, C, device='cuda'))


def test_bad_arguments_raise():
    from hotformerloc_b200 import dwconv as D
    from hotformerloc_b200 import native as N
    from hotformerloc_b200.native import HflError
    n, C, K = 100, 32, 27
    g = torch.Generator().manual_seed(2)
    t = random_table(n, n, K, g)
    data = torch.randn(n, C, device='cuda')
    w = torch.randn(K, 1, C, device='cuda')
    with pytest.raises(HflError):
        D.dwconv_forward_backward(data.t().contiguous().t(), w, t)       # non-contiguous
    with pytest.raises(HflError):
        D.dwconv_forward_backward(data[:, ::2], w[:, :, ::2], t)
    with pytest.raises(HflError):
        D.dwconv_forward_backward(data.double(), w.double(), t)          # wrong dtype
    with pytest.raises(HflError):
        D.dwconv_forward_backward(data, w, t.float())
    with pytest.raises(HflError):
        D.dwconv_forward_backward(data, w[:8], t)                        # K mismatch
    with pytest.raises(HflError):
        D.dwconv_forward_backward(data.cpu(), w, t)
    with pytest.raises(HflError):
        D.inverse_neigh(t[:, ::2])
    with pytest.raises(HflError):
        D.dwconv_weight_backward(data[:50].contiguous(), data, t)        # grad rows != table rows
    # an undersized workspace is reported, not overrun
    L = N.lib()
    need = int(L.hfl_dwconv_wgrad_workspace_bytes(n, K, C))
    assert need > 0
    ws = torch.empty(need, dtype=torch.uint8, device='cuda')
    dw = torch.empty(K, 1, C, device='cuda')
    with pytest.raises(HflError, match='status -3'):
        N.check(L.hfl_dwconv_wgrad(N.ptr(data), N.ptr(data), N.ptr(t), 1, n, n, K, C, N.ptr(dw), N.ptr(ws),
                                   need - 1, N.stream()))
    with pytest.raises(HflError, match='status -1'):
        N.check(L.hfl_dwconv(N.ptr(data), N.ptr(t), 1, N.ptr(w), n, n, 28, C, N.ptr(data), N.stream()))


# --------------------------------------------------------------------------- training scale
@pytest.fixture(scope='module')
def oxford_batch():
    from hotformerloc_b200.octree import build_batch
    g = torch.Generator().manual_seed(7)
    clouds = [M.lidar_cloud(4096, g) for _ in range(128)]      # batch_split_size of the training cfg
    return build_batch(clouds, 9).finalize()


def test_training_scale(oxford_batch):
    from hotformerloc_b200 import dwconv as D
    t = oxford_batch.ne_table(7)
    n, C = t.shape[0], 128
    assert n >= 500_000
    torch.manual_seed(3)
    data, grad = torch.randn(n, C, device='cuda'), torch.randn(n, C, device='cuda')
    w = torch.randn(27, 1, C, device='cuda')
    t64 = t.long()
    out = D.dwconv_forward_backward(data, w, t64)
    ref, scale = ref64(data, w, t64)
    assert ((out.double() - ref).abs() <= 1e-5 * scale + 1e-30).all()
    del ref, scale
    # input gradient: the forward over the inverse table; the fp64 statement scatters through t
    gd = D.dwconv_forward_backward(grad, w, D.inverse_neigh(t64))
    gi = torch.zeros(n, C, dtype=torch.float64, device='cuda')
    gs = torch.zeros_like(gi)
    for k in range(27):
        m = t64[:, k] >= 0
        p = grad.double()[m] * w.double()[k, 0]
        gi.index_add_(0, t64[m, k], p)
        gs.index_add_(0, t64[m, k], p.abs())
    assert ((gd.double() - gi).abs() <= 1e-5 * gs + 1e-30).all()
    del gi, gs
    dw = D.dwconv_weight_backward(grad, data, t64)
    ref_w, scale_w = wgrad64(grad, data, t64)
    assert ((dw.double() - ref_w).abs() <= 1e-4 * scale_w + 1e-30).all()
    assert torch.equal(D.dwconv_weight_backward(grad, data, t64), dw)      # deterministic
    assert torch.equal(D.dwconv_weight_backward(grad, data, t), dw)        # int32 table, same bits


# --------------------------------------------------------------------------- module round trip
@pytest.mark.parametrize('use_bias', [False, True])
def test_module_state_dict_round_trip(fixture_octree, use_bias):
    from hotformerloc_b200 import dwconv as D
    octree, depth, C = fixture_octree, 5, 64
    torch.manual_seed(5)
    mine = D.OctreeDWConv(C, [3], nempty=True, use_bias=use_bias).cuda()
    if use_bias:
        with torch.no_grad():
            mine.bias.uniform_(-1, 1)
    ref = S.OctreeDWConv(C, [3], 1, True, use_bias).cuda()
    assert set(ref.state_dict()) == set(mine.state_dict())
    ref.load_state_dict(mine.state_dict())
    data = torch.randn(octree.n(depth), C, device='cuda')
    with torch.no_grad():
        assert torch.allclose(mine(data, octree, depth), ref(data, octree, depth), atol=1e-5)
    other = D.OctreeDWConv(C, [3], nempty=True, use_bias=use_bias).cuda()
    other.load_state_dict(ref.state_dict())
    with torch.no_grad():
        assert torch.equal(other(data, octree, depth), mine(data, octree, depth))
