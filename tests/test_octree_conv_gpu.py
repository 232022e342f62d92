"""GPU parity of the training octree convolution (hotformerloc_b200.octree_conv, csrc/octree_conv_train.cu)
against float64 statements on real octree tables of both presets' layer shapes.

Every element is held to (s + 2) 2^-24 sum |terms|, with s the kernel's longest fp32 addition chain into
that element as csrc/octree_conv_train.cu documents it: Cin + K for the forward, Cout + K for the input
gradient and R + 32 + chunks for the weight gradient.  One-defect variants of the float64 statement
(a dropped pair, a pair on the wrong tap, a dropped row chunk, two swapped taps) must break that bound,
which shows it is sharp enough to catch them."""
import json
import math
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import model_ref as M
from oracle import octree_ref as R

pytestmark = pytest.mark.gpu

U = 2.0 ** -24
BB = 'backbone.backbone'

# name: submap sizes, generator seed, octree depth, preset
BATCHES = {
    'oxford_6': ([4096, 30, 4096, 20, 2000, 3000], 3, 9, 'oxford'),
    'cswild_4x30k': ([30000] * 4, 1, 7, 'cs-wild-places'),
    'oxford_128': ([4096] * 128, 7, 9, 'oxford'),
}
# (name, input depth offset from the octree depth, stride, Cin, Cout): the model's layers in order
LAYERS = [('convs.0', 0, 1, 3, 32), ('downsamples.0', 0, 2, 32, 64), ('convs.1', 1, 1, 64, 64),
          ('downsamples.1', 1, 2, 64, 128), ('proj', 2, 1, 128, 128), ('downsample.0', 2, 2, 128, 256),
          ('hotf_down.0', 3, 2, 256, 256), ('hotf_down.1', 4, 2, 256, 256)]
_clouds, _octs = {}, {}


def clouds(name):
    if name not in _clouds:
        sizes, seed, _, _ = BATCHES[name]
        g = torch.Generator().manual_seed(seed)
        _clouds[name] = [M.lidar_cloud(n, g) for n in sizes]
    return _clouds[name]


def octree(name):
    if name not in _octs:
        from hotformerloc_b200.octree import build_batch
        _octs[name] = build_batch(clouds(name), BATCHES[name][2]).finalize()
    return _octs[name]


def table(o, depth, stride):
    return o.ne_table(depth) if stride == 1 else o.child_table(depth)


def wgrad_chunks(n, K, cin, cout):
    """The weight gradient's row partition (wgrad_chunks in csrc/octree_conv_train.cu)."""
    c = min(-(-n // 256), (1 << 25) // (K * cin * cout), 1024)
    return max(c, 1)


def ref64(data, w, neigh, dout):
    """float64 out, ddata, dW and their sum |terms|, per tap."""
    x, W, g = data.double(), w.double(), dout.double()
    n_in, (K, cin, cout) = x.shape[0], W.shape
    out = torch.zeros(neigh.shape[0], cout, dtype=torch.float64, device=x.device)
    out_s, dd, dd_s = torch.zeros_like(out), torch.zeros_like(x), torch.zeros_like(x)
    dw, dw_s = torch.zeros_like(W), torch.zeros_like(W)
    for k in range(K):
        e = neigh[:, k].long()
        m = (e >= 0) & (e < n_in)
        rows, src = m.nonzero()[:, 0], e[m]
        xs = x[src]
        out.index_add_(0, rows, xs @ W[k])
        out_s.index_add_(0, rows, xs.abs() @ W[k].abs())
        dd.index_add_(0, src, g[rows] @ W[k].t())
        dd_s.index_add_(0, src, g[rows].abs() @ W[k].abs().t())
        dw[k] = xs.t() @ g[rows]
        dw_s[k] = xs.abs().t() @ g[rows].abs()
    return out, out_s, dd, dd_s, dw, dw_s


def bounds(neigh, cin, cout):
    n, K = neigh.shape
    c = wgrad_chunks(n, K, cin, cout)
    return cin + K + 2, cout + K + 2, -(-n // c) + 32 + c + 2


def excess(a, r, scale, s):
    """(|a - r|) / (s 2^-24 scale), elementwise; <= 1 is within the bound."""
    return (a.double() - r).abs() / (s * U * scale + 1e-300)


def run_native(data, w, neigh, dout):
    from hotformerloc_b200.octree_conv import octree_conv
    x = data.clone().requires_grad_()
    ww = w.clone().requires_grad_()
    out = octree_conv(x, ww, neigh)
    out.backward(dout)
    return out.detach(), x.grad, ww.grad


def layer_inputs(o, depth, stride, cin, cout, seed):
    neigh = table(o, depth, stride)
    g = torch.Generator(device='cuda').manual_seed(seed)
    n_in = o.n(depth)
    data = torch.randn(n_in, cin, device='cuda', generator=g)
    w = torch.randn(neigh.shape[1], cin, cout, device='cuda', generator=g) / math.sqrt(cin)
    dout = torch.randn(neigh.shape[0], cout, device='cuda', generator=g)
    return data, w, neigh, dout


CASES = [(b, *l) for b in BATCHES for l in LAYERS]


@pytest.mark.parametrize('batch,layer,dd,stride,cin,cout', CASES, ids=[f'{c[0]}-{c[1]}' for c in CASES])
def test_matches_float64(batch, layer, dd, stride, cin, cout):
    o = octree(batch)
    depth = o.depth - dd
    data, w, neigh, dout = layer_inputs(o, depth, stride, cin, cout, seed=dd * 10 + stride)
    out, ddata, dw = run_native(data, w, neigh, dout)
    r_out, s_out, r_dd, s_dd, r_dw, s_dw = ref64(data, w, neigh, dout)
    b_out, b_dd, b_dw = bounds(neigh, cin, cout)
    worst = []
    for name, a, r, s, b in (('out', out, r_out, s_out, b_out), ('ddata', ddata, r_dd, s_dd, b_dd),
                             ('dW', dw, r_dw, s_dw, b_dw)):
        x = excess(a, r, s, b)
        worst.append(x.max().item())
        assert bool((x <= 1).all()), f'{name}: max err / bound = {worst[-1]:.3g}'
    occ = int(((neigh >= 0) & (neigh < data.shape[0])).sum())
    print(f'{batch} {layer} @{depth}: n_out {neigh.shape[0]}, pairs/row {occ / max(neigh.shape[0], 1):.2f}, '
          f'max err/bound out {worst[0]:.3g} ddata {worst[1]:.3g} dW {worst[2]:.3g}')


def _fraction_broken(a, r, s, b, affected):
    x = excess(a, r, s, b)[affected]
    return (x > 1).double().mean().item(), x.numel()


@pytest.mark.parametrize('batch', ['oxford_6', 'cswild_4x30k'])
@pytest.mark.parametrize('layer', ['convs.0', 'proj', 'downsample.0'])
def test_one_defect_breaks_the_bound(batch, layer):
    _, dd, stride, cin, cout = next(l for l in LAYERS if l[0] == layer)
    o = octree(batch)
    depth = o.depth - dd
    data, w, neigh, dout = layer_inputs(o, depth, stride, cin, cout, seed=5)
    out, ddata, dw = run_native(data, w, neigh, dout)
    r_out, s_out, r_dd, s_dd, r_dw, s_dw = ref64(data, w, neigh, dout)
    b_out, b_dd, b_dw = bounds(neigh, cin, cout)
    occ = (neigh >= 0).nonzero()
    K = neigh.shape[1]
    i, k = [int(v) for v in occ[len(occ) // 2]]
    j = int(neigh[i, k])
    wrong = (k + 1) % K
    x64, w64, g64 = data[j].double(), w.double(), dout[i].double()
    # out: drop the pair (i, k), or apply it with tap `wrong`
    for name, delta in (('drop', -(x64 @ w64[k])), ('wrong tap', x64 @ (w64[wrong] - w64[k]))):
        fr, cnt = _fraction_broken(out[i], r_out[i] + delta, s_out[i], b_out, delta.abs() > 0)
        assert fr >= 0.9, f'out, {name}: only {fr:.2f} of {cnt} affected elements break the bound'
    # ddata: the same pair seen from the input row j
    for name, delta in (('drop', -(g64 @ w64[k].t())), ('wrong tap', g64 @ (w64[wrong] - w64[k]).t())):
        fr, cnt = _fraction_broken(ddata[j], r_dd[j] + delta, s_dd[j], b_dd, delta.abs() > 0)
        assert fr >= 0.9, f'ddata, {name}: only {fr:.2f} of {cnt} affected elements break the bound'
    # dW: drop the row chunk holding row i, or swap tap k with another occupied tap
    n = neigh.shape[0]
    c = wgrad_chunks(n, K, cin, cout)
    rows = -(-n // c)
    lo = (i // rows) * rows
    part = neigh[lo:lo + rows]
    _, _, _, _, r_part, _ = ref64(data, w, part, dout[lo:lo + rows])
    hit = (part >= 0).any(0)
    fr, cnt = _fraction_broken(dw[hit], (r_dw - r_part)[hit], s_dw[hit], b_dw, r_part[hit].abs() > 0)
    assert fr >= 0.9, f'dW, dropped chunk: only {fr:.2f} of {cnt} affected elements break the bound'
    counts = (neigh >= 0).sum(0)
    k2 = int(torch.argsort(counts, descending=True)[1]) if int(counts.argmax()) == k else int(counts.argmax())
    swapped = r_dw.clone()
    swapped[[k, k2]] = r_dw[[k2, k]]
    aff = torch.zeros_like(r_dw, dtype=torch.bool)
    aff[[k, k2]] = (r_dw[k] - r_dw[k2]).abs().unsqueeze(0) > 0
    fr, cnt = _fraction_broken(dw, swapped, s_dw, b_dw, aff)
    assert fr >= 0.9, f'dW, swapped taps {k} / {k2}: only {fr:.2f} of {cnt} affected elements break the bound'


@pytest.mark.parametrize('batch', ['oxford_6', 'cswild_4x30k'])
def test_tables_match_get_neigh_and_oracle(batch):
    o = octree(batch)
    r = R.build_batch(clouds(batch), o.depth)
    for d in range(o.full_depth + 1, o.depth + 1):
        assert torch.equal(o.child_table(d).long(), o.get_neigh(d, '222', 2, True))
        assert np.array_equal(o.child_table(d).cpu().numpy(), r.get_neigh(d, '222', 2, nempty=True))
        assert np.array_equal(o.ne_table(d).cpu().numpy(), r.get_neigh(d, '333', 1, nempty=True))


def test_child_table_on_fixture_octree(golden_dir):
    from hotformerloc_b200.octree import build_batch
    fx = np.load(os.path.join(golden_dir, 'octree_fixtures.npz'))
    o = build_batch([fx['t4_points'], fx['t5_points']], 6, 3, 'cuda').finalize()
    for d in range(o.full_depth + 1, o.depth + 1):
        assert torch.equal(o.child_table(d).long(), o.get_neigh(d, '222', 2, True))


@pytest.mark.parametrize('layer', ['convs.1', 'downsamples.1'])
def test_deterministic_and_table_dtypes(layer):
    _, dd, stride, cin, cout = next(l for l in LAYERS if l[0] == layer)
    o = octree('cswild_4x30k')
    data, w, neigh, dout = layer_inputs(o, o.depth - dd, stride, cin, cout, seed=9)
    a = run_native(data, w, neigh, dout)
    b = run_native(data, w, neigh, dout)
    c = run_native(data, w, neigh.long(), dout)
    for x, y, z in zip(a, b, c):
        assert torch.equal(x, y) and torch.equal(x, z)


def test_edge_cases():
    from hotformerloc_b200.native import HflError
    from hotformerloc_b200.octree_conv import octree_conv
    g = torch.Generator(device='cuda').manual_seed(3)
    # n = 0 output rows and n = 0 input rows
    for n_out, n_in in ((0, 50), (0, 0)):
        x = torch.randn(n_in, 16, device='cuda', generator=g, requires_grad=True)
        w = torch.randn(27, 16, 8, device='cuda', generator=g, requires_grad=True)
        y = octree_conv(x, w, torch.empty(n_out, 27, dtype=torch.int32, device='cuda'))
        assert y.shape == (n_out, 8)
        y.sum().backward()
        assert torch.equal(x.grad, torch.zeros_like(x)) and torch.equal(w.grad, torch.zeros_like(w))
    # rows whose taps are all empty (and out-of-range entries) give zeros
    t = torch.randint(0, 300, (200, 27), device='cuda', generator=g, dtype=torch.int64)
    t[torch.rand(200, 27, device='cuda', generator=g) < 0.5] = -1
    t[17] = -1
    t[18] = 300
    x = torch.randn(300, 48, device='cuda', generator=g)
    w = torch.randn(27, 48, 40, device='cuda', generator=g)
    out = octree_conv(x, w, t)
    assert (out[17] == 0).all() and (out[18] == 0).all()
    r_out, s_out, *_ = ref64(x, w, t, torch.zeros(200, 40, device='cuda'))
    assert bool((excess(out, r_out, s_out, 48 + 27 + 2) <= 1).all())
    # Cin = 3 with the input gradient requested: the input-gradient call writes 3 columns
    o = octree('oxford_6')
    data, w3, neigh, dout = layer_inputs(o, o.depth, 1, 3, 32, seed=4)
    out, ddata, dw = run_native(data, w3, neigh, dout)
    _, _, r_dd, s_dd, _, _ = ref64(data, w3, neigh, dout)
    assert ddata.shape == (data.shape[0], 3)
    assert bool((excess(ddata, r_dd, s_dd, 32 + 27 + 2) <= 1).all())
    # a stride-2 table with one child per parent: every input row has exactly one consumer
    n_par = 500
    child = torch.full((n_par, 8), -1, dtype=torch.int32, device='cuda')
    child[torch.arange(n_par, device='cuda'), torch.randint(0, 8, (n_par,), device='cuda', generator=g)] = \
        torch.arange(n_par, dtype=torch.int32, device='cuda')
    x = torch.randn(n_par, 64, device='cuda', generator=g)
    w8 = torch.randn(8, 64, 128, device='cuda', generator=g)
    go = torch.randn(n_par, 128, device='cuda', generator=g)
    out, dx, dw8 = run_native(x, w8, child, go)
    r = ref64(x, w8, child, go)
    for a, rr, s, b in zip((out, dx, dw8), r[0::2], r[1::2], bounds(child, 64, 128)):
        assert bool((excess(a, rr, s, b) <= 1).all())
    # non-contiguous inputs are made contiguous: same bits
    xt = x.t().contiguous().t()
    assert not xt.is_contiguous()
    assert torch.equal(octree_conv(xt, w8, child), out)
    assert torch.equal(octree_conv(x, w8.transpose(1, 2).contiguous().transpose(1, 2), child), out)
    # bad arguments raise before any launch
    with pytest.raises(HflError):
        octree_conv(x.double(), w8, child)
    with pytest.raises(HflError):
        octree_conv(x, w8[:4], child)                              # K mismatch
    with pytest.raises(HflError):
        octree_conv(x, w8, child[:, :4].contiguous())              # K = 4 unsupported
    with pytest.raises(HflError):
        octree_conv(x, w8, child.float())
    with pytest.raises(HflError):
        octree_conv(x.cpu(), w8, child)
    with pytest.raises(HflError):
        octree_conv(x[:, :32].contiguous(), w8, child)             # Cin mismatch


def test_status_codes():
    from hotformerloc_b200 import native as N
    L = N.lib()
    x = torch.randn(10, 8, device='cuda')
    w = torch.randn(27, 8, 8, device='cuda')
    t = torch.zeros(10, 27, dtype=torch.int32, device='cuda')
    out = torch.empty(10, 8, device='cuda')
    with pytest.raises(N.HflError, match='status -1'):
        N.check(L.hfl_octree_conv_train_fwd(N.ptr(x), N.ptr(t), 0, N.ptr(w), 10, 10, 9, 8, 8, N.ptr(out), N.stream()))
    with pytest.raises(N.HflError, match='status -1'):
        N.check(L.hfl_octree_conv_train_fwd(N.ptr(x), N.ptr(t), 0, N.ptr(w), 10, 10, 27, 8, 257, N.ptr(out),
                                            N.stream()))
    N.check(L.hfl_octree_conv_train_fwd(N.ptr(x), N.ptr(t), 0, N.ptr(w), 0, 10, 27, 8, 8, N.ptr(out), N.stream()))
    need = int(L.hfl_octree_conv_train_wgrad_workspace_bytes(10, 27, 8, 8))
    ws = torch.empty(need, dtype=torch.uint8, device='cuda')
    dw = torch.empty(27, 8, 8, device='cuda')
    with pytest.raises(N.HflError, match='status -3'):
        N.check(L.hfl_octree_conv_train_wgrad(N.ptr(x), N.ptr(t), 0, N.ptr(x), 10, 10, 27, 8, 8, N.ptr(dw), N.ptr(ws),
                                              need - 1, N.stream()))
    N.check(L.hfl_octree_conv_train_fwd(N.ptr(x), N.ptr(t), 0, N.ptr(w), 10, 10, 27, 8, 8, N.ptr(out), N.stream()))
    torch.cuda.synchronize()
    assert torch.allclose(out, (x[0] @ w.sum(0)).expand(10, 8), rtol=1e-5, atol=1e-5)   # every tap hits row 0


def test_memory_at_oxford_minibatch_proj():
    """proj of the 128 x 4096 Oxford minibatch: forward + backward stay O(n (Cin + Cout)) -- no
    (n, 27, Cin) gather buffer."""
    from hotformerloc_b200 import native as N
    from hotformerloc_b200.octree_conv import octree_conv
    o = octree('oxford_128')
    depth = o.depth - 2
    neigh = o.ne_table(depth)
    n, cin, cout = neigh.shape[0], 128, 128
    assert n > 500_000
    x = torch.randn(n, cin, device='cuda', requires_grad=True)
    w = torch.randn(27, cin, cout, device='cuda', requires_grad=True)
    dout = torch.randn(n, cout, device='cuda')
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    base = torch.cuda.memory_stats()['requested_bytes.all.current']
    torch.cuda.reset_peak_memory_stats()
    octree_conv(x, w, neigh).backward(dout)
    torch.cuda.synchronize()
    peak = torch.cuda.memory_stats()['requested_bytes.all.peak'] - base
    ws = int(N.lib().hfl_octree_conv_train_wgrad_workspace_bytes(n, 27, cin, cout))
    # out, ddata, the inverse table, W^T, dW and the workspace
    allowed = 4 * (n * cout + n * cin + n * 27 + 2 * 27 * cin * cout) + ws + (1 << 20)
    gather = n * 27 * cin * 4
    assert peak <= allowed, f'peak {peak / 2**20:.1f} MiB > {allowed / 2**20:.1f} MiB'
    print(f'n {n}: peak {peak / 2**20:.1f} MiB, bound {allowed / 2**20:.1f} MiB, gather buffer {gather / 2**30:.2f} GiB')


# --------------------------------------------------------------------------- stem + downsample
def _ln(x, mod_or_sd, p=None):
    return F.layer_norm(x, (x.shape[-1],), mod_or_sd[p + '.weight'], mod_or_sd[p + '.bias'], 1e-5)


def native_stem(mods, x, o, D):
    d = D
    for i in range(2):
        for name in (f'convs.{i}', f'downsamples.{i}'):
            conv, norm = mods[name]
            x = F.relu(norm(conv(x, o, d)))
        d -= 1
    conv, norm = mods['proj']
    x = F.relu(norm(conv(x, o, d)))
    conv, norm = mods['downsample.0']
    return norm(conv(x, o, d))


def oracle_stem(cx, x, D):
    d = D
    for i in range(2):
        x = cx.conv_norm_relu(x, f'{BB}.patch_embed.convs.{i}', d, '333', 1)
        x = cx.conv_norm_relu(x, f'{BB}.patch_embed.downsamples.{i}', d, '222', 2)
        d -= 1
    x = cx.conv_norm_relu(x, f'{BB}.patch_embed.proj', d, '333', 1)
    return cx.downsample(x, f'{BB}.downsample.0', d)


def assert_close(name, a, r):
    err = (a.double() - r).abs()
    tol = 1e-4 * r.abs() + 2e-5 * r.abs().max()
    assert bool((err <= tol).all()), f'{name}: max err / tol = {(err / tol).max().item():.3g}'


def test_stem_and_downsample_match_the_oracle_and_train_like_the_statement(golden_dir):
    from hotformerloc_b200.octree_conv import OctreeConv
    shapes = json.load(open(os.path.join(golden_dir, 'state_shapes_oxford.json')))
    sd = M.synthetic_state_dict(shapes, mode='stress')
    names = {f'convs.{i}': f'{BB}.patch_embed.convs.{i}' for i in range(2)}
    names.update({f'downsamples.{i}': f'{BB}.patch_embed.downsamples.{i}' for i in range(2)})
    names.update({'proj': f'{BB}.patch_embed.proj', 'downsample.0': f'{BB}.downsample.0'})
    sd = {k: v for k, v in sd.items() if any(k.startswith(p + '.') for p in names.values())}
    mods, params = {}, {}
    for short, p in names.items():
        w = sd[p + '.conv.weights']
        down = w.shape[0] == 8
        conv = OctreeConv(w.shape[1], w.shape[2], [2] if down else [3], 2 if down else 1, nempty=True,
                          use_bias=p + '.conv.bias' in sd)
        conv.load_state_dict({k[len(p) + 6:]: v for k, v in sd.items() if k.startswith(p + '.conv.')})
        norm = torch.nn.LayerNorm(w.shape[2])
        norm.load_state_dict({k[len(p) + 6:]: v for k, v in sd.items() if k.startswith(p + '.norm.')})
        mods[short] = (conv.cuda(), norm.cuda())
        for k, v in list(conv.named_parameters()):
            params[f'{p}.conv.{k}'] = v
        for k, v in list(norm.named_parameters()):
            params[f'{p}.norm.{k}'] = v
    assert set(params) == set(sd)
    cl = clouds('oxford_6')
    o = octree('oxford_6')
    r = R.build_batch(cl, o.depth)
    feat = torch.from_numpy(r.input_feature_P())
    out = native_stem(mods, feat.cuda(), o, o.depth)
    g = torch.Generator().manual_seed(11)
    wl = torch.randn(out.shape, generator=g)
    scale = 1.0 / math.sqrt(out.numel())
    (out * wl.cuda()).sum().mul(scale).backward()

    sd64 = {k: v.double().requires_grad_() for k, v in sd.items()}
    out64 = oracle_stem(M._Ctx(sd64, r, None), feat.double(), o.depth)
    (out64 * wl.double()).sum().mul(scale).backward()
    assert_close('output', out.detach().cpu(), out64.detach())
    for k, p in params.items():
        assert_close(f'd {k}', p.grad.cpu(), sd64[k].grad)

    sd32 = {k: v.clone().requires_grad_() for k, v in sd.items()}
    out32 = oracle_stem(M._Ctx(sd32, r, None), feat, o.depth)
    (out32 * wl).sum().mul(scale).backward()
    torch.optim.SGD(list(params.values()), lr=0.1).step()
    with torch.no_grad():
        for k, p in params.items():
            ref = sd32[k]
            assert_close(f'{k} after one step', p.cpu(), (ref - 0.1 * ref.grad).double())
            assert not torch.equal(p.cpu(), ref), f'{k} did not move'
