"""GPU parity of the relay-token self-attention op (hotformerloc_b200.relay_token_attention,
csrc/rt_attn_train.cu) against float64 torch autograd statements: the core of
oracle.model_ref._attention (-1000 mask) over the padded (B, Nmax) layout of oracle.model_ref.rt_layout,
and oracle.model_ref.rtsa_block for the whole block.  RT counts come from real batches built by the
oracle's octree (oracle.octree_ref), including a submap without RTs and the padding windows (id B)."""
import math

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import model_ref as M
from oracle import octree_ref as R

pytestmark = pytest.mark.gpu

HD = 16


def assert_close(name, a, r):
    err = (a.double() - r).abs()
    tol = 1e-5 + 1e-4 * r.abs()
    worst = (err / tol).max().item() if err.numel() else 0.0
    assert bool((err <= tol).all()), f'{name}: max |err| / (1e-5 + 1e-4 |ref|) = {worst:.3g}'
    return worst


# name: submap sizes, generator seed, octree depth, level depths, K, dilation
BATCHES = {
    'oxford_6': ([4096, 30, 4096, 20, 2000, 3000], 3, 9, (6, 5, 4), 48, 4),
    'oxford_128': ([4096] * 128, 7, 9, (6, 5, 4), 48, 4),
    'one_262k': ([262144], 11, 9, (6, 5, 4), 48, 4),
}
_batches = {}


def batch(name):
    """(layout, padded oracle index (B, Nmax), padded oracle ids (B, Nmax)) of a named batch."""
    if name not in _batches:
        from hotformerloc_b200.relay_token_attention import rt_layout
        sizes, seed, depth, depths, K, dil = BATCHES[name]
        g = torch.Generator().manual_seed(seed)
        o = R.build_batch([M.lidar_cloud(n, g) for n in sizes], depth)
        index, ids = M.rt_layout([M.make_level(o, d, K, dil) for d in depths], o.batch_size)
        layout = rt_layout([o.batch_nnum_nempty[d] for d in depths], K, dil, 'cuda')
        _batches[name] = (layout, index.cuda(), ids.cuda())
    return _batches[name]


def synthetic(lens, seed=0):
    """A layout over one level whose sequences have the given lengths (packed order = level order), ids
    random in {b, B}, and its padded (B, Nmax) index and ids."""
    from hotformerloc_b200.relay_token_attention import RelayTokenLayout
    B = len(lens)
    cu = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    T = int(cu[-1])
    g = torch.Generator().manual_seed(seed)
    owner = np.repeat(np.arange(B), lens)
    ids = np.where(torch.rand(T, generator=g).numpy() < 0.1, B, owner)
    nmax = max(max(lens), 1)
    index = torch.full((B, nmax), -1, dtype=torch.int64)
    ids_pad = torch.full((B, nmax), 10000, dtype=torch.int64)
    for b in range(B):
        index[b, :lens[b]] = torch.arange(cu[b], cu[b + 1])
        ids_pad[b, :lens[b]] = torch.from_numpy(ids[cu[b]:cu[b + 1]])
    d = lambda a: torch.from_numpy(np.asarray(a, dtype=np.int32)).cuda()
    layout = RelayTokenLayout(d(cu), d(ids), d(np.arange(T)), d(np.arange(T)), [np.asarray(lens)], T, max(lens))
    return layout, index.cuda(), ids_pad.cuda()


def core_ref(xp, ids, H):
    """The attention core of _attention (oracle/model_ref.py) from qkv to before proj, on padded
    (B, Nmax, 3C) rows, in xp's dtype and on its device."""
    N, L, C3 = xp.shape
    C = C3 // 3
    q, k, v = xp.view(N, L, 3, H, C // H).permute(2, 0, 3, 1, 4)
    bias = torch.zeros(N, 1, L, L, dtype=xp.dtype, device=xp.device)
    bias = bias.masked_fill((ids.unsqueeze(2) != ids.unsqueeze(1)).unsqueeze(1), -1000.0)
    att = (q @ k.transpose(-1, -2)) * ((C // H) ** -0.5) + bias
    return (att.softmax(-1) @ v).transpose(1, 2).reshape(N, L, C)


def run_ref64(qkv_cat, dout_cat, index, ids_pad, H):
    """float64 statement: rows of the level concatenation -> padded (B, Nmax) by the oracle's index ->
    core -> back to the concatenation's rows, as rtsa_block does."""
    qkv = qkv_cat.double().requires_grad_()
    real = index >= 0
    xp = qkv[index.clamp(min=0)] * real.unsqueeze(-1)
    op = core_ref(xp, ids_pad, H)
    o = torch.zeros(qkv.shape[0], qkv.shape[1] // 3, dtype=torch.float64, device=qkv.device)
    o = o.index_put((index[real],), op[real])
    o.backward(dout_cat.double())
    return o.detach(), qkv.grad


def run_native(qkv_cat, dout_cat, layout, H, ids=None):
    """pack -> relay_token_attention -> unpack on the concatenation's rows; (o, dqkv) in that order."""
    from hotformerloc_b200.relay_token_attention import RelayTokenAttentionFunction
    qkv = qkv_cat.clone().requires_grad_()
    x = layout.pack(list(qkv.split(layout.windows)))
    o = RelayTokenAttentionFunction.apply(x, layout.cu, layout.ids if ids is None else ids, H)
    o = torch.cat(layout.unpack(o))
    o.backward(dout_cat)
    return o.detach(), qkv.grad


def inputs(T, H, seed=0):
    g = torch.Generator(device='cuda').manual_seed(seed)
    return (torch.randn(T, 3 * HD * H, device='cuda', generator=g),
            torch.randn(T, HD * H, device='cuda', generator=g))


CASES = {  # name: batch or synthetic sequence lengths, H
    'oxford_6_H16': ('oxford_6', 16),
    'oxford_6_H8': ('oxford_6', 8),
    'oxford_6_H1': ('oxford_6', 1),
    'oxford_128_H16': ('oxford_128', 16),
    'one_262k_H16': ('one_262k', 16),
    'long_and_empty_H2': ([0, 4096, 0, 0, 37, 0], 2),
}


@pytest.mark.parametrize('case', list(CASES))
def test_matches_float64_statement(case):
    src, H = CASES[case]
    layout, index, ids_pad = batch(src) if isinstance(src, str) else synthetic(src)
    lens = np.diff(layout.cu.cpu().numpy())
    if case == 'oxford_6_H16':
        assert lens.tolist() == [164, 2, 161, 0, 93, 128]
        assert int((layout.ids == layout.batch_size).sum()) > 0, 'expected padding-window RTs'
    if case == 'oxford_128_H16':
        assert layout.total > 20000
    if case == 'one_262k_H16':
        assert layout.max_len > 1800
    assert layout.max_len == index.shape[1]
    qkv, dout = inputs(layout.total, H)
    o, dqkv = run_native(qkv, dout, layout, H)
    ro, rdqkv = run_ref64(qkv, dout, index, ids_pad, H)
    e_o = assert_close('o', o, ro)
    e_q = assert_close('dqkv', dqkv, rdqkv)
    print(f'{case}: T {layout.total}, Nmax {layout.max_len}, max err/tol o {e_o:.3g}, dqkv {e_q:.3g}')


def test_no_relay_tokens():
    from hotformerloc_b200.relay_token_attention import relay_token_attention, rt_layout
    layout = rt_layout([[0, 0], [0, 0], [0, 0]], 48, 4, 'cuda')
    assert layout.total == 0
    qkv = torch.zeros(0, 3 * HD * 4, device='cuda', requires_grad=True)
    o = relay_token_attention(qkv, layout, 4)
    assert o.shape == (0, HD * 4)
    o.sum().backward()
    assert qkv.grad.shape == qkv.shape


def test_deterministic_and_index_dtypes():
    layout, _, _ = batch('oxford_6')
    H = 16
    qkv, dout = inputs(layout.total, H, seed=1)
    o1, q1 = run_native(qkv, dout, layout, H)
    o2, q2 = run_native(qkv, dout, layout, H)
    assert torch.equal(o1, o2) and torch.equal(q1, q2)
    o3, q3 = run_native(qkv, dout, layout, H, ids=layout.ids.long())
    assert torch.equal(o1, o3) and torch.equal(q1, q3)


def test_misaligned_view():
    from hotformerloc_b200.relay_token_attention import relay_token_attention
    layout, _, _ = batch('oxford_6')
    H = 8
    qkv, dout = inputs(layout.total, H, seed=2)
    store = torch.empty(qkv.numel() + 1, device='cuda')
    mis = store[1:].view_as(qkv)
    mis.copy_(qkv)
    assert mis.data_ptr() % 16 and mis.is_contiguous()
    a = relay_token_attention(qkv, layout, H)
    b = relay_token_attention(mis, layout, H)
    assert torch.equal(a, b)


def test_offsets_are_clamped():
    """cu with a decreasing pair and an entry above T: through the C ABI, the sequences are those of the
    sanitised offsets (each entry clamped into [0, T], never below the previous one)."""
    from hotformerloc_b200 import native as N
    T, H = 400, 2
    C = HD * H
    cu = [0, 100, 60, 60, 300, T + 50]
    san = [0, 100, 100, 100, 300, T]
    B = len(cu) - 1
    layout, index, ids_pad = synthetic(list(np.diff(san)), seed=3)
    qkv, dout = inputs(T, H, seed=3)
    L = N.lib()
    nb = int(L.hfl_rt_attn_train_workspace_bytes(T, B, H))
    ws = torch.empty(nb, dtype=torch.uint8, device='cuda')
    cu_d = torch.tensor(cu, dtype=torch.int32, device='cuda')
    o = torch.empty(T, C, device='cuda')
    lse = torch.empty(T, H, device='cuda')
    dqkv = torch.empty(T, 3 * C, device='cuda')
    N.check(L.hfl_rt_attn_train_fwd(N.ptr(qkv), N.ptr(cu_d), N.ptr(layout.ids), 0, B, T, H, N.ptr(o), N.ptr(lse),
                                    N.ptr(ws), nb, N.stream()))
    N.check(L.hfl_rt_attn_train_bwd(N.ptr(qkv), N.ptr(cu_d), N.ptr(layout.ids), 0, N.ptr(o), N.ptr(lse),
                                    N.ptr(dout), B, T, H, N.ptr(dqkv), N.ptr(ws), nb, N.stream()))
    ro, rdqkv = run_ref64(qkv, dout, index, ids_pad, H)
    assert_close('o', o, ro)
    assert_close('dqkv', dqkv, rdqkv)


def test_memory_at_training_scale():
    """The 128-submap Oxford minibatch: peak memory over forward plus backward stays within o, lse, dqkv
    and the workspace, plus 1 MB -- no (B, H, Nmax, Nmax) tensor."""
    from hotformerloc_b200 import native as N
    from hotformerloc_b200.relay_token_attention import relay_token_attention
    layout, _, _ = batch('oxford_128')
    T, H, B = layout.total, 16, layout.batch_size
    C = HD * H
    qkv = torch.randn(T, 3 * C, device='cuda', requires_grad=True)
    dout = torch.randn(T, C, device='cuda')
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    base = torch.cuda.memory_stats()['requested_bytes.all.current']
    torch.cuda.reset_peak_memory_stats()
    out = relay_token_attention(qkv, layout, H)
    out.backward(dout)
    torch.cuda.synchronize()
    peak = torch.cuda.memory_stats()['requested_bytes.all.peak'] - base
    ws = int(N.lib().hfl_rt_attn_train_workspace_bytes(T, B, H))
    allowed = (T * C + T * H + T * 3 * C) * 4 + ws + (1 << 20)
    dense = B * H * layout.max_len ** 2 * 4
    assert peak <= allowed, f'peak {peak / 2**20:.1f} MiB > {allowed / 2**20:.1f} MiB'
    print(f'T {T}: peak {peak / 2**20:.1f} MiB, bound {allowed / 2**20:.1f} MiB, '
          f'one (B, H, Nmax, Nmax) fp32 tensor {dense / 2**20:.1f} MiB')


def block_state_dict(C, prefix):
    shapes = {'norm1.weight': (C,), 'norm1.bias': (C,), 'rt_attention.qkv.weight': (3 * C, C),
              'rt_attention.qkv.bias': (3 * C,), 'rt_attention.proj.weight': (C, C), 'rt_attention.proj.bias': (C,),
              'norm2.weight': (C,), 'norm2.bias': (C,), 'mlp.fc1.weight': (4 * C, C), 'mlp.fc1.bias': (4 * C,),
              'mlp.fc2.weight': (C, 4 * C), 'mlp.fc2.bias': (C,)}
    return M.synthetic_state_dict({prefix + k: v for k, v in shapes.items()}, mode='stress')


def native_block(blk, rts, layout):
    x = layout.pack(rts)
    x = x + blk.rt_attention(blk.norm1(x), layout)
    x = x + blk.mlp.fc2(F.gelu(blk.mlp.fc1(blk.norm2(x))))
    return layout.unpack(x)


def test_block_matches_rtsa_block_and_trains_like_the_statement():
    from hotformerloc_b200.models.hotformerloc import _RTSABlock
    from hotformerloc_b200.relay_token_attention import RTAttention
    layout, index, ids_pad = batch('oxford_6')
    C, H = 256, 16
    prefix = 'backbone.backbone.hotf_stage.rtsa_blocks.3.'
    sd = block_state_dict(C, prefix)
    blk = _RTSABlock(C)
    blk.rt_attention = RTAttention(C, H)
    blk.load_state_dict({k[len(prefix):]: v for k, v in sd.items()})
    blk = blk.cuda()
    g = torch.Generator(device='cuda').manual_seed(6)
    rts = [torch.randn(n, C, device='cuda', generator=g) for n in layout.windows]
    w = [torch.randn(n, C, device='cuda', generator=g) for n in layout.windows]
    scale = 1.0 / math.sqrt(layout.total * C)
    index_c, ids_c = index.cpu(), ids_pad.cpu()

    # forward and gradients against the float64 statement
    sd64 = {k: v.double().requires_grad_() for k, v in sd.items()}
    rts64 = [r.detach().double().cpu().requires_grad_() for r in rts]
    out64 = M.rtsa_block(M._Ctx(sd64, None, None), rts64, prefix[:-1], index_c, ids_c, H)
    (sum((o * wi.double().cpu()).sum() for o, wi in zip(out64, w)) * scale).backward()
    rts_n = [r.clone().requires_grad_() for r in rts]
    out = native_block(blk, rts_n, layout)
    for j, (a, r) in enumerate(zip(out, out64)):
        assert_close(f'block output level {j}', a.detach().cpu(), r.detach())
    (sum((o * wi).sum() for o, wi in zip(out, w)) * scale).backward()
    for j, (a, r) in enumerate(zip(rts_n, rts64)):
        assert_close(f'd rts level {j}', a.grad.cpu(), r.grad)
    for k, p in blk.named_parameters():
        assert_close(f'd {k}', p.grad.cpu(), sd64[prefix + k].grad)

    # one SGD step on the same loss against the fp32 statement
    sd32 = {k: v.clone().requires_grad_() for k, v in sd.items()}
    out32 = M.rtsa_block(M._Ctx(sd32, None, None), [r.cpu() for r in rts], prefix[:-1], index_c, ids_c, H)
    (sum((o * wi.cpu()).sum() for o, wi in zip(out32, w)) * scale).backward()
    opt = torch.optim.SGD(blk.parameters(), lr=0.1)
    opt.step()
    with torch.no_grad():
        for k, p in blk.named_parameters():
            ref = sd32[prefix + k]
            assert_close(f'{k} after one step', p.cpu(), (ref - 0.1 * ref.grad).double())
            assert not torch.equal(p.cpu(), ref), f'{k} did not move'
