"""GPU parity of the attention-pooling head (hotformerloc_b200.attention_pool, csrc/attn_pool_train.cu) against
a float64 torch autograd statement of the per-segment loop of oracle.model_ref.attn_pool_mixer.  The segment
counts are the batch_nnum_nempty rows of real batches (depths 6, 5 and 4 of depth-9 octrees, the pyramid levels
of the Oxford cfg); the edge cases are built from them."""
import math
import tempfile
from types import SimpleNamespace

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import model_ref as M

pytestmark = pytest.mark.gpu


def pool_ref(x, counts, query):
    """The per-segment loop of attn_pool_mixer in x's dtype: softmax(C^-0.5 q seg^T) seg per segment."""
    outs = []
    for seg in x.split([int(c) for c in counts]):
        att = (query @ seg.t()) * (query.shape[1] ** -0.5)
        outs.append(att.softmax(-1) @ seg)
    return torch.stack(outs)


def assert_close(name, a, r):
    err = (a.double() - r).abs()
    tol = 1e-5 + 1e-4 * r.abs()
    worst = (err / tol).max().item() if err.numel() else 0.0
    assert bool((err <= tol).all()), f'{name}: max |err| / (1e-5 + 1e-4 |ref|) = {worst:.3g}'
    return worst


def assert_maxabs_close(name, a, r, rel=1e-4):
    err = (a.double() - r).abs().max().item()
    bound = rel * r.abs().max().item()
    assert err <= bound, f'{name}: max-abs err {err:.3g} > {rel:g} max|ref| = {bound:.3g}'
    return err / max(r.abs().max().item(), 1e-300)


@pytest.fixture(scope='module')
def mixed():
    """Oxford-cfg depth-9 batch with 30- and 20-point submaps (the window-attention tests' mixed batch)."""
    from hotformerloc_b200.octree import build_batch
    g = torch.Generator().manual_seed(3)
    sizes = [4096, 30, 4096, 20, 2000, 3000]
    return build_batch([M.lidar_cloud(n, g) for n in sizes], 9).finalize()


@pytest.fixture(scope='module')
def oxford128():
    """One Oxford training minibatch: batch_split_size = 128 submaps of 4096 points."""
    from hotformerloc_b200.octree import build_batch
    g = torch.Generator().manual_seed(7)
    return build_batch([M.lidar_cloud(4096, g) for _ in range(128)], 9).finalize()


def level_counts(o, d):
    return [int(c) for c in o.batch_nnum_nempty[d]]


def edge_counts(name, mixed, oxford128):
    c6, c4 = level_counts(mixed, 6), level_counts(mixed, 4)
    if name == 'empty_segments':                 # empty submaps first, between and last
        return [0] + [v for c in c4 for v in (c, 0, 0)]
    if name == 'one_token_segments':
        return [1, 1] + c4 + [1, 0, 1]
    if name == 'long_segment':                    # one segment of >= 20 000 tokens: many chunks
        o6 = level_counts(oxford128, 6)
        m = int(np.searchsorted(np.cumsum(o6), 20000)) + 1     # the first m submaps' tokens as one segment
        return [o6[m], sum(o6[:m]), 3]
    if name == 'B1':
        return [c6[0]]
    if name == 'B1500':                           # more segments than one round of the plan's block scan
        return [c4[i % len(c4)] if i % 7 == 0 else (i % 5 if i % 3 else 0) for i in range(1500)]
    raise KeyError(name)


# name: (batch, depth or edge case, k, C)
CASES = {
    'oxford_l0_k74': ('mixed', 6, 74, 256),
    'oxford_l1_k36': ('mixed', 5, 36, 256),
    'oxford_l2_k18': ('mixed', 4, 18, 256),
    'k148_l0': ('mixed', 6, 148, 256),
    'k72_l1': ('mixed', 5, 72, 256),
    'k36_l2': ('mixed', 4, 36, 256),
    'minibatch128_l0_k74': ('oxford128', 6, 74, 256),
    'minibatch128_l0_k148': ('oxford128', 6, 148, 256),
    'k1': ('mixed', 6, 1, 256),
    'C128': ('mixed', 5, 36, 128),
    'C32_k256': ('mixed', 4, 256, 32),
    'C96_k5': ('mixed', 5, 5, 96),
    'C512_k40': ('mixed', 5, 40, 512),
    'B1': ('edge', 'B1', 74, 256),
    'empty_segments': ('edge', 'empty_segments', 18, 256),
    'one_token_segments': ('edge', 'one_token_segments', 36, 256),
    'long_segment': ('edge', 'long_segment', 74, 256),
    'B1500': ('edge', 'B1500', 18, 256),
}


def make_inputs(case, mixed, oxford128, seed=0):
    src, d, k, C = CASES[case]
    if src == 'edge':
        counts = edge_counts(d, mixed, oxford128)
    else:
        counts = level_counts(mixed if src == 'mixed' else oxford128, d)
    n, B = sum(counts), len(counts)
    g = torch.Generator(device='cuda').manual_seed(seed)
    x = torch.randn(n, C, device='cuda', generator=g)
    query = torch.randn(k, C, device='cuda', generator=g)
    dout = torch.randn(B, k, C, device='cuda', generator=g)
    return dict(x=x, query=query, counts=counts, dout=dout)


def run_native(a):
    from hotformerloc_b200.attention_pool import attention_pool
    x = a['x'].clone().requires_grad_()
    q = a['query'].clone().requires_grad_()
    out = attention_pool(x, a['counts'], q)
    out.backward(a['dout'])
    return out.detach(), x.grad, q.grad


def run_ref64(a):
    x = a['x'].double().requires_grad_()
    q = a['query'].double().requires_grad_()
    out = pool_ref(x, a['counts'], q)
    out.backward(a['dout'].double())
    return out.detach(), x.grad, q.grad


@pytest.mark.parametrize('case', list(CASES))
def test_matches_float64_statement(mixed, oxford128, case):
    a = make_inputs(case, mixed, oxford128)
    o, dx, dq = run_native(a)
    ro, rdx, rdq = run_ref64(a)
    assert o.shape == ro.shape
    e_o = assert_close('out', o, ro)
    e_x = assert_close('dx', dx, rdx)
    e_q = assert_maxabs_close('dquery', dq, rdq)
    empty = [b for b, c in enumerate(a['counts']) if c == 0]
    if empty:
        assert not o[empty].any(), 'an empty segment must pool to zero'
    print(f'{case}: n {a["x"].shape[0]}, B {len(a["counts"])}, max segment {max(a["counts"])}, '
          f'err/tol out {e_o:.3g}, dx {e_x:.3g}, dquery max-abs / max|ref| {e_q:.3g}')


def test_counts_forms_agree(mixed, oxford128):
    """counts as the octree's CPU tensor row, a numpy array and a list give the same result."""
    from hotformerloc_b200.attention_pool import attention_pool
    a = make_inputs('oxford_l1_k36', mixed, oxford128)
    ref = attention_pool(a['x'], a['counts'], a['query'])
    for c in (mixed.batch_nnum_nempty[5], np.asarray(a['counts'], dtype=np.int32), tuple(a['counts'])):
        assert torch.equal(attention_pool(a['x'], c, a['query']), ref)


@pytest.mark.parametrize('case', ['minibatch128_l0_k148', 'long_segment', 'C512_k40'])
def test_deterministic(mixed, oxford128, case):
    a = make_inputs(case, mixed, oxford128, seed=1)
    o1, x1, q1 = run_native(a)
    o2, x2, q2 = run_native(a)
    assert torch.equal(o1, o2) and torch.equal(x1, x2) and torch.equal(q1, q2)


def test_misaligned_views_match_aligned_tensors(mixed, oxford128):
    """x, query and the incoming gradient may be contiguous views at any 4-byte offset."""
    from hotformerloc_b200.attention_pool import attention_pool
    a = make_inputs('oxford_l1_k36', mixed, oxford128, seed=2)
    o, dx, dq = run_native(a)

    def shifted(t):
        buf = torch.empty(t.numel() + 1, device='cuda')
        v = buf[1:].view(t.shape)
        v.copy_(t)
        assert v.data_ptr() % 16 != 0
        return v

    x = shifted(a['x']).requires_grad_()
    q = shifted(a['query']).requires_grad_()
    out = attention_pool(x, a['counts'], q)
    out.backward(shifted(a['dout']))
    assert torch.equal(out, o) and torch.equal(x.grad, dx) and torch.equal(q.grad, dq)


def test_no_tokens():
    from hotformerloc_b200.attention_pool import attention_pool
    x = torch.zeros(0, 256, device='cuda', requires_grad=True)
    q = torch.randn(18, 256, device='cuda', requires_grad=True)
    out = attention_pool(x, [0, 0, 0], q)
    assert out.shape == (3, 18, 256) and not out.any()
    out.sum().backward()
    assert x.grad.shape == (0, 256)
    assert torch.equal(q.grad, torch.zeros_like(q))


@pytest.mark.parametrize('k', [74, 148])
def test_memory_at_training_scale(oxford128, k):
    """Level 0 of one Oxford training minibatch: peak memory over forward plus backward, beyond the inputs,
    stays within the op's output, gradients, the log-sum-exp and both workspaces, plus 1 MB."""
    from hotformerloc_b200 import native as N
    from hotformerloc_b200.attention_pool import attention_pool
    counts = level_counts(oxford128, 6)
    n, B, C = sum(counts), len(counts), 256
    x = torch.randn(n, C, device='cuda', requires_grad=True)
    q = torch.randn(k, C, device='cuda', requires_grad=True)
    dout = torch.randn(B, k, C, device='cuda')
    ws_f = int(N.lib().hfl_attn_pool_train_fwd_workspace_bytes(n, B, k, C))
    ws_b = int(N.lib().hfl_attn_pool_train_bwd_workspace_bytes(n, B, k, C))
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    base = torch.cuda.memory_stats()['requested_bytes.all.current']
    torch.cuda.reset_peak_memory_stats()
    out = attention_pool(x, counts, q)
    out.backward(dout)
    torch.cuda.synchronize()
    peak = torch.cuda.memory_stats()['requested_bytes.all.peak'] - base
    f32 = 4
    # x, q and dout exist before base: the bound is out + lse + dx + dq + both workspaces + 1 MB, so a kept
    # (B, k, Nmax) probability tensor (about 150 MB at k = 148) would not fit
    allowed = (out.numel() + B * k + x.numel() + q.numel()) * f32 + ws_f + ws_b + (1 << 20)
    nmax = max(counts)
    mask = B * nmax * nmax * 8
    assert peak <= allowed, f'peak {peak / 2**20:.1f} MiB > {allowed / 2**20:.1f} MiB'
    print(f'k {k}: n {n}, B {B}, Nmax {nmax}; peak {peak / 2**20:.1f} MiB (bound {allowed / 2**20:.1f} MiB; '
          f'workspaces fwd {ws_f / 2**20:.1f} MiB, bwd {ws_b / 2**20:.1f} MiB); the reference\'s (B, Nmax, Nmax) '
          f'int64 mask {mask / 2**20:.1f} MiB, its padded (B, Nmax, C) fp32 features {B * nmax * C * 4 / 2**20:.1f} MiB')


@pytest.fixture(scope='module')
def oxford_model():
    from hotformerloc_b200.config.presets import write_configs
    from hotformerloc_b200.misc.utils import ModelParams
    from hotformerloc_b200.models.model_factory import model_factory
    d = tempfile.mkdtemp(prefix='hfl_apool_')
    paths = write_configs(d, 'oxford', dataset_folder=d)
    torch.manual_seed(0)
    return model_factory(ModelParams(paths['model_config'])).cuda().eval()


def pooling_state(model):
    p = 'pooling.pooling.'
    return {k[len(p):]: v for k, v in model.state_dict().items() if k.startswith(p)}


def make_head(model):
    from hotformerloc_b200.attention_pool import PyramidAttnPool
    pw = model.pooling.pooling
    head = PyramidAttnPool(256, 256, 3, pw.k_pooled_tokens).cuda()
    head.load_state_dict(pooling_state(model))
    return head


def level_feats(o, C=256, seed=5):
    g = torch.Generator(device='cuda').manual_seed(seed)
    return {d: torch.randn(o.n(d), C, device='cuda', generator=g) for d in (6, 5, 4)}


def test_module_forward_matches_oracle(mixed, oxford_model):
    head = make_head(oxford_model)
    feats = level_feats(mixed)
    y = head(feats, mixed)
    sd = {f'pooling.pooling.{k}': v.detach().double().cpu() for k, v in head.state_dict().items()}
    cx = SimpleNamespace(sd=sd, oct=SimpleNamespace(batch_size=mixed.batch_size))
    levels = [SimpleNamespace(counts=np.asarray(level_counts(mixed, d))) for d in (6, 5, 4)]
    ref = M.attn_pool_mixer(cx, [feats[d].double().cpu() for d in (6, 5, 4)], levels)
    assert y.shape == ref.shape == (mixed.batch_size, 256)
    assert_maxabs_close('module forward', y.detach().cpu(), ref)


def test_module_sgd_step_matches_the_statement(mixed, oxford_model):
    from hotformerloc_b200.models.hotformerloc import PyramidAttnPoolWrapper
    head = make_head(oxford_model)
    ref = PyramidAttnPoolWrapper(256, 256, 3, head.k_pooled_tokens).cuda()
    ref.load_state_dict(head.state_dict())
    feats = level_feats(mixed, seed=6)
    w = torch.randn(mixed.batch_size, 256, device='cuda', generator=torch.Generator(device='cuda').manual_seed(8))

    # fp32 torch statement of the reference formulation, on a copy of the parameters
    toks = [pool_ref(feats[d], level_counts(mixed, d), ap.query) for d, ap in zip((6, 5, 4), ref.attpool)]
    t = torch.cat(toks, 1)
    de = ref.descriptor_extractor
    for layer in de.mix:
        t = t + layer.mix(t)
    t = de.row_proj(de.channel_proj(t.permute(0, 2, 1)).permute(0, 2, 1)).flatten(1)
    ((t * w).sum() / math.sqrt(w.numel())).backward()
    expected = {k: (v - 0.1 * v.grad).detach() for k, v in ref.named_parameters()}

    before = {k: v.detach().clone() for k, v in head.named_parameters()}
    opt = torch.optim.SGD(head.parameters(), lr=0.1)
    opt.zero_grad()
    ((head(feats, mixed) * w).sum() / math.sqrt(w.numel())).backward()
    opt.step()
    with torch.no_grad():
        for k, v in head.named_parameters():
            assert_close(f'{k} after one step', v, expected[k].double())
            assert not torch.equal(v, before[k]), f'{k} did not move'


def test_same_function_as_the_inference_head(mixed, oxford_model):
    """The training head on the backbone's local features against HOTFormerLoc's (bf16) inference head."""
    head = make_head(oxford_model)
    with torch.no_grad():
        local, _, o = oxford_model.backbone(None, mixed, mixed.depth)
        g = F.normalize(head(local, o), dim=1)
        ref = oxford_model({'octree': mixed})['global']
    cos = F.cosine_similarity(g, ref.float(), dim=1)
    print(f'min cosine training head vs inference head {cos.min().item():.6f}')
    assert cos.min().item() >= 0.999


def test_bad_arguments_raise_before_any_launch():
    from hotformerloc_b200 import native as N
    from hotformerloc_b200.attention_pool import attention_pool
    from hotformerloc_b200.native import HflError
    C, k = 64, 8
    x = torch.randn(10, C, device='cuda')
    q = torch.randn(k, C, device='cuda')
    counts = [4, 0, 6]
    attention_pool(x, counts, q)
    bad = [
        dict(x=x.double()),
        dict(q=q.half()),
        dict(x=torch.randn(2 * C, 10, device='cuda').t()[:, :C]),                      # non-contiguous
        dict(q=torch.randn(C, k, device='cuda').t()),
        dict(x=x.cpu()),
        dict(q=q.cpu()),
        dict(x=x.cpu(), q=q.cpu()),
        dict(counts=[4, -1, 7]),
        dict(counts=[4, 0, 5]),                                                          # sums to 9, n = 10
        dict(counts=torch.tensor(counts, device='cuda')),                               # device counts
        dict(counts=[4.0, 0.0, 6.0]),
        dict(counts=[]),
        dict(q=torch.randn(257, C, device='cuda')),                                     # k > 256
        dict(q=torch.randn(0, C, device='cuda')),                                       # k = 0
        dict(x=torch.randn(10, 48, device='cuda'), q=torch.randn(k, 48, device='cuda')),  # C % 32 != 0
        dict(x=torch.randn(10, 544, device='cuda'), q=torch.randn(k, 544, device='cuda')),  # C > 512
        dict(q=torch.randn(k, 2 * C, device='cuda')),                                   # channel mismatch
    ]
    for b in bad:
        a = dict(x=x, q=q, counts=counts)
        a.update(b)
        l0 = N.launch_count()
        with pytest.raises(HflError):
            attention_pool(a['x'], a['counts'], a['q'])
        assert N.launch_count() == l0, f'a launch happened before the error for {list(b)}'
