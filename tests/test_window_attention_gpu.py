"""GPU parity of the window attention core (hotformerloc_b200.window_attention, csrc/window_attn_train.cu)
against a float64 torch autograd statement built from oracle.model_ref._rpe_bias and the core of
oracle.model_ref._attention.  Windows, ids and coordinates come from real batches cut as
oracle.model_ref.make_level / window_rows do, including windows that span two or three submaps and
all-padding windows."""
import math
import tempfile

import pytest
import torch
import torch.nn.functional as F

from oracle import model_ref as M

pytestmark = pytest.mark.gpu

HD = 16


def level_windows(o, d, K, dil, pad_dil, hat):
    """(xyz (N_win, K, 3), ids (N_win, K + hat)) int64 of depth d: tokens padded to a multiple of
    K pad_dil with (0, 0, 0, batch) rows (make_level), windows by window_rows, relay id = first token's."""
    n = o.n(d)
    blk = K * pad_dil
    n_pad = -(-n // blk) * blk
    tok = o.tokens(d, n_pad).long()
    rows = M.window_rows(n_pad, K, dil).cuda()
    xyz, ids = tok[rows, :3].contiguous(), tok[rows, 3].contiguous()
    if hat:
        ids = torch.cat([ids[:, :1], ids], 1).contiguous()
    return xyz, ids


def core_ref(qkv, xyz, ids, table, K, dil, hat, H):
    """The attention core of _attention (oracle/model_ref.py) from qkv to before proj, with the bias of
    _rpe_bias, in qkv's dtype and on its device."""
    N, L, C3 = qkv.shape
    C = C3 // 3
    q, k, v = qkv.view(N, L, 3, H, C // H).permute(2, 0, 3, 1, 4)
    bias = torch.zeros(N, 1, L, L, dtype=qkv.dtype, device=qkv.device)
    bias = bias.masked_fill((ids.unsqueeze(2) != ids.unsqueeze(1)).unsqueeze(1), -1000.0)
    if table is not None:
        rpe = M._rpe_bias({'t.rpe_table': table}, 't', xyz, K, dil)
        if hat:
            rpe = F.pad(rpe, (1, 0, 1, 0))
        bias = bias + rpe
    att = (q @ k.transpose(-1, -2)) * ((C // H) ** -0.5) + bias
    return (att.softmax(-1) @ v).transpose(1, 2).reshape(N, L, C)


def assert_close(name, a, r):
    err = (a.double() - r).abs()
    tol = 1e-5 + 1e-4 * r.abs()
    worst = (err / tol).max().item() if err.numel() else 0.0
    assert bool((err <= tol).all()), f'{name}: max |err| / (1e-5 + 1e-4 |ref|) = {worst:.3g}'
    return worst


def assert_table_close(a, r):
    err = (a.double() - r).abs().max().item()
    bound = 1e-4 * r.abs().max().item()
    assert err <= bound, f'd rpe_table: max-abs err {err:.3g} > 1e-4 max|ref| = {bound:.3g}'
    return err / max(r.abs().max().item(), 1e-300)


@pytest.fixture(scope='module')
def batch():
    """Oxford-cfg depth-9 batch; the 30- and 20-point submaps are shorter than a window, so some
    windows span three submaps, and padding to 4 K leaves all-padding windows at depths 6 and 7."""
    from hotformerloc_b200.octree import build_batch
    g = torch.Generator().manual_seed(3)
    sizes = [4096, 30, 4096, 20, 2000, 3000]
    return build_batch([M.lidar_cloud(n, g) for n in sizes], 9).finalize()


# name: depth, K, H, dil (window_rows), padding multiple of K, hat, rpe
CASES = {
    'oxford_octf_dil1': (7, 48, 8, 1, 1, False, True),
    'oxford_octf_dil4': (7, 48, 8, 4, 4, False, True),
    'oxford_hosa': (6, 48, 16, 1, 4, True, True),
    'cswild_hosa': (6, 64, 16, 1, 4, True, True),
    'no_rpe': (7, 48, 8, 1, 1, False, False),
    'L97_H1': (7, 96, 1, 1, 4, True, True),
}


def make_inputs(o, case, seed=0):
    d, K, H, dil, pad_dil, hat, use_rpe = CASES[case]
    xyz, ids = level_windows(o, d, K, dil, pad_dil, hat)
    n_win, L, C = ids.shape[0], K + int(hat), HD * H
    bnd = int(0.8 * K * dil ** 0.5)
    g = torch.Generator(device='cuda').manual_seed(seed)
    qkv = torch.randn(n_win, L, 3 * C, device='cuda', generator=g)
    table = (torch.randn(3 * (2 * bnd + 1), H, device='cuda', generator=g) * 0.5) if use_rpe else None
    dout = torch.randn(n_win, L, C, device='cuda', generator=g)
    return dict(qkv=qkv, xyz=xyz, ids=ids, table=table, bnd=bnd, hat=hat, H=H, K=K, dil=dil, dout=dout)


def run_native(x, xyz=None, ids=None):
    from hotformerloc_b200.window_attention import window_attention
    qkv = x['qkv'].clone().requires_grad_()
    table = x['table'].clone().requires_grad_() if x['table'] is not None else None
    o = window_attention(qkv, x['xyz'] if xyz is None else xyz, x['ids'] if ids is None else ids, table,
                         x['bnd'], x['hat'], x['H'])
    o.backward(x['dout'])
    return o.detach(), qkv.grad, (table.grad if table is not None else None)


def run_ref64(x):
    qkv = x['qkv'].double().requires_grad_()
    table = x['table'].double().requires_grad_() if x['table'] is not None else None
    o = core_ref(qkv, x['xyz'], x['ids'], table, x['K'], x['dil'], x['hat'], x['H'])
    o.backward(x['dout'].double())
    return o.detach(), qkv.grad, (table.grad if table is not None else None)


@pytest.mark.parametrize('case', list(CASES))
def test_matches_float64_statement(batch, case):
    x = make_inputs(batch, case)
    ids = x['ids'][:, int(x['hat']):]
    spans = torch.stack([(ids == b).any(1) for b in range(batch.batch_size)], 1).sum(1)
    if case.startswith('oxford') or case == 'cswild_hosa':
        assert int(spans.max()) >= 2
    if x['hat']:
        assert bool((ids == batch.batch_size).all(1).any()), 'expected all-padding windows'
    o, dqkv, dtab = run_native(x)
    ro, rdqkv, rdtab = run_ref64(x)
    e_o = assert_close('o', o, ro)
    e_q = assert_close('dqkv', dqkv, rdqkv)
    if x['table'] is not None:
        assert_table_close(dtab, rdtab)
    print(f'{case}: n_win {o.shape[0]}, max err/tol o {e_o:.3g}, dqkv {e_q:.3g}')


def test_windows_span_three_submaps(batch):
    x = make_inputs(batch, 'oxford_octf_dil1')
    spans = torch.stack([(x['ids'] == b).any(1) for b in range(batch.batch_size)], 1).sum(1)
    assert int(spans.max()) >= 3


def test_no_windows():
    from hotformerloc_b200.window_attention import window_attention
    H, K, bnd = 1, 96, 76
    qkv = torch.zeros(0, K + 1, 3 * HD * H, device='cuda', requires_grad=True)
    table = torch.randn(3 * (2 * bnd + 1), H, device='cuda', requires_grad=True)
    xyz = torch.zeros(0, K, 3, dtype=torch.int64, device='cuda')
    ids = torch.zeros(0, K + 1, dtype=torch.int64, device='cuda')
    o = window_attention(qkv, xyz, ids, table, bnd, True, H)
    assert o.shape == (0, K + 1, HD * H)
    o.sum().backward()
    assert qkv.grad.shape == qkv.shape
    assert torch.equal(table.grad, torch.zeros_like(table))


@pytest.mark.parametrize('case', ['oxford_octf_dil4', 'oxford_hosa'])
def test_deterministic_and_index_dtypes(batch, case):
    x = make_inputs(batch, case, seed=1)
    o1, q1, t1 = run_native(x)
    o2, q2, t2 = run_native(x)
    assert torch.equal(q1, q2) and torch.equal(t1, t2)
    o3, q3, t3 = run_native(x, xyz=x['xyz'].int(), ids=x['ids'].int())
    assert torch.equal(o1, o3) and torch.equal(q1, q3) and torch.equal(t1, t3)


def test_memory_at_training_scale():
    """Oxford level 7, one training minibatch (batch_split_size = 128 submaps of 4096 points): peak
    memory over forward plus backward stays within the op's inputs, outputs, gradients, the
    log-sum-exp and the workspace, plus 1 MB -- no (N_win, H, L, L) tensor."""
    from hotformerloc_b200 import native as N
    from hotformerloc_b200.octree import build_batch
    from hotformerloc_b200.window_attention import window_attention
    g = torch.Generator().manual_seed(7)
    o = build_batch([M.lidar_cloud(4096, g) for _ in range(128)], 9).finalize()
    K, H, bnd = 48, 8, 38
    xyz, ids = level_windows(o, 7, K, 1, 1, False)
    del o
    n_win, C = ids.shape[0], HD * H
    assert n_win > 10000
    qkv = torch.randn(n_win, K, 3 * C, device='cuda', requires_grad=True)
    table = torch.randn(3 * (2 * bnd + 1), H, device='cuda', requires_grad=True)
    dout = torch.randn(n_win, K, C, device='cuda')
    # bytes the tensors request: max_memory_allocated also counts the caching allocator's block
    # rounding (a large block is not split when less than 1 MB would remain)
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    base = torch.cuda.memory_stats()['requested_bytes.all.current']
    torch.cuda.reset_peak_memory_stats()
    out = window_attention(qkv, xyz, ids, table, bnd, False, H)
    out.backward(dout)
    torch.cuda.synchronize()
    peak = torch.cuda.memory_stats()['requested_bytes.all.peak'] - base
    ws = int(N.lib().hfl_window_attn_train_bwd_workspace_bytes(H, bnd, 1))
    f32 = 4
    allowed = (out.numel() + n_win * H * K + qkv.numel() + table.numel()) * f32 + ws + (1 << 20)
    dense = n_win * H * K * K * f32
    assert peak <= allowed, f'peak {peak / 2**20:.1f} MiB > {allowed / 2**20:.1f} MiB'
    print(f'n_win {n_win}: peak {peak / 2**20:.1f} MiB, bound {allowed / 2**20:.1f} MiB, '
          f'one (N_win, H, L, L) fp32 tensor {dense / 2**20:.1f} MiB')


@pytest.fixture(scope='module')
def oxford_state_dict():
    from hotformerloc_b200.config.presets import write_configs
    from hotformerloc_b200.misc.utils import ModelParams
    from hotformerloc_b200.models.model_factory import model_factory
    d = tempfile.mkdtemp(prefix='hfl_wattn_')
    paths = write_configs(d, 'oxford', dataset_folder=d)
    torch.manual_seed(0)
    return model_factory(ModelParams(paths['model_config'])).state_dict()


def sub_dict(sd, prefix):
    return {k[len(prefix):]: v for k, v in sd.items() if k.startswith(prefix)}


# block prefix, depth, K, H, dilation, hat
BLOCKS = {
    'octf_dil4': ('backbone.backbone.octf_stage.0.blocks.1.attention.', 7, 48, 8, 4, False),
    'hosa': ('backbone.backbone.hotf_stage.hosa_blocks.0.3.attention.', 6, 48, 16, 1, True),
}


@pytest.mark.parametrize('block', list(BLOCKS))
def test_module_loads_pretrained_and_trains_like_the_statement(batch, oxford_state_dict, block):
    from hotformerloc_b200.window_attention import OctreeAttention
    prefix, d, K, H, dil, hat = BLOCKS[block]
    C = HD * H
    sd = sub_dict(oxford_state_dict, prefix)
    mod = OctreeAttention(C, K, H, dilation=dil, hat=hat).cuda()
    mod.load_state_dict(sd)
    with torch.no_grad():                      # give the RPE a visible effect (trained tables are not ~0)
        mod.rpe.rpe_table.normal_(0, 0.5, generator=torch.Generator(device='cuda').manual_seed(4))
    xyz, ids = level_windows(batch, d, K, dil, 4 if hat else dil, hat)
    g = torch.Generator(device='cuda').manual_seed(5)
    x = torch.randn(ids.shape[0], K + int(hat), C, device='cuda', generator=g)
    w = torch.randn(x.shape, device='cuda', generator=g)

    # forward against the oracle's float64 statement through qkv and proj
    p = {f'a.{k}': v.detach().double().cpu() for k, v in mod.state_dict().items()}
    rpe = M._rpe_bias(p, 'a.rpe', xyz.cpu(), K, dil)
    if hat:
        rpe = F.pad(rpe, (1, 0, 1, 0))
    ref = M._attention(x.double().cpu(), ids.cpu(), p, 'a', H, rpe)
    y = mod(x, xyz, ids)
    assert_close('module forward', y.detach().cpu(), ref)

    # one SGD step on a toy loss against the fp32 torch statement
    params = {k: v.detach().clone().requires_grad_() for k, v in mod.named_parameters()}
    qkv = F.linear(x, params['qkv.weight'], params['qkv.bias'])
    o = core_ref(qkv, xyz, ids, params['rpe.rpe_table'], K, dil, hat, H)
    ((F.linear(o, params['proj.weight'], params['proj.bias']) * w).sum() / math.sqrt(w.numel())).backward()
    opt = torch.optim.SGD(mod.parameters(), lr=0.1)
    opt.zero_grad()
    ((y * w).sum() / math.sqrt(w.numel())).backward()
    opt.step()
    with torch.no_grad():
        for k, v in mod.named_parameters():
            assert_close(f'{k} after one step', v, (params[k] - 0.1 * params[k].grad).double())
            assert not torch.equal(v, params[k]), f'{k} did not move'


def test_bad_arguments_raise():
    from hotformerloc_b200.native import HflError
    from hotformerloc_b200.window_attention import window_attention
    H, K, bnd = 2, 8, 6
    C = HD * H
    qkv = torch.randn(3, K, 3 * C, device='cuda')
    xyz = torch.zeros(3, K, 3, dtype=torch.int64, device='cuda')
    ids = torch.zeros(3, K, dtype=torch.int64, device='cuda')
    table = torch.randn(3 * (2 * bnd + 1), H, device='cuda')
    window_attention(qkv, xyz, ids, table, bnd, False, H)
    bad = [
        dict(qkv=torch.randn(3, K, 3 * C + 3, device='cuda')),                         # C != 16 H
        dict(qkv=torch.randn(3, 129, 3 * C, device='cuda'),
             xyz=torch.zeros(3, 129, 3, dtype=torch.int64, device='cuda'),
             ids=torch.zeros(3, 129, dtype=torch.int64, device='cuda')),               # L > 128
        dict(hat=True),                                                                  # xyz has L rows, not L - 1
        dict(table=torch.randn(3 * (2 * bnd + 3), H, device='cuda')),                   # table for another bnd
        dict(table=torch.randn(3 * (2 * bnd + 1), H + 1, device='cuda')),               # table for another H
        dict(qkv=qkv.double()),
        dict(qkv=qkv.half()),
        dict(ids=ids.float()),
        dict(xyz=xyz.to(torch.int16)),
        dict(table=table.double()),
        dict(qkv=qkv.cpu()),
        dict(ids=ids.cpu()),
        dict(table=table.cpu()),
        dict(qkv=torch.randn(3, 3 * C, K, device='cuda').transpose(1, 2)),             # non-contiguous
        dict(xyz=torch.zeros(3, 3, K, dtype=torch.int64, device='cuda').transpose(1, 2)),
        dict(H=17),
        dict(bnd=-1),
    ]
    for b in bad:
        a = dict(qkv=qkv, xyz=xyz, ids=ids, table=table, bnd=bnd, hat=False, H=H)
        a.update(b)
        if 'H' in b and 'table' not in b:
            a['qkv'] = torch.randn(3, K, 3 * HD * b['H'], device='cuda')
        with pytest.raises(HflError):
            window_attention(a['qkv'], a['xyz'], a['ids'], a['table'], a['bnd'], a['hat'], a['H'])
