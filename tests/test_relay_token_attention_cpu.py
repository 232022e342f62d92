"""Device-free checks of the relay-token self-attention op (hotformerloc_b200.relay_token_attention): the
host layout against oracle.model_ref.rt_layout, the inference engine's tables after their move onto the
shared ownership rule, the host argument checks and the module's parameters."""
import numpy as np
import pytest
import torch

from oracle import model_ref as M
from oracle import octree_ref as R

# name: submap sizes, generator seed, octree depth, level depths, patch size K, dilation
BATCHES = {
    'oxford_6': ([4096, 30, 4096, 20, 2000, 3000], 3, 9, (6, 5, 4), 48, 4),
    'cswild_6x30k': ([30000] * 6, 1, 7, (4, 3, 2), 64, 4),
    'oxford_b1': ([4096], 5, 9, (6, 5, 4), 48, 4),
}


@pytest.fixture(scope='module', params=list(BATCHES))
def batch(request):
    sizes, seed, depth, depths, K, dil = BATCHES[request.param]
    g = torch.Generator().manual_seed(seed)
    oct_ = R.build_batch([M.lidar_cloud(n, g) for n in sizes], depth)
    return request.param, oct_, depths, K, dil


def oracle_packed(oct_, depths, K, dil):
    """oracle.model_ref.rt_layout's padded (B, Nmax) index / ids mapped to packed rows, and cu."""
    levels = [M.make_level(oct_, d, K, dil) for d in depths]
    index, ids = M.rt_layout(levels, oct_.batch_size)
    real = index >= 0
    lens = real.sum(1).numpy()
    return (index[real].numpy(), ids[real].numpy(), np.concatenate([[0], np.cumsum(lens)]),
            [lv.num_windows for lv in levels])


def test_layout_matches_oracle(batch):
    from hotformerloc_b200.relay_token_attention import _layout_tables
    name, oct_, depths, K, dil = batch
    counts = [oct_.batch_nnum_nempty[d] for d in depths]
    own, index, inverse = _layout_tables([torch.as_tensor(np.asarray(c)) for c in counts], K, dil)
    r_index, r_ids, r_cu, r_nw = oracle_packed(oct_, depths, K, dil)
    assert np.array_equal(index, r_index)
    assert np.array_equal(own.ids, r_ids)
    assert np.array_equal(own.cu, r_cu)
    assert all(np.array_equal(a, b) for a, b in zip(own.num_windows, r_nw))
    assert np.array_equal(inverse[index], np.arange(own.total))
    assert own.total == sum(-(-int(np.sum(c)) // (K * dil)) * dil for c in counts)
    lens = np.diff(own.cu)
    assert own.max_len == lens.max()
    B = oct_.batch_size
    if name == 'oxford_6':
        assert lens.tolist() == [164, 2, 161, 0, 93, 128]
        # the padding windows' RTs (id B) sit in the last submap's sequence
        assert (own.ids == B).any() and (own.ids[own.cu[-2]:] == B).any()
        assert not (own.ids[:own.cu[-2]] == B).any()
    if name == 'cswild_6x30k':
        assert own.num_windows[2].tolist() == [1, 0, 1, 0, 1, 1]
        last = own.ids[own.cu[-2]:]
        assert (last == B).sum() >= 1
    if name == 'oxford_b1':
        assert own.cu.tolist() == [0, own.total]


def engine_tables_before(counts, K, dil):
    """The engine's relay-token tables as _Engine._host_tables computed them before it called
    rt_ownership (restated verbatim), with the level geometry of _Engine.forward."""
    B = counts[0].size
    blk = K * dil
    nl = [int(c.sum()) for c in counts]
    npad = [-(-v // blk) * blk for v in nl]
    nwin = [v // K for v in npad]
    R_ = np.concatenate([[0], np.cumsum([v * (K + 1) for v in nwin])]).astype(np.int64)
    L = len(counts)
    nws, starts = [], []
    for j in range(L):
        cum = np.cumsum(counts[j])
        cum[-1] += npad[j] - nl[j]
        boundary = -(-cum // K)
        nw = np.diff(np.concatenate([[0], boundary]))
        nws.append(nw)
        starts.append(np.cumsum(nw) - nw)
    tot = np.sum(nws, axis=0)
    cu = np.concatenate([[0], np.cumsum(tot)]).astype(np.int32)
    total_rt = int(cu[-1])
    rt_rows = np.empty(total_rt, dtype=np.int32)
    ids = np.empty(total_rt, dtype=np.int32)
    prefix = np.zeros(B, dtype=np.int64)
    for j in range(L):
        wi = np.arange(nwin[j], dtype=np.int64)
        owner = np.repeat(np.arange(B, dtype=np.int64), nws[j])
        pos = cu[owner] + prefix[owner] + (wi - starts[j][owner])
        rt_rows[pos] = R_[j] + wi * (K + 1)
        first_pad = -(-nl[j] // K)
        ids[pos] = np.where(wi >= first_pad, B, owner)
        prefix += nws[j]
    return dict(rt_rows=rt_rows, ids=ids, cu=cu, max_len=int(tot.max()), num_windows=nws), npad, nwin, R_


def test_engine_tables_unchanged(batch):
    from hotformerloc_b200.models.hotformerloc import _Engine
    _, oct_, depths, K, dil = batch
    counts = [np.asarray(oct_.batch_nnum_nempty[d], dtype=np.int64) for d in depths]
    before, npad, nwin, R_ = engine_tables_before(counts, K, dil)
    own, rt_rows = _Engine._rt_tables(counts, npad, nwin, R_, K)
    assert np.array_equal(rt_rows, before['rt_rows'])
    assert np.array_equal(own.ids.astype(np.int32), before['ids'])
    assert np.array_equal(own.cu.astype(np.int32), before['cu'])
    assert own.max_len == before['max_len']
    assert all(np.array_equal(a, b) for a, b in zip(own.num_windows, before['num_windows']))


def test_layout_host_checks_raise_before_the_device_is_queried():
    from hotformerloc_b200.native import HflError
    from hotformerloc_b200.relay_token_attention import rt_layout
    good = [[100, 200], [30, 40]]
    cases = [
        (dict(counts=[[100, 200], [30, 40, 5]]), 'same number of submaps'),
        (dict(counts=[[100, -1], [30, 40]]), 'non-negative'),
        (dict(counts=[[100.0, 200.0], [30, 40]]), 'integers'),
        (dict(counts=[torch.tensor([100.0, 200.0]), [30, 40]]), 'integers'),
        (dict(counts=[[[100, 200]], [30, 40]]), '1-D'),
        (dict(counts=[[], []]), '1-D'),
        (dict(counts=[]), 'non-empty'),
        (dict(K=0), 'patch_size'),
        (dict(dil=1.5), 'dilation'),
        (dict(device='cpu'), 'CUDA device'),
    ]
    if torch.cuda.is_available():
        cases.append((dict(counts=[torch.tensor([100, 200], device='cuda'), [30, 40]]), 'host tensor'))
    for b, msg in cases:
        a = dict(counts=good, K=48, dil=4, device='cuda')
        a.update(b)
        with pytest.raises(HflError, match=msg):
            rt_layout(a['counts'], a['K'], a['dil'], a['device'])


def test_attention_host_checks_raise_before_the_device_is_queried():
    from hotformerloc_b200.native import HflError
    from hotformerloc_b200.relay_token_attention import (RelayTokenLayout, _layout_tables,
                                                          relay_token_attention)
    own, index, inverse = _layout_tables([[100, 200], [30, 40]], 48, 4)
    t = lambda a: torch.from_numpy(a.astype(np.int32))
    layout = RelayTokenLayout(t(own.cu), t(own.ids), t(index), t(inverse), own.num_windows, own.total, own.max_len)
    T, H = own.total, 2
    qkv = torch.zeros(T, 3 * 16 * H)
    cases = [
        (dict(qkv=qkv.double()), 'float32'),
        (dict(qkv=torch.zeros(T + 1, 3 * 16 * H)), 'shape'),
        (dict(qkv=torch.zeros(T, 3 * 16 * H + 3)), 'shape'),
        (dict(qkv=torch.zeros(3 * 16 * H, T).t()), 'contiguous'),
        (dict(H=0), 'num_heads'),
        (dict(H=17), 'num_heads'),
        (dict(H=2.0), 'num_heads'),
        (dict(layout=None), 'RelayTokenLayout'),
        (dict(), 'CUDA'),
    ]
    for b, msg in cases:
        a = dict(qkv=qkv, layout=layout, H=H)
        a.update(b)
        with pytest.raises(HflError, match=msg):
            relay_token_attention(a['qkv'], a['layout'], a['H'])


def test_module_has_the_reference_parameters():
    from hotformerloc_b200.models.hotformerloc import _RTSABlock
    from hotformerloc_b200.relay_token_attention import RTAttention
    ref = _RTSABlock(256).rt_attention
    m = RTAttention(256, 16)
    assert {k: tuple(v.shape) for k, v in m.state_dict().items()} == \
        {k: tuple(v.shape) for k, v in ref.state_dict().items()}
    m.load_state_dict(ref.state_dict())
    with pytest.raises(ValueError):
        RTAttention(256, 8)                       # dim != 16 num_heads
    with pytest.raises(ValueError):
        RTAttention(272, 17)                      # more than 16 heads
