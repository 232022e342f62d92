"""Device-free checks of the attention-pooling head (hotformerloc_b200.attention_pool)."""
import pytest
import torch


@pytest.mark.parametrize('k_pooled_tokens', [(74, 36, 18), (148, 72, 36)])
def test_module_builds_without_device_with_reference_parameters(k_pooled_tokens):
    from hotformerloc_b200.attention_pool import PyramidAttnPool
    from hotformerloc_b200.models.hotformerloc import PyramidAttnPoolWrapper
    m = PyramidAttnPool(256, 256, 3, k_pooled_tokens)
    ref = PyramidAttnPoolWrapper(256, 256, 3, k_pooled_tokens)
    shapes = {k: tuple(v.shape) for k, v in m.state_dict().items()}
    assert shapes == {k: tuple(v.shape) for k, v in ref.state_dict().items()}
    assert [shapes[f'attpool.{j}.query'] for j in range(3)] == [(k, 256) for k in k_pooled_tokens]
    m.load_state_dict(ref.state_dict())


def test_model_pooling_tensors_load():
    """The pooling.pooling.* tensors of a model built from a shipped cfg load unchanged."""
    import tempfile
    from hotformerloc_b200.attention_pool import PyramidAttnPool
    from hotformerloc_b200.config.presets import write_configs
    from hotformerloc_b200.misc.utils import ModelParams
    from hotformerloc_b200.models.model_factory import model_factory
    d = tempfile.mkdtemp(prefix='hfl_apool_cpu_')
    model = model_factory(ModelParams(write_configs(d, 'wild-places', dataset_folder=d)['model_config']))
    p = 'pooling.pooling.'
    sd = {k[len(p):]: v for k, v in model.state_dict().items() if k.startswith(p)}
    m = PyramidAttnPool(256, 256, 3, (148, 72, 36))
    m.load_state_dict(sd)
    assert all(torch.equal(v, sd[k]) for k, v in m.state_dict().items())


def test_unsupported_shapes_raise_value_error():
    from hotformerloc_b200.attention_pool import PyramidAttnPool
    with pytest.raises(ValueError):
        PyramidAttnPool(1024, 1024, 1, (16,))          # C > 512
    with pytest.raises(ValueError):
        PyramidAttnPool(256, 256, 1, (512,))           # k > 256


def test_host_checks_raise_before_the_device_is_queried():
    from hotformerloc_b200.attention_pool import attention_pool
    from hotformerloc_b200.native import HflError
    x, q = torch.zeros(10, 64), torch.zeros(8, 64)
    cases = [
        (dict(counts=[4, -1, 7]), 'non-negative'),
        (dict(counts=[4, 0, 5]), 'sum to'),
        (dict(counts=[4.0, 6.0]), 'integers'),
        (dict(counts=[[4, 6]]), '1-D'),
        (dict(x=x.double()), 'float32'),
        (dict(q=torch.zeros(257, 64)), 'k'),
        (dict(x=torch.zeros(10, 48), q=torch.zeros(8, 48)), 'multiple of 32'),
        (dict(q=torch.zeros(8, 96)), 'channels'),
        (dict(x=torch.zeros(64, 10).t()), 'contiguous'),
        (dict(), 'CUDA'),
    ]
    for b, msg in cases:
        a = dict(x=x, q=q, counts=[4, 0, 6])
        a.update(b)
        with pytest.raises(HflError, match=msg):
            attention_pool(a['x'], a['counts'], a['q'])
