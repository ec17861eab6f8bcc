"""GPU parity of calc_Q / calc_Qw / calc_Qe / calc_Qy (mmif_quality_index) with the oracle of oracle/quality_index.py:
the golden metric cases, the 21 sample pairs x 3 fused images, the smallest shapes, constant and all-zero images,
batches, CPU inputs, launch sharing and determinism.  Scalars pass the dual gate of gates.py; Q_Y also gets the slack
that a window whose float64 S(a,b) lies within rounding of the 0.75 threshold can move it by."""
import numpy as np
import pytest
import torch

import cases
import gates
import samples
from oracle import quality_index as QI

pytestmark = pytest.mark.gpu
FUNCS = (('q', 'calc_Q'), ('qw', 'calc_Qw'), ('qe', 'calc_Qe'), ('qy', 'calc_Qy'))


def _mods():
    import mmif_b200  # noqa: F401
    from mmif_b200 import _lib as L
    from mmif_b200.core import metric as MM
    return L, MM


def T(x):
    return torch.from_numpy(np.ascontiguousarray(x)).to(torch.float32)


def _values(MM, a, b, f):
    return {k: getattr(MM, fn)(a, b, f) for k, fn in FUNCS}


def _check(name, a, b, f):
    """a, b, f: CPU float32 (N,1,H,W).  The four device values against the fp32 / fp64 oracle on the whole batch."""
    _, MM = _mods()
    dev = torch.device('cuda')
    got = _values(MM, a.to(dev), b.to(dev), f.to(dev))
    r32 = QI.quality_indices(a, b, f)
    r64 = QI.quality_indices(a.double(), b.double(), f.double())
    for k, _ in FUNCS:
        assert got[k].dtype == torch.float32 and got[k].dim() == 0 and got[k].device.type == 'cuda'
        allow = (lambda: QI.qy_tie_slack(a, b, f)) if k == 'qy' else None
        gates.assert_scalar(f'{name}/{k}', got[k].item(), r32[k].item(), r64[k].item(), allowance=allow)
    return got


@pytest.mark.parametrize('name', cases.METRIC_CASES)
def test_golden_metric_cases(name):
    _check(name, *(T(x) for x in cases.metric_case(name)))


@pytest.mark.parametrize('kind', samples.KINDS)
@pytest.mark.parametrize('name', samples.names())
def test_sample_pairs(name, kind):
    a, b, f = (T(x) for x in samples.case(name, kind))
    _check(f'{name}/{kind}', a, b, f)


@pytest.mark.parametrize('h,w', [(11, 11), (11, 12), (12, 11), (12, 12), (11, 300), (300, 12), (12, 131)])
def test_smallest_shapes(h, w):
    a, b, f = (T(cases.u8(60 + k, (1, 1, h, w))) for k in range(3))
    _check(f'{h}x{w}', a, b, f)


def test_constant_and_zero_images():
    full = lambda v, h=40, w=52: torch.full((1, 1, h, w), float(v))
    tex = T(cases.u8(70, (1, 1, 40, 52)))
    for name, (a, b, f) in {'zeros': (full(0), full(0), full(0)), 'const': (full(17), full(200), full(90)),
                            'const_sources': (full(30), full(30), tex), 'zero_fused': (tex, tex.flip(-1), full(0)),
                            'one_flat_source': (full(128), tex, tex)}.items():
        got = _check(name, a, b, f)
        if name == 'zeros':
            assert all(got[k].item() == 1.0 for k, _ in FUNCS)


def test_batch_of_four_is_one_population():
    a = T(np.concatenate([cases.natural(80 + i, (1, 1, 97, 131)) for i in range(4)]))
    b = T(np.concatenate([cases.natural(90 + i, (1, 1, 97, 131)) for i in range(4)]))
    f = T(np.floor((a.numpy() + b.numpy()) * np.float32(0.5)))
    _check('batch4', a, b, f)
    _, MM = _mods()
    dev = torch.device('cuda')
    per = [MM._dev_rows(MM._qidx(*(x[i:i + 1].to(dev) for x in (a, b, f))))[0] for i in range(4)]
    whole = MM._qidx(*(x.to(dev) for x in (a, b, f)))[2]
    for i in range(4):                                 # the batched launch's per-pair rows equal single-pair launches
        assert torch.equal(whole[i], per[i])


def test_input_layouts_and_cpu_inputs_equal_cuda_inputs():
    L, MM = _mods()
    a, b, f = (T(x) for x in cases.metric_case('natural_max_120x152'))
    dev = torch.device('cuda')
    ref = _values(MM, a.to(dev), b.to(dev), f.to(dev))
    host = _values(MM, a, b, f)
    for k, _ in FUNCS:
        assert host[k].device.type == 'cpu' and host[k].dtype == torch.float32
        assert torch.equal(host[k], ref[k].cpu()), k
    for view in (lambda x: x[:, 0], lambda x: x[0, 0]):
        got = _values(MM, *(view(x).to(dev) for x in (a, b, f)))
        assert all(torch.equal(got[k], ref[k]) for k, _ in FUNCS)


def test_one_launch_for_the_four_calls_on_one_triple():
    L, MM = _mods()
    dev = torch.device('cuda')
    a, b, f = (T(x).to(dev) for x in cases.metric_case('u8_200x216'))
    torch.cuda.synchronize()
    c0 = L.launch_counts()
    for _, fn in FUNCS:
        getattr(MM, fn)(a, b, f)
    c1 = L.launch_counts()
    assert c1['metric'] - c0['metric'] == 1 and L.kernel_launches(c0, c1) == 1, (c0, c1)


def test_run_to_run_bit_equal():
    _, MM = _mods()
    dev = torch.device('cuda')
    a, b, f = (T(x).to(dev) for x in samples.case(samples.names()[0], 'avg_noise'))
    first = _values(MM, a, b, f)
    for _ in range(3):
        again = _values(MM, a.clone(), b.clone(), f.clone())      # new tensors: the memo cannot serve them
        assert all(torch.equal(first[k], again[k]) for k, _ in FUNCS)
    raw1 = MM._qidx(a.clone(), b.clone(), f.clone())[2]
    raw2 = MM._qidx(a.clone(), b.clone(), f.clone())[2]
    assert torch.equal(raw1, raw2)


def test_too_small_images_raise():
    L, MM = _mods()
    dev = torch.device('cuda')
    for h, w in ((10, 40), (40, 10)):
        x = torch.rand(1, 1, h, w, device=dev) * 255
        with pytest.raises(L.MmifError):
            MM.calc_Q(x, x.clone(), x.clone())
