"""Gradients of the metric functions (core/metric.py) against the reference's autograd: oracle/fusion_metric.py evaluated
with requires_grad in float64 (the truth) and in float32 (the reference's own error).  Gate: over the elements where
the fp64 gradient is finite, max|new - fp64| / max|fp64| <= max(1e-5, the fp32 reference's error); the NaN mask must
equal the fp64 oracle's."""
import numpy as np
import pytest
import torch

import cases
from oracle import fusion_metric as OM

pytestmark = pytest.mark.gpu
RTOL = 1e-5


def _mods():
    import mmif_b200  # noqa: F401
    from mmif_b200 import _lib as L
    from mmif_b200.core import metric as MM
    return MM, L


def _case(name):
    return [torch.from_numpy(np.ascontiguousarray(x)).float() for x in cases.metric_case(name)]


def _batch3():
    """Three samples of one shape, one population for the metrics (their values are combined over the batch)."""
    g = torch.Generator().manual_seed(7)
    a = torch.randint(0, 256, (3, 1, 64, 80), generator=g).float()
    b = torch.randint(0, 256, (3, 1, 64, 80), generator=g).float()
    f = torch.floor((a + b) / 2) + torch.rand(3, 1, 64, 80, generator=g)
    f[1] = f[1] * 0.5 + 40.0                    # samples of different statistics
    return [a, b, f]


def _oracle_grads(fn, imgs, dtype):
    xs = [t.to(dtype).clone().requires_grad_(True) for t in imgs]
    fn(*xs).backward()
    return [None if x.grad is None else x.grad.numpy().astype(np.float64) for x in xs]


def _ours(fn, imgs, device='cuda'):
    xs = [t.to(device).clone().requires_grad_(True) for t in imgs]
    out = fn(*xs)
    out.backward()
    return out, [x.grad for x in xs]


def gate(name, new, r32, r64):
    new = np.asarray(new.detach().cpu().numpy() if torch.is_tensor(new) else new, dtype=np.float64)
    assert np.array_equal(np.isnan(new), np.isnan(r64)), \
        f'{name}: NaN mask differs ({int(np.isnan(new).sum())} vs {int(np.isnan(r64).sum())} NaN elements)'
    fin = np.isfinite(r64)
    if not fin.any():
        return
    scale = np.abs(r64[fin]).max()
    if scale == 0.0:
        assert np.all(new[fin] == 0.0), name
        return
    err = np.abs(new[fin] - r64[fin]).max() / scale
    e32 = np.nanmax(np.abs(r32[fin] - r64[fin])) / scale
    assert err <= max(RTOL, e32), f'{name}: max-norm error {err:.3e} (fp32 reference {e32:.3e})'


def check(name, fn_new, fn_ref, imgs):
    _, got = _ours(fn_new, imgs)
    r64 = _oracle_grads(fn_ref, imgs, torch.float64)
    r32 = _oracle_grads(fn_ref, imgs, torch.float32)
    for k, g in enumerate(got):
        if g is None or r64[k] is None:           # not an argument of the call: no gradient on either side
            assert g is None and r64[k] is None, f'{name}/d{k}'
            continue
        gate(f'{name}/d{k}', g, r32[k], r64[k])


def _funcs(MM):
    """(name, ours, oracle) on (a, b, f)."""
    return [
        ('mean', lambda a, b, f: MM.calc_mean(f), lambda a, b, f: OM.mean(f)),
        ('std', lambda a, b, f: MM.calc_std(f), lambda a, b, f: OM.std(f)),
        ('ag', lambda a, b, f: MM.calc_ag(f), lambda a, b, f: OM.avg_gradient(f)),
        ('sf', lambda a, b, f: MM.calc_sf(f), lambda a, b, f: OM.spatial_freq(f)),
        ('mse', lambda a, b, f: MM.calc_mse(a, f) + 2.0 * MM.calc_mse(b, f), lambda a, b, f: OM.mse(a, f) + 2.0 * OM.mse(b, f)),
        ('psnr', lambda a, b, f: MM.calc_psnr((MM.calc_mse(a, f) + MM.calc_mse(b, f)) * 0.5),
         lambda a, b, f: OM.psnr((OM.mse(a, f) + OM.mse(b, f)) * 0.5)),
        ('cc', lambda a, b, f: MM.calc_cc(a, f) - 0.5 * MM.calc_cc(b, f), lambda a, b, f: OM.corrcoef(a, f) - 0.5 * OM.corrcoef(b, f)),
        ('scd', lambda a, b, f: MM.calc_scd(a, b, f), lambda a, b, f: OM.scd(a, b, f)),
        ('ssim', lambda a, b, f: MM.calc_ssim(a, f), lambda a, b, f: OM.ssim(a, f)),
        ('ssim_pad', lambda a, b, f: MM.calc_ssim(b, f, use_padding=True), lambda a, b, f: OM.ssim(b, f, use_padding=True)),
        ('ssim_full', lambda a, b, f: (lambda s: s[0] + 0.3 * s[1])(MM.calc_ssim(a, f, full=True)),
         lambda a, b, f: (lambda s: s[0] + 0.3 * s[1])(OM.ssim(a, f, full=True))),
        ('msssim', lambda a, b, f: MM.calc_msssim(a, f), lambda a, b, f: OM.msssim(a, f)),
        ('msssim_pad', lambda a, b, f: MM.calc_msssim(b, f, use_padding=True), lambda a, b, f: OM.msssim(b, f, use_padding=True)),
    ]


FUNC_NAMES = ['mean', 'std', 'ag', 'sf', 'mse', 'psnr', 'cc', 'scd', 'ssim', 'ssim_pad', 'ssim_full', 'msssim', 'msssim_pad']


@pytest.mark.parametrize('func', FUNC_NAMES)
@pytest.mark.parametrize('name', cases.METRIC_CASES + ['batch3'])
def test_against_fp64_oracle(name, func):
    MM, _ = _mods()
    imgs = _batch3() if name == 'batch3' else _case(name)
    _, new, ref = next(t for t in _funcs(MM) if t[0] == func)
    check(f'{name}/{func}', new, ref, imgs)


@pytest.mark.parametrize('use_padding', [False, True])
@pytest.mark.parametrize('name', ['frac_72x90', 'ir_crop', 'batch3'])
def test_ssim_maps(name, use_padding):
    """size_average=False: the SSIM and CS maps, each weighted per position by a fixed random map."""
    MM, _ = _mods()
    imgs = _batch3() if name == 'batch3' else _case(name)
    n, _, h, w = imgs[0].shape
    hh, ww = (h, w) if use_padding else (h - 10, w - 10)
    g = torch.Generator().manual_seed(3)
    w1, w2 = torch.rand(n, 1, hh, ww, generator=g), torch.rand(n, 1, hh, ww, generator=g) - 0.5

    def new(a, b, f):
        s, cs = MM.calc_ssim(a, f, use_padding=use_padding, size_average=False, full=True)
        return (s * w1.cuda()).sum() + (cs * w2.cuda()).sum()

    def ref(a, b, f):
        s, cs = OM.ssim(a, f, use_padding=use_padding, size_average=False, full=True)
        return (s * w1.to(s)).sum() + (cs * w2.to(s)).sum()
    check(f'{name}/maps/{use_padding}', new, ref, imgs)


def test_msssim_shrunk_window_levels():
    """u8_64x80: levels 3 and 4 (8x10, 4x5) shrink the window to 8 and 4 taps, sigma 1.5 (metric.py:299, 323-325)."""
    MM, _ = _mods()
    imgs = _case('u8_64x80')
    check('u8_64x80/msssim', lambda a, b, f: MM.calc_msssim(a, f), lambda a, b, f: OM.msssim(a, f), imgs)
    check('small_ssim', lambda a, b, f: MM.calc_ssim(a, f), lambda a, b, f: OM.ssim(a, f),
          [t[..., :9, :10].contiguous() for t in imgs])                         # a 9-tap window for calc_ssim itself


def test_degenerate_nan_masks():
    """Constant images: std / sf / cc gradients NaN everywhere.  Flat blocks: AG NaN exactly on the stencils' pixels."""
    MM, _ = _mods()
    g = torch.Generator().manual_seed(11)
    a = torch.randint(0, 256, (1, 1, 32, 40), generator=g).float()
    c = torch.full((1, 1, 32, 40), 100.0)
    for nm, new, ref, imgs in (('std', lambda x, y: MM.calc_std(y), lambda x, y: OM.std(y), (a, c)),
                               ('sf', lambda x, y: MM.calc_sf(y), lambda x, y: OM.spatial_freq(y), (a, c)),
                               ('cc_f', lambda x, y: MM.calc_cc(x, y), lambda x, y: OM.corrcoef(x, y), (a, c)),
                               ('cc_a', lambda x, y: MM.calc_cc(x, y), lambda x, y: OM.corrcoef(x, y), (c, a))):
        _, got = _ours(new, imgs)
        r64 = _oracle_grads(ref, imgs, torch.float64)
        for k, gk in enumerate(got):
            if nm in ('std', 'sf') and k == 0:
                continue                      # a is not an argument of the call
            assert torch.isnan(gk).all(), (nm, k)
            assert np.isnan(r64[k]).all(), (nm, k)
    f = torch.randint(0, 256, (1, 1, 16, 16), generator=g).float()
    f[0, 0, 4:8, 6:10] = 37.0                 # a flat 4x4 block: 9 stencils -> 15 pixels
    _, (gf,) = _ours(lambda x: MM.calc_ag(x), [f])
    r64 = _oracle_grads(lambda x: OM.avg_gradient(x), [f], torch.float64)[0]
    assert int(torch.isnan(gf).sum()) == 15 and int(np.isnan(r64).sum()) == 15
    imgs = _case('natural_flat_97x131')
    check('natural_flat/ag', lambda a, b, f: MM.calc_ag(f), lambda a, b, f: OM.avg_gradient(f), imgs)


def _launches(before, after):
    """Kernel launches per counter (the tensor-map counters are encodings and memo hits, not launches)."""
    return {k: after[k] - before[k] for k in after if not k.startswith('tmap')}


def _eval_seq(M, a, b, f, oracle=False):
    """eval.py:29-75's differentiable metrics in its call order, summed."""
    if oracle:
        mse = (OM.mse(a, f) + OM.mse(b, f)) * 0.5
        return (OM.std(f) + OM.avg_gradient(f) + OM.spatial_freq(f) + mse + OM.psnr(mse)
                + (OM.corrcoef(a, f) + OM.corrcoef(b, f)) * 0.5 + OM.scd(a, b, f)
                + (OM.ssim(a, f) + OM.ssim(b, f)) * 0.5 + (OM.msssim(a, f) + OM.msssim(b, f)) * 0.5)
    sd, ag, sf = M.calc_std(f), M.calc_ag(f), M.calc_sf(f)
    mse = (M.calc_mse(a, f) + M.calc_mse(b, f)) * 0.5
    psnr = M.calc_psnr(mse)
    cc = (M.calc_cc(a, f) + M.calc_cc(b, f)) * 0.5
    scd = M.calc_scd(a, b, f)
    ssim = (M.calc_ssim(a, f) + M.calc_ssim(b, f)) * 0.5
    msssim = (M.calc_msssim(a, f) + M.calc_msssim(b, f)) * 0.5
    return sd + ag + sf + mse + psnr + cc + scd + ssim + msssim, [sd, ag, sf, mse, psnr, cc, scd, ssim, msssim]


@pytest.mark.parametrize('name', ['u8_rand_f_97x131', 'polar_odd_153', 'batch3'])
def test_eval_sequence(name):
    MM, L = _mods()
    imgs = _batch3() if name == 'batch3' else _case(name)
    plain = [t.cuda() for t in imgs]
    c0 = L.launch_counts()
    _, vals0 = _eval_seq(MM, *plain)
    c1 = L.launch_counts()
    xs = [t.cuda().requires_grad_(True) for t in imgs]
    total, vals = _eval_seq(MM, *xs)
    c2 = L.launch_counts()
    assert _launches(c0, c1) == _launches(c1, c2), 'forward launches differ with grad'
    for v0, v in zip(vals0, vals):
        assert v0.grad_fn is None and v.grad_fn is not None
        assert torch.equal(v0, v.detach())
    total.backward()
    c3 = L.launch_counts()
    assert c3['metric'] - c2['metric'] == 8, 'one mmif_stats_bwd per statistics node (sd ag sf mse x2 cc x2 scd)'
    r64 = _oracle_grads(lambda a, b, f: _eval_seq(None, a, b, f, True), imgs, torch.float64)
    r32 = _oracle_grads(lambda a, b, f: _eval_seq(None, a, b, f, True), imgs, torch.float32)
    for k, x in enumerate(xs):
        gate(f'{name}/eval/d{k}', x.grad, r32[k], r64[k])


def test_routing_through_the_triple():
    """calc_cc(a, f) after calc_scd(a, b, f) is served by the triple's launch; its gradient reaches a and f only."""
    MM, L = _mods()
    a, b, f = (t.cuda().requires_grad_(True) for t in _case('frac_72x90'))
    MM.calc_scd(a, b, f)
    c0 = L.launch_counts()
    cc = MM.calc_cc(a, f)
    assert L.launch_counts()['metric'] == c0['metric']           # from the memo
    ga, gb, gf = torch.autograd.grad(cc, (a, b, f), allow_unused=True)
    assert gb is None and ga is not None and gf is not None
    r64 = _oracle_grads(lambda x, y: OM.corrcoef(x, y), [a.detach().cpu(), f.detach().cpu()], torch.float64)
    r32 = _oracle_grads(lambda x, y: OM.corrcoef(x, y), [a.detach().cpu(), f.detach().cpu()], torch.float32)
    gate('routed/cc/da', ga, r32[0], r64[0])
    gate('routed/cc/df', gf, r32[1], r64[1])


def test_no_grad_paths_unchanged():
    MM, L = _mods()
    imgs = _case('polar_crop')
    plain = [t.cuda() for t in imgs]
    c0 = L.launch_counts()
    _, vals0 = _eval_seq(MM, *plain)
    c1 = L.launch_counts()
    xs = [t.cuda().requires_grad_(True) for t in imgs]
    with torch.no_grad():
        _, vals = _eval_seq(MM, *xs)
    c2 = L.launch_counts()
    assert _launches(c0, c1) == _launches(c1, c2)
    for v0, v in zip(vals0, vals):
        assert v.grad_fn is None and not v.requires_grad and torch.equal(v0, v)


def test_cpu_inputs_get_cpu_gradients():
    """eval.py passes CPU tensors.  (psnr is left out of the sum: torch's CPU and CUDA log10 may differ in the last bit.)"""
    MM, _ = _mods()
    imgs = _case('u8_200x216')

    def seq(a, b, f):
        _, v = _eval_seq(MM, a, b, f)
        return v[0] + v[1] + v[2] + v[3] + v[5] + v[6] + v[7] + v[8]
    xc = [t.clone().requires_grad_(True) for t in imgs]
    total_c = seq(*xc)
    total_c.backward()
    xg = [t.cuda().requires_grad_(True) for t in imgs]
    total_g = seq(*xg)
    total_g.backward()
    assert total_c.device.type == 'cpu'
    for c, g in zip(xc, xg):
        assert c.grad.device.type == 'cpu' and c.grad.dtype == torch.float32 and c.grad.shape == c.shape
        assert torch.equal(c.grad.view(torch.int32), g.grad.cpu().view(torch.int32))     # bit for bit, AG NaNs included


def test_backward_is_deterministic():
    MM, _ = _mods()
    imgs = _case('natural_max_120x152')
    grads = []
    for _ in range(2):
        xs = [t.cuda().requires_grad_(True) for t in imgs]
        total, _ = _eval_seq(MM, *xs)
        total.backward()
        grads.append([x.grad.clone() for x in xs])
    for g0, g1 in zip(*grads):
        assert torch.equal(g0.view(torch.int32), g1.view(torch.int32))


def test_other_metrics_stay_detached():
    MM, _ = _mods()
    a, b, f = (t.cuda().requires_grad_(True) for t in _case('ir_crop'))
    for v in (MM.calc_Qabf(a, b, f), MM.calc_Nabf(a, b, f), MM.calc_Labf(a, b, f), MM.calc_viff(a, b, f),
              MM.calc_entropy(f), MM.calc_cross_ent(a, f), MM.calc_mul_info(a, f)):
        assert v.grad_fn is None and not v.requires_grad
