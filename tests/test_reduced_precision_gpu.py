"""bfloat16 / float16 images through the loss modules (an autocast training step).  Widening to float32 is exact, so every
value must be bit-identical to the float32 path run on img.float(), and every gradient bit-identical to that path's gradient
.to(dtype): the gates are torch.equal, no tolerance."""
import numpy as np
import pytest
import torch

import cases

pytestmark = pytest.mark.gpu

HALF = (torch.bfloat16, torch.float16)
W_TRAIN = (1.0, 0.01, 0.1)          # the training configuration: SSIMLoss 1.0, PixelLoss 0.01 'max', GradLoss 0.1 'max'


def _mods():
    import mmif_b200  # noqa: F401
    from mmif_b200 import _lib as L
    from mmif_b200.core import loss as ML
    return L, ML


def _objective(ML):
    return (ML.SSIMLoss('ssim', weight=W_TRAIN[0]), ML.PixelLoss('l1', weight=W_TRAIN[1]), ML.GradLoss('l1', weight=W_TRAIN[2]))


def _three(mods, a, b, f):
    return (mods[0](a, b, f), mods[1](a, b, f, mode='max'), mods[2](a, b, f, mode='max'))


def _run(mods, a, b, f, backward):
    """Three loss values and d/df after `backward(l1, l2, l3)` on a fresh leaf copy of f."""
    F_ = f.detach().clone().requires_grad_(True)
    ls = _three(mods, a, b, F_)
    backward(*ls)
    return [t.detach().clone() for t in ls], F_.grad


def _check(got, ref, dtype):
    (lg, gg), (lr, gr) = got, ref
    for x, y in zip(lg, lr):
        assert x.dtype == torch.float32 and torch.equal(x, y), (x.item(), y.item())
    assert gg.dtype == dtype, gg.dtype
    want = gr.to(dtype)
    assert torch.equal(gg, want), (gg.float() - want.float()).abs().max().item()


def _inputs(name):
    if name == 'nontma_2x97x203':                   # W % 4 != 0: the plain-load ring, scalar narrow / widen tails
        g = torch.Generator().manual_seed(97)
        return tuple(torch.rand(2, 1, 97, 203, generator=g) for _ in range(3))
    if name == 'config2_8x256x256':                 # the per-rank training shape of config 2
        g = torch.Generator().manual_seed(256)
        return tuple(torch.rand(8, 1, 256, 256, generator=g) for _ in range(3))
    return tuple(torch.from_numpy(np.ascontiguousarray(x)) for x in cases.loss_case(name))


OBJECTIVE_CASES = cases.LOSS_CASES + ['nontma_2x97x203', 'config2_8x256x256']


def _total(l1, l2, l3):
    (l1 + l2 + l3).backward()


@pytest.mark.parametrize('src_half', [False, True], ids=['f32_sources', 'half_sources'])
@pytest.mark.parametrize('dtype', HALF, ids=['bf16', 'f16'])
@pytest.mark.parametrize('name', OBJECTIVE_CASES)
def test_training_objective_equals_float32_path(name, dtype, src_half):
    L, ML = _mods()
    mods = _objective(ML)
    a, b, f = (t.cuda() for t in _inputs(name))
    fh = f.to(dtype)
    ah, bh = (a.to(dtype), b.to(dtype)) if src_half else (a, b)
    ref = _run(mods, ah.float(), bh.float(), fh.float(), _total)
    got = _run(mods, ah, bh, fh, _total)
    _check(got, ref, dtype)


@pytest.mark.parametrize('dtype', HALF, ids=['bf16', 'f16'])
@pytest.mark.parametrize('name', ['rand_3x64x96', 'unbounded_f', 'nontma_2x97x203'])
def test_other_backward_cases_equal_float32_path(name, dtype):
    L, ML = _mods()
    mods = _objective(ML)
    a, b, f = (t.cuda() for t in _inputs(name))
    fh = f.to(dtype)

    def unequal(l1, l2, l3):
        (l1 + 2 * l2 + l3).backward()

    def only_pixel(l1, l2, l3):
        l2.backward()

    _check(_run(mods, a, b, fh, unequal), _run(mods, a, b, fh.float(), unequal), dtype)
    _check(_run(mods, a, b, fh, only_pixel), _run(mods, a, b, fh.float(), only_pixel), dtype)

    # a retained graph backpropagated twice: the second backward recomputes (from the saved half-precision image)
    def twice(fx):
        F_ = fx.detach().clone().requires_grad_(True)
        tot = sum(_three(mods, a, b, F_))
        tot.backward(retain_graph=True)
        g1 = F_.grad.clone()
        F_.grad = None
        tot.backward()
        return g1, F_.grad
    (g1, g2), (r1, r2) = twice(fh), twice(fh.float())
    for g, r in ((g1, r1), (g2, r2)):
        assert g.dtype == dtype and torch.equal(g, r.to(dtype))

    # no gradient wanted: the forward-only kernel
    with torch.no_grad():
        c0 = L.launch_counts()
        lh = _three(mods, a, b, fh)
        c1 = L.launch_counts()
        lr = _three(mods, a, b, fh.float())
    assert c1['loss_fwd'] - c0['loss_fwd'] == 1 and c1['loss_single_pass'] == c0['loss_single_pass'], (c0, c1)
    for x, y in zip(lh, lr):
        assert torch.equal(x, y)

    # large upstream gradients (a GradScaler scale): the float16 products overflow to +-inf exactly where .to() does
    for scale in (65536.0, 2.0 ** 30):
        def scaled(l1, l2, l3):
            ((l1 + l2 + l3) * scale).backward()
        got, ref = _run(mods, a, b, fh, scaled), _run(mods, a, b, fh.float(), scaled)
        _check(got, ref, dtype)
        if dtype == torch.float16 and scale == 2.0 ** 30:
            assert torch.isinf(got[1]).any()


def test_launch_counts_of_a_training_step():
    L, ML = _mods()
    mods = _objective(ML)
    a, b, f = (t.cuda() for t in _inputs('rand_3x64x96'))
    _run(mods, a, b, f.to(torch.bfloat16), _total)       # warm-up (tensor maps, first-use attributes)
    _run(mods, a, b, f, _total)
    keys = ('loss_fwd', 'loss_single_pass', 'loss_bwd', 'rescale', 'aux')

    def delta(fx):
        c0 = L.launch_counts()
        _run(mods, a, b, fx, _total)
        c1 = L.launch_counts()
        return {k: c1[k] - c0[k] for k in keys}
    # bfloat16 imgf, float32 sources (autocast): widen + single pass + narrow, nothing else
    assert delta(f.to(torch.bfloat16)) == {'loss_fwd': 0, 'loss_single_pass': 1, 'loss_bwd': 0, 'rescale': 0, 'aux': 2}
    # float32: the single pass and its in-place rescale, as before
    assert delta(f) == {'loss_fwd': 0, 'loss_single_pass': 1, 'loss_bwd': 0, 'rescale': 1, 'aux': 0}


class _Net(torch.nn.Module):
    def __init__(self):
        super().__init__()
        self.c1 = torch.nn.Conv2d(2, 8, 3, padding=1)
        self.c2 = torch.nn.Conv2d(8, 1, 3, padding=1)

    def forward(self, a, b):
        return self.c2(torch.relu(self.c1(torch.cat([a, b], dim=1))))


@pytest.mark.parametrize('dtype', HALF, ids=['bf16', 'f16'])
def test_autocast_training_loop(dtype):
    L, ML = _mods()
    mods = _objective(ML)
    torch.manual_seed(3)
    net = _Net().cuda()
    opt = torch.optim.Adam(net.parameters(), lr=1e-3)
    scaler = torch.amp.GradScaler('cuda') if dtype == torch.float16 else None
    g = torch.Generator(device='cuda').manual_seed(4)
    a, b = (torch.rand(4, 1, 64, 80, device='cuda', generator=g) for _ in range(2))
    losses = []
    for _ in range(4):
        opt.zero_grad(set_to_none=True)
        with torch.autocast('cuda', dtype=dtype):
            f = net(a, b)
            assert f.dtype == dtype
            tot = sum(_three(mods, a, b, f))
        if scaler is None:
            tot.backward()
            for p in net.parameters():
                assert p.grad is not None and torch.isfinite(p.grad).all()
            opt.step()
        else:
            scaler.scale(tot).backward()
            scaler.step(opt)
            scaler.update()
        losses.append(tot.item())
    assert all(np.isfinite(losses)), losses


def _modules_cases(ML):
    """(label, callable(img1, img2, imgf) -> scalar or tuple, which inputs want a gradient)"""
    out = []
    for mode in ('ssim', 'w-ssim', 'ms-ssim', 'msw-ssim'):
        for pad in (False, True):
            m = ML.SSIMLoss(mode, use_padding=pad)
            out.append((f'SSIMLoss-{mode}-pad{int(pad)}', lambda x, y, f, m=m: m(x, y, f), (2,)))
    d = ML.SSIM()
    out.append(('SSIM-dict', lambda x, y, f, d=d: sum(v.sum() for v in d(x, f).values()), (0, 2)))
    d7 = ML.SSIM(win_size=7, use_padding=True)
    out.append(('SSIM-dict-win7-pad', lambda x, y, f, d=d7: sum(v.sum() for v in d(x, f).values()), (2,)))
    mp = ML.SSIM(size_average=False)
    out.append(('SSIM-maps', lambda x, y, f, m=mp: sum(v.sum() for v in m(x, f).values()), (0, 2)))
    out.append(('calc_ssim', lambda x, y, f: ML.calc_ssim(x, f, win_size=5)['ssim'].sum(), (2,)))
    out.append(('calc_msssim', lambda x, y, f: ML.calc_msssim(x, f).sum(), (2,)))
    ms = ML.MS_SSIM(use_padding=True)
    out.append(('MS_SSIM-pad', lambda x, y, f, m=ms: m(x, f).sum(), (2,)))
    for sa in (False, True):
        mw = ML.MSW_SSIM(size_average=sa)
        out.append((f'MSW_SSIM-avg{int(sa)}', lambda x, y, f, m=mw: m(x, y, f), (2,)))
    for nm in ('l1', 'l2'):
        tv, nl = ML.TVLoss(nm, weight=0.5), ML.NormLoss(nm, weight=0.5)
        out.append((f'TVLoss-{nm}', lambda x, y, f, m=tv: m(f), (2,)))
        out.append((f'NormLoss-{nm}', lambda x, y, f, m=nl: m(f), (2,)))
    return out


def _module_run(fn, ins, wants):
    xs = [t.detach().clone().requires_grad_(k in wants) for k, t in enumerate(ins)]
    v = fn(*xs)
    v.backward()
    return v.detach(), [xs[k].grad for k in wants]


def test_other_modules_equal_float32_path():
    L, ML = _mods()
    g = torch.Generator().manual_seed(11)
    a, b, f = (torch.rand(2, 1, 180, 200, generator=g).cuda() for _ in range(3))
    ah, bh, fh = (t.to(torch.bfloat16) for t in (a, b, f))
    for label, fn, wants in _modules_cases(ML):
        vr, gr = _module_run(fn, (ah.float(), bh.float(), fh.float()), wants)
        vh, gh = _module_run(fn, (ah, bh, fh), wants)
        assert torch.equal(vh, vr), (label, vh, vr)
        for k, x, r in zip(wants, gh, gr):
            assert x.dtype == torch.bfloat16, (label, k, x.dtype)
            assert torch.equal(x, r.to(torch.bfloat16)), (label, k, (x.float() - r).abs().max().item())
    # the no-gradient forms: the SSIM dict through the fused launch, the maps through the map kernel
    with torch.no_grad():
        for fn in (lambda x, y: ML.SSIM()(x, y), lambda x, y: ML.SSIM(size_average=False)(x, y)):
            dh, dr = fn(ah, fh), fn(ah.float(), fh.float())
            for k in ('ssim', 'cs', 'sigma'):
                assert torch.equal(dh[k], dr[k]), k


def test_bf16_training_step_captures_into_a_cuda_graph():
    L, ML = _mods()
    mods = _objective(ML)
    g = torch.Generator().manual_seed(21)
    a0, b0, f0 = (torch.rand(4, 1, 96, 160, generator=g).cuda() for _ in range(3))
    a1, b1, f1 = (torch.rand(4, 1, 96, 160, generator=g).cuda() for _ in range(3))
    sa, sb = a0.clone(), b0.clone()
    sf = f0.to(torch.bfloat16).requires_grad_(True)

    def step(A, B_, F_):
        tot = sum(_three(mods, A, B_, F_))
        tot.backward()
        return tot

    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(3):
            sf.grad = None
            step(sa, sb, sf)
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    sf.grad = None
    with torch.cuda.graph(graph):
        stot = step(sa, sb, sf)
    for A, B_, F_ in ((a1, b1, f1), (a0, b0, f0)):
        sa.copy_(A)
        sb.copy_(B_)
        with torch.no_grad():
            sf.copy_(F_.to(torch.bfloat16))
        graph.replay()
        torch.cuda.synchronize()
        Fe = F_.to(torch.bfloat16).requires_grad_(True)
        etot = step(A, B_, Fe)
        assert stot.item() == etot.item()
        assert sf.grad.dtype == torch.bfloat16 and torch.equal(sf.grad, Fe.grad)


def test_other_dtypes_and_host_tensors_still_raise():
    L, ML = _mods()
    x = torch.rand(1, 1, 32, 32, device='cuda')
    mods = _objective(ML)
    for bad in (x.double(), (x * 255).to(torch.int32), (x * 255).to(torch.uint8)):
        with pytest.raises(L.MmifError):
            _three(mods, x, x, bad)
        with pytest.raises(L.MmifError):
            ML.SSIMLoss('w-ssim')(x, x, bad)
        with pytest.raises(L.MmifError):
            ML.SSIM()(x, bad)
        with pytest.raises(L.MmifError):
            ML.TVLoss()(bad)
        with pytest.raises(L.MmifError):
            ML.NormLoss()(bad)
    with pytest.raises(L.MmifError):
        _three(mods, x, x.double(), x.to(torch.bfloat16))      # a float64 source too
    h = x.cpu().to(torch.bfloat16)
    with pytest.raises(L.MmifError, match='CUDA'):
        _three(mods, h, h, h)
    with pytest.raises(L.MmifError, match='CUDA'):
        ML.NormLoss()(h)
    from mmif_b200.core import metric as MM
    with pytest.raises(L.MmifError, match='float32 expected'):
        MM.calc_ssim(x.to(torch.bfloat16), x)
