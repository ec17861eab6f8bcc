"""How a loss + gradient launch cuts the images into CTAs, checked on the kernels themselves against the fp64 oracle.

bwd_geom() (csrc/fusion_loss.cu) picks per shape `nstrip` strips of 108 gradient columns, `n_tall` tall segments of T rows
followed by short segments of s rows and, for the warp-specialised kernel, a fine class: the last F strips of every
sample cut into `nsf` segments of `fr` rows.  Each kernel decodes its CTA index into (class, segment, sample, strip) and
derives from it the first row, the segment height, the batch count and the partial-sum slot of the single-pass loss sums.
A wrong term there either leaves rows unwritten, owns them twice (the loss sums count them twice) or makes two CTAs share
a partial-sum slot.  The shapes of the other GPU tests reach only uniform segments without a fine class or a single fine
strip, so this file runs every such class on purpose:
  1. forced geometries (MMIF_WS_GEOM) on the warp-specialised kernel, in all five of its instantiations;
  2. the 2-CTA kernel on a shape where its own search gives mixed tall + short segments, on every launch it still serves;
  3. the per-rank batches bench.py launches (8 and 64 x 3072 x 4096);
  4. (no GPU) a guard that the shapes and strings used here still reach every class.
Every output starts as NaN, so an element no CTA writes fails the finiteness check."""
import contextlib
import ctypes

import numpy as np
import pytest
import torch

import gates
from oracle import fusion_loss as OL
from test_single_pass_gpu import W3, check_block, check_total_grad

gpu = pytest.mark.gpu

# MmifLossCfg modes (pixel_combine, grad_combine, pixel_norm, grad_norm): the training objective (the FAST
# instantiations) and the general Sobel path (warp-specialised up to 32 Mpix per launch, 2-CTA above)
FAST = ('max', 'max', 'l1', 'l1')
GENERAL = ('avg', 'avg', 'l2', 'l2')
UPSTREAM = (1.5, -0.25, 3.0)          # unequal upstream gradients: mmif_fusion_loss_bwd recomputes

# instantiation of fusion_loss_ws_kernel<WIN, FAST, ZMODE> -> (modes, want_grad, upstream)
INSTS = {'<11,true,2>': (FAST, 2, None), '<11,true,1>': (FAST, 1, None), '<11,true,0>': (FAST, 0, UPSTREAM),
         '<11,false,1>': (GENERAL, 1, None), '<11,false,0>': (GENERAL, 0, UPSTREAM)}

# MMIF_WS_GEOM="T,n_tall,s[,F,fr]" -> what it decodes to at 611 / 613 rows: (nseg, n_tall, T, s, F, fr, nsf)
FORCED = {
    '16,0,16': (39, 0, 16, 16, 0, None, None),          # 16-row segments everywhere (2 batches of 8 rows + halo)
    '64,3,24': (21, 3, 64, 24, 0, None, None),          # mixed tall + short, ragged last segment
    '616,1,616': (1, 1, 616, 616, 0, None, None),       # one segment for the whole image
    '128,2,40,1,48': (11, 2, 128, 40, 1, 48, 13),       # mixed + one fine strip
    '96,7,96,2,32': (7, 7, 96, 96, 2, 32, 20),          # two fine strips
    '200,3,200,3,16': (4, 3, 200, 200, 3, 16, 39),      # three fine strips of 16 rows
    '64,2,136,1,616': (6, 2, 64, 136, 1, 616, 1),       # short taller than tall; a single-segment fine class
}
# 2 x 611 x 976: TMA ring, a last strip 4 columns wide, a ragged last segment; 1 x 613 x 1001: plain-load ring (W % 4 != 0)
FORCED_SHAPES = [(2, 611, 976), (1, 613, 1001)]
# candidates for the 2-CTA kernel's mixed geometry; the first one its search cuts into tall + short segments is used
TWO_CTA_CANDIDATES = [(8, 256, 2048), (8, 384, 1500), (8, 777, 1000), (4, 384, 3000)]
GENERAL_2CTA_SHAPE = (3, 3072, 4096)      # above 32 Mpix: the general modes run on the 2-CTA kernel without any switch
# per-rank batches of bench.py (global batch 64 of 3072 x 4096) on 8 ranks and on 1, and the samples whose whole gradient
# is compared with the oracle
BENCH = {(8, 3072, 4096): (0, 7), (64, 3072, 4096): (0, 31, 63)}


def _mods():
    import mmif_b200  # noqa: F401
    from mmif_b200 import _lib as L
    from mmif_b200.core import loss as ML
    return L, ML


def geometry(B, H, W, kernel=1):
    """mmif_loss_geometry: (nstrip, nseg, n_tall, T, s, F, fr, nsf, CTAs per sample, strip width); kernel 1 = the
    warp-specialised kernel, 0 = the 2-CTA kernel."""
    L, _ = _mods()
    out = (ctypes.c_int * 10)()
    L.check(L.load().mmif_loss_geometry(B, H, W, kernel, out))
    return tuple(out)


def is_mixed(g):
    return 0 < g[2] < g[1] and g[3] != g[4]


def two_cta_mixed_shape():
    for shape in TWO_CTA_CANDIDATES:
        g = geometry(*shape, kernel=0)
        if is_mixed(g):
            return shape, g
    pytest.fail(f'the 2-CTA search cuts none of {TWO_CTA_CANDIDATES} into tall + short segments: pick new shapes')


def assert_decodes_to(g, want, what):
    nseg, n_tall, T, s, F, fr, nsf = want
    assert g[1:6] == (nseg, n_tall, T, s, F) and (F == 0 or g[6:8] == (fr, nsf)), (what, g, want)


@contextlib.contextmanager
def no_tf32():
    keep = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    try:
        yield
    finally:
        torch.backends.cudnn.allow_tf32 = keep


def make_inputs(shape, device='cpu'):
    """continuous random pairs with f = 0.5 (a + b) + noise: L1 sign ties are rare"""
    B, H, W = shape
    g = torch.Generator(device=device).manual_seed(B * 1000003 + H * 1009 + W)
    a, b, n = (torch.rand(B, 1, H, W, device=device, generator=g) for _ in range(3))
    f = 0.5 * (a + b) + 0.2 * (n - 0.5)
    return a.cuda(), b.cuda(), f.cuda()


def secondary_terms(a, b, f, modes):
    pc, gc, pn, gn = modes
    return OL.pixel_loss(a, b, f, pn, W3[1], pc), OL.grad_loss(a, b, f, gn, W3[2], gc)


def oracle_terms(a, b, f, modes):
    return (OL.ssim_loss(a, b, f, 'ssim', weight=W3[0]), *secondary_terms(a, b, f, modes))


def ssim_dict(a, b, f):
    """per-sample (ssim, cs, sigma) of (a, f) and of (b, f): the order of the loss block's per-sample entries, (6, B)"""
    w = OL.window2d(11, 1.5)
    d1, d2 = OL.ssim(a, f, window=w, data_range=1.0), OL.ssim(b, f, window=w, data_range=1.0)
    return torch.stack([d1['ssim'], d1['cs'], d1['sigma'], d2['ssim'], d2['cs'], d2['sigma']]).double().cpu().numpy()


def launch(a, b, f, modes, want_grad, upstream=None):
    """One launch through the C ABI, with the workspace size queried now (it follows a forced geometry).
    upstream None: mmif_fusion_loss_fwd(want_grad) -> (loss block + float32 mirror, dF_unit);
    otherwise mmif_fusion_loss_bwd with those upstream gradients -> (None, dF).  Outputs start as NaN."""
    L, ML = _mods()
    lib = L.load()
    B, _, H, W = f.shape
    st = L.stream_ptr(f.device)
    cfg = ML._cfg(1.0, *modes, *W3)
    ws = torch.zeros(lib.mmif_loss_workspace_bytes(B, H, W), dtype=torch.uint8, device='cuda')
    g = torch.full_like(f, float('nan'))
    before = L.launch_counts()
    if upstream is None:
        cfg.want_grad = want_grad
        out = torch.full((lib.mmif_loss_out_doubles(B),), float('nan'), dtype=torch.float64, device='cuda')
        L.check(lib.mmif_fusion_loss_fwd(a.data_ptr(), b.data_ptr(), f.data_ptr(), B, H, W, ctypes.byref(cfg), out.data_ptr(),
                                         g.data_ptr(), ws.data_ptr(), ws.numel(), st))
        counter = 'loss_single_pass'
    else:
        up = torch.tensor(upstream, dtype=torch.float32, device='cuda')
        L.check(lib.mmif_fusion_loss_bwd(a.data_ptr(), b.data_ptr(), f.data_ptr(), B, H, W, ctypes.byref(cfg), up.data_ptr(), None,
                                         g.data_ptr(), ws.data_ptr(), ws.numel(), st))
        out, counter = None, 'loss_bwd'
    torch.cuda.synchronize()
    assert L.launch_counts()[counter] == before[counter] + 1
    return out, g


# ------------------------------------------------------------------------------------------------ small-shape checks
_ORACLE = {}


def oracle(shape, modes):
    """inputs and the whole-batch oracle of one shape and mode set (cached): fp32 and fp64 loss values, per-sample SSIM
    dicts, fp64 per-term gradients and the fp32 per-term gradients (numpy)"""
    key = (shape, modes)
    if key not in _ORACLE:
        a, b, f = make_inputs(shape)
        with no_tf32():
            f32 = f.clone().requires_grad_(True)
            t32 = oracle_terms(a, b, f32, modes)
            g32 = np.stack([torch.autograd.grad(t, f32, retain_graph=True)[0].cpu().numpy() for t in t32])
            ad, bd = a.double(), b.double()
            fd = f.double().requires_grad_(True)
            t64 = oracle_terms(ad, bd, fd, modes)
            g64 = np.stack([torch.autograd.grad(t, fd, retain_graph=True)[0].cpu().numpy() for t in t64])
            with torch.no_grad():
                d32, d64 = ssim_dict(a, b, f), ssim_dict(ad, bd, fd)
        _ORACLE[key] = dict(abf=(a, b, f), np=tuple(t.cpu().numpy() for t in (a, b, f)), r32=[t.item() for t in t32],
                            r64=[t.item() for t in t64], d32=d32, d64=d64, g32=g32, g64=g64)
    return _ORACLE[key]


def check_vs_oracle(name, inst, out, g, ref):
    """every element written; loss block and per-sample entries against the fp32 / fp64 oracle; the gradient through the
    tie-aware gate of the single-pass tests"""
    modes, want_grad, upstream = INSTS[inst]
    got = g.cpu().numpy()
    assert np.isfinite(got).all(), f'{name}: {int((~np.isfinite(got)).sum())} gradient elements not written'
    a, b, f = ref['np']
    B = f.shape[0]
    if upstream is None:
        nd = 4 + 6 * B
        blk = out[:nd].cpu().numpy()
        mirror = out[nd:].view(torch.float32)[:nd].cpu().numpy()
        check_block(name, blk, mirror, ref['r32'], ref['r64'], *((ref['d32'], ref['d64']) if want_grad == 1 else ()))
        if want_grad == 2:        # the SSIM means per sample; cs / sigma are not summed
            ps = blk[4:].reshape(B, 6)
            for n in range(B):
                for j in (0, 3):
                    gates.assert_scalar(f'{name}/dict[{j},{n}]', ps[n, j], ref['d32'][j, n], ref['d64'][j, n])
            assert (ps[:, [1, 2, 4, 5]] == 0).all()
        up = (1.0, 1.0, 1.0)
    else:
        up = upstream
    w = np.asarray(up).reshape(3, 1, 1, 1, 1)
    check_total_grad(name, got, a, b, f, w * ref['g64'], (w * ref['g32']).sum(axis=0),
                     w=tuple(abs(u) * x for u, x in zip(up, W3)))


def check_consistent(name, res, base):
    """a geometry may move only the per-segment tile-shift constants: loss block to 1e-6, gradient to 2e-6 of max|g|"""
    (o, g), (o0, g0) = res, base
    if o is not None:
        nd = 4 + 6 * g.shape[0]
        rel = ((o[:nd] - o0[:nd]).abs() / o0[:nd].abs().clamp_min(1e-12)).max().item()
        assert rel <= 1e-6, f'{name}: loss block differs from the automatic geometry by {rel:.3e}'
    err = (g - g0).abs().max().item() / g0.abs().max().item()
    assert err <= 2e-6, f'{name}: gradient differs from the automatic geometry by {err:.3e} of max|g|'


_AUTO = {}


def auto_run(shape, inst):
    if (shape, inst) not in _AUTO:
        modes, want_grad, upstream = INSTS[inst]
        _AUTO[shape, inst] = launch(*oracle(shape, modes)['abf'], modes, want_grad, upstream)
    return _AUTO[shape, inst]


@gpu
@pytest.mark.parametrize('geom', ['auto'] + list(FORCED))
@pytest.mark.parametrize('inst', list(INSTS))
@pytest.mark.parametrize('shape', FORCED_SHAPES, ids=lambda s: 'x'.join(map(str, s)))
def test_warp_specialised_kernel_forced_geometry_vs_fp64_oracle(shape, inst, geom, monkeypatch):
    """fusion_loss_ws_kernel under each forced row-segment geometry (and the automatic one) against the fp64 oracle, and
    against the automatic geometry's outputs."""
    monkeypatch.delenv('MMIF_LOSS_WS', raising=False)
    monkeypatch.delenv('MMIF_WS_GEOM', raising=False)
    modes, want_grad, upstream = INSTS[inst]
    ref = oracle(shape, modes)
    auto_geo = geometry(*shape)
    base = auto_run(shape, inst)
    name = f'{shape} {inst} {geom}'
    if geom == 'auto':
        res = base
    else:
        monkeypatch.setenv('MMIF_WS_GEOM', geom)
        g = geometry(*shape)
        assert_decodes_to(g, FORCED[geom], 'the forced geometry did not take effect')
        res = launch(*ref['abf'], modes, want_grad, upstream)
        monkeypatch.delenv('MMIF_WS_GEOM')
        assert geometry(*shape) == auto_geo, 'a forced geometry was left in the memo'
        name += f' -> {g[:8]}'
    check_vs_oracle(name, inst, *res, ref)
    if geom != 'auto':
        check_consistent(name, res, base)


# ------------------------------------------------------------------------------------- the 2-CTA kernel, mixed segments
@gpu
@pytest.mark.parametrize('inst', ['<11,true,1>', '<11,true,0>'])
def test_two_cta_kernel_on_its_mixed_geometry(inst, monkeypatch):
    """fusion_loss_bwd_kernel (MMIF_LOSS_WS=0) where its search cuts tall + short segments: the single pass and the
    recomputing backward against the fp64 oracle and against the warp-specialised kernel."""
    shape, g0 = two_cta_mixed_shape()
    modes, want_grad, upstream = INSTS[inst]
    ref = oracle(shape, modes)
    monkeypatch.delenv('MMIF_WS_GEOM', raising=False)
    monkeypatch.setenv('MMIF_LOSS_WS', '0')
    res = launch(*ref['abf'], modes, want_grad, upstream)
    monkeypatch.setenv('MMIF_LOSS_WS', '1')
    name = f'{shape} 2-CTA {inst} {g0[:5]}'
    check_vs_oracle(name, inst, *res, ref)
    check_consistent(name, res, launch(*ref['abf'], modes, want_grad, upstream))


def oracle_per_sample(a, b, f, modes, grad_samples=()):
    """The fp64 oracle one sample at a time (every loss term is a mean over the whole batch, every sample has the same
    size): the three batch loss values, the per-sample SSIM dicts (6, B) and, for the listed samples, d(total)/d imgf =
    the single sample's gradient / B."""
    B = f.shape[0]
    vals, dic, grads = np.zeros((3, B)), np.zeros((6, B)), {}
    with no_tf32():
        for n in range(B):
            x1, x2, y = (t[n:n + 1].double() for t in (a, b, f))
            with torch.no_grad():
                dic[:, n] = ssim_dict(x1, x2, y)[:, 0]
                pix, grd = secondary_terms(x1, x2, y, modes)
            # SSIMLoss('ssim') of one sample from its two SSIM means (what OL.ssim_loss computes), without a second pass
            vals[:, n] = [W3[0] * (1.0 - 0.5 * (dic[0, n] + dic[3, n])), pix.item(), grd.item()]
            if n in grad_samples:
                yd = y.clone().requires_grad_(True)
                grads[n] = torch.autograd.grad(sum(oracle_terms(x1, x2, yd, modes)), yd)[0][0] / B
    return vals.mean(axis=1), dic, grads


def check_large(name, out, g, ref, want_grad):
    """loss head and per-sample entries to 1e-5 of the fp64 oracle, every element finite, the whole gradient of the
    sampled images: at most 1e-4 of the elements beyond 1e-5 max|g| (L1 sign ties), median error below 1e-6 max|g|"""
    vals, dic, grads = ref
    B = g.shape[0]
    assert torch.isfinite(g).all(), f'{name}: gradient elements not written'
    blk = out[:4 + 6 * B].cpu().numpy()
    assert np.isfinite(blk).all()
    for k, nm in enumerate(('ssim', 'pixel', 'grad')):
        gates.assert_scalar(f'{name}/{nm}', blk[k], vals[k], vals[k])
    ps = blk[4:].reshape(B, 6)
    for j in (range(6) if want_grad == 1 else (0, 3)):
        for n in range(B):
            gates.assert_scalar(f'{name}/dict[{j},{n}]', ps[n, j], dic[j, n], dic[j, n])
    for n, g64 in grads.items():
        d = (g[n].double() - g64).abs()
        scale = g64.abs().max()
        frac = (d > 1e-5 * scale).double().mean().item()
        assert frac <= 1e-4, f'{name} sample {n}: {frac:.2e} of the elements beyond 1e-5 max|g|, max {(d.max() / scale).item():.3e}'
        assert (d.median() / scale).item() < 1e-6, f'{name} sample {n}: median error {(d.median() / scale).item():.3e}'


@gpu
def test_two_cta_kernel_general_modes_above_32_mpix(monkeypatch):
    """avg / l2 on their real route: above 32 Mpix per launch they run on fusion_loss_bwd_kernel<11, false, true, false>,
    whose search cuts this shape into tall + short segments."""
    monkeypatch.delenv('MMIF_LOSS_WS', raising=False)
    B, H, W = GENERAL_2CTA_SHAPE
    assert B * H * W > 32 << 20
    g0 = geometry(B, H, W, kernel=0)
    assert is_mixed(g0), g0
    a, b, f = make_inputs(GENERAL_2CTA_SHAPE, device='cuda')
    out, g = launch(a, b, f, GENERAL, 1)
    check_large(f'{GENERAL_2CTA_SHAPE} 2-CTA general {g0[:5]}', out, g, oracle_per_sample(a, b, f, GENERAL, range(B)), 1)


@gpu
@pytest.mark.parametrize('mode', ['w-ssim', 'ms-ssim', 'msw-ssim'])
def test_extended_ssim_losses_on_the_two_cta_mixed_geometry(mode):
    """The SSIM-only extended backward launches ('w-ssim', MS-SSIM level 0, the 11-tap window of 'msw-ssim') run on
    the 2-CTA kernel; through the drop-in module on the shape where it cuts tall + short segments, against the oracle
    on the GPU (loss through the parity gate; gradient: see the gate below)."""
    L, ML = _mods()
    shape, _ = two_cta_mixed_shape()
    a, b, f = make_inputs(shape)
    F_ = f.clone().requires_grad_(True)
    ln = ML.SSIMLoss(mode)(a, b, F_)
    c0 = L.launch_counts()
    gn, = torch.autograd.grad(ln, F_)
    assert L.launch_counts()['ssim_bwd_ext'] > c0['ssim_bwd_ext']
    assert torch.isfinite(gn).all()
    with no_tf32():
        f32 = f.clone().requires_grad_(True)
        l32 = OL.ssim_loss(a, b, f32, mode)
        g32, = torch.autograd.grad(l32, f32)
        fd = f.double().requires_grad_(True)
        l64 = OL.ssim_loss(a.double(), b.double(), fd, mode)
        g64, = torch.autograd.grad(l64, fd)
    gates.assert_scalar(f'{shape} {mode}', ln.item(), l32.item(), l64.item())
    scale = g64.abs().max()
    d = (gn.double() - g64).abs() / scale
    ref_err = ((g32.double() - g64).abs().max() / scale).item()
    # The 3-tap window of 'msw-ssim' has local variances ~0.002 against E[x^2] ~0.33, so an fp32 variance loses ~160 ulp
    # and ANY fp32 evaluation reaches ~1e-5 max|g| at a few scattered elements (the fp32 oracle: 1.2e-5 here, at 2e-6 of
    # the elements).  Two fp32 evaluations draw that tail independently, so the tail may reach twice the fp32 oracle's
    # error; the bulk is held to the gate of the full-size test.  A decoding defect misplaces or drops whole rows: O(1).
    mx, frac, med = d.max().item(), (d > gates.RTOL).double().mean().item(), d.median().item()
    assert mx <= max(gates.RTOL, 2 * ref_err), f'{shape} {mode}: grad max-norm err {mx:.3e} (fp32 oracle: {ref_err:.3e})'
    assert frac <= 1e-4 and med < 1e-6, f'{shape} {mode}: {frac:.2e} of the elements beyond 1e-5 max|g|, median {med:.2e}'


# ------------------------------------------------------------------------------------------------ the benchmarked launches
@gpu
@pytest.mark.parametrize('shape', list(BENCH), ids=lambda s: 'x'.join(map(str, s)))
def test_benchmarked_launches_vs_fp64_oracle(shape, monkeypatch):
    """The launches bench.py times (want_grad = 2, as the drop-in passes) and want_grad = 1 with the per-sample entries,
    against the oracle evaluated one sample at a time."""
    monkeypatch.delenv('MMIF_LOSS_WS', raising=False)
    monkeypatch.delenv('MMIF_WS_GEOM', raising=False)
    geo = geometry(*shape)
    a, b, f = make_inputs(shape, device='cuda')
    ref = oracle_per_sample(a, b, f, FAST, BENCH[shape])
    res = {}
    for wg in (2, 1):
        out, g = launch(a, b, f, FAST, wg)
        check_large(f'{shape} <11,true,{wg}> {geo[:8]}', out, g, ref, wg)
        res[wg] = (out, g)
    (o2, g2), (o1, g1) = res[2], res[1]
    assert torch.equal(g1, g2) and torch.equal(o1[:4], o2[:4])


# ------------------------------------------------------------------------------------------------ coverage guard (no GPU)
def owned_once(H, nseg, n_tall, T, s):
    rows = np.zeros(H, dtype=np.int32)
    for seg in range(nseg):
        i0 = seg * T if seg < n_tall else n_tall * T + (seg - n_tall) * s
        rows[i0:min(i0 + (T if seg < n_tall else s), H)] += 1
    return (rows == 1).all()


def test_geometry_coverage_of_the_gpu_tests(monkeypatch):
    """The geometries the GPU tests above launch still reach every class of the CTA decoding.  A retune of the geometry
    search that moves them onto easier geometries fails here, on a machine without a GPU."""
    monkeypatch.delenv('MMIF_WS_GEOM', raising=False)
    ws = []                                     # (shape, geometry) of every warp-specialised launch above
    for shape in FORCED_SHAPES:
        ws.append((shape, geometry(*shape)))
        for s, want in FORCED.items():
            monkeypatch.setenv('MMIF_WS_GEOM', s)
            g = geometry(*shape)
            assert_decodes_to(g, want, (shape, s))
            assert owned_once(shape[1], *g[1:5]) and (g[5] == 0 or owned_once(shape[1], g[7], g[7], g[6], g[6])), (shape, s, g)
            ws.append((shape, g))
        monkeypatch.delenv('MMIF_WS_GEOM')
    bench = [geometry(*shape) for shape in BENCH]
    ws += list(zip(BENCH, bench))
    assert {g[5] for _, g in ws} >= {0, 1, 2, 3}, 'fine classes of 0, 1, 2 and 3 strips'
    assert any(g[2] == g[1] > 1 for _, g in ws), 'all segments tall'
    assert any(g[2] == 0 and g[1] > 1 for _, g in ws), 'all segments short'
    assert any(is_mixed(g) and g[3] > g[4] for _, g in ws) and any(is_mixed(g) and g[3] < g[4] for _, g in ws), 'mixed'
    assert any(g[1] == 1 for _, g in ws), 'one segment for the whole image'
    assert any(g[3] == g[4] == 16 for _, g in ws), '16-row segments'
    assert any(W % 4 and W % 108 for (_, _, W), _ in ws), 'the plain-load ring and a ragged last strip'
    assert any(W % 4 == 0 and W % 108 for (_, _, W), _ in ws), 'the TMA ring with a ragged last strip'
    # bench.py's per-rank batches: full-height coarse strips plus a fine class of several segments (DESIGN.md section 4)
    assert sorted(BENCH) == [(8, 3072, 4096), (64, 3072, 4096)]
    for g in bench:
        assert g[1] == g[2] == 1 and g[5] >= 1 and g[7] > 1, g
    # the 2-CTA kernel
    two_cta_mixed_shape()
    B, H, W = GENERAL_2CTA_SHAPE
    assert B * H * W > 32 << 20 and is_mixed(geometry(B, H, W, kernel=0))
