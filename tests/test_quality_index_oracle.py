"""CPU checks of oracle/quality_index.py (Piella's Q / Q_W / Q_E and Yang's Q_Y) on cases that can be worked out by
hand, and the agreement of its float32 and float64 evaluations on the golden metric cases."""
import numpy as np
import pytest
import torch

import cases
from oracle import quality_index as QI

D = torch.float64


def _u8(seed, h=24, w=30, n=1):
    return torch.from_numpy(np.random.default_rng(seed).integers(0, 256, (n, 1, h, w)).astype(np.float64))


def test_q0_of_an_image_with_itself_is_one():
    x = _u8(1)
    mx, my, vx, vy, cxy = QI.box_moments(x, x)
    q = QI.q0(mx, my, vx, vy, cxy)
    assert (vx > 0).all()
    assert torch.allclose(q, torch.ones_like(q), rtol=0, atol=1e-12)


@pytest.mark.parametrize('dt', [torch.float32, torch.float64])
def test_identical_images_score_one(dt):
    a = _u8(2, 40, 52, n=2).to(dt)
    r = QI.quality_indices(a, a, a)
    tol = 1e-12 if dt == torch.float64 else 1e-5
    for k in ('q', 'qw', 'qe', 'qy'):
        assert abs(r[k].item() - 1.0) <= tol, (k, r[k].item())


def test_swapping_the_sources_changes_nothing():
    a, b, f = _u8(3), _u8(4), _u8(5)
    r1, r2 = QI.quality_indices(a, b, f), QI.quality_indices(b, a, f)
    for k in r1:
        assert r1[k].item() == pytest.approx(r2[k].item(), rel=1e-14, abs=1e-15), k


def test_degenerate_q0_branches():
    one = lambda v: torch.full((1, 1, 8, 8), float(v), dtype=D)
    cb = torch.tensor([[(-1.0) ** (i + j) for j in range(8)] for i in range(8)], dtype=D)[None, None]
    # both windows constant (variance sum 0), means 3 and 5: 2 mx my / (mx^2 + my^2)
    assert QI.q0(*QI.box_moments(one(3), one(5))).item() == pytest.approx(2 * 15 / 34, abs=1e-15)
    # zero means, non-zero variances (checkerboards of +-1 and +-2): 2 cov / (vx + vy)
    assert QI.q0(*QI.box_moments(cb, 2 * cb)).item() == pytest.approx(2 * 2 / (1 + 4), abs=1e-15)
    # both sums 0 (all-zero windows): 1
    assert QI.q0(*QI.box_moments(one(0), one(0))).item() == 1.0
    # both sums non-zero: the full formula on a hand case (x = 1 + cb, y = 1 - cb: mu 1, var 1, cov -1 -> -1)
    assert QI.q0(*QI.box_moments(1 + cb, 1 - cb)).item() == pytest.approx(-1.0, abs=1e-15)


def test_weight_is_one_half_at_zero_saliency_and_weighted_q_falls_back_to_q():
    z = torch.zeros(3, dtype=D)
    assert QI.weight(z, z).tolist() == [0.5, 0.5, 0.5]
    assert QI.weight(torch.tensor([1.0], dtype=D), torch.tensor([3.0], dtype=D)).item() == 0.25
    a = torch.full((1, 1, 16, 20), 40.0, dtype=D)
    b = torch.full((1, 1, 16, 20), 90.0, dtype=D)
    f = _u8(6, 16, 20)
    term, c = QI.piella_terms(a, b, f)
    assert c.sum().item() == 0.0
    r = QI.quality_indices(a, b, f)
    assert r['qw'].item() == r['q'].item()
    # the edge images of constant sources are all zero as well: Q_E = Q_W * Q(a', b', f')
    ea, eb, ef = QI.edges(a), QI.edges(b), QI.edges(f)
    assert ea.abs().max().item() == 0.0 and eb.abs().max().item() == 0.0
    assert r['qe'].item() == pytest.approx(r['qw'].item() * QI.piella_q(ea, eb, ef).item(), rel=1e-14)


def test_box_part_of_q_by_hand_on_11x11():
    a, b, f = _u8(7, 11, 11), _u8(8, 11, 11), _u8(9, 11, 11)
    A, B, Fz = (x[0, 0].numpy() for x in (a, b, f))
    terms = []
    for i in range(4):
        for j in range(4):
            wa, wb, wf = (x[i:i + 8, j:j + 8].ravel() for x in (A, B, Fz))

            def q0(x, y):
                mx, my = x.mean(), y.mean()
                vx, vy = ((x - mx) ** 2).mean(), ((y - my) ** 2).mean()
                cxy = ((x - mx) * (y - my)).mean()
                return 4 * cxy * mx * my / ((vx + vy) * (mx * mx + my * my))

            sa, sb = wa.var(), wb.var()
            lam = sa / (sa + sb)
            terms.append(lam * q0(wa, wf) + (1 - lam) * q0(wb, wf))
    assert len(terms) == 16
    assert QI.piella_q(a, b, f).item() == pytest.approx(np.mean(terms), rel=1e-12)


def test_batch_is_one_population():
    a, b, f = _u8(10, n=3), _u8(11, n=3), _u8(12, n=3)
    r = QI.quality_indices(a, b, f)
    term, c = QI.piella_terms(a, b, f)
    assert r['q'].item() == pytest.approx(term.mean().item(), rel=1e-14)
    assert r['qw'].item() == pytest.approx(((c * term).sum() / c.sum()).item(), rel=1e-14)
    per = [QI.yang_qy(a[i:i + 1], b[i:i + 1], f[i:i + 1]).item() for i in range(3)]
    assert r['qy'].item() == pytest.approx(np.mean(per), rel=1e-13)     # equal window counts per pair


# Measured largest float32-vs-float64 differences on these cases: Q_W 4e-7 and Q_E 2e-7 relative; Q 7e-6 relative on
# ir_crop (near-flat 8x8 windows of an infrared image, where E[x^2] - mu^2 in float32 keeps ~1e-3 of a variance that is
# ~1e-2); Q_Y 4e-6 on natural_flat_97x131 (the metric SSIM maps' own float32 arithmetic, as oracle.fusion_metric.ssim).
@pytest.mark.parametrize('name', cases.METRIC_CASES)
def test_float32_and_float64_agree_on_the_golden_cases(name):
    a, b, f = (torch.from_numpy(x) for x in cases.metric_case(name))
    r32 = QI.quality_indices(a, b, f)
    r64 = QI.quality_indices(a.double(), b.double(), f.double())
    for k, tol in (('q', 1e-5), ('qw', 1e-6), ('qe', 1e-6), ('qy', 1e-5)):
        assert abs(r32[k].item() - r64[k].item()) <= tol * max(abs(r64[k].item()), 1e-2), (k, r32[k].item(), r64[k].item())
