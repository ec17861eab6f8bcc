"""Oracle of the window-based fusion quality indices: Piella & Heijmans' Q, Q_W and Q_E (ICIP 2003) and Yang et al.'s
Q_Y (Information Fusion 2008), as surveyed by Liu et al. (TPAMI 2012).  There is no reference implementation of these
indices in the reference code base, so this module is their definition.  Plain torch ops, dtype-generic: float32 inputs
give the float32 arithmetic, float64 inputs the truth.

Conventions.  Images a, b (sources) and f (fused) are float32 (N,1,H,W) with nominal values 0..255.

- Box moments.  w ranges over every valid 8x8 window: stride 1, no padding, (H-7)(W-7) positions.  Weights are 1/64.
  sigma^2 is the population variance (divide by 64); sigma_xy is the population covariance.
- Q0 (Wang-Bovik universal index).  Q0(x,y|w) = 4 sigma_xy mu_x mu_y / ((sigma_x^2+sigma_y^2)(mu_x^2+mu_y^2)).
  Degenerate cases follow Wang's img_qi.m:
  - variance sum 0 and mean-square sum != 0: 2 mu_x mu_y / (mu_x^2+mu_y^2);
  - variance sum != 0 and mean-square sum 0: 2 sigma_xy / (sigma_x^2+sigma_y^2);
  - both 0: 1.
- Saliency.  s(x|w) = sigma_x^2.
- Weight lambda.  lambda(w) = s(a|w) / (s(a|w) + s(b|w)), or 0.5 when both are 0.
- Q = mean over w of [lambda Q0(a,f|w) + (1-lambda) Q0(b,f|w)].
- Q_W = sum_w c(w) [lambda Q0(a,f|w) + (1-lambda) Q0(b,f|w)].  Here c(w) = C(w) / sum C and
  C(w) = max(s(a|w), s(b|w)).  When sum C = 0, Q_W = Q.
- Q_E = Q_W(a,b,f) * Q_W(a',b',f').  Here x' = sqrt(gx^2 + gy^2) is the Sobel magnitude of metric.py:192-206: reflect
  pad, fp32 (the exponent alpha = 1).
- Q_Y.  S(x,y|w) is the metric SSIM map (11-tap Gaussian, sigma 1.5, C1 = (0.01*255)^2, C2 = (0.03*255)^2, valid).
  lambda is formed as above from that window's Gaussian variances.  Q_Y = mean over w of:
  - lambda S(a,f) + (1-lambda) S(b,f) where S(a,b|w) >= 0.75;
  - max(S(a,f), S(b,f)) elsewhere.
- Batches (N > 1).  One population, as every reference metric here (metric._combine_batch):
  - Q and Q_Y: mean over all windows of all pairs.
  - Q_W: sum C over the whole batch.
  - Q_E: the product of the two batch-wide Q_W values.
- Shapes.  H, W >= 11 (the Q_Y window).

Two arithmetic details that leave the definitions unchanged: the box moments are taken of x - min(x) per sample (the
variances and covariances do not depend on the shift, and it keeps E[x^2] - mu^2 from cancelling in float32), and a
variance that rounding makes negative is clamped at 0 (as the SSIM maps clamp theirs).

TEST INFRASTRUCTURE — see ``oracle/__init__.py``.
"""
import torch
import torch.nn.functional as F

from .fusion_loss import blur
from .fusion_metric import metric_window, sobel_polar

BOX = 8
QY_WIN = 11
QY_THRESHOLD = 0.75


def _box(x):
    return F.avg_pool2d(x, BOX, stride=1)


def box_moments(x, y):
    """(mu_x, mu_y, var_x, var_y, cov_xy) maps over every valid 8x8 window, (N,1,H-7,W-7)."""
    cx = x.amin(dim=(-2, -1), keepdim=True)
    cy = y.amin(dim=(-2, -1), keepdim=True)
    u, v = x - cx, y - cy
    mu_u, mu_v = _box(u), _box(v)
    var_u = (_box(u * u) - mu_u * mu_u).clamp(min=0)
    var_v = (_box(v * v) - mu_v * mu_v).clamp(min=0)
    cov = _box(u * v) - mu_u * mu_v
    return mu_u + cx, mu_v + cy, var_u, var_v, cov


def q0(mx, my, vx, vy, cxy):
    """Wang-Bovik universal index per window with img_qi.m's degenerate branches."""
    vs, ms = vx + vy, mx * mx + my * my
    one = torch.ones_like(vs)
    full = 4.0 * cxy * mx * my / torch.where((vs == 0) | (ms == 0), one, vs * ms)
    lum = 2.0 * mx * my / torch.where(ms == 0, one, ms)
    struct = 2.0 * cxy / torch.where(vs == 0, one, vs)
    out = torch.where((vs != 0) & (ms != 0), full, torch.where(vs == 0, lum, struct))
    return torch.where((vs == 0) & (ms == 0), one, out)


def weight(sa, sb):
    """lambda = sa / (sa + sb), 0.5 where both saliencies are 0."""
    d = sa + sb
    return torch.where(d == 0, torch.full_like(d, 0.5), sa / torch.where(d == 0, torch.ones_like(d), d))


def piella_terms(a, b, f):
    """(term, C) maps: term = lambda Q0(a,f) + (1-lambda) Q0(b,f), C = max(s(a), s(b))."""
    ma, mfa, va, vfa, caf = box_moments(a, f)
    mb, mfb, vb, vfb, cbf = box_moments(b, f)
    lam = weight(va, vb)
    term = lam * q0(ma, mfa, va, vfa, caf) + (1.0 - lam) * q0(mb, mfb, vb, vfb, cbf)
    return term, torch.maximum(va, vb)


def edges(x):
    """Sobel magnitude of metric.py:192-206 (reflect pad)."""
    return sobel_polar(x)[0]


def _weighted(term, c):
    sc = c.sum()
    return term.mean() if sc == 0 else (c * term).sum() / sc


def piella_q(a, b, f):
    return piella_terms(a, b, f)[0].mean()


def piella_qw(a, b, f):
    return _weighted(*piella_terms(a, b, f))


def piella_qe(a, b, f):
    return piella_qw(a, b, f) * piella_qw(edges(a), edges(b), edges(f))


def ssim_parts(x, y, data_range=255.0):
    """Metric SSIM map of (x, y) and the clamped Gaussian variances of x and y, each (N,1,H-10,W-10)
    (metric.py:316-364 with the 11-tap window, as oracle.fusion_metric.ssim)."""
    w = metric_window(QY_WIN).to(x)
    mu_x, mu_y = blur(x, w), blur(y, w)
    xx, yy, xy = mu_x * mu_x, mu_y * mu_y, mu_x * mu_y
    var_x = (blur(x * x, w) - xx).clamp(min=0)
    var_y = (blur(y * y, w) - yy).clamp(min=0)
    cov = blur(x * y, w) - xy
    c1, c2 = (0.01 * data_range) ** 2, (0.03 * data_range) ** 2
    s = ((2.0 * xy + c1) * (2.0 * cov + c2)) / ((xx + yy + c1) * (var_x + var_y + c2))
    return s, var_x, var_y


def yang_terms(a, b, f):
    """Per-window Q_Y terms and the S(a,b) map that selects between the two forms."""
    s_af, va, _ = ssim_parts(a, f)
    s_bf, vb, _ = ssim_parts(b, f)
    s_ab = ssim_parts(a, b)[0]
    lam = weight(va, vb)
    blend = lam * s_af + (1.0 - lam) * s_bf
    return torch.where(s_ab >= QY_THRESHOLD, blend, torch.maximum(s_af, s_bf)), s_ab, blend, torch.maximum(s_af, s_bf)


def yang_qy(a, b, f):
    return yang_terms(a, b, f)[0].mean()


def quality_indices(a, b, f):
    """dict q, qw, qe, qy (0-dim tensors of the input dtype) of the batch as one population."""
    term, c = piella_terms(a, b, f)
    eterm, ec = piella_terms(edges(a), edges(b), edges(f))
    qw = _weighted(term, c)
    return {'q': term.mean(), 'qw': qw, 'qe': qw * _weighted(eterm, ec), 'qy': yang_qy(a, b, f)}


def qy_tie_slack(a, b, f, tol=1e-5):
    """Largest change of Q_Y that rounding of S(a,b) across the 0.75 threshold can cause: the windows whose float64
    S(a,b) lies within `tol` of it, each moved from one form to the other, over the window count."""
    q, s_ab, blend, mx = yang_terms(a.double(), b.double(), f.double())
    near = (s_ab - QY_THRESHOLD).abs() <= tol
    return float(((blend - mx).abs() * near).sum() / q.numel())
