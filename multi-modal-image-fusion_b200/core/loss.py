"""Drop-in mirror of the reference ``core/loss.py`` call surface on the B200 kernels.

Same class names, constructor arguments, ``forward`` signatures, return types and error
behaviour as the reference (loss.py:16-19); the arithmetic runs in libmmif_b200.so.  The three
training modules share ONE launch per step: the first of ``SSIMLoss / PixelLoss / GradLoss`` called on a
new (img1, img2, imgf) triple launches the single-pass kernel (the three loss values AND
d(l1 + l2 + l3)/d imgf when imgf wants a gradient; the forward-only kernel otherwise), the other two read
their scalar from the same result (memo keyed on tensor identity and version), and a single autograd node
with three outputs receives all three upstream gradients: ``total.backward()`` is an in-place rescale that
exits at once for unit upstream; unequal upstream gradients or a retained graph recompute.

Built on the same kernels: 'w-ssim' (per-sample gamma weights in the backward kernel), 'ms-ssim'
(one SSIM forward/backward launch per pyramid level + pooling adjoints), use_padding=True (reflect-pad
operator + its adjoint, applied per pyramid level / per window for 'ms-ssim' / 'msw-ssim'), size_average=False
(SSIM / CS / sigma maps), data_range=None auto-detect, TVLoss and NormLoss forward/backward, SSIM(win_size) for the
windows 11/9/7/5/3 on the strip kernels and for ANY other window of 2..17 taps (odd or even) on the generic kernels
(mmif_ssim_generic_*), with a dict that is differentiable w.r.t. both images through all three entries, per-sample or as
size_average=False maps.  'msw-ssim' runs the same forward / backward kernels with the 11/9/7/5/3 windows and per-position
weights.  Every module takes float32, bfloat16 or float16 images (an autocast training step): a bfloat16 / float16 input is
widened to float32 on the device on entry (exact, so the values are those of the float32 path on img.float()) and its
gradient is narrowed from float32 to the input's dtype by mmif_narrow on exit.  Not built (raise NotImplementedError, never a
silent fallback): gradients of the fused objective w.r.t. the sources, SSIM windows above 17 taps, MS_SSIM(size_average=False), MSW_SSIM(size_average=False) with windows other than 11/9/7/5/3.
"""
import ctypes
import threading
import weakref

import torch
import torch.nn as nn

from .. import _lib as L

__all__ = ['SSIM', 'MS_SSIM', 'MSW_SSIM', 'SSIMLoss', 'PixelLoss', 'GradLoss', 'TVLoss', 'NormLoss']

eps = 1e-7


def _cfg(data_range, pixel_combine, grad_combine, pixel_norm, grad_norm, w_ssim=1.0, w_pixel=1.0, w_grad=1.0):
    c = L.MmifLossCfg()
    c.w_ssim, c.w_pixel, c.w_grad = float(w_ssim), float(w_pixel), float(w_grad)
    c.data_range = float(data_range)
    c.pixel_combine, c.grad_combine = L.COMBINE[pixel_combine], L.COMBINE[grad_combine]
    c.pixel_norm, c.grad_norm = L.NORM[pixel_norm], L.NORM[grad_norm]
    return c


_cfg_structs = {}


def _cfg_ref(cfg_key, want_grad):
    """(struct, byref, address) for a configuration: built once — a training loop presents the same one every step."""
    k = (cfg_key, want_grad)
    hit = _cfg_structs.get(k)
    if hit is None:
        c = _cfg(*cfg_key)
        c.want_grad = 2 if want_grad else 0       # 2: the modules read the three loss values only (include/mmif_b200.h)
        hit = _cfg_structs[k] = (c, ctypes.byref(c), ctypes.addressof(c))
        if len(_cfg_structs) > 256:
            _cfg_structs.pop(next(iter(_cfg_structs)))
    return hit


_ws_bytes = {}


def _loss_ws(lib, dev, stream, B, H, W):
    n = _ws_bytes.get((B, H, W))
    if n is None:
        n = _ws_bytes[(B, H, W)] = lib.mmif_loss_workspace_bytes(B, H, W)
    if n == 0:
        raise L.MmifError(f'unsupported shape {(B, H, W)}: H and W must be >= 11')
    return L.workspace(dev, n, 'loss', (B, H, W), stream)


class _FusedObjective(torch.autograd.Function):
    """(img1, img2, imgf) -> (w1 (1 - mean ssim), w2 pixel norm, w3 grad norm, per-sample ssim dict block).

    `want_grad` is decided by the CALLER (`_Memo.lookup`), where the user's grad mode is visible — inside
    `Function.forward` grad mode is always off.  With it the forward runs the single-pass kernel (loss values AND
    d(l1+l2+l3)/d imgf in one launch); backward then only rescales that buffer if the three upstream gradients are
    equal — decided on the device, so there is no host sync — and recomputes otherwise (unequal upstream, or the
    second backward of a retained graph: the buffer is handed to autograd by the first)."""

    @staticmethod
    def forward(ctx, img1, img2, imgf, cfg_key, want_grad):
        lib = L.load()
        x1, B, H, W = L.as_loss_f32_3d(img1, 'img1')
        x2, _, _, _ = L.as_loss_f32_3d(img2, 'img2')
        y, _, _, _ = L.as_loss_f32_3d(imgf, 'imgf')
        if x2.shape != x1.shape or y.shape != x1.shape:
            raise L.MmifError(f'shape mismatch: {tuple(img1.shape)} {tuple(img2.shape)} {tuple(imgf.shape)}')
        dev = y.device
        L.ensure_device(dev)
        want_grad = bool(want_grad and ctx.needs_input_grad[2])
        _, cref, caddr = _cfg_ref(cfg_key, want_grad)
        dF_unit = torch.empty_like(y) if want_grad else None
        nd = L.LOSS_HEAD + L.LOSS_PER_SAMPLE * B
        out = torch.empty(nd + (nd + 1) // 2, dtype=torch.float64, device=dev)
        stream = L.stream_int(dev)
        ws = _loss_ws(lib, dev, stream, B, H, W)
        fc = L.fastcall()
        L.call(dev, fc.loss_fwd if fc is not None else lib.mmif_fusion_loss_fwd, x1.data_ptr(), x2.data_ptr(), y.data_ptr(), B, H, W,
               caddr if fc is not None else cref, out.data_ptr(), dF_unit.data_ptr() if want_grad else None, ws.data_ptr(),
               ws.numel(), stream)
        # a bfloat16 / float16 input is kept as it came: only a recomputing backward needs its float32 widening again
        ctx.save_for_backward(*(x if t.dtype == torch.float32 else t for t, x in ((img1, x1), (img2, x2), (imgf, y))))
        ctx.dF_unit = dF_unit
        ctx.single_pass = want_grad          # which kernel served the forward (the tests assert on it)
        ctx.cfg_key, ctx.dims, ctx.in_shape = cfg_key, (B, H, W), imgf.shape
        ctx.set_materialize_grads(False)
        out32 = out[nd:].view(torch.float32)          # the kernel's own float32 mirror of the block: no conversion launches
        _memo.vec = out32[:4]
        per_sample = out32[L.LOSS_HEAD:nd].view(B, L.LOSS_PER_SAMPLE)
        ctx.mark_non_differentiable(per_sample)
        return out32[0], out32[1], out32[2], per_sample

    @staticmethod
    def backward(ctx, g_ssim, g_pix, g_grad, _g_ps):
        lib = L.load()
        s1, s2, sf = ctx.saved_tensors
        B, H, W = ctx.dims
        dev, dtype = sf.device, sf.dtype
        ups, ptrs = [], []
        for g in (g_ssim, g_pix, g_grad):       # device scalars as autograd hands them over: no stack / zeros launches
            if g is None:
                ptrs.append(None)
                continue
            if g.dtype != torch.float32 or g.device != dev:
                g = g.to(device=dev, dtype=torch.float32)
            g = g.contiguous()
            ups.append(g)
            ptrs.append(g.data_ptr())
        if not ups:
            return None, None, torch.zeros(ctx.in_shape, dtype=dtype, device=dev), None, None
        _, cref, caddr = _cfg_ref(ctx.cfg_key, False)
        # The single-pass buffer is consumed by the first backward: it is rescaled IN PLACE (nothing to do at all for
        # the unit upstream of total.backward()) and handed to autograd; a second backward (retain_graph) recomputes.
        unit, ctx.dF_unit = ctx.dF_unit, None
        tok = getattr(ctx, 'memo_token', None)
        if tok is not None:
            tok[0] = False          # this graph has been backpropagated: a later call on the same tensors builds a fresh one
        if dtype != torch.float32 and unit is not None and ptrs[0] is not None and ptrs[0] == ptrs[1] == ptrs[2]:
            # total.backward() of a bfloat16 / float16 imgf (the same pointer test as mmif_fusion_loss_bwd3): the rescale of the
            # single-pass buffer and the narrowing are one launch, the whole backward
            return None, None, L.narrow_grad(unit, dtype, ups[0]).view(ctx.in_shape), None, None
        x1, x2, y = (s if s.dtype == torch.float32 else L.as_loss_f32(s) for s in (s1, s2, sf))
        dF = unit if unit is not None else torch.empty_like(y)
        stream = L.stream_int(dev)
        ws = _loss_ws(lib, dev, stream, B, H, W)
        fc = L.fastcall()
        L.call(dev, fc.loss_bwd3 if fc is not None else lib.mmif_fusion_loss_bwd3, x1.data_ptr(), x2.data_ptr(), y.data_ptr(), B, H, W,
               caddr if fc is not None else cref, ptrs[0], ptrs[1], ptrs[2], unit.data_ptr() if unit is not None else None,
               dF.data_ptr(), ws.data_ptr(), ws.numel(), stream)
        return None, None, L.narrow_grad(dF, dtype).view(ctx.in_shape), None, None


SINGLE_PASS = True   # set False to force the two-kernel (forward, then recomputing backward) path


class _Memo(threading.local):
    """One-entry memo PER THREAD so loss_fn1/2/3 called back to back (train.py:64-68) cost one launch."""

    def __init__(self):
        self.key, self.refs, self.value, self.vec, self.token = None, None, None, None, None
        # what the sibling modules asked for last time: the guess for the next fused launch
        self.hint = {'pixel': ('max', 'l1'), 'grad': ('max', 'l1'), 'data_range': 1.0,
                     'w_ssim': 1.0, 'w_pixel': 0.01, 'w_grad': 0.1}

    def lookup(self, img1, img2, imgf, cfg_key):
        want_grad = bool(SINGLE_PASS and imgf.requires_grad and torch.is_grad_enabled())    # the CALLER's grad mode
        key = (img1.data_ptr(), img1._version, img2.data_ptr(), img2._version, imgf.data_ptr(), imgf._version,
               imgf.shape, imgf.device, imgf.dtype, cfg_key, imgf.requires_grad and torch.is_grad_enabled(), want_grad)
        # a hit needs the same tensors (identity + version) AND a graph that has not been backpropagated yet: the reference
        # builds a new graph on every call, so loss(...).backward() twice on the same tensors must keep working
        if self.key == key and self.token[0] and all(r() is t for r, t in zip(self.refs, (img1, img2, imgf))):
            return self.value
        if img1.requires_grad or img2.requires_grad:
            raise NotImplementedError('gradients w.r.t. the source images are not built (train.py never needs them)')
        value = _FusedObjective.apply(img1, img2, imgf, cfg_key, want_grad)
        self.token = [True]
        if value[0].grad_fn is not None:
            value[0].grad_fn.memo_token = self.token          # shared with the backward (which runs on autograd's thread)
        self.key, self.value = key, value
        self.refs = tuple(weakref.ref(t) for t in (img1, img2, imgf))
        return value


_memo = _Memo()


def last_loss_vector():
    """The float32 device vector [l_ssim, l_pixel, l_grad, l_ssim + l_pixel + l_grad] the most recent fused launch of this
    thread wrote (a view of the kernel's output block, no copy): what train.py:92-96 all-reduces as four separate scalars
    is ONE 16-byte vector here — see dist_utils.reduce_loss_vector."""
    if _memo.vec is None:
        raise L.MmifError('no fused loss has been computed on this thread yet')
    return _memo.vec


def ingest_u8(img_u8, device=None, out=None):
    """uint8 image tensor (host — pinned for an asynchronous copy — or device) -> float32 device tensor img / 255, the
    scaling data/dataset.py applies on the host, bit-identical (IEEE float32 division on the device): a quarter of the
    host->device bytes for the sources of a training step."""
    lib = L.load()
    if img_u8.dtype != torch.uint8:
        raise L.MmifError(f'uint8 expected, got {img_u8.dtype}')
    dev = img_u8.device if img_u8.is_cuda else (torch.device(device) if device is not None else torch.device('cuda', torch.cuda.current_device()))
    L.ensure_device(dev)
    src = img_u8.contiguous().to(dev, non_blocking=True)
    dst = out if out is not None else torch.empty(src.shape, dtype=torch.float32, device=dev)
    L.call(dev, lib.mmif_widen_u8_unit, src.data_ptr(), src.numel(), dst.data_ptr(), L.stream_int(dev))
    return dst


def _fused(img1, img2, imgf, data_range=None, pixel=None, grad=None, w_ssim=None, w_pixel=None, w_grad=None):
    if not (img1.is_cuda and img2.is_cuda and imgf.is_cuda):
        for t, nm in ((img1, 'img1'), (img2, 'img2'), (imgf, 'imgf')):
            L.require_cuda(t, nm)
    h = _memo.hint
    if data_range is not None:
        h['data_range'] = float(data_range)
    if pixel is not None:
        h['pixel'] = pixel
    if grad is not None:
        h['grad'] = grad
    if w_ssim is not None:
        h['w_ssim'] = float(w_ssim)
    if w_pixel is not None:
        h['w_pixel'] = float(w_pixel)
    if w_grad is not None:
        h['w_grad'] = float(w_grad)
    cfg_key = (h['data_range'], h['pixel'][0], h['grad'][0], h['pixel'][1], h['grad'][1], h['w_ssim'], h['w_pixel'], h['w_grad'])
    return _memo.lookup(img1, img2, imgf, cfg_key)


SSIM_WINDOWS = (11, 9, 7, 5, 3)     # windows the SSIM kernels are instantiated for (the MSW_SSIM set, loss.py:214)


def _fwd_per_sample(x1, x2, y, data_range, win=11):
    """SSIM-only forward (no gradient, no pixel / Sobel terms) -> (B, 6) float64 per-sample means:
    ssim1, cs1, sigma1, ssim2, cs2, sigma2."""
    lib = L.load()
    B, H, W = y.shape
    dev = y.device
    if win not in SSIM_WINDOWS or min(H, W) < 11:   # any other window / an image under 11 pixels: the generic kernels, one pair at a time
        return torch.cat([_generic_fwd(x1, y, data_range, win), _generic_fwd(x2, y, data_range, win)], dim=1)
    out = torch.empty(lib.mmif_loss_out_doubles(B), dtype=torch.float64, device=dev)
    nws = lib.mmif_loss_workspace_bytes(B, H, W)
    if nws == 0:
        raise L.MmifError(f'unsupported shape {(B, H, W)}: H and W must be >= 11 at every level')
    ws = L.workspace(dev, nws, 'loss', (B, H, W))
    L.call(dev, lib.mmif_ssim_fwd_win, x1.data_ptr(), x2.data_ptr(), y.data_ptr(), B, H, W, int(win), float(data_range),
           out.data_ptr(), ws.data_ptr(), ws.numel(), L.stream_int(dev))
    return out[L.LOSS_HEAD:L.LOSS_HEAD + B * L.LOSS_PER_SAMPLE].view(B, L.LOSS_PER_SAMPLE)


def _ssim_bwd_ex(x1, x2, y, data_range, gout1, pair_w, cs_only, scale, win=11):
    lib = L.load()
    B, H, W = y.shape
    dev = y.device
    if win not in SSIM_WINDOWS or min(H, W) < 11:   # generic kernels: per-sample upstream (of the window MEAN) = gout1 * scale * pair weight
        dF = None
        for k, src in enumerate((x1, x2)):
            g = (gout1.to(torch.float32).reshape(1) * float(scale)).expand(B)
            if pair_w is not None:
                g = g * pair_w[:, k].to(torch.float32)
            _, d = _generic_bwd(src, y, data_range, win, None if cs_only else g, g if cs_only else None, None, False, False, True)
            dF = d if dF is None else dF.add_(d)
        return dF
    dF = torch.empty_like(y)
    ws = L.workspace(dev, lib.mmif_loss_workspace_bytes(B, H, W), 'loss', (B, H, W))
    pw = pair_w.to(torch.float32).contiguous() if pair_w is not None else None
    with torch.cuda.device(dev):
        L.check(lib.mmif_ssim_bwd_ex_win(x1.data_ptr(), x2.data_ptr(), y.data_ptr(), B, H, W, int(win), float(data_range),
                                         gout1.data_ptr(), pw.data_ptr() if pw is not None else None, int(cs_only), float(scale),
                                         dF.data_ptr(), ws.data_ptr(), ws.numel(), L.stream_ptr(dev)))
    return dF


def _prep3(img1, img2, imgf):
    for t, nm in ((img1, 'img1'), (img2, 'img2'), (imgf, 'imgf')):
        L.require_cuda(t, nm)
    if img1.requires_grad or img2.requires_grad:
        raise NotImplementedError('gradients w.r.t. the source images are not built (train.py never needs them)')
    x1, B, H, W = L.as_loss_f32_3d(img1.detach(), 'img1')
    x2, _, _, _ = L.as_loss_f32_3d(img2.detach(), 'img2')
    y, _, _, _ = L.as_loss_f32_3d(imgf.detach(), 'imgf')
    if x2.shape != x1.shape or y.shape != x1.shape:
        raise L.MmifError(f'shape mismatch: {tuple(img1.shape)} {tuple(img2.shape)} {tuple(imgf.shape)}')
    L.ensure_device(y.device)
    return x1.view(B, H, W), x2.view(B, H, W), y.view(B, H, W)


class _WeightedSSIM(torch.autograd.Function):
    """SSIMLoss('w-ssim') (loss.py:259-266): gamma_b = sigma1_b / (sigma1_b + sigma2_b) comes from the
    SOURCE images only, so it is a per-sample constant of the backward."""

    @staticmethod
    def forward(ctx, img1, img2, imgf, data_range, win=11):
        x1, x2, y = _prep3(img1, img2, imgf)
        ps = _fwd_per_sample(x1, x2, y, data_range, win).to(torch.float32)
        gamma = ps[:, 2] / (ps[:, 2] + ps[:, 5]).clamp_(min=eps)
        ctx.save_for_backward(x1, x2, y, gamma)
        ctx.data_range, ctx.in_shape, ctx.win, ctx.dtype = data_range, imgf.shape, win, imgf.dtype
        return (gamma * ps[:, 0]).mean() + ((1.0 - gamma) * ps[:, 3]).mean()

    @staticmethod
    def backward(ctx, g):
        x1, x2, y, gamma = ctx.saved_tensors
        pw = torch.stack([gamma, 1.0 - gamma], dim=1)
        g1 = g.to(torch.float32).reshape(1).contiguous()
        dF = _ssim_bwd_ex(x1, x2, y, ctx.data_range, g1, pw, 0, 1.0 / y.shape[0], ctx.win)
        return None, None, L.narrow_grad(dF, ctx.dtype).view(ctx.in_shape), None, None


def _loss_sigma(win):
    return 1.5 if win == 11 else 0.15 * (win - 1)        # loss.py:34


def _generic_fwd(x, y, data_range, win, want_maps=False, sigma=None):
    """mmif_ssim_generic_fwd on (B,H,W) device tensors -> (B,3) float64 per-sample [ssim, cs, sigma], or the three maps.
    sigma: the window's Gaussian sigma, by default the loss rule (the metric functions pass 1.5)."""
    lib = L.load()
    B, H, W = y.shape
    dev = y.device
    sigma = _loss_sigma(win) if sigma is None else sigma
    L.ensure_window_taps(win, sigma)
    if want_maps:
        maps = [torch.empty(B, 1, H - win + 1, W - win + 1, dtype=torch.float32, device=dev) for _ in range(3)]
        L.call(dev, lib.mmif_ssim_generic_fwd, x.data_ptr(), y.data_ptr(), B, H, W, int(win), float(sigma), float(data_range), None,
               maps[0].data_ptr(), maps[1].data_ptr(), maps[2].data_ptr(), None, 0, L.stream_int(dev))
        return maps
    per = torch.empty(B, 3, dtype=torch.float64, device=dev)
    ws = L.workspace(dev, lib.mmif_ssim_generic_workspace_bytes(B, H, W, int(win)), 'ssim_generic', (B, H, W, int(win)))
    L.call(dev, lib.mmif_ssim_generic_fwd, x.data_ptr(), y.data_ptr(), B, H, W, int(win), float(sigma), float(data_range), per.data_ptr(),
           None, None, None, ws.data_ptr(), ws.numel(), L.stream_int(dev))
    return per


def _generic_bwd(x, y, data_range, win, g_ssim, g_cs, g_sigma, maps, want_dx, want_dy, sigma=None):
    """mmif_ssim_generic_bwd: upstream gradients (per-sample (B,) or per-position maps, any may be None) -> (dx, dy).
    sigma: the window's Gaussian sigma, by default the loss rule (the metric functions pass 1.5)."""
    lib = L.load()
    B, H, W = y.shape
    dev = y.device
    sigma = _loss_sigma(win) if sigma is None else sigma
    L.ensure_window_taps(win, sigma)
    gs = [None if g is None else g.to(device=dev, dtype=torch.float32).contiguous() for g in (g_ssim, g_cs, g_sigma)]
    coef = torch.empty(lib.mmif_ssim_generic_coef_doubles(B, H, W, int(win)), dtype=torch.float64, device=dev)
    dx = torch.empty_like(x) if want_dx else None
    dy = torch.empty_like(y) if want_dy else None
    L.call(dev, lib.mmif_ssim_generic_bwd, x.data_ptr(), y.data_ptr(), B, H, W, int(win), float(sigma), float(data_range),
           *(None if g is None else g.data_ptr() for g in gs), 1 if maps else 0, dx.data_ptr() if want_dx else None,
           dy.data_ptr() if want_dy else None, coef.data_ptr(), L.stream_int(dev))
    return dx, dy


class _SSIMGeneric(torch.autograd.Function):
    """calc_ssim of the loss module (loss.py:52-110) for ANY window size and either output form, differentiable w.r.t. both
    images and through all three entries — the complete, slower path (direct k x k evaluation) behind SSIM(win_size=...)
    for windows other than 11/9/7/5/3, for images smaller than the window (the reference shrinks the window to
    min(win, H, W), loss.py:67-71), and for gradients through the size_average=False maps."""

    @staticmethod
    def forward(ctx, img1, img2, data_range, win, size_average):
        x, B, H, W = L.as_loss_f32_3d(img1.detach(), 'img1')
        y, _, _, _ = L.as_loss_f32_3d(img2.detach(), 'img2')
        if y.shape != x.shape:
            raise L.MmifError(f'shape mismatch: {tuple(img1.shape)} {tuple(img2.shape)}')
        L.ensure_device(x.device)
        x, y = x.view(B, H, W), y.view(B, H, W)
        k = min(int(win), H, W)                                    # loss.py:67-71
        ctx.save_for_backward(x, y)
        ctx.meta = (data_range, k, bool(size_average), img1.shape, img2.shape)
        ctx.dtypes = (img1.dtype, img2.dtype)
        ctx.set_materialize_grads(False)
        if size_average:
            per = _generic_fwd(x, y, data_range, k).to(torch.float32)
            return per[:, 0].contiguous(), per[:, 1].contiguous(), per[:, 2].contiguous()
        return tuple(_generic_fwd(x, y, data_range, k, want_maps=True))

    @staticmethod
    def backward(ctx, g_ssim, g_cs, g_sigma):
        x, y = ctx.saved_tensors
        data_range, k, size_average, s1, s2 = ctx.meta
        if g_ssim is None and g_cs is None and g_sigma is None:
            return None, None, None, None, None
        dx, dy = _generic_bwd(x, y, data_range, k, g_ssim, g_cs, g_sigma, not size_average, ctx.needs_input_grad[0],
                              ctx.needs_input_grad[1])
        return (L.narrow_grad(dx, ctx.dtypes[0]).view(s1) if dx is not None else None), \
            (L.narrow_grad(dy, ctx.dtypes[1]).view(s2) if dy is not None else None), None, None, None


class _PlainSSIM(torch.autograd.Function):
    """mean_b (ssim(img1, imgf) + ssim(img2, imgf)) / 2 with gradient w.r.t. imgf: the SSIM-only kernels (no pixel /
    Sobel work) — what SSIMLoss('ssim', use_padding=True) needs after its reflect padding."""

    @staticmethod
    def forward(ctx, img1, img2, imgf, data_range):
        x1, x2, y = _prep3(img1, img2, imgf)
        ps = _fwd_per_sample(x1, x2, y, data_range).to(torch.float32)
        ctx.save_for_backward(x1, x2, y)
        ctx.data_range, ctx.in_shape, ctx.dtype = data_range, imgf.shape, imgf.dtype
        return (ps[:, 0].mean() + ps[:, 3].mean()) * 0.5

    @staticmethod
    def backward(ctx, g):
        x1, x2, y = ctx.saved_tensors
        g1 = g.to(torch.float32).reshape(1).contiguous()
        pw = torch.full((y.shape[0], 2), 0.5, dtype=torch.float32, device=y.device)
        dF = _ssim_bwd_ex(x1, x2, y, ctx.data_range, g1, pw, 0, 1.0 / y.shape[0])
        return None, None, L.narrow_grad(dF, ctx.dtype).view(ctx.in_shape), None


class _SSIMDict(torch.autograd.Function):
    """SSIM.forward (loss.py:163-185 -> calc_ssim, loss.py:52-110) with size_average=True, differentiable:
    (img1, img2) -> per-sample (ssim, cs, sigma).  SSIM and CS are symmetric in their arguments, so the gradient
    w.r.t. either image is the 'fused image' gradient of the SSIM-only backward kernel with the other image as the
    source and the upstream per-sample gradients as pair weights; sigma = clamp(var(img1), 1e-4) does not depend on img2."""

    @staticmethod
    def forward(ctx, img1, img2, data_range, win=11):
        x, B, H, W = L.as_loss_f32_3d(img1.detach(), 'img1')
        y, _, _, _ = L.as_loss_f32_3d(img2.detach(), 'img2')
        if y.shape != x.shape:
            raise L.MmifError(f'shape mismatch: {tuple(img1.shape)} {tuple(img2.shape)}')
        L.ensure_device(x.device)
        x, y = x.view(B, H, W), y.view(B, H, W)
        ps = _fwd_per_sample(x, x, y, data_range, win).to(torch.float32)
        ctx.save_for_backward(x, y)
        ctx.data_range, ctx.shape1, ctx.shape2, ctx.win = data_range, img1.shape, img2.shape, win
        ctx.dtypes = (img1.dtype, img2.dtype)
        ctx.set_materialize_grads(False)
        return ps[:, 0].clone(), ps[:, 1].clone(), ps[:, 2].clone()

    @staticmethod
    def backward(ctx, g_ssim, g_cs, g_sigma):
        x, y = ctx.saved_tensors
        one = torch.ones(1, dtype=torch.float32, device=x.device)

        def wrt(src, tgt):          # d/d tgt of sum_n g_ssim[n] ssim_n + g_cs[n] cs_n
            out = None
            for g, cs_only in ((g_ssim, 0), (g_cs, 1)):
                if g is None:
                    continue
                pw = torch.stack([g.to(torch.float32).reshape(-1), torch.zeros_like(g, dtype=torch.float32).reshape(-1)], dim=1)
                d = _ssim_bwd_ex(src, src, tgt, ctx.data_range, one, pw, cs_only, 1.0, ctx.win)
                out = d if out is None else out + d
            return out if out is not None else torch.zeros_like(tgt)

        g1 = g2 = None
        if ctx.needs_input_grad[1]:
            g2 = L.narrow_grad(wrt(x, y), ctx.dtypes[1]).view(ctx.shape2)
        if ctx.needs_input_grad[0]:
            g1 = wrt(y, x) if (g_ssim is not None or g_cs is not None) else None
            if g_sigma is not None:             # sigma = clamp(var(img1), 1e-4) depends on img1 only: the generic backward
                ds, _ = _generic_bwd(x, y, ctx.data_range, ctx.win, None, None, g_sigma.reshape(-1), False, True, False)
                g1 = ds if g1 is None else g1.add_(ds)
            g1 = L.narrow_grad(g1, ctx.dtypes[0]).view(ctx.shape1) if g1 is not None else None
        return g1, g2, None, None


def _pad_raw(x, pad):
    """(B,H,W) -> reflect-padded (B,H+2p,W+2p); F.pad(.., 'reflect') of use_padding=True (loss.py:45-47)."""
    lib = L.load()
    B, H, W = x.shape
    if pad >= H or pad >= W:
        raise L.MmifError(f'reflect padding {pad} needs H, W > {pad}, got {(H, W)} (torch raises here too)')
    out = torch.empty(B, H + 2 * pad, W + 2 * pad, dtype=torch.float32, device=x.device)
    with torch.cuda.device(x.device):
        L.check(lib.mmif_reflect_pad(x.data_ptr(), B, H, W, pad, out.data_ptr(), L.stream_ptr(x.device)))
    return out


def _pad_bwd_raw(g, pad):
    """Adjoint of _pad_raw: (B,H+2p,W+2p) gradient folded back onto (B,H,W)."""
    lib = L.load()
    B, Hp, Wp = g.shape
    H, W = Hp - 2 * pad, Wp - 2 * pad
    out = torch.empty(B, H, W, dtype=torch.float32, device=g.device)
    with torch.cuda.device(g.device):
        L.check(lib.mmif_reflect_pad_bwd(g.data_ptr(), B, H, W, pad, out.data_ptr(), L.stream_ptr(g.device)))
    return out


def _halve(x):
    lib = L.load()
    B, H, W = x.shape
    out = torch.empty(B, (H + 1) // 2, (W + 1) // 2, dtype=torch.float32, device=x.device)
    with torch.cuda.device(x.device):
        L.check(lib.mmif_halve(x.data_ptr(), B, H, W, out.data_ptr(), L.stream_ptr(x.device)))
    return out


class _MSSSIM(torch.autograd.Function):
    """calc_msssim of the loss module (loss.py:113-160) for the pairs (img1, imgf), (img2, imgf):
    returns the two per-sample MS-SSIM vectors.  use_padding reflect-pads EVERY level by 5 before its
    blur (calc_ssim -> _gaussian_fn, loss.py:45-47) while the pyramid pools the unpadded level
    (loss.py:147-153).  Backward: one SSIM-backward launch per level (cs on levels 0..3, ssim on level
    4, per-sample chain-rule factors) + the padding and pooling adjoints."""

    @staticmethod
    def forward(ctx, img1, img2, imgf, data_range, use_padding=False, win=11):
        x1, x2, y = _prep3(img1, img2, imgf)
        wts = torch.tensor([0.0448, 0.2856, 0.3001, 0.2363, 0.1333], dtype=torch.float32, device=y.device)
        levels, vals, ranges = [], [], []
        pad = win // 2
        for lvl in range(5):
            if min(y.shape[-2:]) < (pad + 1 if use_padding else win):
                raise L.MmifError(f'ms-ssim: level {lvl} is {tuple(y.shape[-2:])}, too small for the {win}-tap window '
                                  '(the reference fails here too)')
            lx1, lx2, ly = (_pad_raw(x1, pad), _pad_raw(x2, pad), _pad_raw(y, pad)) if use_padding else (x1, x2, y)
            dr = _auto_range(x1) if data_range is None else data_range     # per level, from the level's img1 (loss.py:60-65)
            ranges.append(dr)
            ps = _fwd_per_sample(lx1, lx2, ly, dr, win)
            vals.append(torch.stack([ps[:, 1], ps[:, 4]], dim=1) if lvl < 4 else torch.stack([ps[:, 0], ps[:, 3]], dim=1))
            levels.append((lx1, lx2, ly))
            if lvl < 4:
                x1, x2, y = _halve(x1), _halve(x2), _halve(y)
        v = torch.stack(vals, dim=0).to(torch.float32)              # (5, B, 2)
        vc = v.clamp(min=eps)
        ms = torch.prod(vc ** wts.view(5, 1, 1), dim=0)              # (B, 2)
        ctx.levels, ctx.ranges, ctx.in_shape, ctx.use_padding, ctx.win = levels, ranges, imgf.shape, use_padding, win
        ctx.dtype = imgf.dtype
        ctx.save_for_backward(v, vc, ms, wts)
        return ms[:, 0].contiguous(), ms[:, 1].contiguous()

    @staticmethod
    def backward(ctx, g1, g2):
        lib = L.load()
        v, vc, ms, wts = ctx.saved_tensors
        B = ms.shape[0]
        zero = torch.zeros(B, dtype=torch.float32, device=ms.device)
        g = torch.stack([zero if g1 is None else g1.to(torch.float32), zero if g2 is None else g2.to(torch.float32)], dim=1)
        one = torch.ones(1, dtype=torch.float32, device=ms.device)
        fac = g.unsqueeze(0) * wts.view(5, 1, 1) * ms.unsqueeze(0) / vc * (v >= eps).to(torch.float32)   # (5, B, 2)
        grads = []
        for lvl, (x1, x2, y) in enumerate(ctx.levels):
            gl = _ssim_bwd_ex(x1, x2, y, ctx.ranges[lvl], one, fac[lvl], 1 if lvl < 4 else 0, 1.0, ctx.win)
            grads.append(_pad_bwd_raw(gl, ctx.win // 2) if ctx.use_padding else gl)
        for lvl in range(4, 0, -1):
            Bn, H, W = grads[lvl - 1].shape
            with torch.cuda.device(ms.device):
                L.check(lib.mmif_halve_bwd(grads[lvl].data_ptr(), Bn, H, W, grads[lvl - 1].data_ptr(), L.stream_ptr(ms.device)))
        return None, None, L.narrow_grad(grads[0], ctx.dtype).view(ctx.in_shape), None, None, None


class _MSWSSIM(torch.autograd.Function):
    """MSW_SSIM.forward (loss.py:226-237): windows 11/9/7/5/3 (sigma by loss.py:34), per-position
    gamma = sigma1/(sigma1+sigma2) from the SOURCE variances (a constant of the backward).
    use_padding reflect-pads by win//2 per window (loss.py:45-47), so every window sees H x W positions."""

    @staticmethod
    def forward(ctx, img1, img2, imgf, data_range, win_sizes, use_padding=False):
        lib = L.load()
        x1, x2, y = _prep3(img1, img2, imgf)
        B, H, W = y.shape
        dev = y.device
        total = torch.zeros((), dtype=torch.float64, device=dev)
        for k in win_sizes:
            p = k // 2 if use_padding else 0
            a1, a2, ay = (_pad_raw(x1, p), _pad_raw(x2, p), _pad_raw(y, p)) if p else (x1, x2, y)
            Hp, Wp = ay.shape[-2:]
            nws = lib.mmif_loss_workspace_bytes(B, Hp, Wp)
            if nws == 0:
                raise L.MmifError(f'unsupported shape {(B, Hp, Wp)}')
            ws = L.workspace(dev, nws, 'loss', (B, Hp, Wp))
            sums = torch.empty(B * 8, dtype=torch.float64, device=dev)
            with torch.cuda.device(dev):
                L.check(lib.mmif_mswssim_fwd(a1.data_ptr(), a2.data_ptr(), ay.data_ptr(), B, Hp, Wp, int(k), float(data_range),
                                             sums.data_ptr(), ws.data_ptr(), ws.numel(), L.stream_ptr(dev)))
            total = total + sums.view(B, 8)[:, 0].sum() / (B * (Hp - k + 1) * (Wp - k + 1))
        ctx.save_for_backward(x1, x2, y)
        ctx.data_range, ctx.win_sizes, ctx.in_shape, ctx.use_padding = data_range, tuple(win_sizes), imgf.shape, use_padding
        ctx.dtype = imgf.dtype
        return (total / len(win_sizes)).to(torch.float32)

    @staticmethod
    def backward(ctx, g):
        lib = L.load()
        x1, x2, y = ctx.saved_tensors
        B, H, W = y.shape
        dev = y.device
        dF = torch.empty_like(y)
        g1 = g.to(torch.float32).reshape(1).contiguous()
        scale = 1.0 / (B * len(ctx.win_sizes))
        for i, k in enumerate(ctx.win_sizes):
            p = k // 2 if ctx.use_padding else 0
            a1, a2, ay = (_pad_raw(x1, p), _pad_raw(x2, p), _pad_raw(y, p)) if p else (x1, x2, y)
            Hp, Wp = ay.shape[-2:]
            ws = L.workspace(dev, lib.mmif_loss_workspace_bytes(B, Hp, Wp), 'loss', (B, Hp, Wp))
            dst = torch.empty_like(ay) if p else dF
            with torch.cuda.device(dev):
                L.check(lib.mmif_mswssim_bwd(a1.data_ptr(), a2.data_ptr(), ay.data_ptr(), B, Hp, Wp, int(k), float(ctx.data_range),
                                             g1.data_ptr(), scale, 1 if (i and not p) else 0, dst.data_ptr(), ws.data_ptr(),
                                             ws.numel(), L.stream_ptr(dev)))
            if p:
                folded = _pad_bwd_raw(dst, p)
                dF = folded if i == 0 else dF.add_(folded)
        return None, None, L.narrow_grad(dF, ctx.dtype).view(ctx.in_shape), None, None, None


class _Widen(torch.autograd.Function):
    """bfloat16 / float16 -> float32 whose backward narrows the float32 gradient once.  For a module that feeds one input to
    several autograd nodes: their float32 gradients are summed in float32, as on the float32 path, before the narrowing."""

    @staticmethod
    def forward(ctx, x):
        ctx.dtype = x.dtype
        return L.as_loss_f32(x.detach(), 'img')

    @staticmethod
    def backward(ctx, g):
        return L.narrow_grad(g.contiguous(), ctx.dtype)


def _widen_shared(t):
    return t if t.dtype == torch.float32 else _Widen.apply(t)


class _ReflectPad(torch.autograd.Function):
    """F.pad(img, (p,p,p,p), 'reflect') of use_padding=True (loss.py:45-47)."""

    @staticmethod
    def forward(ctx, img, pad):
        lib = L.load()
        L.require_cuda(img, 'img')
        x, B, H, W = L.as_loss_f32_3d(img.detach(), 'img')
        out = torch.empty(B, 1, H + 2 * pad, W + 2 * pad, dtype=torch.float32, device=x.device)
        with torch.cuda.device(x.device):
            L.check(lib.mmif_reflect_pad(x.data_ptr(), B, H, W, pad, out.data_ptr(), L.stream_ptr(x.device)))
        ctx.dims, ctx.pad, ctx.in_shape, ctx.dtype = (B, H, W), pad, img.shape, img.dtype
        return out

    @staticmethod
    def backward(ctx, g):
        lib = L.load()
        B, H, W = ctx.dims
        g = g.contiguous()
        out = torch.empty(B, H, W, dtype=torch.float32, device=g.device)
        with torch.cuda.device(g.device):
            L.check(lib.mmif_reflect_pad_bwd(g.data_ptr(), B, H, W, ctx.pad, out.data_ptr(), L.stream_ptr(g.device)))
        return L.narrow_grad(out, ctx.dtype).view(ctx.in_shape), None


def _pad3(img1, img2, imgf, win_size=11):
    p = win_size // 2
    return _ReflectPad.apply(img1, p), _ReflectPad.apply(img2, p), _ReflectPad.apply(imgf, p)


class _TV(torch.autograd.Function):
    """TVLoss (loss.py:347-358) forward + backward."""

    @staticmethod
    def forward(ctx, x, norm, weight):
        lib = L.load()
        L.require_cuda(x, 'x')
        if x.dim() < 2 or (x.dtype != torch.float32 and x.dtype not in L.HALF_DTYPES):
            raise L.MmifError('TVLoss needs a float32, bfloat16 or float16 tensor with at least 2 dims')
        h, w = x.shape[-2:]
        xc = L.as_loss_f32(x.detach(), 'x').view(-1, h, w)
        dev = x.device
        L.ensure_device(dev)
        out = torch.empty(1, dtype=torch.float64, device=dev)
        n = xc.shape[0]
        ws = L.workspace(dev, lib.mmif_metric_workspace_bytes(n, h, w), 'metric', (n, h, w))
        with torch.cuda.device(dev):
            L.check(lib.mmif_tv_loss(xc.data_ptr(), n, h, w, L.NORM[norm], float(weight), out.data_ptr(), ws.data_ptr(), ws.numel(),
                                     L.stream_ptr(dev)))
        ctx.save_for_backward(xc)
        ctx.norm, ctx.weight, ctx.in_shape, ctx.dtype = norm, weight, x.shape, x.dtype
        return out[0].to(torch.float32)

    @staticmethod
    def backward(ctx, g):
        lib = L.load()
        xc, = ctx.saved_tensors
        n, h, w = xc.shape
        gx = torch.empty_like(xc)
        g1 = g.to(torch.float32).reshape(1).contiguous()
        with torch.cuda.device(xc.device):
            L.check(lib.mmif_tv_loss_bwd(xc.data_ptr(), n, h, w, L.NORM[ctx.norm], float(ctx.weight), g1.data_ptr(), gx.data_ptr(),
                                         L.stream_ptr(xc.device)))
        return L.narrow_grad(gx, ctx.dtype).view(ctx.in_shape), None, None


def _check_norm(mode):
    if mode not in ('l1', 'l2'):
        raise ValueError("only supported ['l1', 'l2'] mode")


def _auto_range(img):
    """data_range=None auto-detect of the reference (loss.py:60-63)."""
    hi = 255.0 if img.max() > 128 else 1.0
    lo = -1.0 if img.min() < -0.5 else 0.0
    return hi - lo


def _ssim_dict(img1, img2, data_range, use_padding, size_average, win_size=11):
    """calc_ssim of the loss module with the module's own window (loss.py:52-110, 163-185): 11 taps, or 9 / 7 / 5 / 3
    (sigma by loss.py:34) for SSIM(win_size=...)."""
    if use_padding:
        img1, img2 = _ReflectPad.apply(img1, win_size // 2), _ReflectPad.apply(img2, win_size // 2)
        use_padding = False
    if data_range is None:
        data_range = _auto_range(img1)
    needs_grad = torch.is_grad_enabled() and (img1.requires_grad or img2.requires_grad)
    h, w = img1.shape[-2:]
    fast_window = win_size in SSIM_WINDOWS and min(h, w) >= 11             # the strip kernels: their windows, images of 11+ pixels
    if not fast_window or (not size_average and (needs_grad or win_size != 11)):
        # any other window size (odd or even, up to 17 taps), an image smaller than the window (the reference shrinks the
        # window, loss.py:67-71), or maps that must carry gradients: the generic kernels
        if min(h, w) < int(win_size):
            raise RuntimeError(f'image {(h, w)} smaller than the {win_size}-tap window of the module (conv2d fails in the reference too)')
        if not 2 <= int(win_size) <= 17:
            raise NotImplementedError('SSIM windows of 2..17 taps are built')
        for t, nm in ((img1, 'img1'), (img2, 'img2')):
            L.require_cuda(t, nm)
        ss, cs, sg = _SSIMGeneric.apply(img1, img2, data_range, int(win_size), bool(size_average))
        return {'ssim': ss, 'cs': cs, 'sigma': sg}
    if not size_average:
        return ssim_maps(img1, img2, data_range)
    if needs_grad or win_size != 11:
        for t, nm in ((img1, 'img1'), (img2, 'img2')):
            L.require_cuda(t, nm)
        ss, cs, sg = _SSIMDict.apply(img1, img2, data_range, win_size)
        return {'ssim': ss, 'cs': cs, 'sigma': sg}
    _, _, _, ps = _fused(img1, img1, img2, data_range=data_range)
    return {'ssim': ps[:, 0], 'cs': ps[:, 1], 'sigma': ps[:, 2]}


def ssim_maps(img1, img2, data_range):
    """size_average=False of calc_ssim (loss.py:99-108): the dict of (B,1,H-10,W-10) maps."""
    lib = L.load()
    for t, nm in ((img1, 'img1'), (img2, 'img2')):
        L.require_cuda(t, nm)
    x, B, H, W = L.as_loss_f32_3d(img1.detach(), 'img1')
    y, _, _, _ = L.as_loss_f32_3d(img2.detach(), 'img2')
    if y.shape != x.shape:
        raise L.MmifError(f'shape mismatch: {tuple(img1.shape)} {tuple(img2.shape)}')
    dev = x.device
    L.ensure_device(dev)
    nws = lib.mmif_loss_workspace_bytes(B, H, W)
    if nws == 0:
        raise L.MmifError(f'unsupported shape {(B, H, W)}: H and W must be >= 11')
    ws = L.workspace(dev, nws, 'loss', (B, H, W))
    maps = [torch.empty(B, 1, H - 10, W - 10, dtype=torch.float32, device=dev) for _ in range(3)]
    with torch.cuda.device(dev):
        L.check(lib.mmif_ssim_maps(x.data_ptr(), x.data_ptr(), y.data_ptr(), B, H, W, float(data_range), maps[0].data_ptr(),
                                   maps[1].data_ptr(), maps[2].data_ptr(), None, None, None, ws.data_ptr(), ws.numel(),
                                   L.stream_ptr(dev)))
    return {'ssim': maps[0], 'cs': maps[1], 'sigma': maps[2]}


def _window_taps(win_size, window, h, w):
    """The window size calc_ssim / calc_msssim end up with: min(win_size, h, w) when no window is passed (loss.py:67-71,
    128-132), else the size of the passed window, which must be one create_window builds (loss.py:33-39)."""
    if window is None:
        return min(int(win_size), int(h), int(w))
    k = int(window.shape[-1])
    from .._windows import loss_window
    if tuple(window.shape[-2:]) != (k, k) or not torch.equal(window.detach().reshape(k, k).float().cpu(), loss_window(k).reshape(k, k)):
        raise NotImplementedError('only the Gaussian windows of create_window (loss.py:33-39) are built')
    return k


def create_window(win_size):
    """reference loss.py:33-39"""
    from .._windows import loss_window
    return loss_window(win_size)


def calc_ssim(img1, img2, win_size=11, window=None, data_range=None, use_padding=False, size_average=True):
    """reference loss.py:52-110 (the function form: without a window it is built for min(win_size, h, w))."""
    h, w = img1.shape[-2:]
    return _ssim_dict(img1, img2, data_range, use_padding, size_average, _window_taps(win_size, window, h, w))


def calc_msssim(img1, img2, win_size=11, window=None, weights=None, data_range=None, use_padding=False, size_average=True):
    """reference loss.py:113-160 with its default five level weights."""
    if weights is not None and not torch.allclose(weights.detach().float().cpu(), torch.tensor([0.0448, 0.2856, 0.3001, 0.2363, 0.1333])):
        raise NotImplementedError('calc_msssim: the default level weights are built')
    if not size_average:
        raise NotImplementedError('size_average=False is not built yet')
    h, w = img1.shape[-2:]
    k = _window_taps(win_size, window, h, w)
    if not 2 <= k <= 17:
        raise NotImplementedError('SSIM windows of 2..17 taps are built')
    return _MSSSIM.apply(img1, img1, img2, data_range, bool(use_padding), k)[0]


class SSIM(nn.Module):
    '''Structural Similarity Index (reference loss.py:163-185)'''

    def __init__(self, win_size=11, data_range=1.0, use_padding=False, size_average=True):
        super(SSIM, self).__init__()
        self.win_size = win_size
        self.data_range = data_range
        self.use_padding = use_padding
        self.size_average = size_average
        from .._windows import loss_window
        self.register_buffer('window', loss_window(win_size))

    def forward(self, img1, img2):
        return _ssim_dict(img1, img2, self.data_range, self.use_padding, self.size_average, self.win_size)


class MS_SSIM(SSIM):
    '''Multi-Scale Structural Similarity Index (reference loss.py:188-208)'''

    def __init__(self, win_size=11, data_range=1.0, use_padding=False, size_average=True):
        super(MS_SSIM, self).__init__(win_size, data_range, use_padding, size_average)
        self.register_buffer('weights', torch.FloatTensor([0.0448, 0.2856, 0.3001, 0.2363, 0.1333]))

    def forward(self, img1, img2):
        if not 1 < int(self.win_size) <= 17:
            raise NotImplementedError('SSIM windows of 2..17 taps are built')
        if not self.size_average:
            raise NotImplementedError('size_average=False is not built yet')
        return _MSSSIM.apply(img1, img1, img2, self.data_range, bool(self.use_padding), int(self.win_size))[0]


class MSW_SSIM(nn.Module):
    '''Multi-Scale and Weighted Structural Similarity Index (reference loss.py:211-237)'''

    def __init__(self, win_sizes=(11, 9, 7, 5, 3), data_range=1.0, use_padding=False, size_average=False):
        super(MSW_SSIM, self).__init__()
        self.win_sizes = win_sizes
        self.data_range = data_range
        self.use_padding = use_padding
        self.size_average = size_average

    def forward(self, img1, img2, imgf):
        dr = _auto_range(img1) if self.data_range is None else self.data_range
        if self.size_average:
            # size_average=True (loss.py:222-237 with per-sample dict entries): gamma_b = sigma1_b / (sigma1_b + sigma2_b) from the
            # window-MEAN clamped variances of the sources, one weighted SSIM per window size — 'w-ssim' with that window
            if any(not 2 <= int(k) <= 17 for k in self.win_sizes):
                raise NotImplementedError('SSIM windows of 2..17 taps are built')
            img1, img2, imgf = (_widen_shared(t) for t in (img1, img2, imgf))      # one input, one node per window
            acc = 0.0
            for k in self.win_sizes:
                x1, x2, y = _pad3(img1, img2, imgf, int(k)) if self.use_padding else (img1, img2, imgf)
                acc = acc + _WeightedSSIM.apply(x1, x2, y, dr, int(k))
            return acc / len(self.win_sizes)
        if any(k not in (11, 9, 7, 5, 3) for k in self.win_sizes):
            raise NotImplementedError('MSW_SSIM(size_average=False): windows 11, 9, 7, 5, 3 are built')
        return _MSWSSIM.apply(img1, img2, imgf, dr, tuple(self.win_sizes), bool(self.use_padding))


class SSIMLoss(nn.Module):
    '''reference loss.py:240-284'''

    def __init__(self, mode='ssim', data_range=1.0, use_padding=False, weight=1.0):
        super(SSIMLoss, self).__init__()
        self.mode = mode
        self.data_range = data_range
        self.use_padding = use_padding
        self.weight = weight

    def forward(self, img1, img2, imgf):
        if self.mode in ('ssim', 'w-ssim') and self.use_padding:
            img1, img2, imgf = _pad3(img1, img2, imgf)      # reflect pad 5, then the valid-window path (loss.py:45-47)
        dr = _auto_range(img1) if self.data_range is None else self.data_range     # loss.py:60-65
        if self.mode == 'ssim':
            if self.use_padding:        # SSIM-only kernels on the padded images (the fused objective's other terms are not wanted)
                return self.weight * (1.0 - _PlainSSIM.apply(img1, img2, imgf, dr))
            loss, _, _, _ = _fused(img1, img2, imgf, data_range=dr, w_ssim=self.weight)
            return loss
        elif self.mode == 'w-ssim':
            loss = _WeightedSSIM.apply(img1, img2, imgf, dr)
            return self.weight * (1.0 - loss)
        elif self.mode == 'ms-ssim':
            m1, m2 = _MSSSIM.apply(img1, img2, imgf, self.data_range, bool(self.use_padding))
            return self.weight * (1.0 - (m1.mean() + m2.mean()) * 0.5)
        elif self.mode == 'msw-ssim':
            loss = MSW_SSIM((11, 9, 7, 5, 3), dr, self.use_padding)(img1, img2, imgf)
            return self.weight * (1.0 - loss)
        else:
            raise ValueError("only supported ['ssim', 'w-ssim', 'ms-ssim', 'msw-ssim'] mode")


class PixelLoss(nn.Module):
    '''reference loss.py:287-304'''

    def __init__(self, mode='l1', weight=1.0):
        super(PixelLoss, self).__init__()
        self.mode = mode
        self.weight = weight
        self.loss_fn = NormLoss(mode, weight)

    def forward(self, img1, img2, imgf, mode='avg'):
        if mode not in ('avg', 'max'):
            return None  # the reference falls through and returns None (loss.py:294-304)
        _check_norm(self.mode)
        _, pix, _, _ = _fused(img1, img2, imgf, pixel=(mode, self.mode), w_pixel=self.weight)
        return pix


class GradLoss(nn.Module):
    '''reference loss.py:307-344'''

    def __init__(self, mode='l1', weight=1.0):
        super(GradLoss, self).__init__()
        self.mode = mode
        self.weight = weight
        self.loss_fn = NormLoss(mode, weight)
        self.register_buffer('x_sobel', torch.FloatTensor([[-1, 0, 1], [-2, 0, 2], [-1, 0, 1]]).reshape(1, 1, 3, 3))
        self.register_buffer('y_sobel', torch.FloatTensor([[-1, -2, -1], [0, 0, 0], [1, 2, 1]]).reshape(1, 1, 3, 3))

    def forward(self, img1, img2, imgf, mode='avg'):
        if mode not in ('avg', 'max'):
            return None
        _check_norm(self.mode)
        _, _, grd, _ = _fused(img1, img2, imgf, grad=(mode, self.mode), w_grad=self.weight)
        return grd


class TVLoss(nn.Module):
    '''reference loss.py:347-358'''

    def __init__(self, mode='l1', weight=1.0):
        super(TVLoss, self).__init__()
        self.mode = mode
        self.weight = weight
        self.loss_fn = NormLoss(mode, weight)

    def forward(self, x):
        _check_norm(self.mode)
        return _TV.apply(x, self.mode, self.weight)


class _Norm(torch.autograd.Function):
    """NormLoss (loss.py:361-385) forward + backward on the device kernels."""

    @staticmethod
    def forward(ctx, x, mode, weight):
        lib = L.load()
        L.require_cuda(x, 'x')
        xc = L.as_loss_f32(x.detach(), 'NormLoss')
        dev = xc.device
        L.ensure_device(dev)
        out = torch.empty(1, dtype=torch.float64, device=dev)
        ws = L.workspace(dev, lib.mmif_norm_workspace_bytes(), 'norm')
        with torch.cuda.device(dev):
            L.check(lib.mmif_norm_loss(xc.data_ptr(), xc.numel(), L.NORM[mode], float(weight), out.data_ptr(), ws.data_ptr(),
                                       ws.numel(), L.stream_ptr(dev)))
        ctx.save_for_backward(xc)
        ctx.mode, ctx.weight, ctx.in_shape, ctx.dtype = mode, weight, x.shape, x.dtype
        return out[0].to(torch.float32)

    @staticmethod
    def backward(ctx, g):
        lib = L.load()
        xc, = ctx.saved_tensors
        gx = torch.empty_like(xc)
        g1 = g.to(torch.float32).reshape(1).contiguous()
        with torch.cuda.device(xc.device):
            L.check(lib.mmif_norm_loss_bwd(xc.data_ptr(), xc.numel(), L.NORM[ctx.mode], float(ctx.weight), g1.data_ptr(),
                                           gx.data_ptr(), L.stream_ptr(xc.device)))
        return L.narrow_grad(gx, ctx.dtype).view(ctx.in_shape), None, None


class NormLoss(nn.Module):
    '''reference loss.py:361-385: weight * mean(|x|) ('l1') or weight * mean(x^2) ('l2') of any tensor.'''

    def __init__(self, mode='l1', weight=1.0):
        super(NormLoss, self).__init__()
        self.mode = mode
        self.weight = weight

    def forward(self, x):
        _check_norm(self.mode)
        return _Norm.apply(x, self.mode, self.weight)
