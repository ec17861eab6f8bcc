"""ctypes binding of libmmif_b200.so (the C ABI declared in include/mmif_b200.h).

No CPU fallback: if the library is missing or the device is not a B200-class GPU the import of
the compute entry points fails loudly.  PyTorch is used only for device memory and streams."""
import ctypes
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, 'libmmif_b200.so')

SYMBOLS = [
    'mmif_version', 'mmif_last_error', 'mmif_check_device', 'mmif_set_gaussian_taps',
    'mmif_loss_workspace_bytes', 'mmif_loss_out_doubles', 'mmif_fusion_loss_fwd', 'mmif_fusion_loss_bwd',
    'mmif_fusion_loss_bwd3', 'mmif_launch_counts', 'mmif_loss_geometry', 'mmif_ssim_generic_workspace_bytes', 'mmif_ssim_generic_coef_doubles',
    'mmif_ssim_generic_fwd', 'mmif_ssim_generic_bwd',
    'mmif_tv_loss', 'mmif_tv_loss_bwd', 'mmif_ssim_bwd_ex', 'mmif_ssim_fwd_win', 'mmif_ssim_bwd_ex_win', 'mmif_mswssim_fwd', 'mmif_mswssim_bwd', 'mmif_halve', 'mmif_halve_bwd', 'mmif_reflect_pad',
    'mmif_reflect_pad_bwd', 'mmif_metric_workspace_bytes', 'mmif_stats', 'mmif_hist', 'mmif_qabf', 'mmif_qabf_raw', 'mmif_ssim',
    'mmif_msssim', 'mmif_viff', 'mmif_eval_suite', 'mmif_eval_suite_host', 'mmif_ssim_maps', 'mmif_widen_u8', 'mmif_widen_u8_unit',
    'mmif_eval_suite_u8', 'mmif_eval_suite_u8_host', 'mmif_norm_workspace_bytes', 'mmif_norm_loss', 'mmif_norm_loss_bwd', 'mmif_test_post',
    'mmif_widen', 'mmif_narrow', 'mmif_stats_bwd', 'mmif_quality_index_workspace_bytes', 'mmif_quality_index',
]

COMBINE = {'max': 0, 'avg': 1}
NORM = {'l1': 1, 'l2': 2}
LOSS_HEAD, LOSS_PER_SAMPLE = 4, 6
ST_COUNT, EN_COUNT, HIST_WORDS = 16, 12, 3 * 256 + 2 * 65536
MSSSIM_DOUBLES, VIFF_DOUBLES, EVAL_METRICS = 22, 26, 16
QIDX_DOUBLES = 13
HALF_DTYPES = {torch.bfloat16: 1, torch.float16: 2}       # MMIF_DTYPE_BF16, MMIF_DTYPE_F16


class MmifLossCfg(ctypes.Structure):
    _fields_ = [('w_ssim', ctypes.c_float), ('w_pixel', ctypes.c_float), ('w_grad', ctypes.c_float),
                ('data_range', ctypes.c_float), ('pixel_combine', ctypes.c_int32), ('grad_combine', ctypes.c_int32),
                ('pixel_norm', ctypes.c_int32), ('grad_norm', ctypes.c_int32), ('want_grad', ctypes.c_int32),
                ('reserved', ctypes.c_int32)]


class MmifError(RuntimeError):
    pass


_lib = None


def load():
    """Load the shared library once; raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise MmifError(f'{LIB_PATH} not found: build it with `make` (or __graft_entry__.build()); '
                        'there is no CPU fallback for the fusion loss / metric path')
    lib = ctypes.CDLL(LIB_PATH)
    vp, sz, ci, cf = ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int, ctypes.c_float
    lib.mmif_version.restype = ci
    lib.mmif_last_error.restype = ctypes.c_char_p
    lib.mmif_check_device.argtypes = [ci]
    lib.mmif_set_gaussian_taps.argtypes = [ci, ctypes.c_double, vp]
    lib.mmif_loss_workspace_bytes.restype = sz
    lib.mmif_loss_workspace_bytes.argtypes = [ci, ci, ci]
    lib.mmif_loss_out_doubles.restype = sz
    lib.mmif_loss_out_doubles.argtypes = [ci]
    lib.mmif_fusion_loss_fwd.argtypes = [vp, vp, vp, ci, ci, ci, ctypes.POINTER(MmifLossCfg), vp, vp, vp, sz, vp]
    lib.mmif_fusion_loss_bwd.argtypes = [vp, vp, vp, ci, ci, ci, ctypes.POINTER(MmifLossCfg), vp, vp, vp, vp, sz, vp]
    lib.mmif_fusion_loss_bwd3.argtypes = [vp, vp, vp, ci, ci, ci, ctypes.POINTER(MmifLossCfg), vp, vp, vp, vp, vp, vp, sz, vp]
    lib.mmif_launch_counts.argtypes = [ctypes.POINTER(ctypes.c_ulonglong), ci]
    lib.mmif_loss_geometry.argtypes = [ci, ci, ci, ci, ctypes.POINTER(ci)]
    lib.mmif_ssim_generic_workspace_bytes.restype = sz
    lib.mmif_ssim_generic_workspace_bytes.argtypes = [ci, ci, ci, ci]
    lib.mmif_ssim_generic_coef_doubles.restype = sz
    lib.mmif_ssim_generic_coef_doubles.argtypes = [ci, ci, ci, ci]
    lib.mmif_ssim_generic_fwd.argtypes = [vp, vp, ci, ci, ci, ci, ctypes.c_double, cf, vp, vp, vp, vp, vp, sz, vp]
    lib.mmif_ssim_generic_bwd.argtypes = [vp, vp, ci, ci, ci, ci, ctypes.c_double, cf, vp, vp, vp, ci, vp, vp, vp, vp]
    lib.mmif_tv_loss.argtypes = [vp, ci, ci, ci, ci, cf, vp, vp, sz, vp]
    lib.mmif_tv_loss_bwd.argtypes = [vp, ci, ci, ci, ci, cf, vp, vp, vp]
    lib.mmif_ssim_bwd_ex.argtypes = [vp, vp, vp, ci, ci, ci, cf, vp, vp, ci, cf, vp, vp, sz, vp]
    lib.mmif_ssim_fwd_win.argtypes = [vp, vp, vp, ci, ci, ci, ci, cf, vp, vp, sz, vp]
    lib.mmif_ssim_bwd_ex_win.argtypes = [vp, vp, vp, ci, ci, ci, ci, cf, vp, vp, ci, cf, vp, vp, sz, vp]
    lib.mmif_mswssim_fwd.argtypes = [vp, vp, vp, ci, ci, ci, ci, cf, vp, vp, sz, vp]
    lib.mmif_mswssim_bwd.argtypes = [vp, vp, vp, ci, ci, ci, ci, cf, vp, cf, ci, vp, vp, sz, vp]
    lib.mmif_halve.argtypes = [vp, ci, ci, ci, vp, vp]
    lib.mmif_halve_bwd.argtypes = [vp, ci, ci, ci, vp, vp]
    lib.mmif_reflect_pad.argtypes = [vp, ci, ci, ci, ci, vp, vp]
    lib.mmif_reflect_pad_bwd.argtypes = [vp, ci, ci, ci, ci, vp, vp]
    lib.mmif_metric_workspace_bytes.restype = sz
    lib.mmif_metric_workspace_bytes.argtypes = [ci, ci, ci]
    lib.mmif_stats.argtypes = [vp, vp, vp, ci, ci, ci, vp, vp, sz, vp]
    lib.mmif_stats_bwd.argtypes = [vp, vp, vp, ci, ci, ci, vp, vp, vp, vp, vp, vp]
    lib.mmif_hist.argtypes = [vp, vp, vp, ci, ci, ci, vp, vp, vp, sz, vp]
    lib.mmif_qabf.argtypes = [vp, vp, vp, ci, ci, ci, cf, vp, vp, sz, vp]
    lib.mmif_qabf_raw.argtypes = [vp, vp, vp, ci, ci, ci, cf, vp, vp, sz, vp]
    lib.mmif_ssim.argtypes = [vp, vp, vp, ci, ci, ci, ci, cf, ci, vp, vp, sz, vp]
    lib.mmif_msssim.argtypes = [vp, vp, vp, ci, ci, ci, ci, cf, vp, vp, sz, vp]
    lib.mmif_viff.argtypes = [vp, vp, vp, ci, ci, ci, vp, vp, sz, vp]
    lib.mmif_eval_suite.argtypes = [vp, vp, vp, ci, ci, ci, vp, vp, sz, vp]
    lib.mmif_eval_suite_host.argtypes = [vp, vp, vp, ci, ci, ci, vp, vp, vp, vp, sz, vp]
    lib.mmif_ssim_maps.argtypes = [vp, vp, vp, ci, ci, ci, cf, vp, vp, vp, vp, vp, vp, vp, sz, vp]
    lib.mmif_test_post.argtypes = [vp, vp, vp, ci, ci, ci, cf, vp, vp, vp, sz, vp]
    lib.mmif_widen_u8.argtypes = [vp, sz, vp, vp]
    lib.mmif_widen_u8_unit.argtypes = [vp, sz, vp, vp]
    lib.mmif_eval_suite_u8.argtypes = [vp, vp, vp, ci, ci, ci, vp, vp, vp, sz, vp]
    lib.mmif_eval_suite_u8_host.argtypes = [vp, vp, vp, ci, ci, ci, vp, vp, vp, vp, vp, sz, vp]
    lib.mmif_norm_workspace_bytes.restype = sz
    lib.mmif_norm_workspace_bytes.argtypes = []
    lib.mmif_norm_loss.argtypes = [vp, sz, ci, cf, vp, vp, sz, vp]
    lib.mmif_norm_loss_bwd.argtypes = [vp, sz, ci, cf, vp, vp, vp]
    lib.mmif_widen.argtypes = [vp, ci, sz, vp, vp]
    lib.mmif_narrow.argtypes = [vp, vp, sz, ci, vp, vp]
    lib.mmif_quality_index_workspace_bytes.restype = sz
    lib.mmif_quality_index_workspace_bytes.argtypes = [ci, ci, ci]
    lib.mmif_quality_index.argtypes = [vp, vp, vp, ci, ci, ci, vp, vp, sz, vp]
    for name in SYMBOLS:
        getattr(lib, name)  # every declared symbol must be exported
    _lib = lib
    register_reference_taps()
    return lib


def check(rc):
    if rc != 0:
        raise MmifError(f'libmmif_b200 error {rc}: {load().mmif_last_error().decode()}')


def stream_ptr(device):
    return ctypes.c_void_p(torch.cuda.current_stream(device).cuda_stream)


_raw_stream = getattr(torch._C, '_cuda_getCurrentRawStream', None)


def stream_int(device):
    """cudaStream_t of torch's current stream on `device`, as a plain int (the raw getter: 0.2 us against the 11 us of
    building a torch.cuda.Stream object, twice per training step)."""
    if _raw_stream is not None:
        return _raw_stream(device.index if device.index is not None else torch.cuda.current_device())
    return torch.cuda.current_stream(device).cuda_stream


_fast = False


def fastcall():
    """The CPython fast-call binding of the per-step entries (csrc/fastcall.c -> _fastcall.so), or None if it was not built
    (MMIF_NO_FASTCALL=1 forces the ctypes binding).  Same library, same entry points, ~0.5 us instead of ~9 us per call."""
    global _fast
    if _fast is False:
        mod = None
        if not os.environ.get('MMIF_NO_FASTCALL'):
            load()
            try:
                from . import _fastcall as mod
            except Exception:       # not built: ctypes serves the same entries
                mod = None
        _fast = mod
    return _fast


def call(device, fn, *args):
    """Run a library entry with `device` current (kernel launches go to the current device) and check its code."""
    if torch.cuda.current_device() == (device.index if device.index is not None else torch.cuda.current_device()):
        rc = fn(*args)
    else:
        with torch.cuda.device(device):
            rc = fn(*args)
    if rc != 0:
        check(rc)


def launch_counts():
    """dict of the library's launch counters (include/mmif_b200.h MMIF_CNT_*)."""
    buf = (ctypes.c_ulonglong * 16)()
    check(load().mmif_launch_counts(buf, 16))
    names = ('loss_fwd', 'loss_single_pass', 'loss_bwd', 'rescale', 'ssim_bwd_ext', 'moment_fwd', 'metric', 'aux',
             'tmap_encode', 'tmap_hit', 'tmap_fail')
    return {n: int(buf[i]) for i, n in enumerate(names)}


def kernel_launches(before, after):
    """Number of kernels launched between two launch_counts() snapshots."""
    return sum(after[k] - before[k] for k in after if not k.startswith('tmap'))


def require_cuda(t, name='tensor'):
    if not t.is_cuda:
        raise MmifError(f'{name} must be a CUDA tensor (no CPU compute path exists)')


_checked_devices = set()


def ensure_device(device):
    idx = device.index if device.index is not None else torch.cuda.current_device()
    if idx not in _checked_devices:
        check(load().mmif_check_device(idx))
        _checked_devices.add(idx)


_ws_cache = {}
_WS_CACHE_CAP = 16


def workspace(device, nbytes, tag, shape=None, stream=None):
    """Zero-initialised workspace, cached per (device, stream, tag, shape).  The kernels leave their
    counters zeroed, but the carve-up of a workspace depends on the problem shape, so a buffer is
    only ever reused for the shape it was first zeroed for (small LRU)."""
    key = (device.index, stream if stream is not None else torch.cuda.current_stream(device).cuda_stream, tag, shape)
    buf = _ws_cache.pop(key, None)
    if buf is None or buf.numel() < nbytes:
        buf = torch.zeros(max(int(nbytes), 256), dtype=torch.uint8, device=device)
    _ws_cache[key] = buf            # re-insert: most recently used last
    while len(_ws_cache) > _WS_CACHE_CAP:
        _ws_cache.pop(next(iter(_ws_cache)))
    return buf


def as_f32_3d(t, name='image'):
    """(N,1,H,W) / (N,H,W) / (H,W) float32 contiguous view -> (tensor, N, H, W)."""
    if t.dtype != torch.float32:
        raise MmifError(f'{name}: float32 expected, got {t.dtype}')
    dims = _dims_3d(t, name)
    return (t.contiguous(),) + dims


def as_loss_f32(t, name='image'):
    """Input of the loss modules -> float32 contiguous tensor: float32 as it is, bfloat16 / float16 (an autocast training
    step) widened on the device by mmif_widen, which is exact.  Every other dtype raises."""
    if t.dtype == torch.float32:
        return t.contiguous()
    code = HALF_DTYPES.get(t.dtype)
    if code is None:
        raise MmifError(f'{name}: float32, bfloat16 or float16 expected, got {t.dtype}')
    require_cuda(t, name)
    src = t.contiguous()
    dst = torch.empty(src.shape, dtype=torch.float32, device=src.device)
    call(src.device, load().mmif_widen, src.data_ptr(), code, src.numel(), dst.data_ptr(), stream_int(src.device))
    return dst


def as_loss_f32_3d(t, name='image'):
    """as_f32_3d for the loss modules: bfloat16 / float16 images are accepted too and widened (as_loss_f32)."""
    if t.dtype == torch.float32:
        return as_f32_3d(t, name)
    dims = _dims_3d(t, name)
    return (as_loss_f32(t, name),) + dims


def narrow_grad(g, dtype, scale=None):
    """Gradient of a loss-module input: the float32 device tensor `g` itself for a float32 input, else
    round-to-nearest-even of (scale[0] *) g to `dtype`, written by mmif_narrow.  scale: a float32 device scalar or None."""
    if dtype == torch.float32 and scale is None:
        return g
    out = torch.empty(g.shape, dtype=dtype, device=g.device)
    call(g.device, load().mmif_narrow, g.data_ptr(), scale.data_ptr() if scale is not None else None, g.numel(), HALF_DTYPES[dtype],
         out.data_ptr(), stream_int(g.device))
    return out


def _dims_3d(t, name):
    if t.dim() == 4:
        if t.shape[1] != 1:
            raise MmifError(f'{name}: single-channel (N,1,H,W) expected, got {tuple(t.shape)}')
        n, h, w = t.shape[0], t.shape[2], t.shape[3]
    elif t.dim() == 3:
        n, h, w = t.shape
    elif t.dim() == 2:
        n, (h, w) = 1, t.shape
    else:
        raise MmifError(f'{name}: unsupported rank {t.dim()}')
    return int(n), int(h), int(w)


_REFERENCE_WINDOWS = [(11, 1.5), (17, 17 / 5), (9, 9 / 5), (5, 5 / 5), (3, 3 / 5)] + [(k, 1.5) for k in range(1, 11)] \
    + [(k, 0.15 * (k - 1)) for k in (9, 7, 5, 3)]


def set_window_taps(win, sigma, taps):
    """Register a 1-D tap table (float32 torch tensor / sequence of `win` floats) for (win, sigma)."""
    t = torch.as_tensor(taps, dtype=torch.float32).contiguous().cpu()
    if t.numel() != win:
        raise MmifError(f'expected {win} taps, got {t.numel()}')
    check(_lib.mmif_set_gaussian_taps(int(win), float(sigma), t.data_ptr()))


_registered_taps = set()


def ensure_window_taps(win, sigma):
    """Register the reference's own taps of (win, sigma) once (any window size the loss module is asked for)."""
    key = (int(win), float(sigma))
    if key not in _registered_taps:
        from ._windows import gauss_1d
        set_window_taps(win, sigma, gauss_1d(win, sigma))
        _registered_taps.add(key)


def register_reference_taps():
    """Build every window the reference uses with the reference's own torch ops on this host
    (loss.py:24-30, metric.py:290-296, 415-416) and hand the tables to the library."""
    from ._windows import gauss_1d
    for win, sigma in _REFERENCE_WINDOWS:
        if sigma > 0:
            set_window_taps(win, sigma, gauss_1d(win, sigma))
