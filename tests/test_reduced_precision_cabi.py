"""CPU-only checks of the bfloat16 / float16 entries: the argument validation of mmif_widen / mmif_narrow, and the
dtype rules of the loss-side input helper (which dtypes are widened, which still raise)."""
import pytest
import torch

BF16, F16 = 1, 2                 # MMIF_DTYPE_BF16, MMIF_DTYPE_F16
E_NULL, E_MODE, E_ALIGN = -1, -3, -5


def _lib():
    import mmif_b200  # noqa: F401
    from mmif_b200 import _lib as L
    return L, L.load()


def test_widen_return_codes():
    L, lib = _lib()
    before = L.launch_counts()
    assert lib.mmif_widen(None, BF16, 8, 16, None) == E_NULL
    assert lib.mmif_widen(16, BF16, 8, None, None) == E_NULL
    assert b'null' in lib.mmif_last_error()
    for bad in (0, 3, -1):                          # MMIF_DTYPE_F32 is not a source to widen
        assert lib.mmif_widen(16, bad, 8, 16, None) == E_MODE
    assert b'dtype' in lib.mmif_last_error()
    assert lib.mmif_widen(17, BF16, 8, 16, None) == E_ALIGN        # src must be 2-byte aligned
    assert lib.mmif_widen(16, BF16, 8, 18, None) == E_ALIGN         # dst must be 4-byte aligned
    assert b'align' in lib.mmif_last_error()
    assert lib.mmif_widen(16, BF16, 0, 16, None) == 0               # n == 0: nothing to do, nothing launched
    assert lib.mmif_widen(18, F16, 0, 20, None) == 0                # 2-byte src and 4-byte dst alignment suffice
    assert L.launch_counts() == before


def test_narrow_return_codes():
    L, lib = _lib()
    before = L.launch_counts()
    assert lib.mmif_narrow(None, None, 8, BF16, 16, None) == E_NULL
    assert lib.mmif_narrow(16, None, 8, BF16, None, None) == E_NULL
    for bad in (0, 3, -1):                          # MMIF_DTYPE_F32 is not a narrowing target
        assert lib.mmif_narrow(16, None, 8, bad, 16, None) == E_MODE
    assert lib.mmif_narrow(18, None, 8, F16, 16, None) == E_ALIGN   # src must be 4-byte aligned
    assert lib.mmif_narrow(16, 18, 8, F16, 16, None) == E_ALIGN     # so must the scale
    assert lib.mmif_narrow(16, None, 8, F16, 17, None) == E_ALIGN   # dst must be 2-byte aligned
    assert lib.mmif_narrow(16, None, 0, BF16, 16, None) == 0        # n == 0
    assert lib.mmif_narrow(20, 24, 0, F16, 18, None) == 0
    assert L.launch_counts() == before


def test_loss_input_helper_dtype_rules_without_gpu():
    L, _ = _lib()
    x32 = torch.rand(2, 1, 12, 13)
    t, n, h, w = L.as_loss_f32_3d(x32, 'img')                      # float32 passes through untouched
    assert t.data_ptr() == x32.data_ptr() and (n, h, w) == (2, 12, 13)
    for dt in (torch.float64, torch.int32, torch.int64, torch.uint8):
        with pytest.raises(L.MmifError, match='float32, bfloat16 or float16 expected'):
            L.as_loss_f32_3d(x32.to(dt), 'img')
        with pytest.raises(L.MmifError):
            L.as_loss_f32(x32.to(dt), 'x')
    for dt in (torch.bfloat16, torch.float16):
        with pytest.raises(L.MmifError, match='CUDA'):              # no host widening path
            L.as_loss_f32_3d(x32.to(dt), 'img')
        with pytest.raises(L.MmifError, match='float32 expected'):  # the metric-side helper keeps rejecting them
            L.as_f32_3d(x32.to(dt), 'img')
        with pytest.raises(L.MmifError, match='rank'):              # the rank rules come first
            L.as_loss_f32_3d(torch.zeros(2, 2, 2, 2, 2, dtype=dt), 'img')
