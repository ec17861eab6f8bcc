"""CPU-only checks of mmif_stats_bwd's argument validation: the return codes of the gradient entry of the statistics
metrics, and that a call with no gradient requested launches nothing."""
E_NULL, E_SHAPE, E_ALIGN = -1, -2, -5


def _lib():
    import mmif_b200  # noqa: F401
    from mmif_b200 import _lib as L
    return L, L.load()


def test_stats_bwd_return_codes():
    L, lib = _lib()
    before = L.launch_counts()
    img, row, gout, out = 256, 512, 768, 1024            # well-aligned fake device addresses: nothing is dereferenced
    ok = (img, img, img, 1, 8, 8, row, gout)
    assert lib.mmif_stats_bwd(None, img, img, 1, 8, 8, row, gout, out, out, out, None) == E_NULL
    assert lib.mmif_stats_bwd(img, None, img, 1, 8, 8, row, gout, out, out, out, None) == E_NULL
    assert lib.mmif_stats_bwd(img, img, None, 1, 8, 8, row, gout, out, out, out, None) == E_NULL
    assert lib.mmif_stats_bwd(img, img, img, 1, 8, 8, None, gout, out, out, out, None) == E_NULL
    assert lib.mmif_stats_bwd(img, img, img, 1, 8, 8, row, None, out, out, out, None) == E_NULL
    assert b'null' in lib.mmif_last_error()
    for n, h, w in ((0, 8, 8), (1, 0, 8), (1, 8, -1), (1, 1, 8), (1, 8, 1)):   # H, W >= 2: AG / SF need a neighbour
        assert lib.mmif_stats_bwd(img, img, img, n, h, w, row, gout, out, out, out, None) == E_SHAPE
    assert lib.mmif_stats_bwd(img + 2, img, img, 1, 8, 8, row, gout, out, out, out, None) == E_ALIGN
    assert lib.mmif_stats_bwd(*ok[:6], row + 4, gout, out, out, out, None) == E_ALIGN        # row: doubles
    assert lib.mmif_stats_bwd(*ok[:7], gout + 2, out, out, out, None) == E_ALIGN
    assert lib.mmif_stats_bwd(*ok, out, out + 1, out, None) == E_ALIGN
    assert lib.mmif_stats_bwd(*ok, None, None, out + 3, None) == E_ALIGN
    assert b'align' in lib.mmif_last_error()
    assert lib.mmif_stats_bwd(*ok, None, None, None, None) == 0        # no gradient wanted: OK, nothing launched
    assert L.launch_counts() == before
