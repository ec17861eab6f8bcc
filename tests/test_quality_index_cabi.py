"""CPU-only checks of mmif_quality_index's argument validation: its return codes, the workspace size rule, and that a
rejected call launches nothing."""
E_NULL, E_SHAPE, E_WORKSPACE, E_ALIGN = -1, -2, -4, -5


def _lib():
    import mmif_b200  # noqa: F401
    from mmif_b200 import _lib as L
    return L, L.load()


def test_quality_index_return_codes():
    L, lib = _lib()
    before = L.launch_counts()
    img, out, ws = 256, 512, 1024                  # well-aligned fake device addresses: nothing is dereferenced
    need = lib.mmif_quality_index_workspace_bytes(2, 11, 12)
    assert need > 0
    ok = (img, img, img, 2, 11, 12)
    assert lib.mmif_quality_index(None, img, img, 2, 11, 12, out, ws, need, None) == E_NULL
    assert lib.mmif_quality_index(img, None, img, 2, 11, 12, out, ws, need, None) == E_NULL
    assert lib.mmif_quality_index(img, img, None, 2, 11, 12, out, ws, need, None) == E_NULL
    assert lib.mmif_quality_index(*ok, None, ws, need, None) == E_NULL
    assert b'null' in lib.mmif_last_error()
    for n, h, w in ((0, 11, 11), (1, 10, 11), (1, 11, 10), (1, 8, 8), (-1, 20, 20), (1, 11, -3)):   # H, W >= 11: Q_Y window
        assert lib.mmif_quality_index(img, img, img, n, h, w, out, ws, need, None) == E_SHAPE
        assert lib.mmif_quality_index_workspace_bytes(n, h, w) == 0
    assert lib.mmif_quality_index(img + 2, img, img, 2, 11, 12, out, ws, need, None) == E_ALIGN
    assert lib.mmif_quality_index(img, img + 1, img, 2, 11, 12, out, ws, need, None) == E_ALIGN
    assert lib.mmif_quality_index(img, img, img + 3, 2, 11, 12, out, ws, need, None) == E_ALIGN
    assert lib.mmif_quality_index(*ok, out + 4, ws, need, None) == E_ALIGN
    assert lib.mmif_quality_index(*ok, out, ws + 4, need, None) == E_ALIGN
    assert b'align' in lib.mmif_last_error()
    assert lib.mmif_quality_index(*ok, out, None, need, None) == E_WORKSPACE
    assert lib.mmif_quality_index(*ok, out, ws, need - 1, None) == E_WORKSPACE
    assert lib.mmif_quality_index(*ok, out, ws, 0, None) == E_WORKSPACE
    assert b'workspace' in lib.mmif_last_error()
    assert L.launch_counts() == before


def test_quality_index_workspace_grows_with_the_problem():
    _, lib = _lib()
    small = lib.mmif_quality_index_workspace_bytes(1, 11, 11)
    assert small > 0 and small % 8 == 0
    assert lib.mmif_quality_index_workspace_bytes(4, 480, 640) > lib.mmif_quality_index_workspace_bytes(1, 480, 640) > small
