"""CPU tests of the fused GATv2 attention entry points (gno_gatv2_attention, its backward and the two
workspace queries): argument validation returns GNO_ERR_INVALID with a message before any device
work, E = 0 touches nothing, and gno_b200.gatv2_attention refuses CPU tensors (no fallback)."""
import ctypes

import pytest
import torch

GNO_ERR_INVALID = 1


def _csr(N=4, E=8, chunk_len=32):
    from gno_b200 import _lib
    return _lib.gno_csr(N, E, None, None, None, None, chunk_len, 0, None, 0, None)


def _fwd(g, H, F, xl_rows=4, dtype=0):
    from gno_b200 import _lib
    return _lib.lib.gno_gatv2_attention(ctypes.byref(g), None, xl_rows, None, None, H, F, 0.2, 1e-16, None, None,
                                        None, dtype, None, 0, None)


def _bwd(g, H, F, xl_rows=4, dtype=0):
    from gno_b200 import _lib
    return _lib.lib.gno_gatv2_attention_backward(ctypes.byref(g), None, xl_rows, None, None, None, None, None, None,
                                                 H, F, 0.2, None, None, None, None, dtype, None, 0, None)


def _ws(g, H, F):
    from gno_b200 import _lib
    n = ctypes.c_size_t()
    return _lib.lib.gno_gatv2_attention_workspace(ctypes.byref(g), H, F, ctypes.byref(n)), n.value


def _bws(g, H, F, grad_r=1, att=1):
    from gno_b200 import _lib
    n = ctypes.c_size_t()
    rc = _lib.lib.gno_gatv2_attention_backward_workspace(ctypes.byref(g), H, F, grad_r, att, ctypes.byref(n))
    return rc, n.value


def _error():
    from gno_b200 import _lib
    return _lib.lib.gno_last_error()


@pytest.mark.parametrize("H,F", [(0, 8), (-1, 8), (3, 8), (2, -4)])
def test_bad_heads_and_widths_are_invalid(H, F):
    g = _csr()
    for rc in (_fwd(g, H, F), _bwd(g, H, F), _ws(g, H, F)[0], _bws(g, H, F)[0]):
        assert rc == GNO_ERR_INVALID and b"H=" in _error()


def test_negative_sizes_are_invalid():
    assert _fwd(_csr(), 2, 8, xl_rows=-1) == GNO_ERR_INVALID and b"bad sizes" in _error()
    assert _bwd(_csr(), 2, 8, xl_rows=-1) == GNO_ERR_INVALID and b"bad sizes" in _error()
    for g in (_csr(N=-1), _csr(E=-3)):
        assert _fwd(g, 2, 8) == GNO_ERR_INVALID and b"bad sizes" in _error()
        assert _bwd(g, 2, 8) == GNO_ERR_INVALID and b"bad sizes" in _error()
        assert _ws(g, 2, 8)[0] == GNO_ERR_INVALID
        assert _bws(g, 2, 8)[0] == GNO_ERR_INVALID


def test_unknown_dtype_is_invalid():
    assert _fwd(_csr(), 2, 8, dtype=7) == GNO_ERR_INVALID and b"dtype" in _error()
    assert _bwd(_csr(), 2, 8, dtype=7) == GNO_ERR_INVALID and b"dtype" in _error()


def test_null_buffers_are_invalid_when_there_are_edges():
    assert _fwd(_csr(), 2, 8) == GNO_ERR_INVALID and b"NULL" in _error()
    assert _bwd(_csr(), 2, 8) == GNO_ERR_INVALID and b"NULL" in _error()


def test_no_edges_touch_nothing():
    g = _csr(E=0)
    assert _fwd(g, 2, 8) == 0
    assert _bwd(g, 2, 8) == 0
    assert _ws(g, 2, 8) == (0, 0)
    assert _bws(g, 2, 8) == (0, 0)


def test_workspace_sizes():
    g = _csr(N=4, E=100, chunk_len=32)                    # 4 chunks, rows padded to 16 floats
    rc, fwd = _ws(g, 2, 10)                               # acc partials + (m, s) partials
    assert rc == 0 and fwd >= 2 * 4 * 16 * 4 + 2 * 4 * 2 * 8
    rc, own = _bws(g, 2, 10, grad_r=1, att=0)
    assert rc == 0 and own >= 2 * 4 * 16 * 4
    rc, att = _bws(g, 2, 10, grad_r=0, att=1)             # per-CTA grad_att partials only
    assert rc == 0 and att >= 10 * 4
    rc, both = _bws(g, 2, 10)
    assert rc == 0 and both >= own + att - 256
    assert _bws(g, 2, 10, grad_r=0, att=0) == (0, 0)      # da and alpha alone need no workspace


def test_gatv2_attention_refuses_cpu_tensors():
    import gno_b200
    N, H, C = 3, 2, 4
    src = torch.tensor([0, 1, 2, 0])
    dst = torch.tensor([1, 2, 0, 0])
    with pytest.raises(gno_b200.GnoError):
        gno_b200.gatv2_attention(torch.randn(N, H, C), torch.randn(N, H, C), torch.randn(H, C), src, dst)


def test_gatv2_attention_public_signature():
    import inspect

    import gno_b200
    params = inspect.signature(gno_b200.gatv2_attention).parameters
    assert list(params) == ["x_l", "x_r", "att", "src", "dst", "negative_slope"]
    assert params["negative_slope"].default == 0.2
    doc = gno_b200.gatv2_attention.__doc__
    assert "dropout" in doc and "return_attention_weights" in doc
