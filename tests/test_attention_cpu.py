"""CPU tests of the graph-attention entry points (gno_segment_softmax*, gno_segment_reduce_heads,
gno_edge_head_dot): argument validation returns GNO_ERR_INVALID before any device work, and the
torch-level ops refuse CPU tensors (no fallback)."""
import ctypes

import pytest
import torch

GNO_ERR_INVALID = 1


def _csr(N=4, E=8, chunk_len=32):
    from gno_b200 import _lib
    return _lib.gno_csr(N, E, None, None, None, None, chunk_len, 0, None, 0, None)


def test_softmax_entry_points_validate_without_gpu():
    from gno_b200 import _lib
    lib = _lib.lib
    g = _csr()
    n = ctypes.c_size_t()
    assert lib.gno_segment_softmax_workspace(ctypes.byref(g), 3, ctypes.byref(n)) == 0
    assert n.value >= (4 * 3 + 2 * 1 * 3) * 8
    for H in (0, -2):
        assert lib.gno_segment_softmax_workspace(ctypes.byref(g), H, ctypes.byref(n)) == GNO_ERR_INVALID
        assert lib.gno_segment_softmax(ctypes.byref(g), None, None, 8, H, 1e-16, None, 0, None, 0,
                                       None) == GNO_ERR_INVALID
        assert lib.gno_segment_softmax_backward(ctypes.byref(g), None, None, None, 8, H, None, 0, None, 0,
                                                None) == GNO_ERR_INVALID
    assert b"H=" in lib.gno_last_error()
    assert lib.gno_segment_softmax(ctypes.byref(g), None, None, 8, 1, 1e-16, None, 7, None, 0, None) == GNO_ERR_INVALID
    assert b"dtype" in lib.gno_last_error()
    # negative sizes, and fewer original edges than the plan holds
    assert lib.gno_segment_softmax(ctypes.byref(g), None, None, -1, 1, 1e-16, None, 0, None, 0, None) == GNO_ERR_INVALID
    assert lib.gno_segment_softmax(ctypes.byref(g), None, None, 5, 1, 1e-16, None, 0, None, 0, None) == GNO_ERR_INVALID
    bad = _csr(N=-1)
    assert lib.gno_segment_softmax_workspace(ctypes.byref(bad), 1, ctypes.byref(n)) == GNO_ERR_INVALID
    # a rowptr plan (no index) must cover every edge
    assert lib.gno_segment_softmax(ctypes.byref(g), None, None, 9, 1, 1e-16, None, 0, None, 0, None) == GNO_ERR_INVALID
    assert lib.gno_segment_softmax(ctypes.byref(_csr(E=0)), None, None, 0, 2, 1e-16, None, 0, None, 0, None) == 0


def test_head_entry_points_validate_without_gpu():
    from gno_b200 import _lib
    lib = _lib.lib
    g = _csr()
    for H, F in ((0, 8), (-1, 8), (3, 8), (2, -4)):
        assert lib.gno_segment_reduce_heads(ctypes.byref(g), None, 4, None, H, None, F, 0, None, 0,
                                            None) == GNO_ERR_INVALID
        assert lib.gno_edge_head_dot(ctypes.byref(g), None, 4, None, H, F, None, 0, None) == GNO_ERR_INVALID
    assert lib.gno_segment_reduce_heads(ctypes.byref(g), None, 4, None, 2, None, 8, 9, None, 0, None) == GNO_ERR_INVALID
    assert lib.gno_edge_head_dot(ctypes.byref(g), None, 4, None, 2, 8, None, 9, None) == GNO_ERR_INVALID
    assert lib.gno_segment_reduce_heads(ctypes.byref(g), None, -1, None, 2, None, 8, 0, None, 0,
                                        None) == GNO_ERR_INVALID
    assert lib.gno_edge_head_dot(ctypes.byref(g), None, -1, None, 2, 8, None, 0, None) == GNO_ERR_INVALID
    # E = 0: nothing to do, no device touched
    assert lib.gno_edge_head_dot(ctypes.byref(_csr(E=0)), None, 4, None, 2, 8, None, 0, None) == 0


def test_attention_ops_refuse_cpu_tensors():
    import gno_b200
    E, N, H, C = 6, 3, 2, 4
    src = torch.tensor([0, 1, 2, 0, 1, 2])
    dst = torch.tensor([0, 0, 1, 1, 2, 2])
    with pytest.raises(gno_b200.GnoError):
        gno_b200.softmax(torch.randn(E, H), dst)
    with pytest.raises(gno_b200.GnoError):
        gno_b200.softmax(torch.randn(E, H), ptr=torch.tensor([0, 2, 4, 6]))
    with pytest.raises(gno_b200.GnoError):
        gno_b200.attention_aggregate(torch.randn(N, H, C), torch.rand(E, H), src, dst, N)


def test_attention_ops_public_signatures():
    import inspect

    import gno_b200
    assert list(inspect.signature(gno_b200.softmax).parameters) == ["src", "index", "ptr", "num_nodes", "dim"]
    assert list(inspect.signature(gno_b200.attention_aggregate).parameters) == ["x", "alpha", "src", "dst",
                                                                                "dim_size"]
