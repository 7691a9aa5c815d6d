"""CPU tests of multi_aggregate (PNAConv.aggregate's aggregators and degree scalers in one pass):
argument validation in Python and at the C-ABI (gno_multi_aggregate*, GNO_ERR_INVALID with a
message before any device work), the workspace query, CPU refusal (no fallback) and the signature."""
import ctypes
import inspect

import pytest
import torch

GNO_ERR_INVALID = 1
PNA = ("mean", "min", "max", "std")


def _csr(N=4, E=8, chunk_len=32):
    from gno_b200 import _lib
    return _lib.gno_csr(N, E, None, None, None, None, chunk_len, 0, None, 0, None)


def _ints(*v):
    return (ctypes.c_int * len(v))(*v)


def _fwd(g, T=1, F=8, aggs=(1, 2, 3, 5), scls=(0,), dtype=0, x_rows=8, arg_fill=8):
    from gno_b200 import _lib
    a, s = _ints(*aggs), _ints(*scls)
    return _lib.lib.gno_multi_aggregate(ctypes.byref(g), None, x_rows, T, F, a, len(aggs), s, len(scls), 1.0, 1.0,
                                        None, None, None, None, None, arg_fill, dtype, None, 0, None)


def _bwd(g, T=1, F=8, aggs=(1, 2, 3, 5), scls=(0,), dtype=0):
    from gno_b200 import _lib
    a, s = _ints(*aggs), _ints(*scls)
    return _lib.lib.gno_multi_aggregate_backward(ctypes.byref(g), None, 8, T, F, a, len(aggs), s, len(scls), 1.0, 1.0,
                                                 None, None, None, None, None, None, dtype, None)


def _coeffs(g, T=1, F=8, aggs=(1, 2, 3, 5), scls=(0,), dtype=0):
    from gno_b200 import _lib
    a, s = _ints(*aggs), _ints(*scls)
    return _lib.lib.gno_multi_aggregate_coeffs(ctypes.byref(g), T, F, a, len(aggs), s, len(scls), 1.0, 1.0, None,
                                               None, None, None, None, None, None, None, dtype, None)


def _ws(g, T=1, F=8, aggs=(1, 2, 3, 5)):
    from gno_b200 import _lib
    n = ctypes.c_size_t()
    rc = _lib.lib.gno_multi_aggregate_workspace(ctypes.byref(g), T, F, _ints(*aggs), len(aggs), ctypes.byref(n))
    return rc, n.value


def _error():
    from gno_b200 import _lib
    return _lib.lib.gno_last_error()


@pytest.mark.parametrize("aggs,scls,msg", [((), (0,), b"aggregators"), ((6,), (0,), b"unknown aggregator"),
                                           ((-1,), (0,), b"unknown aggregator"), ((1,), (), b"scalers"),
                                           ((1,), (5,), b"unknown scaler"), ((0,) * 9, (0,), b"aggregators")])
def test_bad_aggregator_and_scaler_codes_are_invalid(aggs, scls, msg):
    for call in (_fwd, _bwd, _coeffs):
        assert call(_csr(), aggs=aggs, scls=scls) == GNO_ERR_INVALID and msg in _error()


def test_bad_sizes_and_dtype_are_invalid():
    for kw in (dict(T=0), dict(F=-1), dict(T=1 << 12, F=1 << 12)):
        assert _fwd(_csr(), **kw) == GNO_ERR_INVALID and b"bad sizes" in _error()
        assert _bwd(_csr(), **kw) == GNO_ERR_INVALID and b"bad sizes" in _error()
        assert _ws(_csr(), **kw)[0] == GNO_ERR_INVALID
    for g in (_csr(N=-1), _csr(E=-3)):
        assert _fwd(g) == GNO_ERR_INVALID and b"bad sizes" in _error()
    assert _fwd(_csr(chunk_len=48)) == GNO_ERR_INVALID and b"chunk_len" in _error()
    assert _fwd(_csr(), x_rows=-1) == GNO_ERR_INVALID and b"x_rows" in _error()
    assert _fwd(_csr(), arg_fill=1 << 31) == GNO_ERR_INVALID and b"arg_fill" in _error()
    for call in (_fwd, _bwd, _coeffs):
        assert call(_csr(), dtype=7) == GNO_ERR_INVALID and b"dtype" in _error()


def test_null_buffers_and_missing_state_are_invalid():
    assert _fwd(_csr()) == GNO_ERR_INVALID and b"NULL" in _error()
    assert _bwd(_csr()) == GNO_ERR_INVALID and b"NULL" in _error()
    assert _coeffs(_csr()) == GNO_ERR_INVALID and b"NULL" in _error()


def test_nothing_to_do_touches_nothing():
    assert _fwd(_csr(N=0)) == 0
    assert _fwd(_csr(), F=0) == 0
    assert _bwd(_csr(E=0)) == 0
    assert _coeffs(_csr(N=0)) == 0
    assert _ws(_csr(E=0)) == (0, 0)


def test_workspace_holds_only_the_statistics_asked_for():
    g = _csr(N=4, E=100, chunk_len=32)                   # 4 chunks, two partial slots each
    n = 2 * 4 * 2 * 10                                    # slots x T*F (T = 2, F = 10)
    rc, mom = _ws(g, T=2, F=10, aggs=(1, 5))              # sum and sum of squares
    assert rc == 0 and mom >= 2 * n * 4
    rc, ext = _ws(g, T=2, F=10, aggs=(2,))                # min, max and their winners
    assert rc == 0 and ext >= 4 * n * 4
    rc, both = _ws(g, T=2, F=10, aggs=(1, 2, 3, 5))
    assert rc == 0 and both >= mom + ext
    assert both < mom + ext + 7 * 256


def _graph(E=6, N=3):
    return torch.randn(E, 4), torch.tensor([0, 1, 2, 0, 1, 2][:E])


@pytest.mark.parametrize("kw", [dict(aggregators=("mean", "median")), dict(aggregators=()), dict(aggregators="mean"),
                                dict(scalers=("identity", "sqrt")), dict(scalers=())])
def test_unknown_or_empty_names_raise_value_error(kw):
    import gno_b200
    x, idx = _graph()
    with pytest.raises(ValueError):
        gno_b200.multi_aggregate(x, idx, 3, **kw)


@pytest.mark.parametrize("avg_deg", [None, {"lin": 2.0}, {"log": 1.0}, 3.0])
def test_scalers_other_than_identity_need_avg_deg(avg_deg):
    import gno_b200
    x, idx = _graph()
    with pytest.raises(ValueError, match="avg_deg"):
        gno_b200.multi_aggregate(x, idx, 3, scalers=("identity", "amplification"), avg_deg=avg_deg)


def test_length_tower_and_dtype_mismatches_raise_value_error():
    import gno_b200
    x, idx = _graph()
    with pytest.raises(ValueError, match="messages"):
        gno_b200.multi_aggregate(x[:5], idx, 3)                          # message form: one message per edge
    with pytest.raises(ValueError, match="src"):
        gno_b200.multi_aggregate(x, idx, 3, src=torch.tensor([0, 1]))   # gather form: src as long as index
    with pytest.raises(ValueError, match="towers"):
        gno_b200.multi_aggregate(x.view(6, 2, 1, 2), idx, 3)
    with pytest.raises(ValueError, match="towers"):
        gno_b200.multi_aggregate(x[:, 0], idx, 3)
    with pytest.raises(ValueError, match="float"):
        gno_b200.multi_aggregate(torch.ones(6, 4, dtype=torch.int64), idx, 3)
    with pytest.raises(ValueError, match="float"):
        gno_b200.multi_aggregate(x.double(), idx, 3)
    with pytest.raises(ValueError, match="int64"):
        gno_b200.multi_aggregate(x, idx.to(torch.int32), 3)


def test_multi_aggregate_refuses_cpu_tensors():
    import gno_b200
    x, idx = _graph()
    with pytest.raises(gno_b200.GnoError):
        gno_b200.multi_aggregate(x, idx, 3)
    with pytest.raises(gno_b200.GnoError):
        gno_b200.multi_aggregate(torch.randn(3, 2, 4), idx, 3, src=torch.tensor([0, 1, 2, 2, 1, 0]),
                                 scalers=("identity", "linear"), avg_deg={"lin": 2.0, "log": 1.1})


def test_multi_aggregate_public_signature():
    import gno_b200
    params = inspect.signature(gno_b200.multi_aggregate).parameters
    assert list(params) == ["inputs", "index", "dim_size", "aggregators", "scalers", "avg_deg", "src"]
    assert params["dim_size"].default is None
    assert tuple(params["aggregators"].default) == PNA
    assert tuple(params["scalers"].default) == ("identity",)
    assert params["avg_deg"].default is None and params["src"].default is None
