"""Several aggregators over one neighbourhood in one pass: PNAConv.aggregate's list of aggregators
(sum, mean, min, max, var, std) with degree scalers (identity, amplification, attenuation, linear,
inverse_linear), forward and backward, on the CUDA library (include/gno_b200.h:
gno_multi_aggregate*, gno_multi_aggregate_backward, gno_multi_aggregate_coeffs).

Composed from `scatter`, the default PNA set (mean, min, max, std) reads the [E, F] messages about
seven times and materialises their square; `multi_aggregate` reads each message once and writes
every requested block from the same per-row statistics.  The forward and the message-form
backward use the cached dst-sorted plan of the destination index; the gather-form backward adds
the cached src-sorted plan of the sources, so a training step builds at most two plans once and
reuses them.
"""
import collections.abc
import ctypes

import torch

from . import ops
from ._lib import check, lib
from .plan import _on_device, _ptr, _stream, _workspace, plan_cache

AGGREGATORS = {"sum": 0, "mean": 1, "min": 2, "max": 3, "var": 4, "std": 5}
SCALERS = {"identity": 0, "amplification": 1, "attenuation": 2, "linear": 3, "inverse_linear": 4}
_MAX_LIST = 8
_FLOAT = (torch.float32, torch.float16, torch.bfloat16)


def _codes(names, table, what):
    if isinstance(names, str) or not isinstance(names, collections.abc.Sequence) or len(names) == 0:
        raise ValueError(f"multi_aggregate: {what}s must be a non-empty sequence of names")
    if len(names) > _MAX_LIST:
        raise ValueError(f"multi_aggregate: at most {_MAX_LIST} {what}s")
    out = []
    for n in names:
        if n not in table:
            raise ValueError(f"multi_aggregate: unknown {what} '{n}' (one of {', '.join(table)})")
        out.append(table[n])
    return tuple(out)


def _avg(avg_deg, scls):
    """(avg_lin, avg_log) of PNAConv's avg_deg; required once a scaler other than identity is asked."""
    if all(s == SCALERS["identity"] for s in scls):
        return 1.0, 1.0
    if not isinstance(avg_deg, collections.abc.Mapping) or "lin" not in avg_deg or "log" not in avg_deg:
        raise ValueError('multi_aggregate: scalers other than identity need avg_deg = {"lin": ..., "log": ...}')
    return float(avg_deg["lin"]), float(avg_deg["log"])


class _Spec:
    """What a call computes: towers T, width F, aggregator and scaler codes, avg_deg."""
    __slots__ = ("T", "F", "aggs", "scls", "avg_lin", "avg_log")

    def __init__(self, T, F, aggs, scls, avg_lin, avg_log):
        self.T, self.F, self.aggs, self.scls, self.avg_lin, self.avg_log = T, F, aggs, scls, avg_lin, avg_log

    @property
    def W(self):
        return self.T * self.F

    def args(self):
        a = (ctypes.c_int * len(self.aggs))(*self.aggs)
        s = (ctypes.c_int * len(self.scls))(*self.scls)
        return a, len(self.aggs), s, len(self.scls), self.avg_lin, self.avg_log

    @property
    def second(self):
        return any(a in (AGGREGATORS["var"], AGGREGATORS["std"]) for a in self.aggs)


def _run_forward(x, index, src, N, spec, want_state):
    """out [N, T*S*A*F] and the backward state {mean, var, amin, amax} (None entries when not
    requested; empty dict when want_state is False).  x is [E or N_src, T*F] contiguous."""
    W = spec.W
    out = torch.empty((N, W * len(spec.aggs) * len(spec.scls)), dtype=x.dtype, device=x.device)
    state = {}
    if N == 0 or W == 0:
        return out, state
    plan = plan_cache.get(index, N)
    gidx = plan.perm if src is None else plan.sorted_ids(src)
    csr = plan.csr(gidx, plan.perm)
    if want_state:
        f32 = dict(dtype=torch.float32, device=x.device)
        i32 = dict(dtype=torch.int32, device=x.device)
        state["mean"] = torch.empty((N, W), **f32) if spec.second else None
        state["var"] = torch.empty((N, W), **f32) if spec.second else None
        state["amin"] = torch.empty((N, W), **i32) if AGGREGATORS["min"] in spec.aggs else None
        state["amax"] = torch.empty((N, W), **i32) if AGGREGATORS["max"] in spec.aggs else None
    a, na, s, ns, lin, log = spec.args()
    nbytes = ctypes.c_size_t()
    check(lib.gno_multi_aggregate_workspace(ctypes.byref(csr), spec.T, spec.F, a, na, ctypes.byref(nbytes)))
    ws = _workspace(nbytes.value, x.device) if nbytes.value else None
    st = state.get
    with _on_device(x.device):
        check(lib.gno_multi_aggregate(ctypes.byref(csr), _ptr(x), x.size(0), spec.T, spec.F, a, na, s, ns, lin, log,
                                      _ptr(out), _ptr(st("amin")), _ptr(st("amax")), _ptr(st("mean")),
                                      _ptr(st("var")), plan.E, ops._dtype_id(x), _ptr(ws), nbytes.value,
                                      _stream(x.device)))
    return out, state


def _kept_dst(index, N):
    """index with dropped destinations pointed at row N (the zero row of the [P | Q] table)."""
    return ops._memo("multiagg_kept", index, (N,),
                     lambda: torch.where((index >= 0) & (index < N), index, torch.full_like(index, N)))


def _gather_backward(x, g, index, src, N, spec, state):
    """grad_x[j] = sum over edges e with src[e] = j of P[dst_e] + Q[dst_e] * x_j, plus c_min / c_max
    routed to the winners' source rows (as gather_scatter's min / max backward)."""
    W, dev = spec.W, x.device
    plan = plan_cache.get(index, N)
    pq = torch.empty((N + 1, 2 * W), dtype=torch.float32, device=dev)
    pq[N].zero_()
    f32 = dict(dtype=torch.float32, device=dev)
    cmin = torch.empty((N, W), **f32) if state["amin"] is not None else None
    cmax = torch.empty((N, W), **f32) if state["amax"] is not None else None
    a, na, s, ns, lin, log = spec.args()
    with _on_device(dev):
        check(lib.gno_multi_aggregate_coeffs(ctypes.byref(plan.csr(None, None)), spec.T, spec.F, a, na, s, ns, lin,
                                             log, _ptr(g), _ptr(state["amin"]), _ptr(state["amax"]),
                                             _ptr(state["mean"]), _ptr(state["var"]), _ptr(pq), _ptr(cmin),
                                             _ptr(cmax), ops._dtype_id(x), _stream(dev)))
    n_src = x.size(0)
    plan_t = plan_cache.get(src, n_src)
    d_t = _kept_dst(index, N) if plan.n_dropped else index
    acc = ops.segment_reduce(plan_t, pq, "sum", gidx=plan_t.sorted_ids(d_t))
    grad = torch.addcmul(acc[:, :W], x.to(torch.float32), acc[:, W:])
    if cmin is not None or cmax is not None:
        E = src.numel()
        src_ext = torch.cat([src, src.new_full((1,), -1)])   # winner sentinel E -> -1: dropped
        for w, c in ((state["amin"], cmin), (state["amax"], cmax)):
            if c is not None:
                rows = src_ext[w.to(torch.int64).clamp_(max=E)]
                grad += ops.scatter(c, rows, 0, None, n_src, "sum")
    return grad.to(x.dtype)


class _MultiAggregate(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, index, src, N, spec, want_state):
        out, state = _run_forward(x, index, src, N, spec, want_state)
        ctx.N, ctx.spec, ctx.state = N, spec, state
        ctx.save_for_backward(x, index, src)
        return out

    @staticmethod
    def backward(ctx, grad_out):
        x, index, src = ctx.saved_tensors
        N, spec, state = ctx.N, ctx.spec, ctx.state
        if N == 0 or spec.W == 0 or index.numel() == 0:
            return torch.zeros_like(x), None, None, None, None, None
        g = grad_out.to(x.dtype).contiguous()
        if src is not None:
            return _gather_backward(x, g, index, src, N, spec, state), None, None, None, None, None
        plan = plan_cache.get(index, N)
        grad = torch.zeros_like(x) if plan.n_dropped else torch.empty_like(x)
        a, na, s, ns, lin, log = spec.args()
        with _on_device(x.device):
            check(lib.gno_multi_aggregate_backward(ctypes.byref(plan.csr(plan.perm, plan.perm)), _ptr(x), x.size(0),
                                                   spec.T, spec.F, a, na, s, ns, lin, log, _ptr(g),
                                                   _ptr(state["amin"]), _ptr(state["amax"]), _ptr(state["mean"]),
                                                   _ptr(state["var"]), _ptr(grad), ops._dtype_id(x),
                                                   _stream(x.device)))
        return grad, None, None, None, None, None


def _prepare(inputs, index, dim_size, aggregators, scalers, avg_deg, src):
    aggs = _codes(aggregators, AGGREGATORS, "aggregator")
    scls = _codes(scalers, SCALERS, "scaler")
    avg_lin, avg_log = _avg(avg_deg, scls)
    if inputs.dtype not in _FLOAT:
        raise ValueError(f"multi_aggregate: inputs must be float32, float16 or bfloat16, got {inputs.dtype}")
    if inputs.dim() not in (2, 3):
        raise ValueError(f"multi_aggregate: inputs must be [E, F] or [E, T, F] (towers), got {tuple(inputs.shape)}")
    for name, t in (("index", index), ("src", src)):
        if t is not None and (t.dtype != torch.int64 or t.dim() != 1):
            raise ValueError(f"multi_aggregate: {name} must be a 1-D int64 tensor")
    E = index.numel()
    if src is None and inputs.size(0) != E:
        raise ValueError(f"multi_aggregate: {inputs.size(0)} messages for {E} index entries")
    if src is not None and src.numel() != E:
        raise ValueError(f"multi_aggregate: src has {src.numel()} entries, index {E}")
    ops._need_cuda(inputs, index, src)
    T, F = (1, inputs.size(1)) if inputs.dim() == 2 else (inputs.size(1), inputs.size(2))
    if dim_size is None:  # host sync, as upstream: once per index tensor
        dim_size = ops._memo("dim_size", index, (), lambda: int(index.max()) + 1, capacity=16) if E else 0
    if src is not None:
        ops._check_range(src, inputs.size(0), "multi_aggregate: src")
    return _Spec(T, F, aggs, scls, avg_lin, avg_log), int(dim_size)


def multi_aggregate(inputs, index, dim_size=None, aggregators=("mean", "min", "max", "std"), scalers=("identity",),
                    avg_deg=None, src=None):
    """PNAConv.aggregate: every aggregator of `aggregators` over the messages into each destination,
    concatenated, then one copy per scaler of `scalers`, concatenated:
        out[i, t, (s*A + a)*F + f] = agg_a(messages into i)[t, f] * scale_s(d_i),  d_i = max(deg_i, 1)

    Message form (src=None): inputs [E, F] or [E, T, F] (T towers) in edge order, index int64 [E]
    the destination of each message.  Gather form: message e is inputs[src[e]], inputs node
    features [N_src, F] or [N_src, T, F]; the [E, F] messages are never materialised.

    aggregators: "sum", "mean", "min", "max", "var", "std"; scalers: "identity", "amplification",
    "attenuation", "linear", "inverse_linear" (sequences, kept in order).  avg_deg {"lin", "log"}
    (PNAConv's) is required by any scaler other than identity.  mean = sum / d,
    var = sum(m^2) / d - mean^2, std = sqrt(relu(var) + 1e-5); min / max follow torch_scatter (lowest
    edge wins a tie, NaN never wins, empty row -> 0).  Each scaler block is the unscaled aggregate
    times the scaler.  sum(m) and sum(m^2) accumulate in fp32 (16-bit inputs are not squared in 16
    bits), the scale is applied in fp32 and each output is rounded once.

    Returns [dim_size, S*A*F] or [dim_size, T, S*A*F] in inputs' dtype.  Destinations outside
    [0, dim_size) are dropped with a warning; an out-of-range src raises IndexError.
    Differentiable w.r.t. inputs."""
    spec, N = _prepare(inputs, index, dim_size, aggregators, scalers, avg_deg, src)
    x = inputs.reshape(inputs.size(0), spec.W).contiguous()
    want_state = torch.is_grad_enabled() and inputs.requires_grad
    out = _MultiAggregate.apply(x, index.contiguous(), None if src is None else src.contiguous(), N, spec, want_state)
    SAF = len(spec.aggs) * len(spec.scls) * spec.F
    return out.view(N, spec.T, SAF) if inputs.dim() == 3 else out
