"""
Lowered user terms (genesis_forge_b200/expr.py) op by op at edge values, without a GPU.

Two references:
  * `reference`: a float64 evaluation of the IR.  Each node is computed in float64 from the fp32 / int32 /
    bool values of its operands and rounded to the node's dtype -- the per-node rounding the IR promises.
    For add, sub, mul, div and sqrt that is the correctly rounded fp32 result (double rounding through
    float64 is innocuous for them); fma (norm over 2 / 3 elements) is rounded once, explicitly.  Edge rules
    follow torch-CPU where torch is path independent: casts, ties of clamp / amax / amin, NaN propagation,
    int32 wraparound, the sign rule of `%`, sums starting from +0.
  * torch-CPU float32 running the user's own Python function: the project's semantic reference.

Here both are pinned against each other on a grid of edge values, and the code `function_body` emits is
checked for the torch rules the kernel must follow.  tests/test_gpu_user_terms_edges.py runs the same op
table through the specialised kernel on a B200 and compares it with both.
"""
from __future__ import annotations

import hashlib
import math
import re
import types

import numpy as np
import pytest
import torch

from genesis_forge_b200 import expr
from genesis_forge_b200.managers.observation import UnsupportedTermError
from test_user_terms import evaluate

F64, F32N, I64 = np.float64, np.float32, np.int64
D = 12  # the go2 workloads' action width: env.actions and env.last_actions give 24 fp32 inputs per env
INT_MIN = -(1 << 31)

# ------------------------------------------------------------------------------------------------
# edge values
# ------------------------------------------------------------------------------------------------
_DEN_MIN, _DEN_MAX, _FLT_MIN, _FLT_MAX = 2.0 ** -149, 2.0 ** -126 - 2.0 ** -149, 2.0 ** -126, float(np.finfo(F32N).max)
_HALF_PI = [float(F32N(k * math.pi / 2)) for k in (1, 2, 3, 4, 7, 1000, 65536)]
EDGE = sorted({
    0.0, _DEN_MIN, _DEN_MAX, _FLT_MIN, 1.0, _FLT_MAX, math.inf,
    88.72284, 88.72285, 87.33655, 103.27893, 103.972,  # exp overflow / underflow / last-denormal points
    1e4, 1e30, *_HALF_PI, *(float(np.nextafter(F32N(h), F32N(np.inf))) for h in _HALF_PI),
    *(float(np.nextafter(F32N(h), F32N(0))) for h in _HALF_PI),
    1e-10, 1e-4, 0.1, 0.5, 2.5, 3.0, 8.9, 9.0, 9.1,  # tanh near 0 and +-9, rounding of halves
    2.0 ** 24 - 1, 2.0 ** 24, 2.0 ** 24 + 2, 2147483520.0, 2.0 ** 31, 2147483904.0, 3e9,  # casts
}, key=lambda v: (v, str(v)))
EDGE = EDGE + [-v for v in EDGE] + [math.nan]  # +-0 and +-x of every value, NaN
EDGE_F32 = np.array(EDGE, dtype=F32N)
# integer operands (exact in fp32); the divisor grid has no 0 (and no -1: INT_MIN % -1 overflows)
INT_A = [0, 1, -1, 2, -2, 3, -7, 7, 46341, -46341, 65536, 16777216, 16777218, 2147483520, INT_MIN]
INT_B = [1, 2, -2, 3, -3, 7, -7, 46341, 65536, 2147483520, INT_MIN]


def edge_inputs(n_min: int = 0, seed: int = 0) -> np.ndarray:
    """(N, 24) fp32: columns 0 / 1 every pair of edge values, 2 / 3 every pair of integer operands (cycled),
    4..23 edge values and normal draws.  Row r: env.actions = [:, :12], env.last_actions = [:, 12:]."""
    rng = np.random.default_rng(seed)
    pairs = np.array([(a, b) for a in EDGE_F32 for b in EDGE_F32], dtype=F32N)
    ints = np.array([(a, b) for a in INT_A for b in INT_B], dtype=F32N)
    n = max(len(pairs), n_min)
    n += -n % 4  # lowering needs num_envs % 4 == 0
    x = np.empty((n, 2 * D), dtype=F32N)
    x[:, 0:2] = pairs[np.arange(n) % len(pairs)]
    x[:, 2:4] = ints[np.arange(n) % len(ints)]
    pool = np.concatenate([EDGE_F32, rng.standard_normal(64).astype(F32N) * 3])
    x[:, 4:] = pool[rng.integers(0, len(pool), (n, 2 * D - 4))]
    x[n // 2:, 4:] = (rng.standard_normal((n - n // 2, 2 * D - 4)) * 4).astype(F32N)  # finite rows for long sums
    return x


# ------------------------------------------------------------------------------------------------
# the op table: one user term per op, over the 24 inputs
# ------------------------------------------------------------------------------------------------
def _x(e): return e.actions[:, 0]
def _y(e): return e.actions[:, 1]
def _i(e): return e.actions[:, 2].int()
def _j(e): return e.actions[:, 3].int()


# (name, function, comparison).  Comparisons: "exact" -- bit-exact against both references (NaN as a class);
# "zeros" -- ties of +0 / -0 unspecified (zeros compare by value); "tie" -- exact against float64, zeros by
# value against torch-CPU (a clamp with a tensor bound: torch's vectorised path returns the bound on a tie,
# its scalar path x); "sqrt" -- exact against float64, within
# 1 ulp of torch-CPU; ("ulp", k) -- transcendental, special-value classes exact, finite results within the
# CUDA Programming Guide's k ulp of the float64 result; "bound" -- a reduction over n >= 5 elements, within
# (n-1)*2^-24*sum|x_i| + half an ulp of the float64 sum.
OPS = [
    ("neg", lambda e: -_x(e), "exact"),
    ("abs", lambda e: _x(e).abs(), "exact"),
    ("square", lambda e: _x(e).square(), "exact"),
    ("pow2", lambda e: _x(e) ** 2, "exact"),
    ("sqrt", lambda e: _x(e).sqrt(), "sqrt"),
    ("exp", lambda e: torch.exp(_x(e)), ("ulp", 2)),
    ("log", lambda e: torch.log(_x(e)), ("ulp", 1)),
    ("sin", lambda e: torch.sin(_x(e)), ("ulp", 2)),
    ("cos", lambda e: torch.cos(_x(e)), ("ulp", 2)),
    ("tanh", lambda e: torch.tanh(_x(e)), ("ulp", 2)),
    ("add", lambda e: _x(e) + _y(e), "exact"),
    ("sub", lambda e: _x(e) - _y(e), "exact"),
    ("mul", lambda e: _x(e) * _y(e), "exact"),
    ("div", lambda e: _x(e) / _y(e), "exact"),
    ("div_scalar", lambda e: _x(e) / 3.0, "exact"),
    ("mul_scalar", lambda e: _x(e) * 0.1, "exact"),
    ("rsub_scalar", lambda e: 1.0 - _x(e), "exact"),
    ("minimum", lambda e: torch.minimum(_x(e), _y(e)), "zeros"),
    ("maximum", lambda e: torch.maximum(_x(e), _y(e)), "zeros"),
    ("clamp_lo", lambda e: torch.clamp(_x(e), min=_y(e)), "tie"),
    ("clamp_hi", lambda e: torch.clamp(_x(e), max=_y(e)), "tie"),
    ("clamp_both", lambda e: torch.clamp(_x(e), min=-_y(e).abs(), max=_y(e).abs()), "tie"),
    ("clamp_lo_scalar", lambda e: torch.clamp(_x(e), min=0.0), "exact"),
    ("clamp_hi_scalar", lambda e: _x(e).clamp(max=-0.0), "exact"),
    ("clamp_nan_scalar", lambda e: _x(e).clamp(max=math.nan), "exact"),
    ("clamp_nan_two_scalars", lambda e: _x(e).clip(-1.0, math.nan), "exact"),
    ("where", lambda e: torch.where(_x(e) > _y(e), _x(e), _y(e) * 2.0), "exact"),
    ("lt", lambda e: (_x(e) < _y(e)).float(), "exact"),
    ("le", lambda e: (_x(e) <= _y(e)).float(), "exact"),
    ("gt", lambda e: (_x(e) > _y(e)).float(), "exact"),
    ("ge", lambda e: (_x(e) >= _y(e)).float(), "exact"),
    ("eq", lambda e: (_x(e) == _y(e)).float(), "exact"),
    ("ne", lambda e: (_x(e) != _y(e)).float(), "exact"),
    ("logic", lambda e: (((_x(e) > 0) & (_y(e) < 0)) | ~(_x(e) >= _y(e))).float(), "exact"),
    ("f2i", lambda e: _x(e).int().float(), "exact"),
    ("f2b", lambda e: _x(e).bool().float(), "exact"),
    ("i2f_round", lambda e: (_i(e) + 1).float(), "exact"),
    ("int_add", lambda e: (_i(e) + _j(e)).float(), "exact"),
    ("int_sub", lambda e: (_i(e) - _j(e)).float(), "exact"),
    ("int_mul", lambda e: (_i(e) * _j(e)).float(), "exact"),
    ("int_mod", lambda e: (_i(e) % _j(e)).float(), "exact"),
    ("int_mod_const", lambda e: (_i(e) % -3).float(), "exact"),
    ("int_neg_abs", lambda e: (-_i(e)).float() + _j(e).abs().float(), "exact"),
    ("int_minmax", lambda e: torch.minimum(_i(e), _j(e)).float() - torch.maximum(_i(e), _j(e)).float(), "exact"),
    ("int_clamp", lambda e: torch.clamp(_i(e), min=0, max=65536).float(), "exact"),
    ("int_where_cmp", lambda e: torch.where(_i(e) <= _j(e), _i(e), -_j(e)).float(), "exact"),
    ("int_times_float", lambda e: _i(e) * 2.5, "exact"),
    ("int_true_div", lambda e: _i(e) / _j(e), "exact"),
    ("index", lambda e: e.last_actions[..., 7], "exact"),
    ("sum1", lambda e: e.actions[:, :1].sum(dim=1), "exact"),
    ("sum2", lambda e: e.actions[:, :2].sum(1), "exact"),
    ("sum3", lambda e: e.actions[:, 4:7].sum(1), "exact"),
    ("mean4", lambda e: e.actions[:, 4:8].mean(1), "exact"),
    ("amax2", lambda e: e.actions[:, :2].amax(dim=1), "exact"),
    ("amin2", lambda e: e.actions[:, :2].amin(dim=1), "exact"),
    ("amax4", lambda e: e.last_actions[:, :4].amax(dim=-1), "exact"),
    ("amin3", lambda e: e.last_actions[:, 1:4].amin(dim=1), "exact"),
    ("norm1", lambda e: e.actions[:, :1].norm(dim=1), "exact"),
    ("norm2", lambda e: e.actions[:, :2].norm(dim=1), "exact"),
    ("norm3", lambda e: e.actions[:, 4:7].norm(dim=-1), "exact"),
    ("norm4", lambda e: torch.norm(e.actions[:, 4:8], dim=1), "exact"),
    ("any_all", lambda e: (e.actions[:, 4:8] > 0).any(dim=1).float() + (e.last_actions[:, :3] < 1).all(1).float(),
     "exact"),
    ("sum5", lambda e: e.actions[:, 4:9].sum(1), "bound"),
    ("sum12", lambda e: e.last_actions.sum(1), "bound"),
    ("mean12", lambda e: e.last_actions.mean(1), "bound"),
    ("norm5", lambda e: e.last_actions[:, 2:7].norm(dim=1), "bound"),
    ("norm12", lambda e: e.last_actions.norm(dim=1), "bound"),
]
OP_NAMES = [name for name, _, _ in OPS]
# a live param set to NaN: torch.clamp ignores a NaN Python-scalar bound
PARAM_OPS = [("clamp_nan_param", lambda e, lo=0.5: torch.clamp(_x(e), min=lo), {"lo": math.nan}, "exact")]
TERMINATIONS = [
    ("t_cmp", lambda e: (_x(e) > _y(e)) & ~(_i(e) % _j(e) == 0)),
    ("t_any", lambda e: (e.actions[:, 4:8] > 0.5).any(dim=1) | (_x(e).int() == INT_MIN)),
    ("t_clamp", lambda e: torch.clamp(_x(e), min=0.0).bool() & (e.last_actions.amax(1) >= 1.0)),
]


def fake_env(actions, last_actions):
    return types.SimpleNamespace(actions=actions, last_actions=last_actions)


def trace(fn, kind="reward", params=None, n=64) -> expr.Program:
    """The Program of `fn` over env.actions / env.last_actions (what trace_term builds from an environment)."""
    tr = expr.Tracer(n, kind)
    env = fake_env(tr.source(("actions",), (D,), expr.F32), tr.source(("last_actions",), (D,), expr.F32))
    p = {k: tr.param(k, v) for k, v in (params or {}).items()}
    out = fn(env, **p)
    if kind == "reward" and out.dtype_ != expr.F32:
        out = tr.cast(out, expr.F32)
    nodes, o = expr._live_nodes(tr.nodes, out._id)
    return expr.Program(kind, nodes, o, tr.params, tr.param_types)


def torch_cpu(fn, x: np.ndarray, params=None) -> np.ndarray:
    t = torch.from_numpy(x)
    out = fn(fake_env(t[:, :D], t[:, D:]), **(params or {}))
    return (out.float() if out.dtype != torch.bool else out).numpy()


# ------------------------------------------------------------------------------------------------
# float64 reference of the IR
# ------------------------------------------------------------------------------------------------
def _r32(x):
    return np.asarray(x, F64).astype(F32N)


def _wrap32(x):
    return ((np.asarray(x, I64) + (1 << 31)) % (1 << 32) - (1 << 31)).astype(np.int32)


def _fma32(a, b, c):
    """fp32 fma(a, b, c): a*b is exact in float64, the sum is rounded once to fp32."""
    p = a.astype(F64) * b.astype(F64)
    c = c.astype(F64)
    s = p + c
    bb = s - p
    err = (p - (s - bb)) + (c - bb)  # TwoSum: s + err == p + c exactly
    r = s.astype(F32N)
    other = np.nextafter(r, np.where(s > r.astype(F64), F32N(np.inf), F32N(-np.inf)))
    mid = (r.astype(F64) + other.astype(F64)) / 2
    # s on the midpoint of two fp32 values while p + c is not: the sign of err decides the direction
    tie = np.isfinite(s) & np.isfinite(err) & (err != 0) & (s == mid)
    up = np.maximum(r, other)
    down = np.minimum(r, other)
    return np.where(tie, np.where(err > 0, up, down), r)


def f2i(x):
    """torch-CPU float -> int32: truncation; NaN, +-Inf and |x| >= 2^31 give INT_MIN."""
    x64 = np.asarray(x, F64)
    ok = (x64 > -2147483904.0) & (x64 < 2147483648.0)
    return np.where(ok, np.trunc(np.where(ok, x64, 0.0)), INT_MIN).astype(np.int32)


def _chain_sum(cols):
    acc = _r32(0.0 + cols[0].astype(F64))  # torch's sum starts from +0
    for c in cols[1:]:
        acc = _r32(acc.astype(F64) + c.astype(F64))
    return acc


def _pick_first(cols, better):
    """amax / amin: NaN propagating, the first element kept on a tie."""
    acc = cols[0]
    for c in cols[1:]:
        acc = np.where(np.isnan(acc), acc, np.where(np.isnan(c) | better(c, acc), c, acc))
    return acc


def _node(prog, n, a, sources, params):
    op, dt = n.op, n.dtype
    if op == "src":
        return sources[n.attr]
    if op == "param":
        v = params[prog.params[n.attr]]
        return np.int32(v) if dt == expr.I32 else F32N(v)
    if op in ("const", "constvec"):
        return np.array(n.attr, dtype={expr.F32: F32N, expr.I32: np.int32, expr.BOOL: np.bool_}[dt])
    x = a[0] if a else None
    if op == "cast":
        if dt == expr.BOOL:
            return x != 0
        if dt == expr.F32:
            return _r32(x.astype(F64))
        return f2i(x) if x.dtype == F32N else x.astype(np.int32)
    if op == "not":
        return ~x
    if op in ("neg", "abs", "square") and dt == expr.I32:
        x = x.astype(I64)
        return _wrap32({"neg": -x, "abs": np.abs(x), "square": x * x}[op])
    if op in ("neg", "abs", "square", "sqrt", "exp", "log", "sin", "cos", "tanh"):
        x = x.astype(F64)
        fn = {"neg": np.negative, "abs": np.abs, "square": np.square}.get(op) or getattr(np, op)
        return _r32(fn(x))
    if op == "where":
        return np.where(*a)
    if op == "index":
        return x[(slice(None),) + tuple(s if isinstance(s, int) else slice(*s) for s in n.attr)]
    if op in ("sum", "mean", "any", "all", "amax", "amin", "norm"):
        cols = [np.take(x, k, axis=n.attr + 1) for k in range(x.shape[n.attr + 1])]
        if op in ("any", "all"):
            return (np.any if op == "any" else np.all)(np.stack(cols, -1), axis=-1)
        if dt == expr.I32:
            if op == "sum":
                return _wrap32(sum(c.astype(I64) for c in cols))
            return (np.maximum if op == "amax" else np.minimum).reduce(cols)
        if op in ("amax", "amin"):
            return _pick_first(cols, np.greater if op == "amax" else np.less)
        if op == "norm":
            if len(cols) == 1:
                return np.abs(cols[0])
            if len(cols) <= 3:  # sqrt(fma(z, z, fma(y, y, x*x)))
                acc = _r32(cols[0].astype(F64) ** 2)
                for c in cols[1:]:
                    acc = _fma32(c, c, acc)
                return _r32(np.sqrt(acc.astype(F64)))
            return _r32(np.sqrt(_chain_sum([_r32(c.astype(F64) ** 2) for c in cols]).astype(F64)))
        s = _chain_sum(cols)
        return s if op == "sum" else _r32(s.astype(F64) / len(cols))
    b = a[1]
    if op in ("clamp_lo", "clamp_hi"):
        if dt == expr.I32:
            return (np.maximum if op == "clamp_lo" else np.minimum)(x, b)
        out = np.where((x < b) if op == "clamp_lo" else (x > b), b, x)  # x kept on a tie
        return out if n.attr == "scalar" else np.where(np.isnan(b), b, out)
    if op in ("minimum", "maximum"):
        return (np.minimum if op == "minimum" else np.maximum)(x, b)  # NaN propagating; ties unspecified
    cmp = {"lt": np.less, "le": np.less_equal, "gt": np.greater, "ge": np.greater_equal, "eq": np.equal,
           "ne": np.not_equal, "and": np.logical_and, "or": np.logical_or}
    if op in cmp:
        return cmp[op](x, b)
    if dt == expr.I32:
        x, b = x.astype(I64), b.astype(I64)
        if op == "mod":
            r = np.fmod(x, b)
            return _wrap32(np.where((r != 0) & ((r < 0) != (b < 0)), r + b, r))
        return _wrap32({"add": x + b, "sub": x - b, "mul": x * b}[op])
    x, b = x.astype(F64), b.astype(F64)
    return _r32({"add": x + b, "sub": x - b, "mul": x * b, "div": x / b}[op])


def reference(prog: expr.Program, sources: dict, params=None) -> np.ndarray:
    vals = []
    with np.errstate(all="ignore"):
        for n in prog.nodes:
            vals.append(_node(prog, n, [vals[i] for i in n.args], sources, params or {}))
    return vals[prog.out]


def sources_of(x: np.ndarray) -> dict:
    return {("actions",): x[:, :D], ("last_actions",): x[:, D:]}


def exact_sum_bound(prog: expr.Program, x: np.ndarray):
    """(float64 value, bound, rows it holds for) of a reduction over n >= 5 elements (norm: of the sum of
    squares, then sqrt).  It holds where no partial sum in any order can overflow fp32."""
    red = prog.nodes[prog.out]
    src = prog.nodes[red.args[0]]
    cols = reference(expr.Program(prog.kind, prog.nodes[:red.args[0] + 1], red.args[0], prog.params,
                                  prog.param_types), sources_of(x)).astype(F64)
    terms = cols ** 2 if red.op == "norm" else cols
    n = src.shape[red.attr]
    exact = terms.sum(axis=1)
    bound = (n - 1) * 2.0 ** -24 * np.abs(terms).sum(axis=1)
    rows = np.abs(terms).sum(axis=1) < _FLT_MAX
    if red.op == "mean":
        exact, bound = exact / n, bound / n
    if red.op == "norm":  # sqrt(s + d) - sqrt(s) <= d / (2 sqrt(s)), and <= sqrt(d)
        root = np.sqrt(exact)
        with np.errstate(all="ignore"):
            bound = np.minimum(np.sqrt(bound), bound / (2 * root))
        exact = root
    with np.errstate(all="ignore"):
        half_ulp = 0.5 * np.spacing(np.abs(exact).astype(F32N)).astype(F64)
    return exact, bound + half_ulp, rows


# ------------------------------------------------------------------------------------------------
# comparisons (shared with the GPU tests)
# ------------------------------------------------------------------------------------------------
def ordered(x: np.ndarray) -> np.ndarray:
    """fp32 bit patterns on a line (adjacent floats differ by 1; +0 and -0 are both 0)."""
    i = np.asarray(x, F32N).view(np.int32).astype(I64)
    return np.where(i < 0, -(i & 0x7FFFFFFF), i)


def ulp_dist(a, b) -> np.ndarray:
    """Distance in fp32 steps; 0 where both are NaN."""
    both_nan = np.isnan(np.asarray(a, F32N)) & np.isnan(np.asarray(b, F32N))
    return np.where(both_nan, 0, np.abs(ordered(a) - ordered(b)))


def same_bits(got, want, zeros_by_value=False) -> np.ndarray:
    """Bit equality, NaN compared as a class (CUDA and x86 produce different payloads)."""
    got, want = np.asarray(got), np.asarray(want)
    if got.dtype == np.bool_ or want.dtype == np.bool_:
        return got.astype(np.bool_) == want.astype(np.bool_)
    g, w = got.astype(F32N), want.astype(F32N)
    eq = (g.view(np.int32) == w.view(np.int32)) | (np.isnan(g) & np.isnan(w))
    if zeros_by_value:
        eq |= (g == 0) & (w == 0)
    return eq


def special_class(x):
    x = np.asarray(x, F32N)
    return np.where(np.isnan(x), 0, np.where(np.isposinf(x), 1, np.where(np.isneginf(x), 2, 3)))


def ulp_error_vs_float64(got, exact64) -> np.ndarray:
    """|got - exact| in units of the fp32 spacing at the exact result (finite entries; others 0)."""
    got64 = np.asarray(got, F32N).astype(F64)
    fin = np.isfinite(got64) & np.isfinite(exact64)
    with np.errstate(all="ignore"):
        err = np.abs(got64 - exact64) / np.spacing(np.abs(exact64).astype(F32N)).astype(F64)
    return np.where(fin, err, 0.0)


def exact64(name, x: np.ndarray) -> np.ndarray:
    """Unrounded float64 result of a transcendental op of the table (its input is column 0)."""
    fn = {"exp": np.exp, "log": np.log, "sin": np.sin, "cos": np.cos, "tanh": np.tanh}[name]
    with np.errstate(all="ignore"):
        return fn(x[:, 0].astype(F64))


# ------------------------------------------------------------------------------------------------
# the reference against torch-CPU
# ------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def grid():
    return edge_inputs()


def test_grid_covers_the_edges(grid):
    col = grid[:, 0]
    for v in (0.0, _DEN_MIN, _DEN_MAX, _FLT_MIN, _FLT_MAX, math.inf, 88.72284, 87.33655, 103.27893, 2.0 ** 31):
        for s in (1, -1):
            hit = col == F32N(s * v)
            assert hit.any() and (np.signbit(col[hit]) == (s < 0)).any(), (s, v)
    assert np.isnan(col).any() and len(grid) % 4 == 0
    ties = (grid[:, 0] == grid[:, 1]) & (np.signbit(grid[:, 0]) != np.signbit(grid[:, 1]))
    assert ties.any()  # +0 / -0 pairs for min / max / clamp


@pytest.mark.parametrize("name", OP_NAMES + [p[0] for p in PARAM_OPS])
def test_reference_agrees_with_torch_cpu(name, grid):
    fn, cmp, params = next(((f, c, {}) for n, f, c in OPS if n == name), None) or \
        next((f, c, p) for n, f, p, c in PARAM_OPS if n == name)
    prog = trace(fn, params=params)
    ref = reference(prog, sources_of(grid), params)
    got = torch_cpu(fn, grid, params)
    assert ref.dtype == got.dtype == F32N and ref.shape == got.shape == (len(grid),)
    if cmp in ("exact", "zeros", "tie"):
        bad = ~same_bits(got, ref, zeros_by_value=cmp != "exact")
        assert not bad.any(), (name, grid[bad][:4, :4], got[bad][:4], ref[bad][:4])
    elif cmp == "sqrt":
        assert (special_class(got) == special_class(ref)).all()
        assert ulp_dist(got, ref).max() <= 1
        # the reference itself is the correctly rounded square root
        assert same_bits(ref, _r32(np.sqrt(grid[:, 0].astype(F64)))).all()
    elif cmp == "bound":
        exact, bound, fin = exact_sum_bound(prog, grid)
        assert (np.abs(ref[fin].astype(F64) - exact[fin]) <= bound[fin]).all()
        assert (np.abs(got[fin].astype(F64) - exact[fin]) <= bound[fin]).all()
        special = ~np.isfinite(grid).all(axis=1)
        assert (special_class(got[special]) == special_class(ref[special])).all()
    else:  # transcendental: torch's own accuracy is within 1 ulp of the correctly rounded result
        assert (special_class(got) == special_class(ref)).all(), name
        assert ulp_dist(got, ref).max() <= 1, name
        assert ulp_error_vs_float64(ref, exact64(name, grid)).max() <= 0.5


@pytest.mark.parametrize("name,fn", TERMINATIONS)
def test_termination_reference_agrees_with_torch_cpu(name, fn, grid):
    prog = trace(fn, kind="termination")
    assert prog.nodes[prog.out].dtype == expr.BOOL
    assert (reference(prog, sources_of(grid)) == torch_cpu(fn, grid)).all(), name


def test_torch_evaluator_of_the_ir_matches_on_the_edge_grid(grid):
    """The torch evaluator of tests/test_user_terms.py runs the IR through torch ops: on the edge grid it
    reproduces the Python functions wherever the op is path independent."""
    src = {k: torch.from_numpy(v) for k, v in sources_of(grid).items()}
    for name, fn, cmp in OPS:
        # (torch.norm over a strided slice takes another path; the evaluator clamps one bound at a time)
        if cmp != "exact" or name.startswith(("norm", "clamp")):
            continue
        got = evaluate(trace(fn), src, {})
        assert same_bits(got.float().numpy(), torch_cpu(fn, grid)).all(), name


# leads that show up without a GPU: each row pins one torch-CPU rule the reference follows
@pytest.mark.parametrize("fn,x,want", [
    (lambda e: e.actions[:, :2].norm(dim=1), [0.1, 0.7], None),  # fma chain, not the plain sum of squares
    (lambda e: e.actions[:, :1].norm(dim=1), [1e30], 1e30),  # |x|: no overflow of x*x
    (lambda e: _x(e).int().float(), [math.nan], float(INT_MIN)),
    (lambda e: _x(e).int().float(), [math.inf], float(INT_MIN)),
    (lambda e: _x(e).int().float(), [3e9], float(INT_MIN)),
    (lambda e: torch.clamp(_x(e), min=0.0), [-0.0], -0.0),
    (lambda e: torch.clamp(_x(e), max=-0.0), [0.0], 0.0),
    (lambda e: e.actions[:, :2].amax(dim=1), [-0.0, 0.0], -0.0),
    (lambda e: e.actions[:, :2].amin(dim=1), [0.0, -0.0], 0.0),
    (lambda e: torch.clamp(_x(e), min=math.nan), [2.0], 2.0),
    (lambda e: torch.clamp(_x(e), min=_y(e)), [2.0, math.nan], math.nan),
    (lambda e: e.actions[:, :2].sum(1), [-0.0, -0.0], 0.0),
])
def test_edge_rules_of_the_reference(fn, x, want):
    row = np.zeros((4, 2 * D), dtype=F32N)
    row[:, :len(x)] = x
    ref = reference(trace(fn), sources_of(row))
    got = torch_cpu(fn, row)
    assert same_bits(got, ref).all(), (got, ref)
    if want is not None:
        assert same_bits(ref, np.full(4, want, F32N)).all(), ref


def test_norm_over_two_and_three_elements_is_the_fma_chain():
    rng = np.random.default_rng(5)
    x = rng.standard_normal((20000, 2 * D)).astype(F32N)
    for k in (2, 3):
        fn = lambda e, k=k: e.actions[:, :k].norm(dim=1)  # noqa: E731
        prog = trace(fn)
        ref = reference(prog, sources_of(x))
        assert same_bits(torch_cpu(fn, x), ref).all()
        plain = _r32(np.sqrt(_chain_sum([_r32(x[:, c].astype(F64) ** 2) for c in range(k)]).astype(F64)))
        assert (~same_bits(plain, ref)).sum() > 100  # the plain chain is a different function


# ------------------------------------------------------------------------------------------------
# the code function_body emits
# ------------------------------------------------------------------------------------------------
def code(fn, kind="reward", params=None) -> str:
    return expr.function_body(trace(fn, kind, params), "f")


def test_norm_emits_the_device_utils_chains():
    assert re.search(r"= norm2\(v1_0, v1_1\);", code(lambda e: e.actions[:, :2].norm(dim=1)))
    assert re.search(r"= norm3\(v1_0, v1_1, v1_2\);", code(lambda e: e.actions[:, 4:7].norm(dim=-1)))
    assert re.search(r"= fabsf\(v1_0\);", code(lambda e: e.actions[:, 3:4].norm(dim=1)))
    four = code(lambda e: e.actions[:, :4].norm(dim=1))
    assert "norm" not in four.replace("norm(", "") and four.count("sq(") == 4 and "__fsqrt_rn" in four


def test_float_to_int_casts_use_the_torch_rule():
    text = code(lambda e: _x(e).int().float())
    assert "gfb_user_f2i(" in text and "__float2int_rz" not in text
    assert "__int2float_rn" in text


def test_clamp_emits_the_tie_and_nan_rules():
    assert "gfb_user_clamp_lo(" in code(lambda e: torch.clamp(_x(e), min=_y(e)))
    assert "gfb_user_clamp_hi(" in code(lambda e: torch.clamp(_x(e), max=_y(e)))
    assert "gfb_user_clamp_lo_scalar(" in code(lambda e: torch.clamp(_x(e), min=0.0))
    assert "gfb_user_clamp_hi_scalar(" in code(lambda e, hi=1.0: _x(e).clamp(max=hi), params={"hi": 1.0})
    assert "gfb_user_clamp_hi(" in code(lambda e: _x(e).clamp(max=torch.tensor(1.0)))  # a tensor bound
    text = code(lambda e: torch.minimum(_x(e), _y(e)))
    assert "gfb_user_min(" in text and "clamp" not in text


def test_amax_amin_keep_the_first_element_on_a_tie():
    text = code(lambda e: e.actions[:, :3].amax(dim=1))
    assert "v2_0 = gfb_user_max(v1_1, v2_0);" in text and "v2_0 = gfb_user_max(v1_2, v2_0);" in text
    assert "v2_0 = gfb_user_min(v1_1, v2_0);" in code(lambda e: e.actions[:, :2].amin(dim=1))


def test_float_sums_start_from_plus_zero():
    assert "float v2_0 = add(0.0f, v1_0);" in code(lambda e: e.actions[:, :2].sum(1))
    assert "float v2_0 = add(0.0f, v1_0);" in code(lambda e: e.actions[:, :5].mean(1))


def test_device_helpers_are_defined():
    from pathlib import Path

    text = (Path(expr.__file__).parent / "csrc" / "post_kernel.cuh").read_text()
    for name in ("gfb_user_clamp_lo", "gfb_user_clamp_hi", "gfb_user_clamp_lo_scalar", "gfb_user_clamp_hi_scalar",
                 "gfb_user_f2i"):
        assert f" {name}(float" in text, name


def test_digest_changes_with_the_emitted_code():
    """A term whose code changed gets a new identity, so a specialisation built from older code is not
    matched against it; the identity still follows the expression."""
    for fn in (lambda e: e.actions[:, :3].norm(dim=1), lambda e: torch.clamp(_x(e), min=0.0)):
        prog = trace(fn)
        before = int.from_bytes(hashlib.sha1(prog.text().encode()).digest()[:4], "little") & 0x7FFFFFFF
        assert prog.digest() != before
        assert prog.digest() == trace(fn).digest()
    assert trace(lambda e: torch.clamp(_x(e), min=0.0)).digest() != \
        trace(lambda e: torch.clamp(_x(e), min=torch.tensor(0.0))).digest()


# ------------------------------------------------------------------------------------------------
# refusals
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("fn,needle", [
    (lambda e: (_i(e) % 0).float(), "constant 0"),
    (lambda e: _i(e) * torch.tensor(0.5, dtype=torch.float64), "float64"),
    (lambda e: (_x(e) > 0) + torch.tensor(2.0, dtype=torch.float64), "float64"),
    (lambda e: torch.where(_x(e) > 0, _i(e), torch.tensor(0.5, dtype=torch.float64)), "float64"),
    (lambda e: torch.clamp(_i(e), min=torch.tensor(0.5, dtype=torch.float64)), "float64"),
    (lambda e: _x(e).to(torch.int64).float(), "int64"),
    (lambda e: _x(e).type(torch.int64).float(), "int64"),
    (lambda e: _x(e).long().float(), "long"),
])
def test_refusals(fn, needle):
    with pytest.raises(UnsupportedTermError, match=needle):
        trace(fn)


def test_what_torch_does_in_the_refused_cases():
    i = torch.tensor([3], dtype=torch.int32)
    with pytest.raises(Exception, match="ZeroDivision"):
        i % 0
    assert (i * torch.tensor(0.5, dtype=torch.float64)).dtype is torch.float64
    assert torch.tensor([3e9]).to(torch.int64).item() == 3000000000


def test_int_to_int64_cast_is_still_lowered(grid):
    fn = lambda e: (_i(e) % 3).float() + _i(e).to(torch.int64).float()  # noqa: E731 - int -> int64 stays
    assert same_bits(torch_cpu(fn, grid), reference(trace(fn), sources_of(grid))).all()
