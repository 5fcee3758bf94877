"""
User-defined reward / termination / observation terms lowered into the specialised post-physics kernel.

A user term is a plain Python function of the environment, e.g.

    def speed(env):
        return env.robot.get_vel()[:, 0].abs()

`trace_term` runs it ONCE with symbolic stand-ins for the per-env state it may read (the primary
entity's getters, the first EntityManager's cache and body-frame vectors, the action manager's
getters, env.actions / last_actions / episode_length / max_episode_length, the `command` of
kernel-resampled command managers, contact forces and air-time state, the primary entity's link positions /
velocities (`get_links_pos` / `get_links_vel` with `links_idx_local`, and its link objects' `get_pos` /
`get_vel`; FusedStep._layout_links binds them as per-launch gathers in free GFB_B_USER_STATE slots) and -- rewards
only -- extras["terminations"] / ["time_outs"]).  Every operation on them is recorded as a node of a small
expression IR (`Program`) with torch's shapes and type promotion.  Scalar entries of the term's
params become LIVE slots (the term's p[4] in the packed table), so a curriculum that edits them keeps
the same kernel binary; everything else the function captures is a compile-time constant.

`device_code` turns a Program into one straight-line `__device__` function per term, in torch's
operation order with the kernel's round-to-nearest helpers; reductions accumulate in index order.
The generated functions go into the header of the specialised kernel (spec.py) and are called in the
owner phase of post_kernel, in the GFB_R_USER / GFB_T_USER cases of the term switches.

Observation terms (kind "observation", ManagedEnvironment.fuse_user_observations) may return any
per-env shape of at most MAX_CONST_VEC elements, which is flattened row-major into their columns and cast
to fp32, and may build rows with the layout ops torch.stack / torch.cat over the last dimension,
unsqueeze, None in an index and reshape / view / flatten of a row.  Their params are constants (traced
again when they change).  Their device code comes twice: for the owner phase of post_kernel and, reading
global memory only, for the reset path that re-observes reset envs (spec_kernel.cu).

Class-style reward / termination / observation terms (an MdpFnClass instance,
ManagedEnvironment.fuse_stateful_terms) are traced through `type(inst).__call__` (`trace_stateful`).  A per-env
tensor attribute of the instance -- (N, *s) with at most MAX_CONST_VEC elements a row, fp32 / int32 / bool,
on the env's device and contiguous -- is a source
("state", slot); rebinding it to a value of the same row shape and dtype, `self.x[:] = v` and `self.x.copy_(v)`
are state writes (`Program.writes`), stored to the env's row after the result is computed.  An attribute
that is None and gets a per-env value during the call (lazy initialisation) gives a second, first-call
program (`Program.first`), which the kernel selects while the term's p[0] is 0 (rewards and terminations
only: an observation term's state exists once the build's dry run has called it).  Python-scalar attributes
and params are trace constants.  An observation term stores its state only when `UserCtx::active` says so:
the owner phase passes `active && !reset`, because the reset path evaluates a reset env once more.

Anything outside this subset raises UnsupportedTermError naming the op or source; the term then
stays a host callback (split execution), with exactly the results it had before.
"""
from __future__ import annotations

import hashlib
import math

import numpy as np
import torch

from .managers.observation import UnsupportedTermError

F32, I32, BOOL = "f32", "i32", "bool"
_RANK = {BOOL: 0, I32: 1, F32: 2}
MAX_CONST_VEC = 32  # GFB_MAX_DOFS: small constant vectors (per-joint limits, gains) are folded in
MAX_LIVE_PARAMS = 4  # gfb_reward_term.p / gfb_termination_term.p
MAX_STATE_SLOTS = 8  # GFB_B_USER_STATE0..7
MAX_LINKS = 10  # links of one per-link array: a (N, |U|, 3) row stays within GFB_MAX_DOFS floats
# bumped whenever `function_body` emits different code for the same IR: the digest changes with it
CODEGEN_REVISION = 2


class _ParamControlFlow(Exception):
    """A live parameter reached Python control flow: trace again with params as constants."""


def _f32(x) -> float:
    return float(np.float32(x))


# ------------------------------------------------------------------------------------------------
# IR
# ------------------------------------------------------------------------------------------------
class Node:
    __slots__ = ("op", "args", "attr", "shape", "dtype", "weak", "envless")

    def __init__(self, op, args, attr, shape, dtype, weak=False, envless=False):
        self.op, self.args, self.attr = op, tuple(args), attr
        self.shape, self.dtype, self.weak = tuple(shape), dtype, weak
        self.envless = envless  # a value without the env dim (a constant vector): broadcasting aligns it right

    def text(self, i: int) -> str:
        return f"%{i} = {self.op}({', '.join('%' + str(a) for a in self.args)}; {self.attr!r}) : {self.dtype}{list(self.shape)}{' weak' if self.weak else ''}"


class Program:
    """The IR of one term: nodes in evaluation order, the result node, the live parameter names."""

    def __init__(self, kind: str, nodes: list, out: int, params: list[str], param_types: list[str],
                 writes: list | None = None):
        self.kind, self.nodes, self.out = kind, nodes, out
        self.params, self.param_types = params, param_types
        self.writes = writes or []  # [(state slot, node)]: the env's row of the slot after the call
        self.first = None  # lazily initialised state: the program of the term's first evaluation
        self.bindings: dict = {}  # class-style terms: attribute -> (slot, row shape, dtype, lazy)

    def text(self) -> str:
        head = f"{self.kind} params={self.params} types={self.param_types} out=%{self.out}\n"
        text = head + "\n".join(n.text(i) for i, n in enumerate(self.nodes))
        if self.writes:
            text += "\nwrites " + ", ".join(f"state{slot}=%{i}" for slot, i in self.writes)
        if self.first is not None:
            text += "\nfirst call:\n" + self.first.text()
        return text

    def digest(self) -> int:
        """31-bit identity of the expression and of the code `function_body` emits for it (stored in the
        term's structural `i0` field)."""
        text = f"codegen {CODEGEN_REVISION}\n" + self.text()
        return int.from_bytes(hashlib.sha1(text.encode()).digest()[:4], "little") & 0x7FFFFFFF

    def sources(self) -> list[tuple]:
        return [n.attr for n in self.nodes if n.op == "src"]


# ------------------------------------------------------------------------------------------------
# symbolic values
# ------------------------------------------------------------------------------------------------
def _promote(a: "Sym", b: "Sym") -> str:
    """torch.result_type for two operands; `weak` operands are Python scalars (SURVEY appendix C)."""
    if a.weak == b.weak:
        return a.dtype_ if _RANK[a.dtype_] >= _RANK[b.dtype_] else b.dtype_
    strong, weak = (b, a) if a.weak else (a, b)
    return weak.dtype_ if _RANK[weak.dtype_] > _RANK[strong.dtype_] else strong.dtype_


def _bshape(a: "Sym", b: "Sym", what: str) -> tuple:
    if a.shape_ == b.shape_ or not b.shape_:
        return a.shape_
    if not a.shape_:
        return b.shape_
    return _broadcast([a, b], what)


def _broadcast(xs: list, what: str) -> tuple:
    """torch's broadcasting of the per-env shapes: per-env values of one rank, trailing dims aligned, size-1 dims
    expanded; a value without the env dim (a constant vector) aligns with the trailing per-env dims."""
    shapes = [x.shape_ for x in xs if x.shape_]
    ranks = {len(x.shape_) for x in xs if x.shape_ and not x._node.envless}
    rank = max(len(s) for s in shapes)
    out = []
    for d in range(1, rank + 1):
        sizes = {s[-d] for s in shapes if len(s) >= d} - {1}
        if len(sizes) > 1:
            break
        out.append(sizes.pop() if sizes else 1)
    if len(out) == rank and len(ranks) <= 1 and (not ranks or ranks == {rank}):
        return tuple(reversed(out))
    raise UnsupportedTermError(f"user term: '{what}' of shapes {' and '.join(f'(N, *{s})' for s in shapes)} does "
                               "not broadcast row by row")


def _bidx(out_shape: tuple, shape: tuple) -> list[int]:
    """Per element of `out_shape` (row-major), the flat index into a value of `shape` broadcast to it."""
    if shape == out_shape:
        return list(range(int(np.prod(out_shape)) if out_shape else 1))
    if not shape:
        return [0] * (int(np.prod(out_shape)) if out_shape else 1)
    st = _strides(shape)
    lead = len(out_shape) - len(shape)
    return [sum(combo[lead + d] * st[d] for d in range(len(shape)) if shape[d] != 1)
            for combo in np.ndindex(*out_shape)]


class Sym:
    """A (N, *shape) tensor of the trace.  `weak`: a Python scalar (live param or constant)."""

    __hash__ = object.__hash__

    def __init__(self, tr: "Tracer", nid: int):
        self._tr, self._id = tr, nid

    @property
    def _node(self) -> Node:
        return self._tr.nodes[self._id]

    shape_ = property(lambda self: self._node.shape)
    dtype_ = property(lambda self: self._node.dtype)

    @property
    def weak(self):
        return self._node.weak

    @property
    def dtype(self):
        return {F32: torch.float32, I32: torch.int32, BOOL: torch.bool}[self._node.dtype]

    @property
    def shape(self):
        if self.weak:
            return torch.Size(())
        return torch.Size((self._tr.N,) + self._node.shape)

    @property
    def device(self):
        return self._tr.device

    def size(self, dim=None):
        return self.shape if dim is None else self.shape[dim]

    def dim(self):
        return len(self.shape)

    ndim = property(dim)

    # -- refusals -------------------------------------------------------------------------------
    def _control(self, what):
        if self.weak:
            raise _ParamControlFlow(what)
        raise UnsupportedTermError(f"user term: {what} of a per-env value (data-dependent Python control flow)")

    def __bool__(self):
        self._control("__bool__")

    def __index__(self):
        self._control("__index__")

    def __int__(self):
        self._control("__int__")

    def __float__(self):
        self._control("__float__")

    def __len__(self):
        return self.shape[0] if self.shape else self._control("len()")

    def __iter__(self):
        raise UnsupportedTermError("user term: iteration over a per-env value")

    def __setitem__(self, key, value):
        if id(self) not in self._tr.state_objs:
            raise UnsupportedTermError("user term: in-place write (__setitem__)")
        keys = key if isinstance(key, tuple) else (key,)
        if not all(k == slice(None) or k is Ellipsis for k in keys) or len(keys) > len(self.shape):
            raise UnsupportedTermError(f"user term: partial in-place write of state ([{key!r}] = ...)")
        self._tr.state_write(self, value)

    def copy_(self, src, non_blocking=False):
        if id(self) not in self._tr.state_objs:
            raise UnsupportedTermError("user term: in-place op copy_")
        self._tr.state_write(self, src)
        return self

    def __getattr__(self, name):
        if name.startswith("__"):
            raise AttributeError(name)
        raise UnsupportedTermError(f"user term: tensor method '{name}' is not supported by the expression IR")

    def _inplace(self, *a, **k):
        raise UnsupportedTermError("user term: in-place arithmetic")

    __iadd__ = __isub__ = __imul__ = __itruediv__ = __iand__ = __ior__ = __imod__ = __ipow__ = _inplace

    # -- arithmetic ------------------------------------------------------------------------------
    def __add__(self, o): return self._tr.binary("add", self, o)
    def __radd__(self, o): return self._tr.binary("add", o, self)
    def __sub__(self, o): return self._tr.binary("sub", self, o)
    def __rsub__(self, o): return self._tr.binary("sub", o, self)
    def __mul__(self, o): return self._tr.binary("mul", self, o)
    def __rmul__(self, o): return self._tr.binary("mul", o, self)
    def __truediv__(self, o): return self._tr.binary("div", self, o)
    def __rtruediv__(self, o): return self._tr.binary("div", o, self)
    def __mod__(self, o): return self._tr.binary("mod", self, o)
    def __rmod__(self, o): return self._tr.binary("mod", o, self)
    def __lt__(self, o): return self._tr.binary("lt", self, o)
    def __le__(self, o): return self._tr.binary("le", self, o)
    def __gt__(self, o): return self._tr.binary("gt", self, o)
    def __ge__(self, o): return self._tr.binary("ge", self, o)
    def __eq__(self, o): return self._tr.binary("eq", self, o)
    def __ne__(self, o): return self._tr.binary("ne", self, o)
    def __and__(self, o): return self._tr.binary("and", self, o)
    def __rand__(self, o): return self._tr.binary("and", o, self)
    def __or__(self, o): return self._tr.binary("or", self, o)
    def __ror__(self, o): return self._tr.binary("or", o, self)
    def __neg__(self): return self._tr.unary("neg", self)
    def __invert__(self): return self._tr.unary("not", self)
    def __abs__(self): return self._tr.unary("abs", self)

    def __pow__(self, o):
        if isinstance(o, (int, float)) and not isinstance(o, bool) and o == 2:
            return self._tr.unary("square", self)
        raise UnsupportedTermError(f"user term: '** {o!r}' (only ** 2 is supported)")

    # -- methods ---------------------------------------------------------------------------------
    def abs(self): return self._tr.unary("abs", self)
    def square(self): return self._tr.unary("square", self)
    def sqrt(self): return self._tr.unary("sqrt", self)
    def exp(self): return self._tr.unary("exp", self)
    def log(self): return self._tr.unary("log", self)
    def sin(self): return self._tr.unary("sin", self)
    def cos(self): return self._tr.unary("cos", self)
    def tanh(self): return self._tr.unary("tanh", self)
    def logical_not(self): return self._tr.unary("not", self)
    def float(self): return self._tr.cast(self, F32)
    def int(self): return self._tr.cast(self, I32)
    def bool(self): return self._tr.cast(self, BOOL)
    def detach(self): return self
    def clone(self): return Sym(self._tr, self._id)  # a copy: it does not follow an in-place write of state
    def contiguous(self): return self

    def clamp(self, min=None, max=None): return self._tr.clamp(self, min, max)
    clip = clamp

    def sum(self, dim=None, keepdim=False): return self._tr.reduce("sum", self, dim, keepdim)
    def mean(self, dim=None, keepdim=False): return self._tr.reduce("mean", self, dim, keepdim)
    def any(self, dim=None, keepdim=False): return self._tr.reduce("any", self, dim, keepdim)
    def all(self, dim=None, keepdim=False): return self._tr.reduce("all", self, dim, keepdim)
    def amax(self, dim=None, keepdim=False): return self._tr.reduce("amax", self, dim, keepdim)
    def amin(self, dim=None, keepdim=False): return self._tr.reduce("amin", self, dim, keepdim)

    def norm(self, p=2, dim=None, keepdim=False):
        if p != 2:
            raise UnsupportedTermError(f"user term: norm(p={p!r}) (only the 2-norm is supported)")
        return self._tr.reduce("norm", self, dim, keepdim)

    def minimum(self, o): return self._tr.binary("minimum", self, o)
    def maximum(self, o): return self._tr.binary("maximum", self, o)

    def to(self, *args, **kwargs):
        dtype = kwargs.get("dtype") or next((a for a in args if isinstance(a, torch.dtype)), None)
        return self._cast_to(dtype) if dtype is not None else self

    def type(self, dtype):
        return self._cast_to(dtype)

    def _cast_to(self, dtype):
        if dtype is torch.int64 and self.dtype_ == F32:  # torch keeps |x| >= 2^31; the kernel's int is 32-bit
            raise UnsupportedTermError("user term: float -> int64 cast (int32 holds a different result)")
        return self._tr.cast(self, _dtype_of(dtype))

    def __getitem__(self, key):
        out = self._tr.index(self, key)
        if out is not self and id(self) in self._tr.state_objs:  # a view: it would follow an in-place write
            self._tr.viewed.add(self._tr.state_objs[id(self)][0])
        return out

    # -- layout (observation terms) --------------------------------------------------------------
    def unsqueeze(self, dim): return self._tr.unsqueeze(self, dim)
    def reshape(self, *shape): return self._tr.reshape(self, shape)
    view = reshape
    def flatten(self, start_dim=0, end_dim=-1): return self._tr.flatten(self, start_dim, end_dim)

    def nonzero(self, *a, **k):
        raise UnsupportedTermError("user term: nonzero() (data-dependent shape)")

    # -- torch functions -------------------------------------------------------------------------
    @classmethod
    def __torch_function__(cls, func, types, args=(), kwargs=None):
        kwargs = kwargs or {}
        operands = list(args) + list(kwargs.values())
        tr = next((a._tr for a in operands if isinstance(a, Sym)), None)
        if tr is None:  # the symbolic values sit inside a sequence argument (torch.stack, torch.cat, ...)
            name = getattr(func, "__name__", str(func))
            seq = [a for op in operands if isinstance(op, (list, tuple)) for a in op]
            tr = next((a._tr for a in seq if isinstance(a, Sym)), None)
            if tr is None or tr.kind != "observation" or name not in _LAYOUT_SEQ:
                raise UnsupportedTermError(f"user term: torch function '{name}' of a sequence of per-env values")
        return tr.torch_function(func, args, kwargs)


def _dtype_of(dtype) -> str:
    if dtype in (torch.float32, torch.float):
        return F32
    if dtype in (torch.int32, torch.int64, torch.int):
        return I32
    if dtype is torch.bool:
        return BOOL
    raise UnsupportedTermError(f"user term: dtype {dtype} (float32, int32/int64 and bool are supported)")


_UNARY_TORCH = {
    "abs": "abs", "square": "square", "sqrt": "sqrt", "exp": "exp", "log": "log", "sin": "sin", "cos": "cos",
    "tanh": "tanh", "neg": "neg", "negative": "neg", "logical_not": "not", "bitwise_not": "not",
}
_BINARY_TORCH = {
    "add": "add", "sub": "sub", "subtract": "sub", "mul": "mul", "multiply": "mul", "div": "div", "divide": "div",
    "true_divide": "div", "remainder": "mod", "lt": "lt", "less": "lt", "le": "le", "gt": "gt", "greater": "gt",
    "ge": "ge", "eq": "eq", "ne": "ne", "logical_and": "and", "logical_or": "or", "bitwise_and": "and",
    "bitwise_or": "or", "minimum": "minimum", "maximum": "maximum",
}
_REDUCE_TORCH = {"sum": "sum", "mean": "mean", "any": "any", "all": "all", "amax": "amax", "amin": "amin"}
_LAYOUT_SEQ = ("stack", "cat", "concat", "concatenate")  # over a sequence of values (observation terms only)


def _const_index(k):
    """An index list or integer tensor as a list of ints (a 0-d integer tensor: an int), anything else as is."""
    if isinstance(k, np.ndarray):
        k = torch.from_numpy(k)
    if torch.is_tensor(k):
        if k.dtype is torch.bool:
            raise UnsupportedTermError("user term: a bool mask index (data-dependent shape)")
        if k.is_floating_point() or k.is_complex() or k.dim() > 1:
            raise UnsupportedTermError(f"user term: a {k.dtype} index tensor of shape {tuple(k.shape)} (0-d or 1-D "
                                       "integer tensors only)")
        k = k.detach().cpu()
        if k.dim() == 0:
            return int(k.item())
        k = k.tolist()
    if isinstance(k, (list, tuple)):
        if any(isinstance(i, Sym) for i in k):
            next(i for i in k if isinstance(i, Sym))._control("index")
        if any(isinstance(i, (bool, np.bool_)) for i in k):
            raise UnsupportedTermError("user term: a bool mask index (data-dependent shape)")
        if not all(isinstance(i, (int, np.integer)) for i in k):
            raise UnsupportedTermError(f"user term: index list {k!r} (ints only)")
        if len(k) > MAX_CONST_VEC:
            raise UnsupportedTermError(f"user term: an index list of {len(k)} ids (at most {MAX_CONST_VEC})")
        return [int(i) for i in k]
    return k


# ------------------------------------------------------------------------------------------------
# tracer
# ------------------------------------------------------------------------------------------------
class Tracer:
    def __init__(self, N: int, kind: str, device=torch.device("cpu")):
        self.N, self.kind, self.device = N, kind, device
        self.nodes: list[Node] = []
        self._cse: dict = {}
        self.params: list[str] = []
        self.param_types: list[str] = []
        self.state_objs: dict = {}  # id(Sym) -> (slot, Sym): the instance's state tensors
        self.viewed: set = set()  # state slots a view was taken of

    def add(self, op, args, attr, shape, dtype, weak=False, envless=None) -> Sym:
        key = (op, tuple(args), repr(attr), tuple(shape), dtype, weak)
        nid = self._cse.get(key)
        if nid is None:
            if envless is None:  # (derived from constant vectors alone)
                strong = [self.nodes[i] for i in args if not self.nodes[i].weak]
                envless = bool(strong) and all(n.envless for n in strong)
            nid = len(self.nodes)
            self.nodes.append(Node(op, args, attr, shape, dtype, weak, envless))
            self._cse[key] = nid
        return Sym(self, nid)

    def source(self, key: tuple, shape: tuple, dtype: str) -> Sym:
        return self.add("src", (), key, shape, dtype)

    def state_write(self, sym: Sym, value):
        """`self.x[:] = value` / `self.x.copy_(value)`: the state Sym stands for the written value from now on."""
        slot, _ = self.state_objs[id(sym)]
        if slot in self.viewed:
            raise UnsupportedTermError("user term: in-place write of state a view was taken of")
        v = self.lift(value)
        if v.shape_ != sym.shape_ or (v.weak and sym.shape_):
            raise UnsupportedTermError(f"user term: in-place write of a {tuple(v.shape)} value into state of shape "
                                       f"{tuple(sym.shape)}")
        sym._id = self.cast(v, sym.dtype_)._id

    def full(self, like, value, dtype=None) -> Sym:
        """torch.zeros_like / ones_like / full_like of a per-env value."""
        like = self.lift(like)
        if like.weak:
            raise UnsupportedTermError("user term: *_like of a Python scalar")
        if isinstance(value, Sym) or not isinstance(value, (bool, int, float)):
            raise UnsupportedTermError("user term: full_like with a non-constant fill value")
        dt = _dtype_of(dtype) if dtype is not None else like.dtype_
        value = bool(value) if dt == BOOL else (int(value) if dt == I32 else _f32(value))
        return self.add("full", (), value, like.shape_, dt)

    def param(self, name: str, value) -> Sym:
        dtype = I32 if isinstance(value, int) else F32
        if len(self.params) >= MAX_LIVE_PARAMS:
            raise UnsupportedTermError(f"user term: more than {MAX_LIVE_PARAMS} scalar params")
        self.params.append(name)
        self.param_types.append(dtype)
        return self.add("param", (), len(self.params) - 1, (), dtype, weak=True)

    # -- operands ----------------------------------------------------------------------------------
    def lift(self, x) -> Sym:
        if isinstance(x, Sym):
            return x
        if isinstance(x, bool):
            return self.add("const", (), bool(x), (), BOOL, weak=True)
        if isinstance(x, int):
            if not -(1 << 31) <= x < (1 << 31):
                raise UnsupportedTermError(f"user term: integer constant {x} does not fit int32")
            return self.add("const", (), int(x), (), I32, weak=True)
        if isinstance(x, float):
            return self.add("const", (), float(x), (), F32, weak=True)
        if isinstance(x, np.generic):
            return self.lift(x.item())
        if torch.is_tensor(x):
            t = x.detach().cpu()
            if t.dim() == 0:
                v = t.item()
                dtype = _dtype_of(t.dtype)
                value = bool(v) if dtype == BOOL else (int(v) if dtype == I32 else _f32(v))
                return self.add("const", (), value, (), dtype, weak=True)
            if t.dim() == 1 and t.shape[0] <= MAX_CONST_VEC and t.shape[0] != self.N:
                dtype = _dtype_of(t.dtype)
                vals = tuple(bool(v) if dtype == BOOL else (int(v) if dtype == I32 else _f32(v)) for v in t.tolist())
                return self.add("constvec", (), vals, (t.shape[0],), dtype, envless=True)
            raise UnsupportedTermError(
                f"user term: a concrete tensor of shape {tuple(t.shape)} enters the expression (per-env state the "
                "kernel does not hold: a captured buffer, a further entity, a user-level manager's state)")
        raise UnsupportedTermError(f"user term: operand of type {type(x).__name__}")

    # -- ops ---------------------------------------------------------------------------------------
    def unary(self, op: str, a) -> Sym:
        a = self.lift(a)
        dt = a.dtype_
        if op == "not":
            if dt != BOOL:
                raise UnsupportedTermError("user term: '~' on a non-bool value (bitwise not of integers)")
            out = BOOL
        elif op in ("neg", "abs", "square"):
            if dt == BOOL:
                raise UnsupportedTermError(f"user term: '{op}' of a bool value")
            out = dt
        else:  # transcendental / sqrt: integer inputs become float32
            out = F32
        if a.weak and op != "neg":
            raise _ParamControlFlow(op)  # math on a Python scalar: evaluated in double by the function itself
        x = a if out == dt or op in ("neg", "abs", "square", "not") else self.cast(a, F32)
        return self.add(op, (x._id,), None, a.shape_, out, weak=a.weak)

    def cast(self, a, dtype: str) -> Sym:
        a = self.lift(a)
        if a.dtype_ == dtype:
            return a
        return self.add("cast", (a._id,), dtype, a.shape_, dtype, weak=a.weak)

    def binary(self, op: str, a, b) -> Sym:
        a, b = self.lift(a), self.lift(b)
        if a.weak and b.weak:
            raise _ParamControlFlow(op)  # Python scalars combine in double precision
        shape = _bshape(a, b, op)
        dt = _promote(a, b)
        if op in ("and", "or"):
            if a.dtype_ != BOOL or b.dtype_ != BOOL:
                raise UnsupportedTermError(f"user term: '{op}' of non-bool values (bitwise integer ops)")
            return self.add(op, (a._id, b._id), None, shape, BOOL)
        if op == "div":
            dt = F32  # true division
        if op == "mod" and dt != I32:
            raise UnsupportedTermError("user term: '%' is supported for integers only")
        if op == "mod" and b._node.op == "const" and b._node.attr == 0:
            raise UnsupportedTermError("user term: '%' by the constant 0 (torch raises ZeroDivisionError)")
        if op in ("add", "sub", "mul", "minimum", "maximum") and dt == BOOL:
            raise UnsupportedTermError(f"user term: '{op}' of two bool values")
        ca, cb = self.cast(a, dt), self.cast(b, dt)
        if op in ("lt", "le", "gt", "ge", "eq", "ne"):
            return self.add(op, (ca._id, cb._id), None, shape, BOOL)
        return self.add(op, (ca._id, cb._id), None, shape, dt)

    def nan_dropping(self, op: str, a, b) -> Sym:
        """fmaxf / fminf ("fmax" / "fmin") of fp32 values: a NaN operand gives the other one.  Internal: the
        restated stock terms use them where their kernel case does."""
        a, b = self.cast(self.lift(a), F32), self.cast(self.lift(b), F32)
        return self.add(op, (a._id, b._id), None, _bshape(a, b, op), F32)

    def where(self, c, a, b) -> Sym:
        c, a, b = self.lift(c), self.lift(a), self.lift(b)
        if c.dtype_ != BOOL:
            raise UnsupportedTermError("user term: where() with a non-bool condition")
        if a.weak and b.weak:
            dt = a.dtype_ if _RANK[a.dtype_] >= _RANK[b.dtype_] else b.dtype_
        else:
            dt = _promote(a, b)
        shapes = {s for s in (c.shape_, a.shape_, b.shape_) if s}
        shape = (shapes.pop() if len(shapes) == 1 else _broadcast([c, a, b], "where")) if shapes else ()
        if c.weak:
            raise UnsupportedTermError("user term: where() with a scalar condition")
        return self.add("where", (c._id, self.cast(a, dt)._id, self.cast(b, dt)._id), None, shape, dt)

    def clamp(self, x, lo, hi) -> Sym:
        x = self.lift(x)
        if lo is None and hi is None:
            raise UnsupportedTermError("user term: clamp() without bounds")
        if x.dtype_ == BOOL:
            raise UnsupportedTermError("user term: clamp() of a bool value")
        out = x
        # torch.clamp(x, lo, hi) == min(max(x, lo), hi): x kept on a tie, NaN in x propagating.  A NaN bound
        # propagates, except that torch-CPU ignores it when it is the only bound and a Python scalar (a live
        # param is one): attr "scalar"
        for op, bound in (("clamp_lo", lo), ("clamp_hi", hi)):
            if bound is None:
                continue
            scalar = (lo is None or hi is None) and (isinstance(bound, (int, float, np.generic))
                                                     or (isinstance(bound, Sym) and bound._node.op == "param"))
            bound = self.lift(bound)
            dt = _promote(out, bound)
            out = self.add(op, (self.cast(out, dt)._id, self.cast(bound, dt)._id), "scalar" if scalar else None,
                           _bshape(out, bound, "clamp"), dt)
        return out

    def reduce(self, kind: str, x, dim, keepdim=False) -> Sym:
        x = self.lift(x)
        if keepdim:
            raise UnsupportedTermError(f"user term: {kind}(keepdim=True)")
        if isinstance(dim, (tuple, list)):
            if len(dim) != 1:
                raise UnsupportedTermError(f"user term: {kind} over several dims")
            dim = dim[0]
        rank = len(x.shape_) + 1
        if dim is None or rank == 1:
            raise UnsupportedTermError(f"user term: {kind} over the env dimension")
        if isinstance(dim, Sym):
            dim._control("dim")
        d = dim + rank if dim < 0 else dim
        if not 1 <= d < rank:
            raise UnsupportedTermError(f"user term: {kind}(dim={dim}) of a rank-{rank} value")
        axis = d - 1  # in the per-env shape
        shape = x.shape_[:axis] + x.shape_[axis + 1:]
        dt = x.dtype_
        if kind in ("any", "all"):
            src = self.cast(x, BOOL) if dt != BOOL else x
            return self.add(kind, (src._id,), axis, shape, BOOL)
        if kind == "sum":
            out = I32 if dt in (BOOL, I32) else F32
            return self.add("sum", (self.cast(x, out)._id,), axis, shape, out)
        if kind in ("mean", "norm"):
            if dt != F32:
                raise UnsupportedTermError(f"user term: {kind} of a non-float value")
            return self.add(kind, (x._id,), axis, shape, F32)
        if dt == BOOL:
            raise UnsupportedTermError(f"user term: {kind} of a bool value")
        return self.add(kind, (x._id,), axis, shape, dt)

    # -- layout ops: observation terms build their rows with them ------------------------------------
    def _layout(self, what: str):
        if self.kind != "observation":
            raise UnsupportedTermError(f"user term: {what} (layout ops are lowered in observation terms only)")

    def _as_row(self, shape: tuple, x: Sym) -> Sym:
        """x with the per-env shape `shape` (same elements, row-major)."""
        if tuple(shape) == x.shape_:
            return x
        return self.add("reshape", (x._id,), None, tuple(shape), x.dtype_)

    def _dim(self, dim, rank: int, what: str, extra: int = 0) -> int:
        """A dim argument over the full (N, ...) rank as a per-env axis; the env axis is refused."""
        if isinstance(dim, Sym):
            dim._control("dim")
        if not isinstance(dim, int) or isinstance(dim, bool):
            raise UnsupportedTermError(f"user term: {what}(dim={dim!r})")
        d = dim + rank + extra if dim < 0 else dim
        if not 1 <= d < rank + extra:
            raise UnsupportedTermError(f"user term: {what}(dim={dim}) of a rank-{rank} value (the env dimension "
                                       "stays first)")
        return d - 1

    def unsqueeze(self, x, dim) -> Sym:
        self._layout("unsqueeze")
        x = self.lift(x)
        axis = self._dim(dim, len(x.shape_) + 1, "unsqueeze", extra=1)
        return self._as_row(x.shape_[:axis] + (1,) + x.shape_[axis:], x)

    def reshape(self, x, shape) -> Sym:
        self._layout("reshape / view")
        x = self.lift(x)
        if len(shape) == 1 and isinstance(shape[0], (tuple, list, torch.Size)):
            shape = tuple(shape[0])
        if any(isinstance(v, Sym) for v in shape):
            next(v for v in shape if isinstance(v, Sym))._control("reshape")
        size = int(np.prod(x.shape_)) if x.shape_ else 1
        total = self.N * size
        shape = [int(v) for v in shape]
        if shape.count(-1) > 1:
            raise UnsupportedTermError("user term: reshape with more than one -1")
        known = int(np.prod([v for v in shape if v != -1])) if shape else 1
        if -1 in shape:
            if known == 0 or total % known:
                raise UnsupportedTermError(f"user term: reshape to {tuple(shape)}")
            shape[shape.index(-1)] = total // known
        if not shape or shape[0] != self.N or int(np.prod(shape)) != total:
            raise UnsupportedTermError(f"user term: reshape to {tuple(shape)} (rows of the {self.N} envs only)")
        return self._as_row(tuple(shape[1:]), x)

    def flatten(self, x, start_dim=0, end_dim=-1) -> Sym:
        self._layout("flatten")
        x = self.lift(x)
        rank = len(x.shape_) + 1
        s = start_dim + rank if start_dim < 0 else start_dim
        t = end_dim + rank if end_dim < 0 else end_dim
        if s < 1 or t < s or t >= rank:
            if rank == 1 and s == 1:
                return x
            raise UnsupportedTermError(f"user term: flatten({start_dim}, {end_dim}) (rows of the envs only)")
        a, b = s - 1, t - 1
        return self._as_row(x.shape_[:a] + (int(np.prod(x.shape_[a:b + 1])),) + x.shape_[b + 1:], x)

    def stack_cat(self, name: str, seq, dim) -> Sym:
        self._layout(f"torch.{name}")
        if not isinstance(seq, (list, tuple)) or not seq:
            raise UnsupportedTermError(f"user term: torch.{name} of {type(seq).__name__}")
        xs = [self.lift(v) for v in seq]
        if any(v.weak for v in xs):
            raise UnsupportedTermError(f"user term: torch.{name} of a Python scalar")
        dt = max((v.dtype_ for v in xs), key=_RANK.get)  # torch.result_type of tensors alone
        xs = [self.cast(v, dt) for v in xs]
        if name == "stack":
            shape = xs[0].shape_
            if any(v.shape_ != shape for v in xs):
                raise UnsupportedTermError("user term: torch.stack of values with different shapes")
            axis = self._dim(dim, len(shape) + 1, "stack", extra=1)
            if axis != len(shape):
                raise UnsupportedTermError(f"user term: torch.stack(dim={dim}) (over the last dimension only)")
            return self.add("stack", tuple(v._id for v in xs), None, shape + (len(xs),), dt)
        rank = len(xs[0].shape_) + 1
        if rank == 1:
            raise UnsupportedTermError(f"user term: torch.{name} of (N,) values (it joins envs)")
        axis = self._dim(dim, rank, name)
        if axis != rank - 2 or any(len(v.shape_) != rank - 1 or v.shape_[:-1] != xs[0].shape_[:-1] for v in xs):
            raise UnsupportedTermError(f"user term: torch.{name}(dim={dim}) (over the last dimension only)")
        shape = xs[0].shape_[:-1] + (sum(v.shape_[-1] for v in xs),)
        return self.add("cat", tuple(v._id for v in xs), None, shape, dt)

    def index(self, x: Sym, key) -> Sym:
        if not isinstance(key, tuple):
            key = (key,)
        if any(k is None for k in key[1:]):  # None inserts a size-1 axis: the indexed value, reshaped
            self._layout("None in an index")
            kept = tuple(k for k in key if k is not None)
            out = self.index(x, kept)
            rest = list(key[1:])
            if key[0] is Ellipsis:
                n_tail = sum(1 for k in rest if k is not None)
                rest = [slice(None)] * (len(x.shape_) - n_tail) + rest
            shape, src = [], list(out.shape_)
            for k in rest:
                if k is None:
                    shape.append(1)
                elif isinstance(k, slice) or isinstance(_const_index(k), list):
                    shape.append(src.pop(0))
            shape += src
            return self._as_row(tuple(shape), out)
        return self._index(x, key)

    def _index(self, x: Sym, key: tuple) -> Sym:
        shape = x.shape_
        if not key or not (key[0] == slice(None) or key[0] is Ellipsis):
            raise UnsupportedTermError("user term: indexing that selects envs (only [:, ...] / [..., j] keep every env)")
        rest = list(key[1:]) if key[0] == slice(None) else None
        if key[0] is Ellipsis:  # [..., j]: the trailing dims
            tail = list(key[1:])
            if any(k is Ellipsis for k in tail) or len(tail) > len(shape):
                raise UnsupportedTermError("user term: unsupported index")
            rest = [slice(None)] * (len(shape) - len(tail)) + tail
        if len(rest) > len(shape):
            raise UnsupportedTermError("user term: too many indices")
        rest += [slice(None)] * (len(shape) - len(rest))
        spec, out_shape = [], []
        rest = [_const_index(k) for k in rest]
        if sum(isinstance(k, list) for k in rest) > 1:
            raise UnsupportedTermError("user term: two advanced (list / tensor) indices in one indexing expression")
        for k, n in zip(rest, shape):
            if isinstance(k, Sym):
                k._control("index")
            if isinstance(k, list):  # a constant index list: a gather along the axis, order and duplicates kept
                if any(not -n <= i < n for i in k):
                    raise UnsupportedTermError(f"user term: index list {k} out of range for size {n}")
                spec.append(("list",) + tuple(i % n for i in k))
                out_shape.append(len(k))
                continue
            if isinstance(k, bool) or not isinstance(k, (int, slice)):
                raise UnsupportedTermError(f"user term: index {k!r} (ints, basic slices and constant index lists only)")
            if isinstance(k, int):
                if not -n <= k < n:
                    raise UnsupportedTermError(f"user term: index {k} out of range for size {n}")
                spec.append(k % n)
            else:
                start, stop, step = k.indices(n)
                if step != 1:
                    raise UnsupportedTermError("user term: strided slice")
                spec.append((start, max(start, stop)))
                out_shape.append(max(0, stop - start))
        if all(isinstance(s, tuple) and s == (0, n) for s, n in zip(spec, shape)):
            return x
        return self.add("index", (x._id,), tuple(spec), tuple(out_shape), x.dtype_)

    def torch_function(self, func, args, kwargs):
        name = getattr(func, "__name__", str(func))
        if name in ("__get__",) or name.endswith("__setitem__"):
            raise UnsupportedTermError("user term: in-place write")
        name = name.strip("_") if name.startswith("__") else name
        name = {"radd": "add", "rmul": "mul"}.get(name, name)
        if name.endswith("_") and not name.startswith("_"):
            raise UnsupportedTermError(f"user term: in-place op {name}")
        if name in ("rsub", "rtruediv", "rmod"):
            return self.binary(name[1:].replace("truediv", "div"), args[1], args[0])
        if name in ("truediv",):
            name = "div"
        if name in _UNARY_TORCH and len(args) == 1:
            return self.unary(_UNARY_TORCH[name], args[0])
        if name in _BINARY_TORCH:
            other = args[1] if len(args) > 1 else kwargs.get("other")
            return self.binary(_BINARY_TORCH[name], args[0], other)
        if name in ("where",):
            return self.where(*args[:3])
        if name in ("clamp", "clip"):
            lo = args[1] if len(args) > 1 else kwargs.get("min")
            hi = args[2] if len(args) > 2 else kwargs.get("max")
            return self.clamp(args[0], lo, hi)
        if name in _REDUCE_TORCH:
            dim = args[1] if len(args) > 1 else kwargs.get("dim")
            return self.reduce(_REDUCE_TORCH[name], args[0], dim, kwargs.get("keepdim", False))
        if name in ("norm", "vector_norm"):
            p = kwargs.get("p", kwargs.get("ord", args[1] if len(args) > 1 and name == "norm" else 2))
            if p not in (2, 2.0, None, "fro"):
                raise UnsupportedTermError(f"user term: norm(p={p!r})")
            dim = kwargs.get("dim", args[2] if len(args) > 2 else None)
            return self.reduce("norm", args[0], dim, kwargs.get("keepdim", False))
        if name in _LAYOUT_SEQ:
            seq = args[0] if args else kwargs.get("tensors")
            dim = args[1] if len(args) > 1 else kwargs.get("dim", 0)
            return self.stack_cat("stack" if name == "stack" else "cat", seq, dim)
        if name == "unsqueeze":
            return self.unsqueeze(args[0], args[1] if len(args) > 1 else kwargs.get("dim"))
        if name in ("reshape", "view"):
            return self.reshape(args[0], tuple(args[1:]) if len(args) > 1 else (kwargs.get("shape"),))
        if name == "flatten":
            return self.flatten(args[0], args[1] if len(args) > 1 else kwargs.get("start_dim", 0),
                                args[2] if len(args) > 2 else kwargs.get("end_dim", -1))
        if name == "pow":
            return self.lift(args[0]).__pow__(args[1])
        if name in ("float",):
            return self.cast(args[0], F32)
        if name == "getitem":
            return self.index(self.lift(args[0]), args[1])
        if name == "nonzero":
            raise UnsupportedTermError("user term: nonzero() (data-dependent shape)")
        if name in ("zeros_like", "ones_like", "full_like"):
            value = {"zeros_like": 0, "ones_like": 1}.get(name)
            if value is None:
                value = args[1] if len(args) > 1 else kwargs.get("fill_value")
            return self.full(args[0], value, kwargs.get("dtype"))
        if name == "clone":
            return self.lift(args[0]).clone()
        raise UnsupportedTermError(f"user term: torch function '{name}' is not supported by the expression IR")


# ------------------------------------------------------------------------------------------------
# trace: sources swapped in for the duration of one call
# ------------------------------------------------------------------------------------------------
class _EntityProxy:
    """Stands for the primary entity while a term is traced."""

    def __init__(self, tr: Tracer, dofs_idx, n_dofs: int, robot=None):
        self._tr, self._dofs_idx, self._D, self._robot = tr, dofs_idx, n_dofs, robot

    # -- links: the real link objects (their get_pos / get_vel are swapped for the trace) --------------
    @property
    def links(self):
        return self._robot_or_refuse("links").links

    def get_link(self, name=None, *args, **kwargs):
        return self._robot_or_refuse("get_link").get_link(name, *args, **kwargs)

    def get_links_pos(self, links_idx_local=None, envs_idx=None):
        return self._links("pos", links_idx_local, envs_idx)

    def get_links_vel(self, links_idx_local=None, envs_idx=None):
        return self._links("vel", links_idx_local, envs_idx)

    def _robot_or_refuse(self, what):
        if self._robot is None:
            raise UnsupportedTermError(f"user term: robot.{what} without a primary entity")
        return self._robot

    def _links(self, what, links_idx_local, envs_idx):
        if envs_idx is not None:
            raise UnsupportedTermError(f"user term: robot.get_links_{what}(envs_idx=...)")
        if links_idx_local is None:
            raise UnsupportedTermError(f"user term: robot.get_links_{what}() without links_idx_local (every link of "
                                       "the entity; name the links the term reads)")
        if isinstance(links_idx_local, range):
            links_idx_local = list(links_idx_local)
        ids = _const_index(links_idx_local)
        if not isinstance(ids, list):
            raise UnsupportedTermError(f"user term: robot.get_links_{what}(links_idx_local={links_idx_local!r}) (a "
                                       "list, tuple, range or 1-D integer tensor of local link ids)")
        n = len(self._robot_or_refuse(f"get_links_{what}").links)
        if not ids or any(not 0 <= i < n for i in ids):
            raise UnsupportedTermError(f"user term: robot.get_links_{what}: local link ids {ids} (the entity has {n})")
        if len(set(ids)) > MAX_LINKS:
            raise UnsupportedTermError(f"user term: robot.get_links_{what} of {len(set(ids))} links (at most "
                                       f"{MAX_LINKS})")
        return self._tr.source((f"link_{what}", tuple(ids)), (len(ids), 3), F32)

    def get_pos(self, envs_idx=None):
        return self._plain("pos", 3, envs_idx)

    def get_quat(self, envs_idx=None):
        return self._plain("quat", 4, envs_idx)

    def get_vel(self, envs_idx=None):
        return self._plain("vel", 3, envs_idx)

    def get_ang(self, envs_idx=None):
        return self._plain("ang", 3, envs_idx)

    def _plain(self, key, width, envs_idx):
        if envs_idx is not None:
            raise UnsupportedTermError(f"user term: robot.get_{key}(envs_idx=...)")
        return self._tr.source((key,), (width,), F32)

    def _dofs(self, key, dofs_idx, envs_idx):
        same = dofs_idx is not None and self._dofs_idx is not None and list(dofs_idx) == list(self._dofs_idx)
        if envs_idx is not None or not same or self._D == 0:
            raise UnsupportedTermError(f"user term: robot.get_dofs_{key}() of DOFs other than the action manager's")
        return self._tr.source((f"dof_{key}",), (self._D,), F32)

    def get_dofs_position(self, dofs_idx=None, envs_idx=None):
        return self._dofs("pos", dofs_idx, envs_idx)

    def get_dofs_velocity(self, dofs_idx=None, envs_idx=None):
        return self._dofs("vel", dofs_idx, envs_idx)

    def __getattr__(self, name):
        raise UnsupportedTermError(f"user term: robot.{name} is not a source of the expression IR")


class _AirProxy:
    def __init__(self, tr: Tracer, m: int, n_links: int):
        self._tr, self._m, self._L = tr, m, n_links

    def __getitem__(self, j):
        if not isinstance(j, int) or not 0 <= j < 4:
            raise UnsupportedTermError("user term: air-time state indexing")
        return self._tr.source(("air", self._m, j), (self._L,), F32)


class _Swap:
    """Set attributes for the duration of a trace and put the originals back afterwards."""

    def __init__(self):
        self.saved: list = []

    def set(self, obj, name, value):
        self.saved.append((obj, name, obj.__dict__.get(name, _MISSING)))
        setattr(obj, name, value)

    def set_item(self, d: dict, key, value):
        self.saved.append((d, key, d.get(key, _MISSING)))
        d[key] = value

    def restore(self):
        for obj, name, old in reversed(self.saved):
            if isinstance(obj, dict):
                if old is _MISSING:
                    obj.pop(name, None)
                else:
                    obj[name] = old
            elif old is _MISSING:
                obj.__dict__.pop(name, None)
            else:
                setattr(obj, name, old)
        self.saved = []


_MISSING = object()


class ExprMode:
    """env._tracing while a user term is traced: the manager getters' `_trace_or` lands here."""

    def __init__(self, tr: Tracer, fused):
        self.tr, self.fused = tr, fused

    def source(self, key, compute):
        tr, D = self.tr, self.fused.D
        if key in ("lin_vel_b", "ang_vel_b", "gravity_b"):
            return tr.source((key,), (3,), F32)
        if key in ("dof_pos", "dof_vel", "targets") and D > 0:
            return tr.source((key,), (D,), F32)
        if key == "env_actions" and D > 0:
            return tr.source(("actions",), (D,), F32)
        if isinstance(key, tuple) and key[0] == "command":
            return key[1].command
        # body-frame vectors the kernel does not hold: a further EntityManager's (its own cached quaternion) and
        # those of a term without an entity_manager (the current quaternion); refused without evaluating them
        if isinstance(key, tuple) and isinstance(key[0], str) and key[0].startswith("entity_"):
            raise UnsupportedTermError("user term: a body-frame getter of a further EntityManager (the kernel "
                                       "holds the first manager's pose)")
        if isinstance(key, str) and key.endswith("_uncached"):
            raise UnsupportedTermError("user term: a body-frame term without an entity_manager")
        return compute()

    def stock_call(self, kind: str, fn, params: dict) -> Sym:
        """A stock reward / termination descriptor called inside the traced term (ManagedEnvironment.fuse_stock_calls):
        the unweighted term as IR, `params` normalised as FusedStep.pack normalises a table row."""
        name = getattr(fn, "__name__", type(fn).__name__)
        what = f"user term: stock term {name}"
        if self.tr.kind == "observation":
            raise UnsupportedTermError(f"{what} inside an observation term (stock calls are inlined in rewards and "
                                       "terminations only)")
        restate = _STOCK.get((kind, fn.gfb_opcode))
        if restate is None:
            raise UnsupportedTermError(f"{what}: keeps per-term state in the kernel and is not inlined")
        return restate(_Stock(self, what), params)


class _Stock:
    """What the restatement of one stock term reads: its sources, its managers (checked as FusedStep.pack checks
    a table row's) and the row's fp32 constants."""

    def __init__(self, mode: ExprMode, what: str):
        self.tr, self.fused, self.what = mode.tr, mode.fused, what

    def refuse(self, why: str):
        raise UnsupportedTermError(f"{self.what}: {why}")

    def src(self, key: tuple, shape: tuple = (), dtype: str = F32) -> Sym:
        return self.tr.source(key, shape, dtype)

    def entity(self, p: dict):
        """FusedStep._entity_ok, with the trace's stand-in for the primary entity."""
        fused, em = self.fused, p.get("entity_manager")
        if em is not None:
            if em is not fused.entity_manager:
                self.refuse("the entity_manager is a further EntityManager (the kernel holds the first one's pose)")
            return
        attr = p.get("entity_attr", "robot")
        if not isinstance(getattr(fused.env, attr, None), _EntityProxy):
            self.refuse(f"entity_attr '{attr}' is not the fused step's entity")

    def command(self, mgr) -> Sym:
        fused = self.fused
        k = next((k for k, m in enumerate(fused.commands) if m is mgr), None)
        if k is None:
            self.refuse("its command manager is not registered with this environment")
        if mgr in fused.python_commands or mgr._external_controller is not None:
            self.refuse("its command manager is a user-level or externally controlled one")
        return self.src(("command", k), (int(mgr._command.shape[1]),))

    def contact_norm(self, mgr) -> tuple[int, Sym]:
        """(index, (N, L) force norms of the tracked links): the kernel's st_cnorm."""
        m = next((m for m, c in enumerate(self.fused.contacts) if c is mgr), None)
        if m is None:
            self.refuse("its contact manager is not registered with this environment")
        return m, self.src(("contacts", m), (int(mgr._link_ids.shape[0]), 3)).norm(dim=-1)

    def scalar(self, v, what: str) -> Sym:
        """A row's fp32 p[k]: a live param of the user term stays live, a Python or one-element value is a constant."""
        if isinstance(v, Sym):
            if not v.weak:
                self.refuse(f"a per-env {what}")
            return v
        if torch.is_tensor(v) or isinstance(v, np.ndarray):
            t = torch.as_tensor(v)
            if t.numel() != 1:
                self.refuse(f"a {what} tensor of shape {tuple(t.shape)} (a per-env value the kernel does not hold)")
            v = t.item()
        if isinstance(v, bool) or not isinstance(v, (int, float, np.generic)):
            self.refuse(f"{what} {v!r}")
        return self.tr.lift(_f32(v))

    def dof_deviation(self) -> Sym:
        """sum_d |q_d - default_d| (P.default_dof_pos folded in as a constant vector)."""
        fused = self.fused
        if fused.D == 0:
            self.refuse("no action manager")
        default = tuple(_f32(x) for x in fused.action.kernel_params()["default"].detach().cpu().tolist())
        q = self.src(("dof_pos",), (fused.D,))
        return (q - self.tr.add("constvec", (), default, (fused.D,), F32, envless=True)).abs().sum(dim=1)

    def episode_length(self) -> Sym:
        return self.src(("episode_length",), (), I32)

    def terminated(self) -> Sym:
        if self.tr.kind != "reward":
            self.refuse("reads extras['terminations'], which a termination term does not see")
        return self.src(("terminated",), (), BOOL)


# The stock terms as IR, op for op as their cases in post_kernel.cuh (same operands, same order, the same
# fp32 helpers), so an inlined call has the bits of the stock row evaluated in the same launch.
def _r_base_height(s: _Stock, p):
    s.entity(p)
    off = 0.0
    tm = p["terrain_manager"]
    if tm is not None:
        if tm.height_field is not None:
            s.refuse("a height-field terrain")
        off = float(tm._origin[2])
    if p["height_command"] is not None:
        target = s.command(p["height_command"])[:, 0]
    else:
        target = s.scalar(p["target_height"], "target_height")
    z = s.src(("pos",), (3,))[:, 2]
    return ((z - off) - target).square()


def _r_action_rate(s: _Stock, p):
    # the sum the action kernel wrote for this step (GFB_B_ACTION_RATE): the stock row's value by construction
    if s.tr.kind != "reward":
        s.refuse("reads the action-rate sum, which only the reward phase reads")
    return s.src(("action_rate",))


def _r_stand_still(s: _Stock, p):
    if p["vel_cmd_manager"] is None:
        s.refuse("no vel_cmd_manager")
    c = s.command(p["vel_cmd_manager"])
    return s.dof_deviation() * (c[:, :2].norm(dim=1) < s.scalar(p["command_threshold"], "command_threshold")).float()


def _r_body_sq(key: str, dims: tuple):
    def restate(s: _Stock, p):
        s.entity(p)
        v = s.src((key,), (3,))
        out = v[:, dims[0]].square()
        return out + v[:, dims[1]].square() if len(dims) > 1 else out
    return restate


def _fixed_command(s: _Stock, value, lin: bool) -> list:
    """A command tensor of at most MAX_CONST_VEC elements that is the same for every env: its x, y (lin) or its
    yaw rate, folded in as constants."""
    if isinstance(value, Sym):
        s.refuse("a per-env command")
    t = torch.as_tensor(value, dtype=torch.float32).detach().cpu()
    if t.numel() > MAX_CONST_VEC:
        s.refuse(f"a command tensor of shape {tuple(t.shape)} (a per-env command the kernel does not hold)")
    try:
        t = torch.broadcast_to(t, (1, 2) if lin else (1,)).reshape(-1)
    except RuntimeError:
        s.refuse(f"a command tensor of shape {tuple(t.shape)}")
    return [s.tr.lift(_f32(x)) for x in t.tolist()]


def _r_track(lin: bool):
    def restate(s: _Stock, p):
        s.entity(p)
        if p["vel_cmd_manager"] is not None:
            c = s.command(p["vel_cmd_manager"])
            cmd = [c[:, 0], c[:, 1]] if lin else [c[:, 2]]
        else:
            cmd = _fixed_command(s, p["command"] if lin else p["commanded_ang_vel"], lin)
        if lin:
            v = s.src(("lin_vel_b",), (3,))
            err = (cmd[0] - v[:, 0]).square() + (cmd[1] - v[:, 1]).square()
        else:
            err = (cmd[0] - s.src(("ang_vel_b",), (3,))[:, 2]).square()
        return (-err / s.scalar(p["sensitivity"], "sensitivity")).exp()
    return restate


def _r_feet_air_time(s: _Stock, p):
    mgr = p["contact_manager"]
    m, _ = s.contact_norm(mgr)
    if not mgr._track_air_time:
        s.refuse("its contact manager does not track air time")
    L = int(mgr._link_ids.shape[0])
    last_air, cur_contact = s.src(("air", m, 0), (L,)), s.src(("air", m, 3), (L,))
    made = (cur_contact > 0.0) & (cur_contact < _f32(s.fused.env.dt + 1.0e-8))  # has_made_contact(env.dt)
    a = (last_air - s.scalar(p["time_threshold"], "time_threshold")) * made.float()
    if p["time_threshold_max"] is not None:
        span = p["time_threshold_max"] - p["time_threshold"]  # (a live param here is traced as a constant)
        a = s.tr.nan_dropping("fmin", a, s.scalar(span, "time_threshold_max"))
    v = a.sum(dim=1)
    if p["vel_cmd_manager"] is not None:
        c = s.command(p["vel_cmd_manager"])
        v = v * (c[:, :2].norm(dim=1) > 0.1).float()
    return v


def _r_feet_slide(s: _Stock, p):
    mgr = p["contact_manager"]
    _, cn = s.contact_norm(mgr)
    s.entity({"entity_attr": p["entity_attr"]})
    ids = [int(i) for i in mgr.local_link_ids.tolist()]
    speed = _EntityProxy(s.tr, None, 0, s.fused.primary_entity).get_links_vel(links_idx_local=ids).norm(dim=-1)
    return (speed * (cn > 1.0).float()).sum(dim=1)


def _t_bad_orientation(s: _Stock, p):
    s.entity(p)
    threshold = s.fused._tilt_threshold(p["limit_angle"])  # (a live limit_angle: traced as a constant)
    g = s.src(("gravity_b",), (3,))
    tilt = g[:, :2].norm(dim=1)
    after_grace = ~(s.episode_length() <= int(p["grace_steps"]))
    return after_grace & (tilt == tilt) & (s.tr.nan_dropping("fmin", tilt, 0.99) >= s.scalar(threshold, "limit_angle"))


def _t_base_height_min(s: _Stock, p):
    s.entity(p)
    return s.src(("pos",), (3,))[:, 2] < s.scalar(p["minimum_height"], "minimum_height")


def _t_out_of_bounds(s: _Stock, p):
    s.entity(p)
    if p["terrain_manager"] is None:
        s.refuse("no terrain_manager")
    x_min, x_max, y_min, y_max = p["terrain_manager"].get_bounds(p["subterrain"])
    margin = p["border_margin"]
    lo_x, hi_x = s.scalar(x_min + margin, "bound"), s.scalar(x_max - margin, "bound")
    lo_y, hi_y = s.scalar(y_min + margin, "bound"), s.scalar(y_max - margin, "bound")
    pos = s.src(("pos",), (3,))
    x, y = pos[:, 0], pos[:, 1]
    return (x < lo_x) | (x > hi_x) | (y < lo_y) | (y > hi_y)


def _has_contact(s: _Stock, p):
    _, cn = s.contact_norm(p["contact_manager"])
    return (cn > s.scalar(p["threshold"], "threshold")).sum(dim=1) >= int(p["min_contacts"])


def _contact_force_any(s: _Stock, p):
    _, cn = s.contact_norm(p["contact_manager"])
    return (cn > s.scalar(p["threshold"], "threshold")).any(dim=1)


def _t_timeout(s: _Stock, p):
    ep = s.episode_length()
    if not s.fused.env._base_max_episode_length:
        return s.tr.full(ep, False, torch.bool)
    return ep > s.src(("max_episode_length",), (), I32)


_STOCK = {
    ("reward", "GFB_R_IS_ALIVE"): lambda s, p: (~s.terminated()).float(),
    ("reward", "GFB_R_TERMINATED"): lambda s, p: s.terminated().float(),
    ("reward", "GFB_R_BASE_HEIGHT"): _r_base_height,
    ("reward", "GFB_R_DOF_SIMILAR"): lambda s, p: s.dof_deviation(),
    ("reward", "GFB_R_STAND_STILL"): _r_stand_still,
    ("reward", "GFB_R_LIN_VEL_Z"): _r_body_sq("lin_vel_b", (2,)),
    ("reward", "GFB_R_ANG_VEL_XY"): _r_body_sq("ang_vel_b", (0, 1)),
    ("reward", "GFB_R_FLAT_ORIENTATION"): _r_body_sq("gravity_b", (0, 1)),
    ("reward", "GFB_R_ACTION_RATE"): _r_action_rate,
    ("reward", "GFB_R_TRACK_LIN_VEL"): _r_track(True),
    ("reward", "GFB_R_TRACK_ANG_VEL"): _r_track(False),
    ("reward", "GFB_R_HAS_CONTACT"): lambda s, p: _has_contact(s, p).float(),
    ("reward", "GFB_R_CONTACT_FORCE"): lambda s, p: s.tr.nan_dropping(
        "fmax", s.contact_norm(p["contact_manager"])[1] - s.scalar(p["threshold"], "threshold"), 0.0).sum(dim=1),
    ("reward", "GFB_R_FEET_AIR_TIME"): _r_feet_air_time,
    ("reward", "GFB_R_FEET_SLIDE"): _r_feet_slide,
    ("termination", "GFB_T_TIMEOUT"): _t_timeout,
    ("termination", "GFB_T_BAD_ORIENTATION"): _t_bad_orientation,
    ("termination", "GFB_T_BASE_HEIGHT_MIN"): _t_base_height_min,
    ("termination", "GFB_T_OUT_OF_BOUNDS"): _t_out_of_bounds,
    ("termination", "GFB_T_HAS_CONTACT"): _has_contact,
    ("termination", "GFB_T_CONTACT_FORCE"): _contact_force_any,
    ("termination", "GFB_T_CONTACT_FORCE_GRACE"): lambda s, p: (
        _contact_force_any(s, p) & ~(s.episode_length() <= int(p["grace_steps"]))),
}


def param_kinds(params) -> tuple:
    """Per live-param candidate: int or float (a live param's kernel type, int32 or fp32, follows it)."""
    return tuple(sorted((k, type(v).__name__) for k, v in dict(params or {}).items()
                        if isinstance(v, (int, float)) and not isinstance(v, bool)))


def is_class_term(fn) -> bool:
    """An MdpFnClass instance (or a builtin): not a plain function."""
    return not hasattr(getattr(fn, "__func__", fn), "__code__")


class StateSlots:
    """The GFB_B_USER_STATE slots a class-style term may take: its own (by attribute) first, then free ones."""

    def __init__(self, own: dict, free: list):
        self.own, self.free = dict(own), list(free)

    def slot(self, attr: str) -> int:
        if attr not in self.own:
            if not self.free:
                raise UnsupportedTermError(f"user term: more state tensors than the {MAX_STATE_SLOTS} slots of the "
                                           "ABI (GFB_B_USER_STATE0..7)")
            self.own[attr] = self.free.pop(0)
        return self.own[attr]


def trace_term(fused, kind: str, name: str, item, live_params: bool = True, state: StateSlots | None = None) -> Program:
    """Trace one user-defined reward / termination / observation into a Program (raises UnsupportedTermError).
    `state`: the slots a class-style reward / termination term may bind (None: class-style terms are refused)."""
    env = fused.env
    fn = item.fn
    what = f"{kind} '{name}'"
    if is_class_term(fn):
        if state is None or kind == "observation" or isinstance(fn, type):
            raise UnsupportedTermError(f"{what}: class-style terms keep their own state and are not lowered")
        return _trace_stateful(fused, kind, what, item, state)
    tr = Tracer(fused.N, kind, fused.device)
    params = {}
    for k, v in dict(item.params or {}).items():
        if live_params and isinstance(v, (int, float)) and not isinstance(v, bool):
            params[k] = tr.param(k, v)
        else:
            params[k] = v
    swap = _Swap()
    try:
        _install_sources(fused, tr, swap, kind)
        env._tracing = ExprMode(tr, fused)
        result = fn(env=env, **params) if kind == "observation" else fn(env, **params)
    finally:
        env._tracing = None
        swap.restore()
    if not isinstance(result, Sym):
        raise UnsupportedTermError(f"{what}: the result does not depend on per-env state the kernel holds "
                                   f"({type(result).__name__})")
    return _term_program(tr, kind, what, result)


def trace_stateful(fused, kind: str, name: str, item, state: StateSlots) -> Program:
    """Trace one class-style reward / termination / observation term, binding its per-env tensors to the
    `state` slots (raises UnsupportedTermError)."""
    if isinstance(item.fn, type):
        raise UnsupportedTermError(f"{kind} '{name}': a class, not an instance of it")
    return _trace_stateful(fused, kind, f"{kind} '{name}'", item, state)


def _term_program(tr: Tracer, kind: str, what: str, result, writes: dict | None = None) -> Program:
    """The Program of a term's result (and of its state writes {slot: node})."""
    if not isinstance(result, Sym):
        raise UnsupportedTermError(f"{what}: the result does not depend on per-env state the kernel holds "
                                   f"({type(result).__name__})")
    slots = sorted(writes or {})
    if kind == "observation":
        # flattened row-major into its columns and cast to fp32, as FusedStep.evaluate_external_obs copies it
        if result.weak:
            raise UnsupportedTermError(f"{what}: the result is a Python scalar")
        width = int(np.prod(result.shape_)) if result.shape_ else 1
        if width > MAX_CONST_VEC:
            raise UnsupportedTermError(f"{what}: {width} columns (at most {MAX_CONST_VEC} are lowered)")
        out = tr.cast(tr._as_row((width,), result), F32)._id
        nodes, out, extra = _live_nodes(tr.nodes, out, [writes[s] for s in slots])
        return Program(kind, nodes, out, [], [], list(zip(slots, extra)))
    if result.weak or result.shape_ != ():
        raise UnsupportedTermError(f"{what}: the result has shape {tuple(result.shape)}, not (N,)")
    if kind == "termination" and result.dtype_ != BOOL:
        raise UnsupportedTermError(f"{what}: a termination must return a bool tensor")
    out = result._id
    if kind == "reward" and result.dtype_ != F32:
        out = tr.cast(result, F32)._id
    nodes, out, extra = _live_nodes(tr.nodes, out, [writes[s] for s in slots])
    return Program(kind, nodes, out, tr.params, tr.param_types, list(zip(slots, extra)))


_SCALARS = (bool, int, float, str, bytes, type(None))


def _same(a, b) -> bool:
    return a is b or (type(a) is type(b) and isinstance(a, _SCALARS) and a == b)


def instance_constants(inst) -> tuple:
    """The Python-scalar attributes of a class-style term: trace constants (a change traces it again)."""
    return tuple((k, v) for k, v in vars(inst).items() if isinstance(v, _SCALARS) and v is not None)


def _holds_env_rows(obj, N: int) -> bool:
    values = obj.values() if isinstance(obj, dict) else (obj if isinstance(obj, (list, tuple, set)) else
                                                          vars(obj).values())
    return any(torch.is_tensor(v) and v.dim() >= 1 and v.shape[0] == N for v in values)


def _trace_stateful(fused, kind: str, what: str, item, state: StateSlots) -> Program:
    """
    Trace a class-style term: `type(inst).__call__(inst, env, **params)` (an observation term: `env=env`) with
    the instance's per-env tensors as ("state", slot) sources.  Attributes that are None and get a per-env value
    during the call are initialised lazily: the call is traced once with them None (the first-call program) and
    once more with them as state.  Observation terms have no first-call program: the build's dry run has
    already called them, so such an attribute still None is refused.
    """
    env, inst, N = fused.env, item.fn, fused.N
    params = dict(item.params or {})
    before = dict(vars(inst))
    known = {id(env)} | {id(v) for v in vars(env).values()}
    for mgrs in getattr(env, "managers", {}).values():
        known |= {id(m) for m in (mgrs if isinstance(mgrs, (list, tuple)) else [mgrs])}
    rows: dict = {}  # attribute -> (row shape, dtype) of the per-env tensors
    for attr, v in before.items():
        if torch.is_tensor(v):
            if v.dim() == 0 or v.shape[0] != N:
                continue  # a constant (folded in where it is read); a write to it is refused below
            if v.dtype == torch.int64:
                raise UnsupportedTermError(f"{what}: state self.{attr} is int64 (the kernel's integers are 32-bit)")
            if v.dtype not in (torch.float32, torch.int32, torch.bool):
                raise UnsupportedTermError(f"{what}: state self.{attr} has dtype {v.dtype} (fp32, int32 or bool)")
            if int(np.prod(v.shape[1:])) > MAX_CONST_VEC:
                raise UnsupportedTermError(f"{what}: state self.{attr} has more than {MAX_CONST_VEC} elements a row")
            if v.device != fused.device or not v.is_contiguous():
                raise UnsupportedTermError(f"{what}: state self.{attr} is not a contiguous tensor on {fused.device}")
            rows[attr] = (tuple(v.shape[1:]), _dtype_of(v.dtype))
        elif id(v) not in known and not callable(v) and (isinstance(v, (list, tuple, set, dict))
                                                         or hasattr(v, "__dict__")):
            if _holds_env_rows(v, N):
                raise UnsupportedTermError(f"{what}: per-env state inside a container or sub-object (self.{attr})")
    ptrs = [before[a].untyped_storage().data_ptr() for a in rows]
    if len(set(ptrs)) != len(ptrs):
        raise UnsupportedTermError(f"{what}: two state tensors share storage")

    def run(lazy_rows: dict):
        tr = Tracer(N, kind, fused.device)
        syms, src = {}, {}
        for attr, (shape, dt) in {**rows, **lazy_rows}.items():
            slot = state.slot(attr)
            syms[attr] = tr.source(("state", slot), shape, dt)
            src[attr] = syms[attr]._id
            tr.state_objs[id(syms[attr])] = (slot, syms[attr])
        swap = _Swap()
        try:
            _install_sources(fused, tr, swap, kind)
            env._tracing = ExprMode(tr, fused)
            inst.__dict__.update(syms)
            if kind == "observation":
                result = type(inst).__call__(inst, env=env, **params)
            else:
                result = type(inst).__call__(inst, env, **params)
            after = dict(vars(inst))
        finally:
            env._tracing = None
            swap.restore()
            inst.__dict__.clear()
            inst.__dict__.update(before)
        writes = {}  # slot -> node of the value the env's row holds after the call
        for attr in sorted(set(before) | set(after)):
            old, new = before.get(attr, _MISSING), after.get(attr, _MISSING)
            if attr in syms:
                shape, dt = rows.get(attr) or lazy_rows[attr]
                if not isinstance(new, Sym) or new.weak or new.shape_ != shape or new.dtype_ != dt:
                    got = f"{new.dtype_}{list(new.shape_)}" if isinstance(new, Sym) else type(new).__name__
                    raise UnsupportedTermError(f"{what}: self.{attr} is rebound to {got}, not {dt}{list(shape)} (its "
                                               "row shape and dtype must stay)")
                if new._id != src[attr]:
                    writes[state.slot(attr)] = new._id
            elif old is None and isinstance(new, Sym) and kind == "observation":
                # (the build's dry run has called the term: lazily initialised state exists by now, or the
                #  term did not initialise it there)
                raise UnsupportedTermError(f"{what}: self.{attr} is None when the term is traced (an observation "
                                           "term is lowered with its state initialised)")
            elif old is None and isinstance(new, Sym) and not lazy_rows:  # lazy initialisation (first call)
                if new.weak or int(np.prod(new.shape_)) > MAX_CONST_VEC:
                    raise UnsupportedTermError(f"{what}: self.{attr} is initialised to a value that is not per-env "
                                               f"state of at most {MAX_CONST_VEC} elements a row")
                lazy[attr] = (new.shape_, new.dtype_)
                writes[state.slot(attr)] = new._id
            elif not _same(old, new):
                if torch.is_tensor(old) or torch.is_tensor(new):
                    raise UnsupportedTermError(f"{what}: the call writes self.{attr}, which is not per-env state")
                raise UnsupportedTermError(f"{what}: self.{attr} changes during the call (host state the kernel "
                                           "does not keep)")
        return tr, result, writes

    lazy: dict = {}
    tr, result, writes = run({})
    first = None
    if lazy:
        first = _term_program(tr, kind, what, result, writes)
        tr, result, writes = run(dict(lazy))
    prog = _term_program(tr, kind, what, result, writes)
    prog.first = first
    prog.bindings = {attr: (state.slot(attr), shape, dt, attr in lazy) for attr, (shape, dt) in {**rows, **lazy}.items()}
    return prog


def lower_term(fused, kind: str, name: str, item) -> tuple[Program, bool]:
    """(program, params_live): trace with live params, or once more with params as constants (always for
    observation terms: only their scale and noise are live, as for stock columns)."""
    if kind == "observation":
        try:
            return trace_term(fused, kind, name, item, live_params=False), False
        except _ParamControlFlow as e:
            raise UnsupportedTermError(f"{kind} '{name}': Python scalar arithmetic on '{e}' inside the term") from None
    try:
        return trace_term(fused, kind, name, item, live_params=True), True
    except _ParamControlFlow:
        pass
    try:
        return trace_term(fused, kind, name, item, live_params=False), False
    except _ParamControlFlow as e:
        raise UnsupportedTermError(f"{kind} '{name}': Python scalar arithmetic on '{e}' inside the term") from None


def _live_nodes(nodes: list, out: int, extra: list | None = None) -> tuple:
    """Dead-node elimination + renumbering (`extra`: further roots, returned renumbered as a third item)."""
    keep, stack = set(), [out] + list(extra or [])
    while stack:
        i = stack.pop()
        if i in keep:
            continue
        keep.add(i)
        stack.extend(nodes[i].args)
    order = sorted(keep)
    remap = {old: new for new, old in enumerate(order)}
    new = []
    for old in order:
        n = nodes[old]
        new.append(Node(n.op, [remap[a] for a in n.args], n.attr, n.shape, n.dtype, n.weak))
    if extra is None:
        return new, remap[out]
    return new, remap[out], [remap[i] for i in extra]


def _install_sources(fused, tr: Tracer, swap: _Swap, kind: str):
    env = fused.env
    robot = fused.primary_entity
    dofs_idx = fused.action.dofs_idx if fused.action is not None else None
    proxy = _EntityProxy(tr, dofs_idx, fused.D, robot)
    if robot is not None:
        for attr, value in list(vars(env).items()):
            if value is robot:
                swap.set(env, attr, proxy)
        # the primary entity's link objects, also those a term captured at build time: (N, 3) sources
        for link in getattr(robot, "links", ()):
            for what in ("pos", "vel"):
                swap.set(link, f"get_{what}", _link_getter(tr, what, int(link.idx_local)))
    if fused.entity_manager is not None:
        em = fused.entity_manager
        swap.set(em, "entity", proxy)
        # (rewards and terminations run after the entity phase: the cache IS this step's pose; the observation
        #  of a reset env sees the pre-reset cache next to the post-reset engine state)
        cached = kind == "observation"
        swap.set(em, "_base_pos", tr.source(("base_pos",) if cached else ("pos",), (3,), F32))
        swap.set(em, "_base_quat", tr.source(("base_quat",) if cached else ("quat",), (4,), F32))
    for k, mgr in enumerate(fused.commands):
        if mgr in fused.python_commands or mgr._external_controller is not None:
            continue  # a user-level manager's state stays concrete: refused where it is used
        swap.set(mgr, "_command", tr.source(("command", k), (mgr._command.shape[1],), F32))
    for m, mgr in enumerate(fused.contacts):
        L = int(mgr._link_ids.shape[0])
        swap.set(mgr, "contacts", tr.source(("contacts", m), (L, 3), F32))
        if mgr._track_air_time:
            swap.set(mgr, "_air", _AirProxy(tr, m, L))
    swap.set(env, "episode_length", tr.source(("episode_length",), (), I32))
    if env.max_episode_length is not None:
        swap.set(env, "max_episode_length", tr.source(("max_episode_length",), (), I32))
    if fused.D > 0:
        swap.set(env, "_actions", tr.source(("actions",), (fused.D,), F32))
        swap.set(env, "_last_actions", tr.source(("last_actions",), (fused.D,), F32))
    extras = env.extras
    for key, src in (("terminations", "terminated"), ("time_outs", "truncated")):
        if fused.termination is None:  # nothing publishes the key: reading it fails in the function itself
            swap.set_item(extras, key, _Refused(f"extras['{key}'] without a termination manager"))
        elif kind == "reward":
            swap.set_item(extras, key, tr.source((src,), (), BOOL))
        else:
            swap.set_item(extras, key, _Refused(f"extras['{key}'] inside a {kind} term"))


def _link_getter(tr: Tracer, what: str, local: int):
    def get(envs_idx=None):
        if envs_idx is not None:
            raise UnsupportedTermError(f"user term: link.get_{what}(envs_idx=...)")
        return tr.source((f"link_{what}", (local,)), (3,), F32)
    return get


def link_union(progs) -> dict:
    """{"pos" / "vel": local link ids in first-use order} read by the link sources of `progs` (and their
    first-call programs)."""
    out: dict = {}
    for prog in progs:
        for p in (prog, prog.first):
            for n in (p.nodes if p is not None else ()):
                if n.op == "src" and n.attr[0] in ("link_pos", "link_vel"):
                    ids = out.setdefault(n.attr[0][5:], [])
                    ids += [i for i in n.attr[1] if i not in ids]
    return {k: out[k] for k in ("pos", "vel") if k in out}


def place_links(progs, layout: dict):
    """Write the table's link layout {"pos" / "vel": (slot, U)} into the link sources of `progs`: the attr
    (kind, ids, slot, U) is part of the program's text, so of its identity and of the header."""
    for prog in progs:
        for p in (prog, prog.first):
            for n in (p.nodes if p is not None else ()):
                if n.op == "src" and n.attr[0] in ("link_pos", "link_vel"):
                    slot, U = layout[n.attr[0][5:]]
                    n.attr = (n.attr[0], n.attr[1], slot, tuple(U))


class _Refused:
    def __init__(self, what):
        self._what = what

    def __getattr__(self, name):
        raise UnsupportedTermError(f"user term: {object.__getattribute__(self, '_what')}")

    def _refuse(self, *a, **k):
        raise UnsupportedTermError(f"user term: {self._what}")

    __invert__ = __and__ = __or__ = __rand__ = __ror__ = __getitem__ = __bool__ = _refuse

    @classmethod
    def __torch_function__(cls, func, types, args=(), kwargs=None):
        what = next(a for a in args if isinstance(a, _Refused))._what
        raise UnsupportedTermError(f"user term: {what}")


# ------------------------------------------------------------------------------------------------
# device code
# ------------------------------------------------------------------------------------------------
_CT = {F32: "float", I32: "int", BOOL: "bool"}


def _lit(v, dtype) -> str:
    if dtype == BOOL:
        return "true" if v else "false"
    if dtype == I32:
        return f"({int(v)})"
    v = _f32(v)
    if math.isnan(v):
        return "__int_as_float(0x7fc00000)"
    if math.isinf(v):
        return "__int_as_float(0x7f800000)" if v > 0 else "__int_as_float(0xff800000)"
    return f"{v.hex()}f" if v >= 0 else f"(-{(-v).hex()}f)"


_SLAB = {"pos": "off_pos", "quat": "off_quat", "vel": "off_vel", "ang": "off_ang"}  # staged slab rows (plan.h)


def _src_elems(key: tuple, shape: tuple, lines: list, v: str, glob: bool = False) -> list[str]:
    """C expressions of a source's elements for this env (row-major over `shape`).  `glob`: global memory
    only (the reset path of observation terms, which has no slab, stash or body-frame registers)."""
    n = int(np.prod(shape)) if shape else 1
    name = key[0]
    if name in ("base_pos", "base_quat"):  # the EntityManager's cached pose (observation terms)
        w, eng = (3, "pos") if name == "base_pos" else (4, "quat")
        cache = f"reinterpret_cast<const float*>(c.b.buf[GFB_B_BASE_{eng.upper()}]) + (size_t)c.e * {w}"
        if glob:
            lines.append(f"const float* {v}p = {cache};")
        else:
            # a launch with the entity phase (the only one that stages quat) writes the cache from these rows
            off = f"c.plan.{_SLAB[eng]}"
            engine = f"reinterpret_cast<const float*>(c.b.buf[GFB_B_{eng.upper()}]) + (size_t)c.e * {w}"
            lines.append(f"const float* {v}p = c.plan.off_quat >= 0 ? ({off} >= 0 ? c.S + {off} + c.tid * {w} : "
                         f"{engine}) : {cache};")
        return [f"{v}p[{i}]" for i in range(n)]
    row = {"pos": ("GFB_B_POS", 3), "quat": ("GFB_B_QUAT", 4), "vel": ("GFB_B_VEL", 3), "ang": ("GFB_B_ANG", 3),
           "dof_pos": ("GFB_B_DOF_POS", n), "dof_vel": ("GFB_B_DOF_VEL", n), "targets": ("GFB_B_TARGETS", n),
           "actions": ("GFB_B_ENV_ACTIONS", n), "last_actions": ("GFB_B_ENV_LAST_ACTIONS", n)}
    if name in row:
        buf, w = row[name]
        gaddr = f"reinterpret_cast<const float*>(c.b.buf[{buf}]) + (size_t)c.e * {w}"
        if name in _SLAB and not glob:  # the slab row when the plan stages the array (a compile-time choice)
            off = f"c.plan.{_SLAB[name]}"
            lines.append(f"const float* {v}p = {off} >= 0 ? c.S + {off} + c.tid * {w} : {gaddr};")
        else:
            lines.append(f"const float* {v}p = {gaddr};")
        return [f"{v}p[{i}]" for i in range(n)]
    if name == "command":
        lines.append(f"const float* {v}p = reinterpret_cast<const float*>(c.b.buf[GFB_B_COMMAND0 + {key[1]}]) + "
                     f"(size_t)c.e * {n};")
        return [f"{v}p[{i}]" for i in range(n)]
    if name == "contacts":
        lines.append(f"const float* {v}p = reinterpret_cast<const float*>(c.b.buf[GFB_B_CONTACTS0 + {key[1]}]) + "
                     f"(size_t)c.e * {n};")
        return [f"{v}p[{i}]" for i in range(n)]
    if name == "air":
        m, j = key[1], key[2]
        if glob:  # (4, N, Lc) planes
            lines.append(f"const float* {v}p = reinterpret_cast<const float*>(c.b.buf[GFB_B_AIR0 + {m}]) + "
                         f"(size_t){j} * c.n_envs * {n} + c.e * {n};")
            return [f"{v}p[{l}]" for l in range(n)]
        return [f"c.st[c.plan.st_air[{m}] + {l * 4 + j}]" for l in range(n)]
    if name in ("lin_vel_b", "ang_vel_b", "gravity_b"):
        # the kernel's own register when the plan computes it (same rotation), else rotated here
        reg, need = {"lin_vel_b": ("lin_b", "NEED_LIN"), "ang_vel_b": ("ang_b", "NEED_ANG"),
                     "gravity_b": ("grav_b", "NEED_GRAV")}[name]
        if name == "gravity_b":
            vec = "V3{0.0f, 0.0f, -1.0f}"
        else:
            buf = "GFB_B_VEL" if name == "lin_vel_b" else "GFB_B_ANG"
            lines.append(f"const float* {v}p = reinterpret_cast<const float*>(c.b.buf[{buf}]) + (size_t)c.e * 3;")
            vec = f"V3{{{v}p[0], {v}p[1], {v}p[2]}}"
        if glob:
            lines.append(f"const V3 {v}r = rotate({vec}, c.iw, c.iq);")
        else:
            lines.append(f"const V3 {v}r = (c.plan.needs & {need}) ? c.{reg} : rotate({vec}, c.iw, c.iq);")
        return [f"{v}r.x", f"{v}r.y", f"{v}r.z"]
    if name in ("link_pos", "link_vel"):
        # a per-launch (N, |U|, 3) gather of the engine's link array, bound to a free GFB_B_USER_STATE slot
        if len(key) != 4:
            raise UnsupportedTermError(f"user term: source {key!r} has no link layout")
        ids, slot, U = key[1], key[2], key[3]
        lines.append(f"const float* {v}p = reinterpret_cast<const float*>(c.b.buf[GFB_B_USER_STATE0 + {slot}]) + "
                     f"(size_t)c.e * {len(U) * 3};")
        return [f"{v}p[{U.index(i) * 3 + k}]" for i in ids for k in range(3)]
    if name == "action_rate":  # rewards only: the action kernel's sum for this step, as the stock row reads it
        return ["reinterpret_cast<const float*>(c.b.buf[GFB_B_ACTION_RATE])[c.e]"]
    if name == "episode_length":
        return ["c.ep_len"]
    if name == "max_episode_length":
        return ["c.max_len"]
    if name == "terminated":
        return ["c.terminated"]
    if name == "truncated":
        return ["c.truncated"]
    raise UnsupportedTermError(f"user term: source {key!r}")


def _strides(shape):
    out, s = [], 1
    for n in reversed(shape):
        out.append(s)
        s *= n
    return list(reversed(out))


def _binop(op, a, b, dtype, attr=None):
    if dtype == F32:
        arith = {"add": f"add({a}, {b})", "sub": f"sub({a}, {b})", "mul": f"mul({a}, {b})", "div": f"fdiv({a}, {b})"}
    else:
        arith = {"add": f"({a} + {b})", "sub": f"({a} - {b})", "mul": f"({a} * {b})"}
    if op in arith:
        return arith[op]
    if op == "mod":
        return f"gfb_user_mod({a}, {b})"
    if op in ("fmax", "fmin"):
        return f"{op}f({a}, {b})"
    if op in ("clamp_lo", "clamp_hi") and dtype == F32:
        return f"gfb_user_{op}{'_scalar' if attr == 'scalar' else ''}({a}, {b})"
    if op in ("minimum", "clamp_hi"):
        # NaN propagates (torch.minimum)
        return f"gfb_user_min({a}, {b})" if dtype == F32 else f"min({a}, {b})"
    if op in ("maximum", "clamp_lo"):
        return f"gfb_user_max({a}, {b})" if dtype == F32 else f"max({a}, {b})"
    cmp = {"lt": "<", "le": "<=", "gt": ">", "ge": ">=", "eq": "==", "ne": "!="}
    if op in cmp:
        return f"({a} {cmp[op]} {b})"
    if op == "and":
        return f"({a} && {b})"
    if op == "or":
        return f"({a} || {b})"
    raise UnsupportedTermError(op)


def _unop(op, a, dtype):
    if op == "neg":
        return f"(-{a})"
    if op == "not":
        return f"(!{a})"
    if op == "abs":
        return f"fabsf({a})" if dtype == F32 else f"abs({a})"
    if op == "square":
        return f"sq({a})" if dtype == F32 else f"({a} * {a})"
    fn = {"sqrt": "__fsqrt_rn", "exp": "expf", "log": "logf", "sin": "sinf", "cos": "cosf", "tanh": "tanhf"}[op]
    return f"{fn}({a})"


_PASS = ("sum", "mean", "any", "all", "amax", "amin", "norm", "reshape", "stack", "cat")  # no new variables


def function_body(prog: Program, fname: str, glob: bool = False) -> str:
    """One `__device__` function for the program (straight-line code, one variable per element).  An
    observation term writes its columns to `out`; `glob` reads global memory only (see _src_elems)."""
    lines: list[str] = []
    elems: list[list[str]] = []
    for i, n in enumerate(prog.nodes):
        v = f"v{i}"
        ct = _CT[n.dtype]
        size = int(np.prod(n.shape)) if n.shape else 1
        if n.op == "src" and n.attr[0] == "state":  # the env's row of a class-style term's state
            lines.append(f"const {ct}* {v}p = reinterpret_cast<const {ct}*>(c.b.buf[GFB_B_USER_STATE0 + {n.attr[1]}]) + "
                         f"c.e * {size};")
            exprs = [f"{v}p[{k}]" for k in range(size)]
        elif n.op == "src":
            exprs = _src_elems(n.attr, n.shape, lines, v, glob)
        elif n.op == "full":
            exprs = [_lit(n.attr, n.dtype)] * size
        elif n.op == "reshape":
            exprs = list(elems[n.args[0]])
        elif n.op == "stack":
            parts = [elems[j] for j in n.args]
            exprs = [p[k] for k in range(len(parts[0])) for p in parts]
        elif n.op == "cat":
            parts = [(elems[j], prog.nodes[j].shape[-1]) for j in n.args]
            rows = len(parts[0][0]) // parts[0][1] if parts[0][1] else 0
            exprs = [x for r in range(rows) for p, w in parts for x in p[r * w:(r + 1) * w]]
        elif n.op == "param":
            p = f"c.p[{n.attr}]"
            exprs = [f"((int){p})" if n.dtype == I32 else p]
        elif n.op == "const":
            exprs = [_lit(n.attr, n.dtype)]
        elif n.op == "constvec":
            exprs = [_lit(x, n.dtype) for x in n.attr]
        elif n.op == "cast":
            src = prog.nodes[n.args[0]].dtype
            a = elems[n.args[0]]
            if n.dtype == BOOL:
                exprs = [f"({x} != 0)" for x in a]
            elif n.dtype == F32 and src == I32:
                exprs = [f"__int2float_rn({x})" for x in a]
            elif n.dtype == F32:
                exprs = [f"({x} ? 1.0f : 0.0f)" for x in a]
            elif src == F32:
                exprs = [f"gfb_user_f2i({x})" for x in a]
            else:
                exprs = [f"(int)({x})" for x in a]
        elif n.op in ("neg", "not", "abs", "square", "sqrt", "exp", "log", "sin", "cos", "tanh"):
            exprs = [_unop(n.op, x, n.dtype) for x in elems[n.args[0]]]
        elif n.op == "where":
            c, a, b = (elems[j] for j in n.args)
            ic, ia, ib = (_bidx(n.shape, prog.nodes[j].shape) for j in n.args)
            exprs = [f"({c[ic[k]]} ? {a[ia[k]]} : {b[ib[k]]})" for k in range(size)]
        elif n.op == "index":
            src_shape = prog.nodes[n.args[0]].shape
            a = elems[n.args[0]]
            st = _strides(src_shape)
            ranges = [[s] if isinstance(s, int) else list(s[1:]) if s[0] == "list" else list(range(s[0], s[1]))
                      for s in n.attr]
            exprs = []
            for combo in np.ndindex(*[len(r) for r in ranges]) if ranges else [()]:
                flat = sum(ranges[d][combo[d]] * st[d] for d in range(len(ranges)))
                exprs.append(a[flat])
        elif n.op in ("sum", "mean", "any", "all", "amax", "amin", "norm"):
            src_shape = prog.nodes[n.args[0]].shape
            a = elems[n.args[0]]
            axis = n.attr
            st = _strides(src_shape)
            outs = []
            out_shape = n.shape
            for combo in (np.ndindex(*out_shape) if out_shape else [()]):
                idx = list(combo)
                terms = []
                for r in range(src_shape[axis]):
                    full = idx[:axis] + [r] + idx[axis:]
                    terms.append(a[sum(full[d] * st[d] for d in range(len(src_shape)))])
                outs.append(_reduce_expr(n.op, terms, n.dtype, lines, f"{v}_{len(outs)}"))
            exprs = outs
        else:
            a = elems[n.args[0]]
            b = elems[n.args[1]]
            ia, ib = (_bidx(n.shape, prog.nodes[j].shape) for j in n.args)
            exprs = [_binop(n.op, a[ia[k]], b[ib[k]], prog.nodes[n.args[0]].dtype, n.attr) for k in range(size)]
        # every element is materialised once, in node order (torch's operation order)
        names = []
        for k, x in enumerate(exprs):
            nm = f"{v}_{k}" if n.op not in _PASS else x
            if nm != x:
                lines.append(f"const {ct} {nm} = {x};")
            names.append(nm)
        elems.append(names)
    body = "\n".join("  " + ln for ln in lines)
    stores = []
    # after the result; lanes that shadow env N-1 in a tail slab do not store, nor (observation terms) a reset
    # env in the owner phase: the reset path evaluates it again
    for slot, i in prog.writes:
        ct = _CT[prog.nodes[i].dtype]
        row = elems[i]
        stores.append(f"    {ct}* s{slot} = reinterpret_cast<{ct}*>(c.b.buf[GFB_B_USER_STATE0 + {slot}]) + c.e * "
                      f"{len(row)};")
        stores += [f"    s{slot}[{k}] = {x};" for k, x in enumerate(row)]
    store = ("\n  if (c.active) {\n" + "\n".join(stores) + "\n  }") if stores else ""
    if prog.kind == "observation":
        out = "\n".join(f"  out[{k}] = {x};" for k, x in enumerate(elems[prog.out]))
        return f"__device__ __forceinline__ void {fname}(const UserCtx& c, float* out) {{\n{body}\n{out}{store}\n}}\n"
    ret = elems[prog.out][0]
    rtype = "bool" if prog.kind == "termination" else "float"
    return (f"__device__ __forceinline__ {rtype} {fname}(const UserCtx& c) {{\n{body}{store}\n  return {ret};\n}}\n")


def _reduce_expr(op, terms, dtype, lines, acc) -> str:
    ct = _CT[dtype]
    if op in ("any", "all"):
        j = " || " if op == "any" else " && "
        lines.append(f"const bool {acc} = {j.join(terms) if terms else ('false' if op == 'any' else 'true')};")
        return acc
    if not terms:
        raise UnsupportedTermError(f"user term: {op} over an empty dimension")
    if op == "norm" and len(terms) <= 3:  # torch-CPU: |x|, and the fma chains of device_utils.cuh
        fn = {1: "fabsf", 2: "norm2", 3: "norm3"}[len(terms)]
        lines.append(f"const float {acc} = {fn}({', '.join(terms)});")
        return acc
    if op in ("sum", "mean", "norm"):
        # torch's sum starts from +0 (a row of -0 sums to +0)
        first = f"sq({terms[0]})" if op == "norm" else (f"add(0.0f, {terms[0]})" if dtype == F32 else terms[0])
        lines.append(f"{ct} {acc} = {first};")
        for t in terms[1:]:
            x = f"sq({t})" if op == "norm" else t
            lines.append(f"{acc} = add({acc}, {x});" if dtype == F32 else f"{acc} = {acc} + {x};")
        if op == "mean":
            lines.append(f"{acc} = fdiv({acc}, {_lit(float(len(terms)), F32)});")
        if op == "norm":
            lines.append(f"{acc} = __fsqrt_rn({acc});")
        return acc
    fn = ("gfb_user_max" if op == "amax" else "gfb_user_min") if dtype == F32 else ("max" if op == "amax" else "min")
    lines.append(f"{ct} {acc} = {terms[0]};")
    for t in terms[1:]:
        lines.append(f"{acc} = {fn}({t}, {acc});")  # (on a tie the accumulator: the first element is kept)
    return acc


def device_code(rewards: dict[int, Program], terminations: dict[int, Program],
                observations: list[tuple[int, Program]] = (), obs_words: int = 0) -> str:
    """The user-term functions of one table and their dispatchers, keyed by table row; the observation terms
    as (first word in the (N, obs_words) user-observation row, program), each twice (owner phase, reset path)."""
    parts = []
    for what, progs, fn in (("reward", rewards, "gfb_user_r"), ("termination", terminations, "gfb_user_t")):
        for r, prog in sorted(progs.items()):
            if prog.first is None:
                parts.append(f"/* {what} row {r} */\n" + function_body(prog, f"{fn}{r}"))
                continue
            # lazily initialised state: the first-call program until the host sets the term's p[0]
            rtype = "bool" if prog.kind == "termination" else "float"
            parts.append(f"/* {what} row {r}: first call */\n" + function_body(prog.first, f"{fn}{r}_first"))
            parts.append(f"/* {what} row {r} */\n" + function_body(prog, f"{fn}{r}_steady"))
            parts.append(f"__device__ __forceinline__ {rtype} {fn}{r}(const UserCtx& c) {{\n"
                         f"  return c.p[0] != 0.0f ? {fn}{r}_steady(c) : {fn}{r}_first(c);\n}}\n")
    cases_r = "".join(f"    case {r}: return gfb_user_r{r}(c);\n" for r in sorted(rewards))
    cases_t = "".join(f"    case {t}: return gfb_user_t{t}(c);\n" for t in sorted(terminations))
    parts.append("__device__ __forceinline__ float user_reward(int r, const UserCtx& c) {\n  switch (r) {\n"
                 f"{cases_r}    default: return 0.0f;\n  }}\n}}\n")
    parts.append("__device__ __forceinline__ bool user_termination(int t, const UserCtx& c) {\n  switch (t) {\n"
                 f"{cases_t}    default: return false;\n  }}\n}}\n")
    if observations:
        calls, calls_g = "", ""
        for j, (col0, prog) in enumerate(observations):
            parts.append(f"/* observation term {j}: words {col0}.. */\n" + function_body(prog, f"gfb_user_o{j}"))
            parts.append(function_body(prog, f"gfb_user_og{j}", glob=True))
            calls += f"  gfb_user_o{j}(c, out + {col0});\n"
            calls_g += f"  gfb_user_og{j}(c, out + {col0});\n"
        if any(prog.writes for _, prog in observations):
            # (spec.py defines GFB_SPEC_USER_OBS_STATE for it: the owner phase passes active && !reset)
            parts.append("/* observation terms store state */\n")
        parts.append(f"constexpr int kUserObsWords = {obs_words};\n")
        parts.append(f"__device__ __forceinline__ void user_observations(const UserCtx& c, float* out) {{\n{calls}}}\n")
        parts.append("__device__ __forceinline__ void user_observations_global(const UserCtx& c, float* out) {\n"
                     f"{calls_g}}}\n")
    return "".join(parts)
