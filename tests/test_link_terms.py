"""
Host side of lowered user terms that read per-link state (configs/link_terms.py): link sources of the tracer,
their layout in the GFB_B_USER_STATE slots, row-wise broadcasting and constant index lists, refusals, and the
generated device code.  No GPU needed.
"""
import os
import re
import shutil
import subprocess
import tempfile
import types
from pathlib import Path

import numpy as np
import pytest
import torch

import genesis_forge_b200 as gfb
from configs import link_terms, specs
from configs.env_builder import build_env, dropin_namespace
from genesis_forge_b200 import expr
from genesis_forge_b200.managed_env import ManagedEnvironment
from genesis_forge_b200.managers.config import MdpFnClass
from test_user_terms_edges import EDGE_F32

N = 64
NVCC = shutil.which("nvcc") or ("/usr/local/cuda/bin/nvcc" if os.path.exists("/usr/local/cuda/bin/nvcc") else None)
SWITCHES = ("fuse_user_terms", "fuse_user_observations", "fuse_stateful_terms")
REWARDS = ("foot_clearance", "foot_slip", "feet_spacing", "front_foot", "swing_peak")
OBS = ("feet_rel_base", "foot_speed")


@pytest.fixture()
def cpu_device():
    prev = gfb.gs.device
    gfb.set_device("cpu")
    yield torch.device("cpu")
    gfb.gs.device = prev


@pytest.fixture()
def jit(monkeypatch):
    """The lowering decision needs a compilable specialisation; it is made without compiling anything."""
    from genesis_forge_b200 import spec

    monkeypatch.delenv("GFB_NO_SPEC", raising=False)
    monkeypatch.setattr(spec, "jit_allowed", lambda: True)


def dry_env(spec, monkeypatch, on=True, n=N):
    for name in SWITCHES:
        monkeypatch.setattr(ManagedEnvironment, name, on)
    env = build_env(spec, dropin_namespace(), n, torch.device("cpu"))
    env._dry_run = True
    env.build()
    env._fused._set_program()
    return env


def test_workload_lowers_completely(cpu_device, jit, monkeypatch):
    fused = dry_env(link_terms.link_terms(), monkeypatch)._fused
    assert not fused.user_term_refusals and not fused.external_rows and not fused.external_obs
    assert not fused.split_mode
    assert sorted(n for k, n in fused.user_terms) == sorted(REWARDS + ("feet_below",))
    assert sorted(n for _, n in fused.user_obs) == sorted(OBS)
    feet, calves = (4, 8, 12, 16), (3, 7, 11, 15)
    state = {s for b in fused.stateful.values() for s in b["tensors"]}
    assert state == {0}  # swing_peak's (N, 4) peak
    assert fused._link_layout == {"pos": (7, feet), "vel": (6, feet + calves)}
    assert fused._obs_reads_links and fused._obs_reads_pose
    # the layout is part of every program reading links, so of its identity
    for prog, *_ in list(fused.user_terms.values()) + list(fused.user_obs.values()):
        for key in prog.sources():
            if key[0] in ("link_pos", "link_vel"):
                assert key[2:] == fused._link_layout[key[0][5:]]
    K = gfb._native.K
    robot = fused.primary_entity
    assert fused._link_phases == K["GFB_PHASE_REWARD"] | K["GFB_PHASE_TERMINATION"] | K["GFB_PHASE_OBSERVE"]
    fused._bind_links(True)  # (one gather per link array and launch)
    ptrs = {fused.buffers.buf[K["GFB_B_USER_STATE0"] + s] for s in (6, 7)}
    assert all(ptrs) and len(ptrs) == 2
    fused._bind_links(False)  # a launch that reads none: the placeholder, nothing gathered or kept
    assert {fused.buffers.buf[K["GFB_B_USER_STATE0"] + s] for s in (6, 7)} == {fused._link_placeholder.data_ptr()}
    from genesis_forge_b200 import spec

    macro = spec._user_terms_macro(fused.user_code)
    assert "#define GFB_SPEC_STATE_SLOTS 193u" in macro  # slots 0, 6 and 7
    assert torch.equal(robot.get_links_pos(links_idx_local=list(feet)), robot.get_links_pos(links_idx_local=feet))


def test_switches_off_keep_todays_plans(cpu_device, jit, monkeypatch):
    off = dry_env(link_terms.link_terms(), monkeypatch, on=False)._fused
    assert not off.user_terms and not off.user_obs and not off._link_layout and not off.user_term_refusals
    assert [n for _, n, _ in off.external_rows] == list(REWARDS) + ["feet_below"]
    assert [n for _, n, _, _, _ in off.external_obs] == list(OBS)
    K = gfb._native.K
    assert not any(off.buffers.buf[K["GFB_B_USER_STATE0"] + s] for s in range(8))
    stock_on = dry_env(specs.contacts(), monkeypatch)._fused
    stock_off = dry_env(specs.contacts(), monkeypatch, on=False)._fused
    assert bytes(stock_on.program) == bytes(stock_off.program) and stock_on.split_plan == stock_off.split_plan
    assert not stock_on._link_layout


def test_demotion_unbinds_the_link_slots(cpu_device, jit, monkeypatch):
    on = dry_env(link_terms.link_terms(), monkeypatch)._fused
    off = dry_env(link_terms.link_terms(), monkeypatch, on=False)._fused
    on._demote_user_terms("test")
    assert on._link_layout == {} and not on._obs_reads_links
    assert on.split_plan == off.split_plan
    assert [(k, n) for k, n, _ in on.external_rows] == [(k, n) for k, n, _ in off.external_rows]
    K = gfb._native.K
    assert not any(on.buffers.buf[K["GFB_B_USER_STATE0"] + s] for s in range(8))
    on._engine_buffers()
    on._bind_links(True)
    assert not any(on.buffers.buf[K["GFB_B_USER_STATE0"] + s] for s in range(8))


def test_a_retrace_that_changes_the_links_changes_the_layout_and_identity(cpu_device, jit, monkeypatch):
    def one_link(env, link=4):
        return env.robot.get_links_pos(links_idx_local=[link])[:, 0, 2]

    spec = link_terms.link_terms()
    spec["rewards"] = dict(spec["rewards"], one_link={"fn": one_link, "weight": 1.0, "params": {"link": 4}})
    fused = dry_env(spec, monkeypatch)._fused
    pos = fused._link_layout["pos"]
    row = list(fused.reward.cfg).index("foot_clearance")
    i0 = fused.program.head.reward[row].i0
    fused.reward.cfg["one_link"].params["link"] = 2  # FL_thigh, which no other term reads: traced again
    fused._set_program(force=True)
    assert fused._link_layout["pos"] == (pos[0], pos[1] + (2,))
    assert fused.program.head.reward[row].i0 != i0  # same expression, other columns: another kernel
    assert fused.program.head.reward[row].i0 == fused.user_terms[("reward", "foot_clearance")][0].digest()


def test_a_retrace_past_the_link_limit_keeps_the_table_and_demotes(cpu_device, jit, monkeypatch):
    def first_links(env, n=2):
        return env.robot.get_links_pos(links_idx_local=range(n))[:, :, 2].sum(dim=1)

    spec = link_terms.link_terms()
    spec["rewards"] = dict(spec["rewards"], first_links={"fn": first_links, "weight": 1.0, "params": {"n": 2}})
    fused = dry_env(spec, monkeypatch)._fused
    layout, code = dict(fused._link_layout), fused.user_code
    assert layout["pos"][1] == (4, 8, 12, 16, 0, 1)
    fused.reward.cfg["first_links"].params["n"] = 10  # 12 links in the position array
    fused._set_program(force=True)
    assert fused._link_layout == layout and fused.user_code == code  # the table stays as its binary was built
    why = fused._check_state()  # (before the step's first launch)
    assert "first_links" in why and "at most 10" in why, why
    fused._demote_user_terms(why)
    assert ("reward", "first_links") in {(k, n) for k, n, _ in fused.external_rows} and not fused._link_layout


def test_a_one_term_evaluation_of_a_further_entity_gathers_links_from_the_robot(cpu_device, jit, monkeypatch):
    """A stock term of the prop runs through evaluate_single_term, which points `primary_entity` at the prop: the
    link arrays still come from the robot the layout was built for (the prop has no links to gather)."""
    from configs import second_entity

    spec = link_terms.link_terms()
    spec["rewards"] = dict(spec["rewards"], prop_height={
        "fn": "base_height", "weight": -2.0, "params": {"target_height": 1.3, "entity_attr": "prop"}})
    for name in SWITCHES:
        monkeypatch.setattr(ManagedEnvironment, name, True)
    ns = dropin_namespace()
    env = second_entity.add_prop(build_env(spec, ns, N, torch.device("cpu")), ns)
    env._dry_run = True
    env.build()
    fused = env._fused
    fused._set_program()
    assert [n for _, n, _ in fused.external_rows] == ["prop_height"] and fused._link_layout
    K = gfb._native.K
    robot, prop = fused.primary_entity, env.prop
    assert not hasattr(prop, "get_links_pos")
    fused.primary_entity = prop  # (what evaluate_single_term does for the prop's term)
    try:
        fused._engine_buffers()
        fused._bind_links(True)
    finally:
        fused.primary_entity = robot
    slot, ids = fused._link_layout["vel"]
    bound = fused._keepalive[-1]
    assert fused.buffers.buf[K["GFB_B_USER_STATE0"] + slot] == bound.data_ptr()
    assert torch.equal(bound, robot.get_links_vel(links_idx_local=list(ids)))


# ------------------------------------------------------------------------------------------------
# refusals
# ------------------------------------------------------------------------------------------------
def _refused(monkeypatch, fn, kind="reward", spec=None):
    spec = spec or specs.contacts()
    table = "rewards" if kind == "reward" else "terminations"
    spec[table] = dict(spec[table], probe={"fn": fn, "weight": 1.0} if kind == "reward" else {"fn": fn})
    fused = dry_env(spec, monkeypatch)._fused
    assert (kind, "probe") not in fused.user_terms
    assert (kind, "probe") in {(k, n) for k, n, _ in fused.external_rows}
    return fused.user_term_refusals[(kind, "probe")]


def _pos(e):
    return e.robot.get_pos()


class _ManyState(MdpFnClass):
    def __init__(self, env):
        super().__init__(env)
        for k in range(7):
            setattr(self, f"s{k}", torch.zeros(env.num_envs))

    def __call__(self, env):
        v = env.robot.get_links_pos(links_idx_local=[4])[:, 0, 2]
        for k in range(7):
            setattr(self, f"s{k}", getattr(self, f"s{k}") + v)
        return self.s0 + env.robot.get_links_vel(links_idx_local=[4])[:, 0, 2]


@pytest.mark.parametrize("fn,needle", [
    (lambda e: e.robot.get_links_pos()[:, 0, 0], "get_links_pos"),
    (lambda e: e.robot.get_links_vel()[:, 0, 0], "get_links_vel"),
    (lambda e: e.robot.get_links_pos(links_idx_local=[4], envs_idx=torch.arange(4))[:, 0, 0], "envs_idx"),
    (lambda e: e.robot.get_link("FL_foot").get_pos(envs_idx=torch.arange(4))[:, 0], "envs_idx"),
    (lambda e: e.robot.get_links_pos(links_idx_local=[99])[:, 0, 0], "local link ids"),
    (lambda e: e.robot.get_links_pos(links_idx_local=list(range(11)))[:, :, 2].sum(dim=1), "at most 10"),
    (lambda e: (e.robot.get_links_pos(links_idx_local=list(range(6)))[:, :, 2].sum(dim=1)
                + e.robot.get_links_pos(links_idx_local=list(range(6, 12)))[:, :, 2].sum(dim=1)), "at most 10"),
    (lambda e: e.robot.get_links_pos(links_idx_local=[0.5])[:, 0, 0], "ints only"),
    (lambda e: _pos(e)[:, torch.tensor([True, False, True])].sum(dim=1), "bool mask"),
    (lambda e: e.robot.get_links_pos(links_idx_local=[1, 2])[:, [0, 1], [0, 2]].sum(dim=1), "two advanced"),
    (lambda e: _pos(e)[:, [0, 3]].sum(dim=1), "out of range"),
    (lambda e: _pos(e)[:, [0] * 33].sum(dim=1), "at most 32"),
    (lambda e: _pos(e)[:, [0, e.episode_length]].sum(dim=1), "index"),
    (lambda e: (e.robot.get_links_pos(links_idx_local=[4, 8])[:, :, 2] - _pos(e)[:, 0:3]).sum(dim=1),
     "does not broadcast"),
    (lambda e: (e.robot.get_links_pos(links_idx_local=[4, 8]) - _pos(e)).sum(dim=1).sum(dim=1), "does not broadcast"),
    (_ManyState, "GFB_B_USER_STATE0..7"),
])
def test_refusals_keep_the_callback(fn, needle, cpu_device, jit, monkeypatch):
    why = _refused(monkeypatch, fn)
    assert needle in why, why


def test_links_of_a_further_entity_are_refused(cpu_device, jit, monkeypatch):
    # (the ground plane is an entity of its own: its link reads the engine's concrete state)
    why = _refused(monkeypatch, lambda e: e.scene.plane.get_link("plane").get_pos()[:, 2] + _pos(e)[:, 2])
    assert "concrete tensor" in why and "further entity" in why, why


# ------------------------------------------------------------------------------------------------
# the IR against the Python functions, over steps with resets
# ------------------------------------------------------------------------------------------------
_DT = {expr.F32: torch.float32, expr.I32: torch.int32, expr.BOOL: torch.bool}


def evaluate(prog, source, state=None, params=None):
    """torch-CPU evaluation of a Program: the evaluator of tests/test_user_terms.py with link sources,
    broadcasting and constant index lists; `source(attr)` gives a source's (N, ...) tensor, `state` (slot ->
    tensor) gets the program's writes."""
    vals = []
    for n in prog.nodes:
        a = [vals[i] for i in n.args]
        op = n.op
        if op == "src":
            v = state[n.attr[1]].clone() if n.attr[0] == "state" else source(n.attr).reshape((N,) + n.shape)
        elif op == "param":
            v = params[prog.params[n.attr]]
        elif op == "const":
            v = n.attr
        elif op == "constvec":
            v = torch.tensor(n.attr, dtype=_DT[n.dtype])
        elif op == "full":
            v = torch.full((N,) + n.shape, n.attr, dtype=_DT[n.dtype])
        elif op == "cast":
            v = a[0].to(_DT[n.dtype]) if torch.is_tensor(a[0]) else {"f32": float, "i32": int, "bool": bool}[n.dtype](a[0])
        elif op == "neg":
            v = -a[0]
        elif op == "not":
            v = ~a[0]
        elif op in ("abs", "square", "sqrt", "exp", "log", "sin", "cos", "tanh"):
            v = getattr(torch, op)(a[0])
        elif op == "where":
            v = torch.where(*[x if torch.is_tensor(x) else torch.tensor(x) for x in a])
        elif op == "index":
            v = a[0][(slice(None),) + tuple(s if isinstance(s, int) else list(s[1:]) if s[0] == "list" else slice(*s)
                                            for s in n.attr)]
        elif op in ("sum", "mean", "any", "all", "amax", "amin"):
            v = getattr(torch, op)(a[0], dim=n.attr + 1)
        elif op == "norm":
            v = torch.norm(a[0], dim=n.attr + 1)
        elif op == "reshape":
            v = a[0].reshape((N,) + n.shape)
        elif op in ("stack", "cat"):
            v = torch.stack(a, dim=-1) if op == "stack" else torch.cat(a, dim=-1)
        elif op == "clamp_lo":
            v = torch.clamp(a[0], min=a[1])
        elif op == "clamp_hi":
            v = torch.clamp(a[0], max=a[1])
        elif op in ("minimum", "maximum"):
            v = getattr(torch, op)(a[0], a[1] if torch.is_tensor(a[1]) else torch.tensor(a[1], dtype=a[0].dtype))
        else:
            fn = {"add": torch.add, "sub": torch.sub, "mul": torch.mul, "div": torch.div, "mod": torch.remainder,
                  "lt": torch.lt, "le": torch.le, "gt": torch.gt, "ge": torch.ge, "eq": torch.eq, "ne": torch.ne,
                  "and": torch.logical_and, "or": torch.logical_or}[op]
            x, y = a
            v = fn(x, y) if torch.is_tensor(x) else fn(torch.tensor(x), y)
        vals.append(v)
    for slot, i in prog.writes:
        state[slot] = torch.as_tensor(vals[i], dtype=state[slot].dtype).expand_as(state[slot]).clone()
    return vals[prog.out]


def _engine_sources(fused):
    """Sources as the kernel sees them: the engine's getters, one gather per link array of the layout."""
    robot, cm = fused.primary_entity, fused.contacts[0]
    arrays = {what: (robot.get_links_pos if what == "pos" else robot.get_links_vel)(links_idx_local=list(ids))
              for what, (_, ids) in fused._link_layout.items()}

    def source(attr):
        if attr[0] in ("link_pos", "link_vel"):
            ids, U = attr[1], attr[3]
            return arrays[attr[0][5:]][:, [U.index(i) for i in ids], :]
        return {"pos": robot.get_pos, "vel": robot.get_vel, "contacts": lambda: cm.contacts}[attr[0]]()
    return source


def test_ir_reproduces_the_python_functions_over_steps_with_resets(cpu_device, jit, monkeypatch):
    env = dry_env(link_terms.link_terms(), monkeypatch)
    fused = env._fused
    scene, cm = env.scene, fused.contacts[0]
    inst = fused.reward.cfg["swing_peak"].fn
    twin = type(inst).__new__(type(inst))
    twin.__dict__.update({k: v.clone() if torch.is_tensor(v) else v for k, v in vars(inst).items()})
    (slot, *_), = fused.stateful[("reward", "swing_peak")]["attrs"].values()
    state = {slot: inst.peak.clone()}
    gen = torch.Generator().manual_seed(3)
    fired = 0
    for step in range(12):
        scene.step()
        cm.contacts.copy_(torch.randn(cm.contacts.shape, generator=gen) * 3)
        if step % 3 == 2:  # a reset: the engine moves the links of some envs, the term's state rows restart
            idx = torch.randperm(N, generator=gen)[:N // 4]
            scene.state["links_pos"][idx] = 0.0
            twin.peak[idx] = 0.0
            state[slot][idx] = 0.0
        source = _engine_sources(fused)
        for (kind, name), (prog, *_) in fused.user_terms.items():
            item = (fused.reward.cfg if kind == "reward" else fused.termination.term_cfg)[name]
            fn = twin if name == "swing_peak" else item.fn
            want = (type(fn).__call__(fn, env, **item.params) if fn is twin else fn(env, **item.params))
            got = evaluate(prog, source, state if name == "swing_peak" else None, dict(item.params or {}))
            want = want.float() if kind == "reward" else want
            assert got.dtype == want.dtype and torch.equal(got, want), (name, step)
            fired += int(want.sum()) if kind == "termination" else 0
        assert torch.equal(state[slot], twin.peak), step
        for (g, name), (prog, *_) in fused.user_obs.items():
            want = fused.observations[g].cfg[name].fn(env=env).reshape(N, -1).float()
            assert torch.equal(evaluate(prog, source), want), (name, step)
    assert fired > 0  # the termination is exercised


# ------------------------------------------------------------------------------------------------
# broadcasting and constant index lists at edge values
# ------------------------------------------------------------------------------------------------
def _grid(seed):
    rng = np.random.default_rng(seed)
    pool = np.concatenate([EDGE_F32, rng.standard_normal(32).astype(np.float32)])
    return torch.from_numpy(pool[rng.integers(0, len(pool), (N, 24))])


BROADCAST = [  # (name, function of a (N, 24) input x): observation terms, so reshape builds the shapes
    ("k_1", lambda x: x[:, 0:4] - x[:, 4:5]),
    ("k3_13", lambda x: x[:, 0:12].reshape(N, 4, 3) * x[:, 12:15].reshape(N, 1, 3)),
    ("k3_3", lambda x: x[:, 0:12].reshape(N, 4, 3) + torch.tensor([1.0, -0.0, 2.5])),
    ("k1_13", lambda x: x[:, 0:4].reshape(N, 4, 1) / x[:, 4:7].reshape(N, 1, 3)),
    ("k1_1k", lambda x: torch.maximum(x[:, 0:4].reshape(N, 4, 1), x[:, 4:8].reshape(N, 1, 4)).flatten(1)),
    ("where", lambda x: torch.where(x[:, 0:4].reshape(N, 4, 1) > 0, x[:, 4:7].reshape(N, 1, 3), x[:, 7:8].reshape(N, 1, 1))),
    ("clamp", lambda x: torch.clamp(x[:, 0:6].reshape(N, 2, 3), min=x[:, 6:9].reshape(N, 1, 3))),
    ("cmp", lambda x: (x[:, 0:6].reshape(N, 3, 2) <= x[:, 6:8].reshape(N, 1, 2)).float()),
    ("list", lambda x: x[:, [5, 0, 5, 23]]),
    ("list_neg", lambda x: x[:, [-1, 2]] * 2.0),
    ("tensor_3d", lambda x: x[:, 0:12].reshape(N, 4, 3)[:, torch.tensor([3, 1, 3])]),
    ("tensor_0d", lambda x: x[:, 0:12].reshape(N, 4, 3)[:, torch.tensor(2)]),
    ("list_mid", lambda x: x[:, 0:12].reshape(N, 2, 6)[:, :, [4, 0]]),
    ("list_int", lambda x: x[:, 0:12].reshape(N, 4, 3)[:, [0, 2], 1]),
    ("int_list", lambda x: x[:, 0:24].reshape(N, 2, 4, 3)[:, 1, :, [2, 0]]),
    ("ellipsis", lambda x: x[:, 0:12].reshape(N, 4, 3)[..., [1]] - x[:, 12:16].reshape(N, 4, 1)),
    ("list_none", lambda x: x[:, [1, 3]][:, None, :] + x[:, 4:7].reshape(N, 3, 1)),
]


def _trace_obs(fn):
    tr = expr.Tracer(N, "observation")
    out = fn(tr.source(("actions",), (24,), expr.F32))
    return expr._term_program(tr, "observation", "probe", out)


@pytest.mark.parametrize("name,fn", BROADCAST, ids=[b[0] for b in BROADCAST])
def test_broadcasting_and_index_lists_match_torch_cpu_bit_for_bit(name, fn):
    prog = _trace_obs(fn)
    for seed in range(4):
        x = _grid(seed)
        want = fn(x).reshape(N, -1).float()
        got = evaluate(prog, lambda attr: x)
        assert got.shape == want.shape
        assert torch.equal(got.view(torch.int32), want.view(torch.int32)), (name, seed)


@pytest.mark.parametrize("name,fn", BROADCAST, ids=[b[0] for b in BROADCAST])
def test_generated_code_reads_the_broadcast_elements(name, fn):
    """The device function's element expressions, evaluated as Python over the input row, give torch's values."""
    prog = _trace_obs(fn)
    body = expr.function_body(prog, "f", glob=True)
    x = _grid(0)
    want = fn(x).reshape(N, -1).float()
    helpers = {"sub": lambda a, b: np.float32(a) - np.float32(b), "add": lambda a, b: np.float32(a) + np.float32(b),
               "mul": lambda a, b: np.float32(a) * np.float32(b), "fdiv": lambda a, b: np.float32(a) / np.float32(b),
               "gfb_user_max": lambda a, b: np.float32(np.nan) if np.isnan(a) or np.isnan(b) else max(a, b),
               "gfb_user_clamp_lo": lambda a, b: np.float32(np.nan) if np.isnan(a) or np.isnan(b) else max(a, b),
               "__int2float_rn": np.float32}
    with np.errstate(all="ignore"):
        for e in range(0, N, 7):
            env = dict(helpers, row=x[e].numpy())
            for line in body.splitlines():
                m = re.match(r"\s*const (?:float|bool|int) (v\d+_\d+) = (.*);$", line)
                if m:
                    expr_ = re.sub(r"v0p\[(\d+)\]", r"row[\1]", m.group(2))
                    expr_ = re.sub(r"(-?0x[0-9a-fp.+-]+)f", r"np.float32(float.fromhex('\1'))", expr_)
                    expr_ = re.sub(r"\b(\d+\.\d+)f", r"np.float32(\1)", expr_)
                    expr_ = re.sub(r"\((\S+) \? (.+) : (.+)\)$", r"(\2 if \1 else \3)", expr_)
                    env[m.group(1)] = eval(expr_, {"np": np}, env)
                m = re.match(r"\s*out\[(\d+)\] = (\S+);$", line)
                if m:
                    got = np.float32(eval(re.sub(r"v0p\[(\d+)\]", r"row[\1]", m.group(2)), {"np": np}, env))
                    ref = np.float32(want[e, int(m.group(1))].item())
                    assert got.tobytes() == ref.tobytes() or (np.isnan(got) and np.isnan(ref)), (name, e, line)


# ------------------------------------------------------------------------------------------------
# device code
# ------------------------------------------------------------------------------------------------
@pytest.mark.skipif(NVCC is None, reason="nvcc not available")
def test_generated_header_compiles_for_sm100a_without_spills(cpu_device, jit, monkeypatch):
    from genesis_forge_b200 import spec

    env = dry_env(link_terms.link_terms(), monkeypatch, n=256)
    todo = spec.collect(env, rng_modes=(1,))
    assert len(todo) == 1
    text = next(iter(todo.values()))
    assert "GFB_B_USER_STATE0 + 7]" in text and "GFB_B_USER_STATE0 + 6]" in text
    assert "#define GFB_SPEC_STATE_SLOTS 193u" in text
    with tempfile.TemporaryDirectory() as d:
        header = os.path.join(d, "spec.h")
        Path(header).write_text(text)
        out = subprocess.run([NVCC, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-Xptxas", "-v",
                              "-Xcompiler", "-fPIC", "-shared", "--fmad=false", f'-DGFB_SPEC_HEADER="{header}"',
                              str(spec.PKG / "csrc" / "spec_kernel.cu"), "-o", os.path.join(d, "spec.so")],
                             capture_output=True, text=True)
        assert out.returncode == 0, out.stderr
        lib = __import__("ctypes").CDLL(os.path.join(d, "spec.so"))
        lib.gfb_spec_state_slots.restype = __import__("ctypes").c_uint32
        assert lib.gfb_spec_state_slots() == 193
    post = [ln for ln in out.stderr.splitlines() if "spill" in ln]
    assert post and all("0 bytes spill stores, 0 bytes spill loads" in ln for ln in post), out.stderr
