"""
Host side of the lowered class-style user terms (ManagedEnvironment.fuse_stateful_terms, configs/stateful_terms.py):
tracing of per-env state, the IR with its state writes against the Python instances over several steps, the
refusals, re-tracing on edits, rebinding / demotion and the generated device code.  No GPU needed.
"""
import os
import shutil
import subprocess
import types

import pytest
import torch

import genesis_forge_b200 as gfb
from configs import specs, stateful_terms
from configs.env_builder import build_env, dropin_namespace
from genesis_forge_b200 import expr
from genesis_forge_b200.managed_env import ManagedEnvironment
from genesis_forge_b200.managers.config import MdpFnClass

N = 64
NVCC = shutil.which("nvcc") or ("/usr/local/cuda/bin/nvcc" if os.path.exists("/usr/local/cuda/bin/nvcc") else None)


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


def dry_env(spec, stateful: bool, monkeypatch, n=N, user_terms=False):
    monkeypatch.setattr(ManagedEnvironment, "fuse_stateful_terms", stateful)
    monkeypatch.setattr(ManagedEnvironment, "fuse_user_terms", user_terms)
    env = build_env(spec, dropin_namespace(), n, torch.device("cpu"))
    env._dry_run = True
    env.build()
    env._fused._set_program()
    return env


_STATEFUL = ["joint_accel", "action_jerk", "speed_ema", "tilt_latch", "stuck"]


def test_workload_a_lowers_completely_and_runs_as_one_launch(cpu_device, jit, monkeypatch):
    fused = dry_env(stateful_terms.stateful_terms(), True, monkeypatch)._fused
    assert not fused.user_term_refusals and not fused.external_rows
    assert not fused.split_mode and fused.split_plan == []
    assert sorted(n for _, n in fused.user_terms) == sorted(_STATEFUL)
    P, K = fused.program.head, gfb._native.K
    assert [P.reward[r].op for r in range(P.n_reward)].count(K["GFB_R_USER"]) == 4
    assert [P.termination[t].op for t in range(P.n_termination)].count(K["GFB_T_USER"]) == 1
    slots = sorted(s for b in fused.stateful.values() for s in b["tensors"])
    assert slots == list(range(7))  # joint_accel: prev_vel + gain; action_jerk: prev1 + prev2; 3 more
    for slot in slots:
        assert fused.buffers.buf[K["GFB_B_USER_STATE0"] + slot]
    jerk = fused.user_terms[("reward", "action_jerk")][0]
    assert jerk.first is not None and fused._lazy_started[("reward", "action_jerk")] is False
    row = list(fused.reward.cfg).index("action_jerk")
    assert P.reward[row].p[0] == 0.0  # the first-call program until the kernel has evaluated the term
    gain = fused.user_terms[("reward", "joint_accel")][0]
    assert {s for s, _ in gain.writes} == {gain.bindings["prev_vel"][0]}  # the gain is read only


def test_switch_off_keeps_the_plans_and_the_refusal(cpu_device, jit, monkeypatch):
    off = dry_env(stateful_terms.stateful_terms(), False, monkeypatch, user_terms=True)._fused
    assert off.split_mode and not off.user_terms and not off.stateful
    assert sorted(n for _, n, _ in off.external_rows) == sorted(_STATEFUL)
    assert all("class-style" in off.user_term_refusals[(k, n)] for k, n, _ in off.external_rows)
    K = gfb._native.K
    assert not any(off.buffers.buf[K["GFB_B_USER_STATE0"] + s] for s in range(8))
    plain = dry_env(specs.command_direction(), True, monkeypatch)._fused
    ref = dry_env(specs.command_direction(), False, monkeypatch)._fused
    assert bytes(plain.program) == bytes(ref.program)


def test_stock_body_acceleration_keeps_its_opcode(cpu_device, jit, monkeypatch):
    spec = specs.command_direction()
    spec["rewards"] = dict(spec["rewards"], body_acc={"fn": "body_acceleration_exp", "weight": -0.1,
                                                      "params": {"entity_manager": specs._EM}})
    fused = dry_env(spec, True, monkeypatch)._fused
    K = gfb._native.K
    row = list(fused.reward.cfg).index("body_acc")
    assert fused.program.head.reward[row].op == K["GFB_R_BODY_ACC_EXP"] and not fused.user_terms


# ------------------------------------------------------------------------------------------------
# the IR with its state against the Python instances
# ------------------------------------------------------------------------------------------------
_DT = {expr.F32: torch.float32, expr.I32: torch.int32, expr.BOOL: torch.bool}


def evaluate(prog, sources: dict, state: dict):
    """torch-CPU evaluation of a Program; `state` (slot -> (N, *s) tensor) gets its writes."""
    vals = []
    for n in prog.nodes:
        a = [vals[i] for i in n.args]
        op = n.op
        if op == "src":
            v = state[n.attr[1]].clone() if n.attr[0] == "state" else sources[n.attr]
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
            v = a[0][(slice(None),) + tuple(s if isinstance(s, int) else slice(*s) for s in n.attr)]
        elif op in ("sum", "mean", "any", "all", "amax", "amin"):
            v = getattr(torch, op)(a[0], dim=n.attr + 1)
        elif op == "norm":
            v = torch.norm(a[0], dim=n.attr + 1)
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


def _fake_env(gen, step, dt=0.02):
    f = lambda *s: torch.randn(*s, generator=gen)  # noqa: E731
    src = {("dof_vel",): f(N, 12) * 3, ("actions",): f(N, 12), ("lin_vel_b",): f(N, 3) * 0.1,
           ("gravity_b",): f(N, 3) * 0.1 - torch.tensor([0.0, 0.0, 0.97]), ("command", 0): f(N, 3),
           ("episode_length",): ((torch.arange(N, dtype=torch.int32) + step) % 7 + 1).to(torch.int32)}
    env = types.SimpleNamespace(
        num_envs=N, dt=dt, actions=src[("actions",)], episode_length=src[("episode_length",)],
        action_manager=types.SimpleNamespace(get_dofs_velocity=lambda: src[("dof_vel",)]),
        robot_manager=types.SimpleNamespace(get_linear_velocity=lambda: src[("lin_vel_b",)],
                                            get_projected_gravity=lambda: src[("gravity_b",)]),
        velocity_command=types.SimpleNamespace(command=src[("command", 0)]))
    return src, env


def test_ir_reproduces_the_instances_over_ten_steps(cpu_device, jit, monkeypatch):
    fused = dry_env(stateful_terms.stateful_terms(), True, monkeypatch)._fused
    gen = torch.Generator().manual_seed(11)
    _, env0 = _fake_env(gen, 0)
    refs, states = {}, {}
    for (kind, name), (prog, *_) in fused.user_terms.items():
        item = (fused.reward.cfg if kind == "reward" else fused.termination.term_cfg)[name]
        refs[name] = (type(item.fn)(env0, **item.params), dict(item.params))
        states[name] = {slot: t.clone() for slot, t in fused.stateful[(kind, name)]["tensors"].items()}
    for step in range(10):
        src, env = _fake_env(gen, step, fused.env.dt)
        for (kind, name), (prog, *_) in fused.user_terms.items():
            inst, params = refs[name]
            want = inst(env, **params)
            use = prog.first if (prog.first is not None and step == 0) else prog
            got = evaluate(use, src, states[name])
            if kind == "reward":
                want = want.float()
            assert got.dtype == want.dtype and torch.equal(got, want), (name, step)
            for attr, (slot, *_rest) in prog.bindings.items():
                assert torch.equal(states[name][slot], getattr(inst, attr)), (name, attr, step)


# ------------------------------------------------------------------------------------------------
# refusals
# ------------------------------------------------------------------------------------------------
def _refused(monkeypatch, cls, kind="reward"):
    spec = specs.command_direction()
    table = "rewards" if kind == "reward" else "terminations"
    spec[table] = dict(spec[table], probe={"fn": cls, "weight": 1.0} if kind == "reward" else {"fn": cls})
    fused = dry_env(spec, True, monkeypatch)._fused
    assert (kind, "probe") not in fused.user_terms and not fused.stateful
    assert (kind, "probe") in {(k, n) for k, n, _ in fused.external_rows}
    return fused.user_term_refusals[(kind, "probe")]


def _state_class(init, call):
    return type("Probe", (MdpFnClass,), {"__init__": lambda self, env: (MdpFnClass.__init__(self, env), init(self, env))[0],
                                         "__call__": lambda self, env: call(self, env)})


def _rows(env, *shape, dtype=torch.float32):
    return torch.zeros((env.num_envs,) + shape, dtype=dtype)


SHARED = torch.zeros(N)


def _partial(self, env):
    self.x[:, 0] = env.actions[:, 0]
    return self.x[:, 1]


def _rebind_shape(self, env):
    self.x = env.actions
    return env.actions[:, 0]


def _calls(self, env):
    self.calls += 1
    return env.actions[:, 0]


def _const_write(self, env):
    self.k = env.actions[:, :3]
    return env.actions[:, 0]


def _many(self, env):
    out = env.actions[:, 0]
    for k in range(9):
        setattr(self, f"s{k}", out + k)
    return out


@pytest.mark.parametrize("init,call,needle", [
    (lambda s, e: setattr(s, "x", _rows(e, 2)), _partial, "partial in-place write"),
    (lambda s, e: setattr(s, "x", _rows(e)), _rebind_shape, "row shape and dtype"),
    (lambda s, e: setattr(s, "x", _rows(e, dtype=torch.int64)), lambda s, e: s.x.float(), "int64"),
    (lambda s, e: setattr(s, "k", torch.zeros(3)), _const_write, "not per-env state"),
    (lambda s, e: setattr(s, "calls", 0), _calls, "host state"),
    (lambda s, e: setattr(s, "hist", [_rows(e)]), lambda s, e: e.actions[:, 0], "container or sub-object"),
    (lambda s, e: setattr(s, "sub", types.SimpleNamespace(x=_rows(e))), lambda s, e: e.actions[:, 0],
     "container or sub-object"),
    (lambda s, e: [setattr(s, f"s{k}", _rows(e)) for k in range(9)], _many, "slots"),
    (lambda s, e: (setattr(s, "a", SHARED), setattr(s, "b", SHARED[:])), lambda s, e: s.a + s.b, "share storage"),
])
def test_refusals_keep_the_callback(init, call, needle, cpu_device, jit, monkeypatch):
    why = _refused(monkeypatch, _state_class(init, call))
    assert needle in why, why


def test_two_terms_holding_the_same_storage_are_refused(cpu_device, jit, monkeypatch):
    def init(s, e):
        s.x = SHARED

    cls = _state_class(init, lambda s, e: s.x + e.actions[:, 0])
    spec = specs.command_direction()
    spec["rewards"] = dict(spec["rewards"], one={"fn": cls, "weight": 1.0}, two={"fn": cls, "weight": 1.0})
    fused = dry_env(spec, True, monkeypatch)._fused
    assert ("reward", "one") in fused.stateful and ("reward", "two") not in fused.stateful
    assert "shares storage" in fused.user_term_refusals[("reward", "two")]


def test_observation_class_terms_stay_refused(cpu_device, jit, monkeypatch):
    fused = dry_env(stateful_terms.stateful_terms(), True, monkeypatch)._fused
    item = types.SimpleNamespace(fn=stateful_terms.speed_ema(fused.env), params={})
    with pytest.raises(expr.UnsupportedTermError, match="class-style"):
        expr.trace_term(fused, "observation", "ema", item, state=expr.StateSlots({}, [7]))


# ------------------------------------------------------------------------------------------------
# edits, rebinding, demotion
# ------------------------------------------------------------------------------------------------
def test_params_edit_reinstantiates_and_binds_the_new_tensors(cpu_device, jit, monkeypatch):
    fused = dry_env(stateful_terms.stateful_terms(), True, monkeypatch)._fused
    K = gfb._native.K
    item = fused.reward.cfg["joint_accel"]
    old, digest = item.fn, fused.user_terms[("reward", "joint_accel")][0].digest()
    item.params["scale"] = 2.0e-4  # ConfigItem._rebuild: a new instance, fresh state
    fused._set_program()
    assert item.fn is not old and fused.stateful[("reward", "joint_accel")]["inst"] is item.fn
    slot = fused.stateful[("reward", "joint_accel")]["attrs"]["prev_vel"][0]
    assert fused.buffers.buf[K["GFB_B_USER_STATE0"] + slot] == item.fn.prev_vel.data_ptr()
    assert fused.user_terms[("reward", "joint_accel")][0].digest() != digest  # the scale is a constant


def test_scalar_attribute_edit_traces_again(cpu_device, jit, monkeypatch):
    fused = dry_env(stateful_terms.stateful_terms(), True, monkeypatch)._fused
    row = list(fused.reward.cfg).index("speed_ema")
    digest = fused.program.head.reward[row].i0
    fused.reward.cfg["speed_ema"].fn.rate = 0.2
    fused._set_program()
    assert fused.program.head.reward[row].i0 == fused.user_terms[("reward", "speed_ema")][0].digest() != digest


def test_rebinding_and_demotion_hand_the_callbacks_the_state(cpu_device, jit, monkeypatch):
    fused = dry_env(stateful_terms.stateful_terms(), True, monkeypatch)._fused
    K = gfb._native.K
    ema = fused.reward.cfg["speed_ema"].fn
    slot = fused.stateful[("reward", "speed_ema")]["attrs"]["ema"][0]
    ema.ema = torch.full((N,), 0.5)  # a compatible rebinding: the slot follows it
    assert fused._check_state() is None
    assert fused.buffers.buf[K["GFB_B_USER_STATE0"] + slot] == ema.ema.data_ptr()
    jerk = fused.reward.cfg["action_jerk"].fn
    assert jerk.prev1 is None  # lazily initialised: None until the kernel has evaluated the term
    fused._after_launch_lazy = {("reward", "action_jerk")}
    fused._after_report()
    assert jerk.prev1 is fused.stateful[("reward", "action_jerk")]["tensors"][jerk_slot(fused)]
    assert fused._lazy_started[("reward", "action_jerk")]
    fused._set_program()
    assert fused.program.head.reward[list(fused.reward.cfg).index("action_jerk")].p[0] == 1.0
    prev1 = jerk.prev1
    ema.ema = torch.zeros((N, 2))  # incompatible: the lowered terms become callbacks
    why = fused._check_state()
    assert "speed_ema" in why
    fused._demote_user_terms(why)
    assert fused.split_mode and not fused.stateful and not fused.user_terms
    assert jerk.prev1 is prev1 and ema.ema.shape == (N, 2)  # what the Python __call__ continues from
    assert not any(fused.buffers.buf[K["GFB_B_USER_STATE0"] + s] for s in range(8))


def jerk_slot(fused):
    return fused.stateful[("reward", "action_jerk")]["attrs"]["prev1"][0]


@pytest.mark.skipif(NVCC is None, reason="nvcc not available")
def test_generated_header_compiles_for_sm100a_without_spills(cpu_device, monkeypatch):
    from genesis_forge_b200 import spec

    env = dry_env(stateful_terms.stateful_terms(), True, monkeypatch, n=256)
    todo = spec.collect(env, rng_modes=(0,))
    assert len(todo) == 1
    text = next(iter(todo.values()))
    assert "GFB_SPEC_USER_TERMS" in text and "#define GFB_SPEC_STATE_SLOTS 127u" in text
    key = next(iter(todo))
    header = spec.CACHE / f"spec_{key}.verbose.h"
    spec.CACHE.mkdir(exist_ok=True)
    header.write_text(text)
    try:
        out = subprocess.run([NVCC, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-Xptxas", "-v",
                              "-Xcompiler", "-fPIC", "-shared", "--fmad=false", f'-DGFB_SPEC_HEADER="{header}"',
                              str(spec.PKG / "csrc" / "spec_kernel.cu"), "-o", os.devnull],
                             capture_output=True, text=True)
    finally:
        header.unlink()
    assert out.returncode == 0, out.stderr
    post = [ln for ln in out.stderr.splitlines() if "spill" in ln]
    assert post and all("0 bytes spill stores, 0 bytes spill loads" in ln for ln in post), out.stderr


def test_workload_b_lowers_its_lazily_initialised_contact_term(cpu_device, jit, monkeypatch):
    fused = dry_env(stateful_terms.stateful_contacts(), True, monkeypatch)._fused
    assert not fused.user_term_refusals and not fused.split_mode
    prog = fused.user_terms[("reward", "contact_streak")][0]
    assert prog.first is not None and prog.bindings["streak"][1:] == ((4,), expr.F32, True)
    assert fused.reward.cfg["contact_streak"].fn.streak is None
