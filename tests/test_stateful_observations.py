"""
Host side of the lowered class-style user observation terms (ManagedEnvironment.fuse_stateful_terms,
configs/stateful_observations.py): lowering and slot binding, the IR with its state writes against the Python
instances over several observations, the refusals, group-keyed bindings, re-tracing on edits, rebinding and
demotion, the generated device code, and the unchanged device code of every table without such terms.  No
GPU needed.
"""
import concurrent.futures as cf
import hashlib
import json
import os
import re
import shutil
import subprocess
import tempfile
import types
from pathlib import Path

import pytest
import torch

import genesis_forge_b200 as gfb
from configs import specs, stateful_observations as so, stateful_terms, user_observations, user_terms
from configs.env_builder import build_env, dropin_namespace
from genesis_forge_b200 import expr
from genesis_forge_b200.managed_env import ManagedEnvironment
from genesis_forge_b200.managers.config import MdpFnClass

N = 64
NVCC = shutil.which("nvcc") or ("/usr/local/cuda/bin/nvcc" if os.path.exists("/usr/local/cuda/bin/nvcc") else None)
CUOBJDUMP = shutil.which("cuobjdump") or ("/usr/local/cuda/bin/cuobjdump"
                                          if os.path.exists("/usr/local/cuda/bin/cuobjdump") else None)
GOLDEN = Path(__file__).parent / "golden" / "spec_sass_digests.json"


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


def dry_env(spec, monkeypatch, n=N, stateful=True, **switches):
    monkeypatch.setattr(ManagedEnvironment, "fuse_stateful_terms", stateful)
    for name in ("fuse_user_terms", "fuse_user_observations"):
        monkeypatch.setattr(ManagedEnvironment, name, switches.get(name, False))
    env = build_env(spec, dropin_namespace(), n, torch.device("cpu"))
    env._dry_run = True
    env.build()
    env._fused._set_program()
    return env


def _key(group, name):
    return ("observation", name, 0 if group == "policy" else 1)


def _inst(fused, group, name):
    return fused.observations[0 if group == "policy" else 1].cfg[name].fn


def test_workload_a_lowers_completely(cpu_device, jit, monkeypatch):
    fused = dry_env(so.stateful_observations(), monkeypatch)._fused
    assert not fused.user_term_refusals and not fused.external_obs and not fused.external_rows
    assert not fused.split_mode and fused.split_plan == []
    assert sorted(fused.stateful) == sorted(_key(g, n) for g, n in so.STATE)
    slots = sorted(s for b in fused.stateful.values() for s in b["tensors"])
    assert slots == list(range(8))  # exactly the 8 slots of the ABI
    K = gfb._native.K
    for key, b in fused.stateful.items():
        for attr, (slot, *_rest) in b["attrs"].items():
            assert fused.buffers.buf[K["GFB_B_USER_STATE0"] + slot] == getattr(b["inst"], attr).data_ptr()
    for (group, name), attrs in so.STATE.items():
        prog = fused.user_obs[(_key(group, name)[2], name)][0]
        assert prog.first is None and sorted(prog.bindings) == sorted(attrs)
        written = {a for a, (slot, *_rest) in prog.bindings.items() if slot in {s for s, _ in prog.writes}}
        assert written == set(attrs) - {"freq"}, name  # the clock's frequency is read only
    P = fused.program.head
    assert P.obs_group[0].user_id == P.obs_group[1].user_id != 0
    code = fused.user_code
    assert "/* observation terms store state */" in code
    from genesis_forge_b200 import spec

    assert "#define GFB_SPEC_USER_OBS_STATE 1" in spec._user_terms_macro(code)


def test_workload_a_split_lowers_its_observation_terms_and_runs_split(cpu_device, jit, monkeypatch):
    fused = dry_env(so.stateful_observations_split(), monkeypatch)._fused
    assert fused.split_mode and [n for _, n, _ in fused.external_rows] == ["upright_bonus"]
    assert not fused.external_obs and len(fused.user_obs) == 5 and len(fused.stateful) == 5
    K = gfb._native.K
    observe = [p for cb, p, _ in fused.split_plan if p & K["GFB_PHASE_OBSERVE"]]
    assert len(observe) == 1 and not observe[0] & K["GFB_PHASE_RESET"]  # the observe-only launch stores every env


def test_switch_off_keeps_the_program_and_the_refusal(cpu_device, jit, monkeypatch):
    plain = dry_env(specs.command_direction(), monkeypatch)._fused
    ref = dry_env(specs.command_direction(), monkeypatch, stateful=False)._fused
    assert bytes(plain.program) == bytes(ref.program)
    for mk in (user_observations.user_observations_entity, stateful_terms.stateful_terms):
        on = dry_env(mk(), monkeypatch, fuse_user_observations=True)._fused
        off = dry_env(mk(), monkeypatch, fuse_user_observations=True, stateful=False)._fused
        if mk is user_observations.user_observations_entity:  # no class-style term: the same table
            assert bytes(on.program) == bytes(off.program) and on.user_code == off.user_code
    off = dry_env(so.stateful_observations(), monkeypatch, stateful=False, fuse_user_observations=True)._fused
    assert not off.user_obs and not off.stateful and len(off.external_obs) == 5
    assert all("class-style" in off.user_term_refusals[("observation", n)] for _, n in so.STATE)
    K = gfb._native.K
    assert not any(off.buffers.buf[K["GFB_B_USER_STATE0"] + s] for s in range(8))


# ------------------------------------------------------------------------------------------------
# the IR with its state against the Python instances
# ------------------------------------------------------------------------------------------------
_DT = {expr.F32: torch.float32, expr.I32: torch.int32, expr.BOOL: torch.bool}


def evaluate(prog, sources: dict, state: dict):
    """torch-CPU evaluation of an observation Program ((N, width) fp32); `state` (slot -> tensor) gets its writes."""
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
        elif op == "reshape":
            v = a[0].reshape((N,) + n.shape)
        elif op == "stack":  # (over the last dimension only)
            v = torch.stack(a, dim=-1)
        elif op == "cat":
            v = torch.cat(a, dim=-1)
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


def _fake_env(gen, step, dt):
    f = lambda *s: torch.randn(*s, generator=gen)  # noqa: E731
    src = {("dof_vel",): f(N, 12) * 3, ("targets",): f(N, 12), ("lin_vel_b",): f(N, 3) * 0.2,
           ("episode_length",): ((torch.arange(N, dtype=torch.int32) + step) % 5).to(torch.int32)}
    env = types.SimpleNamespace(
        num_envs=N, dt=dt, episode_length=src[("episode_length",)],
        action_manager=types.SimpleNamespace(get_dofs_velocity=lambda: src[("dof_vel",)],
                                             get_actions=lambda: src[("targets",)]),
        robot_manager=types.SimpleNamespace(get_linear_velocity=lambda: src[("lin_vel_b",)]))
    return src, env


def test_ir_reproduces_the_instances_over_ten_steps(cpu_device, jit, monkeypatch):
    fused = dry_env(so.stateful_observations(), monkeypatch)._fused
    gen = torch.Generator().manual_seed(11)
    refs, states = {}, {}
    for key, b in fused.stateful.items():
        inst = b["inst"]
        twin = type(inst).__new__(type(inst))  # the same state, advanced by the Python __call__
        twin.__dict__.update({k: v.clone() if torch.is_tensor(v) else v for k, v in vars(inst).items()})
        refs[key] = twin
        states[key] = {slot: t.clone() for slot, t in b["tensors"].items()}
    for step in range(10):
        src, env = _fake_env(gen, step, fused.env.dt)
        for key, twin in refs.items():
            g, name = key[2], key[1]
            item = fused.observations[g].cfg[name]
            want = type(twin).__call__(twin, env=env, **item.params).reshape(N, -1).float()
            got = evaluate(fused.user_obs[(g, name)][0], src, states[key])
            assert got.dtype == want.dtype and torch.equal(got, want), (key, step)
            for attr, (slot, *_rest) in fused.stateful[key]["attrs"].items():
                assert torch.equal(states[key][slot], getattr(twin, attr)), (key, attr, step)


# ------------------------------------------------------------------------------------------------
# refusals: the term stays a host column
# ------------------------------------------------------------------------------------------------
def _state_class(init, call):
    return type("Probe", (MdpFnClass,), {"__init__": lambda self, env: (MdpFnClass.__init__(self, env), init(self, env))[0],
                                         "__call__": lambda self, env: call(self, env)})


def _rows(env, *shape, dtype=torch.float32):
    return torch.zeros((env.num_envs,) + shape, dtype=dtype)


def _vel(env):
    return env.action_manager.get_dofs_velocity()


def _partial(self, env):
    self.x[:, 0] = _vel(env)[:, 0]
    return self.x


def _rebind_shape(self, env):  # (grows by a column every call: the build's dry run has made one)
    self.x = torch.cat([self.x, _vel(env)[:, :1]], dim=1)
    return self.x[:, :2]


def _calls(self, env):
    self.calls += 1
    return _vel(env)[:, :2]


def _refused_obs(monkeypatch, cls, spec=None, group="policy"):
    spec = spec or specs.command_direction()
    terms = dict(spec["observations"][group]["terms"], probe={"fn": cls})
    spec["observations"] = dict(spec["observations"], **{group: dict(spec["observations"][group], terms=terms)})
    fused = dry_env(spec, monkeypatch)._fused
    g = list(spec["observations"]).index(group)
    assert (g, "probe") not in fused.user_obs and ("observation", "probe", g) not in fused.stateful
    assert "probe" in [n for _, n, _, _, _ in fused.external_obs]
    return fused, fused.user_term_refusals[("observation", "probe")]


SHARED = torch.zeros(N)


@pytest.mark.parametrize("init,call,needle", [
    (lambda s, e: setattr(s, "x", _rows(e, 2)), _partial, "partial in-place write"),
    (lambda s, e: setattr(s, "x", _rows(e, 2)), _rebind_shape, "row shape and dtype"),
    (lambda s, e: setattr(s, "x", _rows(e, dtype=torch.int64)), lambda s, e: s.x.float(), "int64"),
    (lambda s, e: setattr(s, "calls", 0), _calls, "host state"),
])
def test_refusals_keep_the_host_column(init, call, needle, cpu_device, jit, monkeypatch):
    _, why = _refused_obs(monkeypatch, _state_class(init, call))
    assert needle in why, why


def test_an_attribute_still_none_is_refused(cpu_device, jit, monkeypatch):
    fused = dry_env(specs.command_direction(), monkeypatch)._fused

    def call(s, e):
        if s.x is None:
            s.x = _vel(e).clone()
        return s.x * 2.0

    inst = _state_class(lambda s, e: setattr(s, "x", None), call)(fused.env)
    item = types.SimpleNamespace(fn=inst, params={})
    with pytest.raises(expr.UnsupportedTermError, match="is None when the term is traced"):
        expr.trace_stateful(fused, "observation", "lazy", item, expr.StateSlots({}, [0]))


def test_storage_shared_with_a_reward_term_is_refused(cpu_device, jit, monkeypatch):
    spec = specs.command_direction()
    reward = _state_class(lambda s, e: setattr(s, "x", SHARED), lambda s, e: s.x + e.actions[:, 0])
    spec["rewards"] = dict(spec["rewards"], shared={"fn": reward, "weight": 1.0})
    fused, why = _refused_obs(monkeypatch, _state_class(lambda s, e: setattr(s, "y", SHARED),
                                                        lambda s, e: (s.y + _vel(e)[:, 0]).unsqueeze(1)), spec)
    assert ("reward", "shared") in fused.stateful
    assert "shares storage" in why and "reward 'shared'" in why, why


def test_a_ninth_slot_keeps_that_term_a_host_column(cpu_device, jit, monkeypatch):
    spec = so.stateful_observations()

    def call(s, e):
        s.z = s.z + _vel(e)[:, 0]
        return s.z.unsqueeze(1)

    fused, why = _refused_obs(monkeypatch, _state_class(lambda s, e: setattr(s, "z", _rows(e)), call), spec, "history")
    assert "slots" in why, why
    assert len(fused.stateful) == 5 and len(fused.user_obs) == 5  # the others stay lowered


# ------------------------------------------------------------------------------------------------
# group-keyed bindings, edits, rebinding, demotion
# ------------------------------------------------------------------------------------------------
def test_the_same_class_in_two_groups_is_two_bindings(cpu_device, jit, monkeypatch):
    fused = dry_env(so.stateful_observations(), monkeypatch)._fused
    a, b = fused.stateful[_key("policy", "gait_clock")], fused.stateful[_key("history", "gait_clock")]
    assert a["inst"] is not b["inst"] and not set(a["tensors"]) & set(b["tensors"])
    assert a["attrs"]["phase"][0] != b["attrs"]["phase"][0]


def test_params_and_scalar_edits_trace_again(cpu_device, jit, monkeypatch):
    fused = dry_env(so.stateful_observations(), monkeypatch)._fused
    K = gfb._native.K
    om = fused.observations[1]
    old, uid = om.cfg["gait_clock"].fn, fused._obs_user_id
    om.cfg["gait_clock"].params["seed"] = 9  # ConfigItem._rebuild: a new instance with its own tensors
    new = om.cfg["gait_clock"].fn
    assert new is not old
    assert fused._check_state() is None
    b = fused.stateful[_key("history", "gait_clock")]
    assert b["inst"] is new
    for attr, (slot, *_rest) in b["attrs"].items():
        assert fused.buffers.buf[K["GFB_B_USER_STATE0"] + slot] == getattr(new, attr).data_ptr()
    fused._program_pushed = False
    fused._set_program()
    assert fused._obs_user_id == uid  # the seed only changes the tensors: the same program
    filt = _inst(fused, "policy", "joint_vel_filt")
    filt.alpha = 0.5  # a trace constant
    fused._program_pushed = False
    fused._set_program()
    assert fused._obs_user_id != uid and not fused.split_mode


def test_a_params_edit_to_an_uninitialised_instance_demotes(cpu_device, jit, monkeypatch):
    fused = dry_env(so.stateful_observations(), monkeypatch)._fused
    om = fused.observations[0]
    om.cfg["joint_vel_filt"].params["alpha"] = 0.5  # the new instance's filter is None until it is called
    why = fused._check_state()
    assert why is not None and "None" in why, why
    fused._demote_user_terms(why)
    assert fused.split_mode and not fused.stateful and not fused.user_obs and len(fused.external_obs) == 5
    assert om.cfg["joint_vel_filt"].fn.filt is None  # the Python __call__ initialises it


def test_rebinding_and_demotion_hand_the_host_columns_the_state(cpu_device, jit, monkeypatch):
    fused = dry_env(so.stateful_observations(), monkeypatch)._fused
    K = gfb._native.K
    clock = _inst(fused, "policy", "gait_clock")
    slot = fused.stateful[_key("policy", "gait_clock")]["attrs"]["phase"][0]
    clock.phase = torch.full((N,), 0.25)  # a compatible rebinding: the slot follows it
    assert fused._check_state() is None
    assert fused.buffers.buf[K["GFB_B_USER_STATE0"] + slot] == clock.phase.data_ptr()
    hist = _inst(fused, "policy", "action_history")
    prev1 = hist.prev1
    counter = _inst(fused, "policy", "still_steps")
    counter.count = counter.count.to(torch.int64)  # incompatible: the lowered terms become host columns
    fused.width_probe = True  # (a dry run: the getters return zeros of their shape)
    fused.evaluate_external_obs()  # (checked before the host columns of an observation are evaluated)
    assert fused.split_mode and not fused.stateful and not fused.user_obs
    assert "still_steps" in fused.user_term_refusals[("observation", "still_steps")]
    assert hist.prev1 is not prev1 and clock.phase.shape == (N,)  # the host columns ran once, from that state
    assert not any(fused.buffers.buf[K["GFB_B_USER_STATE0"] + s] for s in range(8))


# ------------------------------------------------------------------------------------------------
# device code
# ------------------------------------------------------------------------------------------------
def _nvcc(text: str, out: str, *extra) -> subprocess.CompletedProcess:
    from genesis_forge_b200 import spec

    with tempfile.TemporaryDirectory() as d:
        header = os.path.join(d, "spec.h")
        Path(header).write_text(text)
        return subprocess.run([NVCC, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", *extra,
                               "-Xcompiler", "-fPIC", "-shared", "--fmad=false", f'-DGFB_SPEC_HEADER="{header}"',
                               str(spec.PKG / "csrc" / "spec_kernel.cu"), "-o", out], capture_output=True, text=True)


@pytest.mark.skipif(NVCC is None, reason="nvcc not available")
@pytest.mark.parametrize("mk", [so.stateful_observations, so.stateful_contact_observations])
def test_generated_header_compiles_for_sm100a_without_spills(mk, cpu_device, jit, monkeypatch):
    from genesis_forge_b200 import spec

    env = dry_env(mk(), monkeypatch, n=256)
    todo = spec.collect(env, rng_modes=(1,))
    assert len(todo) == 1
    text = next(iter(todo.values()))
    assert "#define GFB_SPEC_USER_OBS_STATE 1" in text and "GFB_SPEC_STATE_SLOTS" in text
    out = _nvcc(text, os.devnull, "-Xptxas", "-v")
    assert out.returncode == 0, out.stderr
    post = [ln for ln in out.stderr.splitlines() if "spill" in ln]
    assert post and all("0 bytes spill stores, 0 bytes spill loads" in ln for ln in post), out.stderr


# tables without class-style observation terms: their specialisations (production Philox draws, as bench.py
# runs them) compile to the instructions recorded in tests/golden/spec_sass_digests.json
SASS_TABLES = {
    "command_direction": (specs.command_direction, {}),
    "user_terms": (user_terms.user_terms, {"fuse_user_terms": True}),
    "user_observations": (user_observations.user_observations, {"fuse_user_observations": True}),
    "user_observations_entity": (user_observations.user_observations_entity, {"fuse_user_observations": True}),
    "stateful_terms": (stateful_terms.stateful_terms, {"fuse_stateful_terms": True}),
}


def _sass_digest(text: str) -> str:
    with tempfile.TemporaryDirectory() as d:
        so_path = os.path.join(d, "spec.so")
        out = _nvcc(text, so_path)
        assert out.returncode == 0, out.stderr
        sass = subprocess.run([CUOBJDUMP, "-sass", so_path], check=True, capture_output=True, text=True).stdout
    skip = ("Fatbin", "code for", "arch =", "code version", "host =", "compile_size", "identifier")
    # (the anonymous namespace's mangled name carries a hash of the source path)
    lines = [re.sub(r"_GLOBAL__N__[0-9a-f]+_", "_GLOBAL__N__", ln) for ln in sass.splitlines()
             if ln.strip() and not ln.strip().startswith(skip)]
    return hashlib.sha1("\n".join(lines).encode()).hexdigest()


@pytest.mark.skipif(NVCC is None or CUOBJDUMP is None, reason="nvcc / cuobjdump not available")
def test_existing_specialisations_keep_their_sass(cpu_device, jit, monkeypatch):
    from genesis_forge_b200 import spec

    want = json.loads(GOLDEN.read_text())
    todo = {}
    for name, (mk, switches) in SASS_TABLES.items():
        switches = dict(switches)
        env = dry_env(mk(), monkeypatch, n=256, stateful=switches.pop("fuse_stateful_terms", False), **switches)
        for i, text in enumerate(sorted(spec.collect(env, rng_modes=(1,)).values())):
            assert "GFB_SPEC_USER_OBS_STATE" not in text
            todo[f"{name}#{i}"] = text
    assert sorted(todo) == sorted(want)
    with cf.ThreadPoolExecutor(max_workers=len(todo)) as pool:
        got = dict(zip(todo, pool.map(_sass_digest, todo.values())))
    assert got == want
