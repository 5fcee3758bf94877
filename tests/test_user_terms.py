"""
Host side of the lowered user-defined terms (genesis_forge_b200/expr.py, ManagedEnvironment.fuse_user_terms):
tracing, the IR against the Python functions it came from, refusals, the lowering decision and the
generated device code.  No GPU needed.
"""
import shutil
import types

import pytest
import torch

import genesis_forge_b200 as gfb
from configs import specs, user_terms
from configs.env_builder import build_env, dropin_namespace
from genesis_forge_b200 import expr
from genesis_forge_b200.managed_env import ManagedEnvironment

N = 64


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


def dry_env(spec, fuse: bool, monkeypatch, n=N):
    monkeypatch.setattr(ManagedEnvironment, "fuse_user_terms", fuse)
    env = build_env(spec, dropin_namespace(), n, torch.device("cpu"))
    env._dry_run = True
    env.build()
    env._fused._set_program()
    return env


# ------------------------------------------------------------------------------------------------
# torch-CPU evaluator of the IR (test side)
# ------------------------------------------------------------------------------------------------
_TORCH_DT = {expr.F32: torch.float32, expr.I32: torch.int32, expr.BOOL: torch.bool}


def evaluate(prog: expr.Program, sources: dict, params: dict):
    vals = []
    for n in prog.nodes:
        a = [vals[i] for i in n.args]
        op = n.op
        if op == "src":
            v = sources[n.attr]
        elif op == "param":
            v = params[prog.params[n.attr]]
        elif op == "const":
            v = n.attr
        elif op == "constvec":
            v = torch.tensor(n.attr, dtype=_TORCH_DT[n.dtype])
        elif op == "cast":
            v = a[0].to(_TORCH_DT[n.dtype]) if torch.is_tensor(a[0]) else {"f32": float, "i32": int, "bool": bool}[n.dtype](a[0])
        elif op in ("neg",):
            v = -a[0]
        elif op == "not":
            v = ~a[0]
        elif op in ("abs", "square", "sqrt", "exp", "log", "sin", "cos", "tanh"):
            v = getattr(torch, op)(a[0])
        elif op == "where":
            v = torch.where(*a)
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
            other = a[1] if torch.is_tensor(a[1]) else torch.tensor(a[1], dtype=a[0].dtype)
            v = getattr(torch, op)(a[0], other)
        else:
            fn = {"add": torch.add, "sub": torch.sub, "mul": torch.mul, "div": torch.div, "mod": torch.remainder,
                  "lt": torch.lt, "le": torch.le, "gt": torch.gt, "ge": torch.ge, "eq": torch.eq, "ne": torch.ne,
                  "and": torch.logical_and, "or": torch.logical_or}[op]
            x, y = a
            v = fn(x, y) if torch.is_tensor(x) else fn(torch.tensor(x), y)
        vals.append(v)
    return vals[prog.out]


def _random_state(gen, D=12, L=4):
    """Random sources, and a stand-in environment exposing the same values through the user API."""
    f = lambda *s: torch.randn(*s, generator=gen) * 2  # noqa: E731
    src = {
        ("pos",): f(N, 3) * 5, ("quat",): f(N, 4), ("vel",): f(N, 3), ("ang",): f(N, 3).abs(),
        ("actions",): f(N, D), ("last_actions",): f(N, D), ("command", 0): f(N, 3),
        ("contacts", 0): f(N, L, 3) * 10, ("air", 0, 0): f(N, L).abs() * 0.3,
        ("episode_length",): torch.randint(0, 200, (N,), generator=gen, dtype=torch.int32),
        ("max_episode_length",): torch.randint(900, 1100, (N,), generator=gen, dtype=torch.int32),
        ("terminated",): torch.rand(N, generator=gen) < 0.2, ("truncated",): torch.rand(N, generator=gen) < 0.1,
    }
    src.update({("lin_vel_b",): f(N, 3), ("ang_vel_b",): f(N, 3), ("gravity_b",): f(N, 3) * 0.3,
                ("dof_pos",): f(N, D), ("dof_vel",): f(N, D), ("targets",): f(N, D)})
    robot = types.SimpleNamespace(get_pos=lambda: src[("pos",)], get_quat=lambda: src[("quat",)],
                                  get_vel=lambda: src[("vel",)], get_ang=lambda: src[("ang",)])
    robot_manager = types.SimpleNamespace(
        get_linear_velocity=lambda: src[("lin_vel_b",)], get_angular_velocity=lambda: src[("ang_vel_b",)],
        get_projected_gravity=lambda: src[("gravity_b",)], base_pos=src[("pos",)], base_quat=src[("quat",)])
    action_manager = types.SimpleNamespace(get_dofs_position=lambda: src[("dof_pos",)],
                                           get_dofs_velocity=lambda: src[("dof_vel",)],
                                           get_actions=lambda: src[("targets",)])
    env = types.SimpleNamespace(
        robot_manager=robot_manager, action_manager=action_manager,
        robot=robot, actions=src[("actions",)], last_actions=src[("last_actions",)],
        episode_length=src[("episode_length",)], max_episode_length=src[("max_episode_length",)],
        velocity_command=types.SimpleNamespace(command=src[("command", 0)]),
        foot_contact_manager=types.SimpleNamespace(contacts=src[("contacts", 0)], last_air_time=src[("air", 0, 0)]),
        extras={"terminations": src[("terminated",)], "time_outs": src[("truncated",)]},
    )
    return src, env


def test_workload_lowers_completely_and_runs_as_one_launch(cpu_device, jit, monkeypatch):
    env = dry_env(user_terms.user_terms(), True, monkeypatch)
    fused = env._fused
    assert not fused.user_term_refusals and not fused.external_rows
    assert not fused.split_mode and fused.split_plan == []
    assert len(fused.user_terms) == 11
    P, K = fused.program.head, gfb._native.K
    r_ops = [P.reward[r].op for r in range(P.n_reward)]
    t_ops = [P.termination[t].op for t in range(P.n_termination)]
    assert r_ops.count(K["GFB_R_USER"]) == 8 and t_ops.count(K["GFB_T_USER"]) == 3


def test_the_two_workloads_cover_every_source_and_op(cpu_device, jit, monkeypatch):
    nodes = []
    for spec in (user_terms.user_terms(), user_terms.user_terms_entity()):
        fused = dry_env(spec, True, monkeypatch)._fused
        assert not fused.user_term_refusals and not fused.split_mode
        nodes += [n for entry in fused.user_terms.values() for n in entry[0].nodes]
    seen_src = {n.attr[0] for n in nodes if n.op == "src"}
    assert seen_src == {"pos", "quat", "vel", "ang", "lin_vel_b", "ang_vel_b", "gravity_b", "dof_pos", "dof_vel",
                        "targets", "actions", "last_actions", "command", "contacts", "air", "episode_length",
                        "max_episode_length", "terminated", "truncated"}
    ops = {n.op for n in nodes}
    device_ops = {"add", "sub", "mul", "div", "mod", "neg", "not", "abs", "square", "sqrt", "exp", "log", "sin",
                  "cos", "tanh", "clamp_lo", "clamp_hi", "minimum", "maximum", "where", "lt", "le", "gt", "ge", "eq",
                  "ne", "and", "or", "cast", "index", "sum", "mean", "any", "all", "amax", "amin", "norm", "src",
                  "param", "const", "constvec"}
    assert ops == device_ops


def test_switch_off_keeps_todays_plans(cpu_device, jit, monkeypatch):
    K = gfb._native.K
    head, term, rew, reset, obs = (K["GFB_PHASE_ENTITY"] | K["GFB_PHASE_CONTACT"], K["GFB_PHASE_TERMINATION"],
                                   K["GFB_PHASE_REWARD"] | K["GFB_PHASE_COMMAND"], K["GFB_PHASE_RESET"],
                                   K["GFB_PHASE_OBSERVE"])
    want = {
        "user_terms": [(None, head, False), ("termination", term, False), ("reward", rew | reset, True),
                       ("observe", obs, False)],
        "custom_terms": [(None, head, False), ("termination", term, False), ("reward", rew, False),
                         ("commands", reset, True), ("observe", obs, False)],
        "gait_trainer": [(None, head | term, False), ("reward", rew, False), ("commands", reset, True),
                         ("observe", obs, False)],
    }
    for spec in (user_terms.user_terms(), specs.get("custom_terms"), specs.get("gait_trainer")):
        fused = dry_env(spec, False, monkeypatch)._fused
        assert not fused.user_terms and fused.split_mode
        assert [tuple(p) for p in fused.split_plan] == want[spec["name"]], spec["name"]
    env = dry_env(user_terms.user_terms(), False, monkeypatch)
    assert [name for _, name, _ in env._fused.external_rows] == [
        "contact_z", "level_speed", "action_excess", "clock", "air_time", "smoothness", "progress", "outcome",
        "wandered_off", "slow_start", "dropped"]


def test_custom_terms_keep_only_the_wave_and_clock_callbacks(cpu_device, jit, monkeypatch):
    off = dry_env(specs.get("custom_terms"), False, monkeypatch)._fused
    on = dry_env(specs.get("custom_terms"), True, monkeypatch)._fused
    assert not on.external_rows and not on.user_term_refusals
    assert len(on.python_commands) == len(off.python_commands) == 1  # the `wave` manager; `clock` stays too
    assert [name for _, name, _, _, _ in on.external_obs] == [name for _, name, _, _, _ in off.external_obs]
    assert on.split_mode and len(on.split_plan) < len(off.split_plan)


def test_without_a_compiler_the_terms_stay_callbacks(cpu_device, monkeypatch):
    monkeypatch.setenv("GFB_NO_SPEC", "1")
    fused = dry_env(user_terms.user_terms(), True, monkeypatch)._fused
    assert not fused.user_terms and len(fused.external_rows) == 11 and fused.split_mode


@pytest.mark.parametrize("workload", ["user_terms", "user_terms_entity"])
def test_ir_reproduces_the_python_functions(workload, cpu_device, jit, monkeypatch):
    fused = dry_env(getattr(user_terms, workload)(), True, monkeypatch)._fused
    gen = torch.Generator().manual_seed(7)
    for trial in range(3):
        src, fake = _random_state(gen)
        for (kind, name), (prog, *_) in fused.user_terms.items():
            item = (fused.reward.cfg if kind == "reward" else fused.termination.term_cfg)[name]
            params = dict(item.params or {})
            want = item.fn(fake, **params)
            got = evaluate(prog, src, params)
            if kind == "reward":
                want = want.float()
            assert got.dtype == want.dtype and torch.equal(got, want), (name, trial)


def _refused(monkeypatch, fn, kind="reward", params=None):
    spec = specs.contacts()
    table = "rewards" if kind == "reward" else "terminations"
    spec[table] = dict(spec[table], probe={"fn": fn, "weight": 1.0, "params": params or {}} if kind == "reward"
                       else {"fn": fn, "params": params or {}})
    fused = dry_env(spec, True, monkeypatch)._fused
    assert (kind, "probe") not in fused.user_terms
    assert (kind, "probe") in {(k, n) for k, n, _ in fused.external_rows}
    return fused.user_term_refusals[(kind, "probe")]


STATE = torch.zeros(N)


class ClassTerm:
    def __init__(self, env):
        self.env = env

    def build(self):
        pass

    def __call__(self, env):
        return env.robot.get_pos()[:, 0]


@pytest.mark.parametrize("fn,kind,needle", [
    (lambda env: env.robot.get_pos()[:, 0] + STATE, "reward", "concrete tensor"),
    (lambda env: env.robot.get_pos()[:, 0] if env.robot.get_pos()[:, 0] > 0 else env.robot.get_vel()[:, 0],
     "reward", "__bool__"),
    (lambda env: env.robot.get_pos()[:, env.episode_length], "reward", "index"),
    (lambda env: env.robot.get_pos().nonzero()[:, 0].float(), "reward", "nonzero"),
    (lambda env: env.robot.get_pos().add_(1.0)[:, 0], "reward", "add_"),
    (lambda env: env.robot.get_links_pos()[:, 0, 0], "reward", "get_links_pos"),
    (lambda env: env.robot.get_pos(), "reward", "shape"),
    (lambda env: env.robot.get_pos()[:, 0], "termination", "bool"),
    (lambda env: env.extras["terminations"] & (env.robot.get_pos()[:, 0] > 0), "termination", "extras"),
    (lambda env: env.robot.get_pos()[:, 0].cumsum(0), "reward", "cumsum"),
    (lambda env: torch.stack([env.robot.get_pos()[:, 0], env.robot.get_vel()[:, 1]], dim=1).sum(dim=1), "reward",
     "sequence"),
    (lambda env: torch.cat([env.robot.get_pos(), env.robot.get_vel()], dim=1).sum(dim=1), "reward", "sequence"),
    (lambda env: env.robot.get_pos()[:, 0] * {}["missing"], "reward", "KeyError"),
])
def test_refusals_keep_the_callback(fn, kind, needle, cpu_device, jit, monkeypatch):
    why = _refused(monkeypatch, fn, kind)
    assert needle in why, why


def test_in_place_write_and_direct_stock_call_are_refused(cpu_device, jit, monkeypatch):
    from genesis_forge_b200.mdp import rewards

    def writes(env):
        v = env.robot.get_vel()
        v[:, 0] = 0.0
        return v[:, 1]

    def calls_stock(env):
        return rewards.lin_vel_z_l2(env, entity_manager=env.robot_manager) * 2.0

    assert "in-place" in _refused(monkeypatch, writes)
    assert "stock term" in _refused(monkeypatch, calls_stock)
    assert "class-style" in _refused(monkeypatch, ClassTerm)


def test_param_in_control_flow_is_traced_as_a_constant(cpu_device, jit, monkeypatch):
    def gated(env, scale=2.0):
        x = env.robot.get_pos()[:, 0]
        return x * scale if scale > 1.0 else x

    spec = specs.contacts()
    spec["rewards"] = dict(spec["rewards"], gated={"fn": gated, "weight": 1.0, "params": {"scale": 2.0}})
    fused = dry_env(spec, True, monkeypatch)._fused
    prog, live, traced, _ = fused.user_terms[("reward", "gated")]
    assert not live and prog.params == [] and traced == {"scale": 2.0}
    digest = prog.digest()
    fused.reward.cfg["gated"].params["scale"] = 3.0  # the constant changes: traced again, new identity
    fused._set_program(force=True)
    assert fused.user_terms[("reward", "gated")][0].digest() != digest
    assert fused.program.head.reward[list(fused.reward.cfg).index("gated")].i0 == \
        fused.user_terms[("reward", "gated")][0].digest()


def test_live_params_land_in_the_term_row(cpu_device, jit, monkeypatch):
    fused = dry_env(user_terms.user_terms(), True, monkeypatch)._fused
    row = list(fused.reward.cfg).index("level_speed")
    assert fused.program.head.reward[row].p[0] == pytest.approx(0.5)
    digest = fused.program.head.reward[row].i0
    fused.reward.cfg["level_speed"].params["scale"] = 0.75
    fused._set_program(force=True)
    assert fused.program.head.reward[row].p[0] == pytest.approx(0.75)
    assert fused.program.head.reward[row].i0 == digest  # same expression, same kernel


def test_dtype_promotion_follows_torch(cpu_device):
    tr = expr.Tracer(N, "reward")
    i = tr.source(("episode_length",), (), expr.I32)
    f = tr.source(("vel",), (3,), expr.F32)
    b = tr.source(("terminated",), (), expr.BOOL)
    assert (i * 2).dtype is torch.int32 and (i * 2.0).dtype is torch.float32 and (i / 2).dtype is torch.float32
    assert (b.float() + 1).dtype is torch.float32 and (i % 3).dtype is torch.int32
    assert (f[:, 0] > 1).dtype is torch.bool and (f.sum(dim=1) + i).dtype is torch.float32
    assert torch.where(b, i, 0.5).dtype is torch.float32
    assert (f[..., 1:3]).shape == (N, 2) and f.norm(dim=-1).shape == (N,)


@pytest.mark.skipif(shutil.which("nvcc") is None and not __import__("os").path.exists("/usr/local/cuda/bin/nvcc"),
                    reason="nvcc not available")
@pytest.mark.parametrize("workload", ["user_terms", "user_terms_entity"])
def test_generated_header_compiles_for_sm100a(workload, cpu_device, monkeypatch):
    from genesis_forge_b200 import spec

    env = dry_env(getattr(user_terms, workload)(), True, monkeypatch, n=256)
    todo = spec.collect(env, rng_modes=(0,))
    assert len(todo) == 1 and "GFB_SPEC_USER_TERMS" in next(iter(todo.values()))
    paths = spec.compile_many(todo)
    assert all(p.exists() for p in paths)


def test_a_live_param_changing_between_int_and_float_is_traced_again(cpu_device, jit, monkeypatch):
    def late(env, after=50):
        return (env.episode_length > after).float()

    spec = specs.contacts()
    spec["rewards"] = dict(spec["rewards"], late={"fn": late, "weight": 1.0, "params": {"after": 50}})
    fused = dry_env(spec, True, monkeypatch)._fused
    assert fused.user_terms[("reward", "late")][0].param_types == ["i32"]
    fused.reward.cfg["late"].params["after"] = 62.5
    fused._set_program(force=True)
    assert fused.user_terms[("reward", "late")][0].param_types == ["f32"]
    row = list(fused.reward.cfg).index("late")
    assert fused.program.head.reward[row].p[0] == 62.5
    assert fused.program.head.reward[row].i0 == fused.user_terms[("reward", "late")][0].digest()


def test_extras_without_a_termination_manager_are_refused(cpu_device, jit, monkeypatch):
    def alive(env):
        return (~env.extras["terminations"]).float()

    fused = dry_env(specs.contacts(), True, monkeypatch)._fused
    item = types.SimpleNamespace(fn=alive, params={})
    assert fused._lower_user_term("reward", "alive2", item)  # published by the termination manager
    fused.termination = None  # an environment without one: the function itself would raise KeyError
    assert not fused._lower_user_term("reward", "alive3", item)
    assert "without a termination manager" in fused.user_term_refusals[("reward", "alive3")]


def test_batches_that_cannot_use_the_specialised_kernel_keep_the_callbacks(cpu_device, jit, monkeypatch):
    fused = dry_env(user_terms.user_terms(), True, monkeypatch, n=66)._fused  # num_envs % 4 != 0: no TMA
    assert not fused.user_terms and len(fused.external_rows) == 11 and fused.split_mode
    monkeypatch.setenv("GFB_DISABLE_TMA", "1")
    fused = dry_env(user_terms.user_terms(), True, monkeypatch)._fused
    assert not fused.user_terms and fused.split_mode


def test_demotion_restores_the_split_plan(cpu_device, jit, monkeypatch):
    off = dry_env(user_terms.user_terms(), False, monkeypatch)._fused
    on = dry_env(user_terms.user_terms(), True, monkeypatch)._fused
    assert not on.split_mode
    on._demote_user_terms("test")
    assert on.split_mode and on.split_plan == off.split_plan and not on.user_terms
    assert [(k, n) for k, n, _ in on.external_rows] == [(k, n) for k, n, _ in off.external_rows]
    assert set(on.user_term_refusals) == {(k, n) for k, n, _ in off.external_rows}
    on._set_program(force=True)
    K = gfb._native.K
    ops = {on.program.head.reward[r].op for r in range(on.program.head.n_reward)}
    assert K["GFB_R_USER"] not in ops and K["GFB_R_EXTERNAL"] in ops
