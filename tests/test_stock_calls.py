"""
Stock mdp reward / termination calls inside user terms, inlined into the lowered terms
(ManagedEnvironment.fuse_stock_calls, expr.ExprMode.stock_call): the lowering of both workloads of
configs/stock_calls.py, every covered stock term through an identity wrapper against the oracle port at edge
states, the refusals, live and traced-again params, and the generated code.  No GPU needed.
"""
import math
import os
import shutil
import subprocess
import tempfile
import types
from pathlib import Path

import pytest
import torch

import genesis_forge_b200 as gfb
from configs import specs, stock_calls
from configs.env_builder import build_env, dropin_namespace
from genesis_forge_b200 import expr
from genesis_forge_b200.managed_env import ManagedEnvironment
from genesis_forge_b200.managers.observation import UnsupportedTermError
from genesis_forge_b200.mdp import rewards, terminations
from oracle.manager_port import PortEnv
from test_user_terms import evaluate

N = 64
NVCC = shutil.which("nvcc") or ("/usr/local/cuda/bin/nvcc" if os.path.exists("/usr/local/cuda/bin/nvcc") else None)
SWITCHES = ("fuse_user_terms", "fuse_stateful_terms")
WRAPPERS_A = ("gated_tracking", "upright", "smooth", "alive_yaw", "posture_ema", "lin_vel_z_wrap", "fell",
              "fall_over_wrap")
WRAPPERS_B = ("air_when_moving", "contact_mix", "slide", "hard_hit")


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


def dry_env(spec, monkeypatch, stock=True, n=N):
    for name in SWITCHES:
        monkeypatch.setattr(ManagedEnvironment, name, True)
    monkeypatch.setattr(ManagedEnvironment, "fuse_stock_calls", stock)
    env = build_env(spec, dropin_namespace(), n, torch.device("cpu"))
    env._dry_run = True
    env.build()
    env._fused._set_program()
    return env


def test_both_workloads_lower_completely_into_one_launch(cpu_device, jit, monkeypatch):
    for spec, names in ((stock_calls.stock_calls_a(), WRAPPERS_A), (stock_calls.stock_calls_b(), WRAPPERS_B)):
        fused = dry_env(spec, monkeypatch)._fused
        assert not fused.user_term_refusals and not fused.external_rows, spec["name"]
        assert not fused.split_mode and fused.split_plan == []
        assert sorted(n for _, n in fused.user_terms) == sorted(names)
    assert fused._link_layout == {"vel": (7, (3, 7, 11, 15))}  # feet_slide's calves


def test_switch_off_refuses_every_wrapper_as_today(cpu_device, jit, monkeypatch):
    for spec, names in ((stock_calls.stock_calls_a(), WRAPPERS_A), (stock_calls.stock_calls_b(), WRAPPERS_B)):
        fused = dry_env(spec, monkeypatch, stock=False)._fused
        assert sorted(n for _, n in fused.user_term_refusals) == sorted(names)
        assert all("a direct call of the stock term" in why and why.endswith("is not inlined")
                   for why in fused.user_term_refusals.values())
        assert sorted(n for _, n, _ in fused.external_rows) == sorted(names) and fused.split_mode


def test_programs_without_stock_calls_are_unchanged(cpu_device, jit, monkeypatch):
    """The switch changes nothing for a table whose terms call no stock term: same programs, same header."""
    from configs import link_terms

    codes = [dry_env(link_terms.link_terms(), monkeypatch, stock=on)._fused.user_code for on in (False, True)]
    assert codes[0] == codes[1] and "ACTION_RATE" not in codes[0] and "fmaxf" not in codes[0]


# ------------------------------------------------------------------------------------------------
# identity wrappers against the oracle port
# ------------------------------------------------------------------------------------------------
FLAT = types.SimpleNamespace(height_field=None, _origin=torch.tensor([0.0, 0.0, 0.05]))
BOUNDS = (-5.0, 5.0, -4.0, 4.0)
BOXED = types.SimpleNamespace(get_bounds=lambda subterrain=None: BOUNDS)
FIXED_LIN, FIXED_YAW = torch.tensor([0.5, -0.2]), torch.tensor(0.3)

# name -> (wrapper, oracle term, oracle params); None: a flat terrain, restated in the test
REWARDS = {
    "is_alive": (lambda env: rewards.is_alive(env), "is_alive", {}),
    "terminated": (lambda env: rewards.terminated(env), "terminated", {}),
    "base_height": (lambda env: rewards.base_height(env, target_height=0.3), "base_height", {"target_height": 0.3}),
    "base_height_0d": (lambda env: rewards.base_height(env, target_height=torch.tensor(0.25)), "base_height",
                       {"target_height": torch.tensor(0.25)}),
    "base_height_cmd": (lambda env: rewards.base_height(env, height_command=env.velocity_command), "base_height",
                        {"height_command": "@h"}),
    "base_height_flat": (lambda env: rewards.base_height(env, target_height=0.3, terrain_manager=FLAT), None, None),
    "dof_similar_to_default": (lambda env: rewards.dof_similar_to_default(env, action_manager=env.action_manager),
                               "dof_similar_to_default", {}),
    "lin_vel_z_l2": (lambda env: rewards.lin_vel_z_l2(env, entity_manager=env.robot_manager), "lin_vel_z_l2",
                     {"entity_manager": "@em"}),
    "ang_vel_xy_l2": (lambda env: rewards.ang_vel_xy_l2(env, entity_manager=env.robot_manager), "ang_vel_xy_l2",
                      {"entity_manager": "@em"}),
    "flat_orientation_l2": (lambda env: rewards.flat_orientation_l2(env), "flat_orientation_l2", {}),
    "action_rate_l2": (lambda env: rewards.action_rate_l2(env), "action_rate_l2", {}),
    "track_lin": (lambda env: rewards.command_tracking_lin_vel(env, vel_cmd_manager=env.velocity_command,
                                                               entity_manager=env.robot_manager, sensitivity=0.3),
                  "command_tracking_lin_vel", {"vel_cmd_manager": "@vc", "entity_manager": "@em", "sensitivity": 0.3}),
    "track_lin_fixed": (lambda env: rewards.command_tracking_lin_vel(env, command=FIXED_LIN),
                        "command_tracking_lin_vel", {}),
    "track_ang": (lambda env: rewards.command_tracking_ang_vel(env, vel_cmd_manager=env.velocity_command),
                  "command_tracking_ang_vel", {"vel_cmd_manager": "@vc"}),
    "track_ang_fixed": (lambda env: rewards.command_tracking_ang_vel(env, commanded_ang_vel=FIXED_YAW,
                                                                     sensitivity=0.5),
                        "command_tracking_ang_vel", {"sensitivity": 0.5}),
    "stand_still": (lambda env: rewards.stand_still_joint_deviation_l1(env, vel_cmd_manager=env.velocity_command,
                                                                       action_manager=env.action_manager),
                    "stand_still_joint_deviation_l1", {"vel_cmd_manager": "@vc"}),
    "has_contact": (lambda env: rewards.has_contact(env, env.foot_contact_manager, threshold=1.0, min_contacts=2),
                    "has_contact", {"contact_manager": "@fcm", "threshold": 1.0, "min_contacts": 2}),
    "contact_force": (lambda env: rewards.contact_force(env, env.foot_contact_manager, threshold=1.0),
                      "contact_force", {"contact_manager": "@fcm", "threshold": 1.0}),
    "feet_air_time": (lambda env: rewards.feet_air_time(env, env.foot_contact_manager, time_threshold=0.5,
                                                        time_threshold_max=1.0, vel_cmd_manager=env.velocity_command),
                      "feet_air_time", {"contact_manager": "@fcm", "time_threshold": 0.5, "time_threshold_max": 1.0,
                                        "vel_cmd_manager": "@vc"}),
    "feet_slide": (lambda env: rewards.feet_slide(env, env.foot_contact_manager), "feet_slide",
                   {"contact_manager": "@fcm"}),
}
TERMINATIONS = {
    "timeout": (lambda env: terminations.timeout(env), "timeout", {}),
    "bad_orientation": (lambda env: terminations.bad_orientation(env, limit_angle=20.0, grace_steps=5,
                                                                 entity_manager=env.robot_manager),
                        "bad_orientation", {"limit_angle": 20.0, "grace_steps": 5, "entity_manager": "@em"}),
    "base_height_below_minimum": (lambda env: terminations.base_height_below_minimum(
        env, minimum_height=0.15, entity_manager=env.robot_manager), "base_height_below_minimum",
        {"minimum_height": 0.15, "entity_manager": "@em"}),
    "out_of_bounds": (lambda env: terminations.out_of_bounds(env, terrain_manager=BOXED, border_margin=0.5),
                      "out_of_bounds", {"border_margin": 0.5}),
    "has_contact_t": (lambda env: terminations.has_contact(env, env.foot_contact_manager, threshold=1.0,
                                                           min_contacts=2),
                      "has_contact", {"contact_manager": "@fcm", "threshold": 1.0, "min_contacts": 2}),
    "contact_force_t": (lambda env: terminations.contact_force(env, env.foot_contact_manager, threshold=1.0),
                        "contact_force", {"contact_manager": "@fcm", "threshold": 1.0}),
    "contact_force_grace": (lambda env: terminations.contact_force_with_grace_period(
        env, env.foot_contact_manager, threshold=100.0, grace_steps=10), "contact_force_with_grace_period",
        {"contact_manager": "@fcm", "threshold": 100.0, "grace_steps": 10}),
}


def _wrapped_table():
    spec = specs.contacts()
    spec["rewards"] = dict(spec["rewards"], **{k: {"fn": v[0], "weight": 1.0} for k, v in REWARDS.items()})
    spec["terminations"] = dict(spec["terminations"], **{k: {"fn": v[0]} for k, v in TERMINATIONS.items()})
    return spec


def _edge_state(gen, fused, L=4):
    """Random sources with thresholds hit exactly, NaN and +-Inf in some rows."""
    f = lambda *s: torch.randn(*s, generator=gen)  # noqa: E731
    D = fused.D
    src = {("lin_vel_b",): f(N, 3), ("ang_vel_b",): f(N, 3), ("gravity_b",): f(N, 3) * 0.4, ("pos",): f(N, 3),
           ("dof_pos",): f(N, D), ("command", 0): f(N, 3) * 0.2, ("contacts", 0): f(N, L, 3) * 2,
           ("air", 0, 0): f(N, L).abs(), ("air", 0, 3): f(N, L).abs() * 0.03,
           ("episode_length",): torch.randint(0, 20, (N,), generator=gen, dtype=torch.int32),
           ("max_episode_length",): torch.randint(5, 15, (N,), generator=gen, dtype=torch.int32),
           ("terminated",): torch.rand(N, generator=gen) < 0.3}
    links = f(N, L, 3)
    actions, last = f(N, D), f(N, D)
    # exactly at the thresholds
    src[("contacts", 0)][0:4, :, :] = torch.tensor([1.0, 0.0, 0.0])  # norm == threshold
    src[("contacts", 0)][4, :2, :] = torch.tensor([0.0, 100.0, 0.0])
    src[("air", 0, 3)][5:7, :] = expr._f32(fused.env.dt + 1.0e-8)
    src[("air", 0, 3)][7, :] = 0.0
    src[("air", 0, 0)][8, :] = 0.5
    src[("episode_length",)][9:12] = torch.tensor([5, 10, 0], dtype=torch.int32)
    src[("max_episode_length",)][12] = src[("episode_length",)][12]
    src[("pos",)][13, 2] = expr._f32(0.15)
    src[("pos",)][14, :2] = torch.tensor([BOUNDS[0] + 0.5, BOUNDS[3] - 0.5])
    src[("gravity_b",)][15, :] = torch.tensor([fused._tilt_threshold(20.0), 0.0, -0.9])
    src[("command", 0)][16, :] = torch.tensor([0.06, 0.0, 0.0])
    src[("command", 0)][17, :] = torch.tensor([0.1, 0.0, 0.0])
    src[("pos",)][18, 2] = expr._f32(0.3)
    # non-finite
    for row, v in ((20, math.nan), (21, math.inf), (22, -math.inf)):
        for key in (("lin_vel_b",), ("ang_vel_b",), ("gravity_b",), ("pos",), ("dof_pos",), ("command", 0)):
            src[key][row, 0] = v
        src[("contacts", 0)][row, 1, 2] = v
        src[("air", 0, 0)][row, 2] = v
        src[("air", 0, 3)][row, 3] = v
        links[row, 0, 1] = v
        actions[row, 3] = v
    src[("gravity_b",)][23, :] = torch.tensor([math.nan, math.nan, 0.0])
    src[("action_rate",)] = torch.sum(torch.square(last - actions), dim=1)  # what the action kernel writes
    return src, links, actions, last


class _Sources(dict):
    def __init__(self, src, links):
        super().__init__(src)
        self.links = links

    def __missing__(self, key):  # ("link_vel", ids, slot, U)
        assert key[0] == "link_vel" and list(key[1]) == [3, 7, 11, 15]
        return self.links


def _evaluate(prog, sources: _Sources, params: dict):
    """tests/test_user_terms.py's evaluator, with the internal NaN-dropping ops as torch.fmax / torch.fmin."""
    nodes, sources = list(prog.nodes), _Sources(dict(sources), sources.links)
    for i, n in enumerate(nodes):
        if n.op in ("fmax", "fmin"):
            a, b = (evaluate(expr.Program(prog.kind, nodes[:j + 1], j, prog.params, prog.param_types), sources, params)
                    for j in n.args)
            a, b = (x if torch.is_tensor(x) else torch.tensor(x, dtype=torch.float32) for x in (a, b))
            sources[("fm", i)] = getattr(torch, n.op)(a, b)
            nodes[i] = expr.Node("src", (), ("fm", i), n.shape, n.dtype)
    return evaluate(expr.Program(prog.kind, nodes, prog.out, prog.params, prog.param_types), sources, params)


def _oracle(fused, src, links, actions, last, cmd_dims=3):
    port = object.__new__(PortEnv)
    robot = types.SimpleNamespace(get_pos=lambda: src[("pos",)], get_dofs_position=lambda idx=None: src[("dof_pos",)],
                                  get_links_vel=lambda links_idx_local=None: links)
    fixed = torch.zeros((N, 3))
    fixed[:, :2], fixed[:, 2] = FIXED_LIN, FIXED_YAW
    port.__dict__.update(
        num_envs=N, dt=fused.env.dt, record_margins=False, margins=[], robot=robot, dofs_idx=None,
        default_dofs_pos=fused.action.kernel_params()["default"].float(), base_pos=src[("pos",)],
        actions=actions, last_actions=last, episode_length=src[("episode_length",)],
        max_episode_length=src[("max_episode_length",)], extras={"terminations": src[("terminated",)]},
        t_bounds=BOUNDS, fixed_command=fixed,
        command={"vc": {"command": src[("command", 0)]}, "h": {"command": src[("command", 0)][:, :1]}},
        contact={"fcm": {"contacts": src[("contacts", 0)], "last_air": src[("air", 0, 0)],
                         "cur_contact": src[("air", 0, 3)], "local_link_ids": [3, 7, 11, 15]}},
        _lin_vel=lambda cached=True: src[("lin_vel_b",)], _ang_vel=lambda cached=True: src[("ang_vel_b",)],
        _gravity=lambda cached=True: src[("gravity_b",)])
    return port


def _kernel_rule(name, src):
    """The rows where the kernel case and the reference differ: fmaxf / fminf drop a NaN (post_kernel.cuh
    GFB_R_CONTACT_FORCE, GFB_R_FEET_AIR_TIME), which is what the stock row gives and the inlined call keeps."""
    cn = torch.norm(src[("contacts", 0)], dim=-1)
    if name == "contact_force":
        return torch.fmax(cn - 1.0, torch.tensor(0.0)).sum(dim=1)
    cur = src[("air", 0, 3)]
    made = (cur > 0.0) & (cur < expr._f32(0.02 + 1.0e-8))
    a = torch.fmin((src[("air", 0, 0)] - 0.5) * made.float(), torch.tensor(0.5))
    return a.sum(dim=1) * (torch.norm(src[("command", 0)][:, :2], dim=1) > 0.1).float()


def _same(got, want):
    if got.dtype.is_floating_point:
        return bool(((got == want) | (got.isnan() & want.isnan())).all()) and got.dtype == want.dtype
    return torch.equal(got, want)


def test_identity_wrappers_equal_the_oracle_at_edge_states(cpu_device, jit, monkeypatch):
    fused = dry_env(_wrapped_table(), monkeypatch)._fused
    assert not fused.user_term_refusals
    gen = torch.Generator().manual_seed(11)
    for trial in range(3):
        src, links, actions, last = _edge_state(gen, fused)
        port = _oracle(fused, src, links, actions, last)
        sources = _Sources(src, links)
        for kind, table in (("reward", REWARDS), ("termination", TERMINATIONS)):
            for name, (_, fn, params) in table.items():
                prog = fused.user_terms[(kind, name)][0]
                got = _evaluate(prog, sources, {})
                if fn is None:  # a flat terrain: the origin's fp32 z, then the target (rewards.py:54-90)
                    want = torch.square(src[("pos",)][:, 2] - torch.tensor(0.05) - 0.3)
                elif kind == "reward":
                    want = port._reward_value(fn, params).float()
                else:
                    want = port._termination_value(fn, params)
                if name in ("contact_force", "feet_air_time"):
                    nan = want.isnan()
                    want = torch.where(nan, _kernel_rule(name, src), want)
                assert _same(got, want), (name, trial, got, want)


def test_every_covered_stock_term_is_inlined(cpu_device, jit, monkeypatch):
    fused = dry_env(_wrapped_table(), monkeypatch)._fused
    opcodes = {fn.gfb_opcode for fn in vars(rewards).values() if getattr(fn, "gfb_kind", None) == "reward"} - \
        {"GFB_R_BODY_ACC_EXP"}
    assert {k[1] for k in expr._STOCK if k[0] == "reward"} == opcodes
    assert {k[1] for k in expr._STOCK if k[0] == "termination"} == \
        {fn.gfb_opcode for fn in vars(terminations).values() if getattr(fn, "gfb_kind", None) == "termination"}
    srcs = {n.attr[0] for (k, _), (prog, *_) in fused.user_terms.items() for n in prog.nodes if n.op == "src"}
    assert {"action_rate", "link_vel", "air", "contacts", "command", "terminated"} <= srcs


# ------------------------------------------------------------------------------------------------
# refusals
# ------------------------------------------------------------------------------------------------
def _body_acc(env):
    inst = rewards.body_acceleration_exp.__new__(rewards.body_acceleration_exp)
    return inst(env, entity_manager=env.robot_manager)


class _Unregistered:
    _external_controller = None


@pytest.mark.parametrize("fn,kind,needle", [
    (_body_acc, "reward", "keeps per-term state"),
    (lambda env: rewards.base_height(env, target_height=0.3, terrain_manager=types.SimpleNamespace(
        height_field=torch.zeros(4, 4), _origin=torch.zeros(3))), "reward", "height-field"),
    (lambda env: rewards.base_height(env, target_height=torch.full((N,), 0.3)), "reward", "per-env"),
    (lambda env: rewards.command_tracking_lin_vel(env, command=torch.zeros(N, 2)), "reward", "per-env command"),
    (lambda env: rewards.lin_vel_z_l2(env, entity_manager=types.SimpleNamespace()), "reward",
     "further EntityManager"),
    (lambda env: rewards.lin_vel_z_l2(env, entity_attr="terrain"), "reward", "entity_attr 'terrain'"),
    (lambda env: rewards.command_tracking_ang_vel(env, vel_cmd_manager=_Unregistered()), "reward", "not registered"),
    (lambda env: rewards.contact_force(env, _Unregistered()), "reward", "not registered"),
    (lambda env: rewards.is_alive(env) > 0.5, "termination", "extras"),
    (lambda env: rewards.terminated(env) > 0.5, "termination", "extras"),
])
def test_refusals_keep_the_callback(fn, kind, needle, cpu_device, jit, monkeypatch):
    spec = specs.contacts()
    table = "rewards" if kind == "reward" else "terminations"
    spec[table] = dict(spec[table], probe={"fn": fn, "weight": 1.0} if kind == "reward" else {"fn": fn})
    fused = dry_env(spec, monkeypatch)._fused
    assert (kind, "probe") not in fused.user_terms
    assert (kind, "probe") in {(k, n) for k, n, _ in fused.external_rows}
    why = fused.user_term_refusals[(kind, "probe")]
    assert "stock term" in why and needle in why, why


def test_a_stock_call_in_an_observation_term_is_refused(cpu_device, jit, monkeypatch):
    fused = dry_env(specs.contacts(), monkeypatch)._fused
    mode = expr.ExprMode(expr.Tracer(N, "observation"), fused)
    with pytest.raises(UnsupportedTermError, match="inside an observation term"):
        mode.stock_call("reward", rewards.lin_vel_z_l2, {"entity_attr": "robot", "entity_manager": None})


# ------------------------------------------------------------------------------------------------
# params
# ------------------------------------------------------------------------------------------------
def test_a_live_param_passed_to_a_stock_call_stays_live(cpu_device, jit, monkeypatch):
    fused = dry_env(stock_calls.stock_calls_a(), monkeypatch)._fused
    row = list(fused.reward.cfg).index("gated_tracking")
    prog, live, *_ = fused.user_terms[("reward", "gated_tracking")]
    assert live and prog.params == ["sensitivity"]
    assert any(n.op == "div" and prog.nodes[n.args[1]].op == "param" for n in prog.nodes)
    digest = fused.program.head.reward[row].i0
    assert fused.program.head.reward[row].p[0] == pytest.approx(0.25)
    fused.reward.cfg["gated_tracking"].params["sensitivity"] = 0.4
    fused._set_program(force=True)
    assert fused.program.head.reward[row].p[0] == pytest.approx(0.4)
    assert fused.program.head.reward[row].i0 == digest  # the same binary


def test_a_param_in_the_normalisation_traces_the_term_again(cpu_device, jit, monkeypatch):
    def tilted(env, limit=30.0):
        return terminations.bad_orientation(env, limit_angle=limit, entity_manager=env.robot_manager)

    spec = specs.contacts()
    spec["terminations"] = dict(spec["terminations"], tilted={"fn": tilted, "params": {"limit": 30.0}})
    fused = dry_env(spec, monkeypatch)._fused
    prog, live, traced, _ = fused.user_terms[("termination", "tilted")]
    assert not live and prog.params == [] and traced == {"limit": 30.0}
    row = list(fused.termination.term_cfg).index("tilted")
    digest = fused.program.head.termination[row].i0
    fused.termination.term_cfg["tilted"].params["limit"] = 25.0
    fused._set_program(force=True)
    new = fused.user_terms[("termination", "tilted")][0]
    assert new.digest() != digest and fused.program.head.termination[row].i0 == new.digest()
    consts = {n.attr for n in new.nodes if n.op == "const"}
    assert expr._f32(fused._tilt_threshold(25.0)) in consts


# ------------------------------------------------------------------------------------------------
# generated code
# ------------------------------------------------------------------------------------------------
@pytest.mark.skipif(NVCC is None, reason="nvcc not available")
@pytest.mark.parametrize("workload", ["stock_calls_a", "stock_calls_b"])
def test_generated_header_compiles_for_sm100a_without_spills(workload, cpu_device, jit, monkeypatch):
    from genesis_forge_b200 import spec

    env = dry_env(getattr(stock_calls, workload)(), monkeypatch, n=256)
    todo = spec.collect(env, rng_modes=(1,))
    assert len(todo) == 1
    text = next(iter(todo.values()))
    assert "GFB_SPEC_USER_TERMS" in text and ("GFB_B_ACTION_RATE" in text) == (workload == "stock_calls_a")
    with tempfile.TemporaryDirectory() as d:
        header = os.path.join(d, "spec.h")
        Path(header).write_text(text)
        out = subprocess.run([NVCC, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-Xptxas", "-v",
                              "-Xcompiler", "-fPIC", "-shared", "--fmad=false", f'-DGFB_SPEC_HEADER="{header}"',
                              str(spec.PKG / "csrc" / "spec_kernel.cu"), "-o", os.path.join(d, "spec.so")],
                             capture_output=True, text=True)
        assert out.returncode == 0, out.stderr
    post = [ln for ln in out.stderr.splitlines() if "spill" in ln]
    assert post and all("0 bytes spill stores, 0 bytes spill loads" in ln for ln in post), out.stderr
