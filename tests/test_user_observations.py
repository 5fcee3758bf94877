"""
Host side of the lowered user-defined observation terms (ManagedEnvironment.fuse_user_observations): the
lowering decision, the IR against the Python functions it came from (layout ops and flattening included),
refusals, the switch leaving everything else as it was, demotion and the generated device code.  No GPU.
"""
import shutil
import types

import pytest
import torch

import genesis_forge_b200 as gfb
from configs import specs, user_observations as uo
from configs.env_builder import build_env, dropin_namespace
from genesis_forge_b200 import expr
from genesis_forge_b200.managed_env import ManagedEnvironment
from test_user_terms import N, ClassTerm, _random_state, cpu_device, evaluate, jit  # noqa: F401

K = gfb._native.K


def dry_env(spec, monkeypatch, obs: bool, terms: bool = False, n=N):
    monkeypatch.setattr(ManagedEnvironment, "fuse_user_observations", obs)
    monkeypatch.setattr(ManagedEnvironment, "fuse_user_terms", terms)
    env = build_env(spec, dropin_namespace(), n, torch.device("cpu"))
    env._dry_run = True
    env.build()
    env._fused._set_program()
    return env


def evaluate_obs(prog: expr.Program, sources: dict) -> torch.Tensor:
    """The IR evaluator of tests/test_user_terms.py, node by node, plus the layout ops of observation terms."""
    vals = []
    for n in prog.nodes:
        a = [vals[i] for i in n.args]
        if n.op == "reshape":
            v = a[0].reshape((N,) + n.shape)
        elif n.op == "stack":
            v = torch.stack(a, dim=-1)
        elif n.op == "cat":
            v = torch.cat(a, dim=-1)
        elif not n.args:
            v = evaluate(expr.Program(prog.kind, [n], 0, [], []), sources, {})
        else:  # one node over stand-in sources holding its operands
            args = [expr.Node("src", (), ("arg", j), prog.nodes[i].shape, prog.nodes[i].dtype, prog.nodes[i].weak)
                    for j, i in enumerate(n.args)]
            one = expr.Node(n.op, range(len(args)), n.attr, n.shape, n.dtype, n.weak)
            v = evaluate(expr.Program(prog.kind, args + [one], len(args), [], []),
                         {("arg", j): x for j, x in enumerate(a)}, {})
        vals.append(v)
    return vals[prog.out]


def _state(gen):
    src, env = _random_state(gen)
    src[("base_pos",)], src[("base_quat",)] = src[("pos",)], src[("quat",)]
    env.num_envs = N
    return src, env


@pytest.mark.parametrize("workload", ["user_observations", "user_observations_entity"])
def test_workloads_lower_completely(workload, cpu_device, jit, monkeypatch):
    fused = dry_env(getattr(uo, workload)(), monkeypatch, True)._fused
    assert not fused.user_term_refusals and not fused.external_obs and fused.ext_obs is None
    assert not fused.split_mode and fused.split_plan == []
    P = fused.program.head
    srcs = [fused.program.obs_cols[c].src for c in range(sum(P.obs_group[g].n_cols for g in range(P.n_obs_groups)))]
    assert srcs.count(K["GFB_O_USER"]) == fused.user_obs_width  # one word per column of frame 0
    ids = {P.obs_group[g].user_id for g in range(P.n_obs_groups)}
    assert len(ids) == 1 and 0 not in ids


@pytest.mark.parametrize("workload", ["user_observations", "user_observations_entity"])
def test_ir_reproduces_the_python_functions(workload, cpu_device, jit, monkeypatch):
    fused = dry_env(getattr(uo, workload)(), monkeypatch, True)._fused
    ops = {n.op for prog, *_ in fused.user_obs.values() for n in prog.nodes}
    assert ({"reshape", "stack", "cat"} if workload == "user_observations" else {"reshape", "cat"}) <= ops
    gen = torch.Generator().manual_seed(11)
    for trial in range(3):
        src, fake = _state(gen)
        for (g, name), (prog, _, _, width) in fused.user_obs.items():
            item = fused.observations[g].cfg[name]
            want = item.fn(env=fake).reshape(N, width).float()
            got = evaluate_obs(prog, src)
            assert got.dtype == want.dtype and torch.equal(got, want), (name, trial)


def _refused(monkeypatch, fn, spec=None, prop=False):
    spec = spec or specs.contacts()
    spec["observations"]["policy"]["terms"]["probe"] = {"fn": fn}
    if prop:  # a second EntityManager (configs/second_entity.py)
        from configs import second_entity

        monkeypatch.setattr(ManagedEnvironment, "fuse_user_observations", True)
        ns = dropin_namespace()
        env = second_entity.add_prop(build_env(spec, ns, N, torch.device("cpu")), ns)
        env._dry_run = True
        env.build()
        fused = env._fused
    else:
        fused = dry_env(spec, monkeypatch, True)._fused
    assert not any(name == "probe" for _, name in fused.user_obs)
    assert "probe" in [name for _, name, *_ in fused.external_obs]
    return fused.user_term_refusals[("observation", "probe")]


@pytest.mark.parametrize("fn,needle", [
    (lambda env: env.extras.get("terminations", env.robot.get_pos()[:, 0] > 0).float().unsqueeze(1), "extras"),
    (lambda env: env.robot.get_pos().repeat(1, 2), "repeat"),
    (lambda env: torch.cat([env.robot.get_pos()] * 11, dim=1), "33 columns"),
    (lambda env: torch.stack([env.robot.get_pos()[:, 0], env.robot.get_vel()[:, 0]], dim=0).T, "dim=0"),
    (lambda env: env.robot.get_pos().reshape(-1), "rows of the"),
])
def test_refusals_keep_the_host_column(fn, needle, cpu_device, jit, monkeypatch):
    why = _refused(monkeypatch, fn)
    assert needle in why, why


def test_class_style_and_further_entity_terms_stay_host_columns(cpu_device, jit, monkeypatch):
    from configs import second_entity

    assert "class-style" in _refused(monkeypatch, ClassTerm)
    spec = second_entity.spec()
    why = _refused(monkeypatch, lambda env: env.prop_manager.get_linear_velocity() * 2.0, spec=spec, prop=True)
    assert "further EntityManager" in why, why


def test_stack_and_cat_stay_refused_in_rewards(cpu_device, jit, monkeypatch):
    spec = specs.contacts()
    spec["rewards"]["probe"] = {"fn": lambda env: torch.stack([env.robot.get_pos()[:, 0], env.robot.get_vel()[:, 1]],
                                                              dim=1).sum(dim=1), "weight": 1.0}
    spec["rewards"]["probe2"] = {"fn": lambda env: env.robot.get_pos().unsqueeze(1)[:, 0, 0], "weight": 1.0}
    fused = dry_env(spec, monkeypatch, True, terms=True)._fused
    assert "sequence" in fused.user_term_refusals[("reward", "probe")]
    assert "observation terms only" in fused.user_term_refusals[("reward", "probe2")]


def test_switch_off_keeps_todays_plans(cpu_device, jit, monkeypatch):
    head, term, rew, reset, obs = (K["GFB_PHASE_ENTITY"] | K["GFB_PHASE_CONTACT"], K["GFB_PHASE_TERMINATION"],
                                   K["GFB_PHASE_REWARD"] | K["GFB_PHASE_COMMAND"], K["GFB_PHASE_RESET"],
                                   K["GFB_PHASE_OBSERVE"])
    fused = dry_env(uo.user_observations(), monkeypatch, False)._fused
    assert not fused.user_obs and fused.split_mode
    assert [tuple(p) for p in fused.split_plan] == [(None, head | term | rew | reset, True), ("observe", obs, False)]
    assert [(n, c0, w) for _, n, _, c0, w in fused.external_obs] == [
        ("gait_clock", 0, 2), ("base_height", 2, 1), ("command_scaled", 3, 3), ("feet_down", 7 - 1, 4),
        ("planar_motion", 10, 3), ("air_clock", 13, 1), ("clock", 14, 2), ("quat_tail", 16, 2)]
    custom = dry_env(specs.get("custom_terms"), monkeypatch, False)._fused
    assert [(n, w) for _, n, _, _, w in custom.external_obs] == [("clock", 2), ("ang_vel_fresh", 3)]


def test_switch_on_leaves_tables_without_user_observations_alone(cpu_device, jit, monkeypatch):
    from genesis_forge_b200 import spec as spec_mod

    for name in list(specs.ALL) + list(specs.VARIANTS):
        if name == "custom_terms":  # (has a user observation term)
            continue
        texts = []
        for on in (False, True):
            env = dry_env(specs.get(name), monkeypatch, on, n=256)
            assert not env._fused.user_obs
            texts.append(spec_mod.collect(env, rng_modes=(0,)))
        assert texts[0] == texts[1], name


def test_custom_terms_lower_the_clock_only(cpu_device, jit, monkeypatch):
    fused = dry_env(specs.get("custom_terms"), monkeypatch, True, terms=True)._fused
    assert [name for _, name in fused.user_obs] == ["clock"]
    assert [name for _, name, *_ in fused.external_obs] == ["ang_vel_fresh"]
    assert len(fused.python_commands) == 1 and fused.split_mode  # the `wave` manager stays a callback
    assert ("observation", "ang_vel_fresh") not in fused.user_term_refusals  # (not a user function: not tried)


def test_demotion_restores_the_host_columns(cpu_device, jit, monkeypatch):
    off = dry_env(uo.user_observations(), monkeypatch, False)._fused
    on = dry_env(uo.user_observations(), monkeypatch, True)._fused
    on._demote_user_terms("test")
    assert on.split_mode and on.split_plan == off.split_plan and not on.user_obs
    assert [(n, c0, w) for _, n, _, c0, w in on.external_obs] == [(n, c0, w) for _, n, _, c0, w in off.external_obs]
    assert on.ext_obs.shape == off.ext_obs.shape and on.user_obs_values is None
    assert on.user_term_refusals[("observation", "gait_clock")] == "test"
    on._set_program(force=True)
    P = on.program.head
    n_cols = sum(P.obs_group[g].n_cols for g in range(P.n_obs_groups))
    assert K["GFB_O_USER"] not in {on.program.obs_cols[c].src for c in range(n_cols)}
    assert all(P.obs_group[g].user_id == 0 for g in range(P.n_obs_groups))


def test_a_closure_constant_changes_the_identity(cpu_device, jit, monkeypatch):
    ids = []
    for gain in (2.0, 3.0):
        spec = uo.user_observations()
        spec["observations"]["policy"]["terms"]["base_height"] = {"fn": lambda env, g=gain: env.robot.get_pos()[:, 2:3] * g}
        ids.append(dry_env(spec, monkeypatch, True)._fused.program.head.obs_group[0].user_id)
    assert ids[0] != ids[1]


@pytest.mark.skipif(shutil.which("nvcc") is None and not __import__("os").path.exists("/usr/local/cuda/bin/nvcc"),
                    reason="nvcc not available")
@pytest.mark.parametrize("workload", ["user_observations", "user_observations_entity"])
def test_generated_header_compiles_for_sm100a(workload, cpu_device, monkeypatch):
    from genesis_forge_b200 import spec

    env = dry_env(getattr(uo, workload)(), monkeypatch, True, n=256)
    todo = spec.collect(env, rng_modes=(0,))
    assert len(todo) == 1
    text = next(iter(todo.values()))
    assert "GFB_SPEC_USER_OBS" in text and "user_observations_global" in text
    paths = spec.compile_many(todo)
    assert all(p.exists() for p in paths)


# sha1 of the specialised headers (both draw modes, 256 envs) that the lowered reward / termination terms
# generated before user observation terms could be lowered: with fuse_user_terms alone they must not change
_LOWERED_TERM_HEADERS = {
    "user_terms": ["5ad5c2ea0de07c451ba8c2ea7760eea9cd37f31a", "d83c462caca8e65100772c48b841619ed0e06b3c"],
    "user_terms_entity": ["37b1d4254f3a9d886480944d9882227d58042803", "bbad6fe899744d8f840362cfa7889fb08868b3d8"],
    "custom_terms": ["00b74d5d592aa660e11aea761c7b7f7174afb1f4", "129475cd19efaa41fda93b04d8230a704177c58a",
                     "2a9e9565707f595a3f01d1d87c8acaf460433f6a", "9581b2d8037c4c613ff42a5ac245dbf6f169c89c",
                     "f3cfc1de6fae03560c5a357777eb7fc5ded78f83", "f432b2a75bc4213dc158419e5965148ff52e3ce9"],
}


@pytest.mark.parametrize("workload", sorted(_LOWERED_TERM_HEADERS))
def test_lowered_reward_terms_keep_their_headers(workload, cpu_device, jit, monkeypatch):
    import hashlib

    from configs import user_terms
    from genesis_forge_b200 import spec

    make = specs.get if workload == "custom_terms" else (lambda name: getattr(user_terms, name)())
    env = dry_env(make(workload), monkeypatch, False, terms=True, n=256)
    texts = spec.collect(env).values()
    assert sorted(hashlib.sha1(t.encode()).hexdigest() for t in texts) == _LOWERED_TERM_HEADERS[workload]
    if workload == "user_terms":  # the terms read the staged pos / vel / ang / quat rows where the plan has them
        assert any("c.plan.off_pos >= 0 ? c.S + c.plan.off_pos" in t for t in texts)
