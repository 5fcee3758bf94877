"""
Environments with more than one EntityManager (the reference registry keeps a list,
genesis_forge/managed_env.py:200-220, :269-270, :294-296, :353-354).  Workload: configs/second_entity.py
(the `simple` example plus a prop with its own manager, on_reset item and observation group).

  * the committed trace of the UNMODIFIED reference (tests/golden/second_entity.pt, oracle/make_golden.py)
    is checked against a direct statement of what the second manager must produce (cache taken before
    the reset, velocities read after it) -- CPU;
  * the drop-in's host logic accepts the configuration and routes the prop's terms to host-evaluated
    columns -- CPU, dry run;
  * the CUDA path reproduces the trace -- GPU.
"""
import pytest
import torch

import genesis_forge_b200 as gfb
from configs import second_entity
from configs.env_builder import build_env, dropin_namespace
from genesis_forge_b200 import _native as nat
from genesis_forge_b200.fused import UnsupportedTermError
from genesis_forge_b200.synthetic import ROBOT_MODELS, StateSource
from oracle import geom, make_golden
from oracle.parity import _close


def test_reference_trace_of_the_second_manager():
    """Pins the semantics the drop-in has to reproduce, on the reference's own output."""
    gold = make_golden.load("second_entity")
    n, spec = gold["num_envs"], second_entity.spec()
    source = StateSource(ROBOT_MODELS[spec["robot"]], n, 8, gold["seed"])
    gravity = torch.tensor([0.0, 0.0, -1.0]).expand(n, 3)
    n_reset = 0
    for i, g in enumerate(gold["step"]):
        st = source(i + 1)  # the scene steps before the managers run
        quat = st["quat"][:, [0, 2, 3, 1]]
        cache = g["extra"]
        # entity_manager.py:189-195 runs at the top of the step: the cache holds the PRE-reset pose
        assert torch.equal(cache["base_pos"], st["pos"] + 1.0), i
        assert torch.equal(cache["base_quat"], quat), i
        assert torch.equal(cache["inv_base_quat"], geom.inv_quat(quat)), i
        # the observation group is assembled after the reset: post-reset velocities (zeroed by set_pos /
        # set_quat for the reset envs), rotated by the cached -- pre-reset -- quaternion
        reset = torch.zeros(n, dtype=torch.bool)
        reset[g["reset_idx"]] = True
        n_reset += int(reset.sum())
        keep = (~reset).float().unsqueeze(1)
        inv = geom.inv_quat(quat)
        want = torch.cat([
            geom.transform_by_quat(st["ang"] * 0.5 * keep, inv) * 2.0,
            geom.transform_by_quat(gravity, inv),
            geom.transform_by_quat(st["vel"] * 2.0 * keep, inv) * 0.25,
        ], dim=1)
        assert torch.equal(g["obs"]["prop"][:, :9], want), i
    assert n_reset >= 5  # the trace exercises the reset path


@pytest.fixture()
def cpu_device():
    prev = gfb.gs.device
    gfb.set_device("cpu")
    yield torch.device("cpu")
    gfb.gs.device = prev


def _dropin(n, device, stock_terms=False, **kw):
    ns = dropin_namespace()
    return second_entity.add_prop(build_env(second_entity.spec(stock_terms), ns, n, device, **kw), ns)


def test_dropin_accepts_further_entity_managers(cpu_device):
    env = _dropin(32, cpu_device)
    env._dry_run = True
    env.build()
    fused = env._fused
    assert fused.entity_manager is env.robot_manager and fused.secondary_entities == [env.prop_manager]
    assert env.robot_manager._primary and not env.prop_manager._primary
    # the prop's body-frame terms are host-evaluated columns, the robot's stay kernel sources
    sources = {name: key for name, key, width in env.observation_managers["prop"]._sources}
    widths = {name: width for name, key, width in env.observation_managers["prop"]._sources}
    assert all(sources[f"prop_{t}"] == ("external", f"prop_{t}")
               for t in ("linear_velocity", "projected_gravity", "angular_velocity"))
    assert sources["robot_angular_velocity"] == "ang_vel_b"
    assert set(widths.values()) == {3}
    assert fused.split_mode
    # the further manager's cache was filled by its build() (entity_manager.py:157), by device copies
    assert torch.equal(env.prop_manager.base_pos, env.prop.get_pos())
    assert torch.equal(env.prop_manager.inv_base_quat, geom.inv_quat(env.prop.get_quat()))


def test_stock_terms_of_a_further_entity_become_host_callbacks(cpu_device):
    """Stock mdp terms that refer to the prop are evaluated between the kernel phases (one-term path bound
    to the prop's state); the robot's stay in the kernel."""
    env = _dropin(32, cpu_device, stock_terms=True)
    env._dry_run = True
    env.build()
    fused = env._fused
    fused._set_program()
    external = {(kind, name) for kind, name, _ in fused.external_rows}
    assert external == {("reward", "prop_lin_vel_z"), ("reward", "prop_flat"), ("reward", "prop_height"),
                        ("termination", "prop_tilt")}
    K = nat.K
    ops = {name: op for name, _, op in fused.reward_terms}
    assert ops["prop_flat"] == K["GFB_R_EXTERNAL"] and ops["lin_vel_z"] == K["GFB_R_LIN_VEL_Z"]
    assert {name: op for name, _, op in fused.termination_terms}["fall_over"] == K["GFB_T_BAD_ORIENTATION"]
    assert [callback for callback, _, _ in fused.split_plan] == [None, "termination", "reward", "observe"]


def test_body_acceleration_of_a_further_entity_is_refused(cpu_device):
    ns = dropin_namespace()
    spec = second_entity.spec()
    spec["rewards"]["prop_acc"] = {"fn": "body_acceleration_exp", "weight": 1.0,
                                   "params": {"entity_manager": "@prop_manager"}}
    env = second_entity.add_prop(build_env(spec, ns, 32, cpu_device), ns)
    env._dry_run = True
    with pytest.raises(UnsupportedTermError, match="first EntityManager"):
        env.build()


@pytest.mark.gpu
@pytest.mark.parametrize("stock_terms", [False, True], ids=["getters", "stock_terms"])
def test_cuda_path_reproduces_reference_trace_with_two_entity_managers(stock_terms, cuda_device):
    gold = make_golden.load("second_entity_terms" if stock_terms else "second_entity")
    n = gold["num_envs"]
    gfb.set_device(cuda_device)
    env = _dropin(n, cuda_device, stock_terms=stock_terms, seed=gold["seed"])
    torch.manual_seed(gold["seed"])
    env.build()
    assert env._fused.split_mode and env._fused.secondary_entities == [env.prop_manager]
    obs, extras = env.reset()
    for group, want in gold["reset"]["obs"].items():
        ok, err, _ = _close(extras["observations"][group], want)
        assert ok, f"reset obs[{group}] err {err}"
    gen = torch.Generator().manual_seed(gold["seed"] + 77)
    n_act = env.action_space.shape[0]
    for i, g in enumerate(gold["step"]):
        actions = torch.randn(n, n_act, generator=gen)
        out = env.step(actions.to(cuda_device))
        assert torch.equal(out[2].cpu(), g["terminated"]), f"step {i} terminated"
        assert torch.equal(out[3].cpu(), g["truncated"]), f"step {i} truncated"
        k = int(g["reset_idx"].numel())
        assert torch.equal(env._fused.reset_idx[:k].cpu(), g["reset_idx"]), f"step {i} reset_idx"
        ok, err, _ = _close(out[1], g["rewards"])
        assert ok, f"step {i} rewards err {err}"
        for group, want in g["obs"].items():
            ok, err, _ = _close(out[4]["observations"][group], want)
            assert ok, f"step {i} obs[{group}] err {err}"
        for key, want in g["logging"].items():
            ok, err, _ = _close(torch.as_tensor(out[4]["episode"][key]).reshape(()), want)
            assert ok, f"step {i} extras[{key}] err {err}"
        for key, want in second_entity.prop_cache(env).items():
            assert torch.equal(want, g["extra"][key]), f"step {i} prop {key}"  # copies and sign flips: exact
    assert ("set_pos", 1) in env.prop.calls or any(c[0] == "set_pos" for c in env.prop.calls)
