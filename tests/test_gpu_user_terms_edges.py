"""
Lowered user terms through the specialised kernel on the GPU, op by op at edge values, against the float64
reference of the IR and torch-CPU running the same Python functions (tests/test_user_terms_edges.py).

Harness: env.actions / env.last_actions reach the kernel unchanged, so each env row carries 24 fp32 inputs
chosen here.  Every user reward is one op; its weight makes the packed fp32(weight * dt) exactly 1.0, and the
episode sums are filled with -0.0 before the step, so afterwards row r holds the term's value bit for bit
(-0 + v == v for every v, +-0 included).  The tables have no termination that can fire during the check.
"""
import numpy as np
import pytest
import torch

from test_gpu_user_terms import _user_library
from test_user_terms_edges import (D, OPS, PARAM_OPS, TERMINATIONS, _chain_sum, edge_inputs, exact64,
                                   exact_sum_bound, reference, same_bits, sources_of, special_class, torch_cpu,
                                   ulp_dist, ulp_error_vs_float64)

pytestmark = pytest.mark.gpu

DT = 1 / 50
WEIGHT = 50.0  # fp32(WEIGHT * DT) == 1.0: the summed value is the term's value
TIMEOUT_ONLY = {"timeout": {"fn": "timeout", "time_out": True}}


def _spec(rewards: dict, terminations: dict, contacts: bool, stock_rewards=()) -> dict:
    from configs import specs

    s = specs.contacts() if contacts else specs.command_direction()
    assert s["dt"] == DT
    s.update(name="user_term_edges", max_episode_length_sec=10000, max_episode_random_scaling=0.0)
    s["rewards"] = {**{k: s["rewards"][k] for k in stock_rewards}, **rewards}
    s["terminations"] = terminations
    return s


def _env(spec, n, device, monkeypatch, tile=None):
    import genesis_forge_b200 as gfb
    from configs.env_builder import build_env, dropin_namespace
    from genesis_forge_b200.managed_env import ManagedEnvironment

    monkeypatch.setattr(ManagedEnvironment, "fuse_user_terms", True)
    if tile is not None:
        monkeypatch.setenv("GFB_TILE", str(tile))
    gfb.set_device(device)
    env = build_env(spec, dropin_namespace(), n, device, pool=4, seed=11, n_contacts=8 if spec["contacts"] else 0,
                    apply_setters=False)
    env.build()
    env.reset()
    fused = env._fused
    assert not fused.user_term_refusals, fused.user_term_refusals
    assert not fused.split_mode and not fused.external_rows
    return env


def _rows(env, names):
    cfg = list(env.reward_manager.cfg)
    head = env._fused.program.head
    rows = [cfg.index(n) for n in names]
    assert all(head.reward[r].weight == 1.0 for r in rows)
    return rows


def _step_checked(env, actions):
    """One step that ran the specialised library carrying this table's user code."""
    fused = env._fused
    before = fused.spec_stats()["specialised_launches"]
    out = env.step(actions)
    stats = fused.spec_stats()
    assert stats["specialised_launches"] == before + 1, stats
    assert _user_library(fused) in stats["libraries"], stats
    return out


def _run_inputs(env, x: np.ndarray):
    """env.last_actions = x[:, 12:], env.actions = x[:, :12] in the second step; the episode sums of it."""
    dev = env._fused.device
    t = torch.from_numpy(x).to(dev)
    _step_checked(env, t[:, D:].contiguous())
    env.reward_manager._episode_sums.fill_(-0.0)
    _step_checked(env, t[:, :D].contiguous())
    bits = lambda v: v.cpu().view(torch.int32)  # noqa: E731 - (NaN != NaN: compare the bit patterns)
    assert torch.equal(bits(env.last_actions), bits(t[:, D:])) and torch.equal(bits(env.actions), bits(t[:, :D]))
    return env.reward_manager._episode_sums.cpu().numpy()


CHUNK = 30
TABLES = [OPS[k:k + CHUNK] for k in range(0, len(OPS), CHUNK)]


@pytest.mark.parametrize("table", range(len(TABLES)))
def test_ops_at_edge_values(table, cuda_device, monkeypatch):
    ops = TABLES[table] + (PARAM_OPS if table == 0 else [])
    rewards = {}
    for op in ops:
        name, fn = op[0], op[1]
        rewards[name] = {"fn": fn, "weight": WEIGHT, "params": dict(op[2]) if len(op) == 4 else {}}
    env = _env(_spec(rewards, TIMEOUT_ONLY, contacts=False), len(x := edge_inputs()), cuda_device, monkeypatch)
    sums = _run_inputs(env, x)
    fused = env._fused
    failed = []
    for op, r in zip(ops, _rows(env, [op[0] for op in ops])):
        name, fn, cmp = op[0], op[1], op[-1]
        params = dict(op[2]) if len(op) == 4 else {}
        prog = fused.user_terms[("reward", name)][0]
        got = sums[r]
        ref = reference(prog, sources_of(x), params)
        cpu = torch_cpu(fn, x, params)
        vs_cpu = same_bits(got, cpu, zeros_by_value=cmp in ("zeros", "tie"))
        if cmp in ("exact", "zeros", "tie", "sqrt"):
            ok = same_bits(got, ref, zeros_by_value=cmp == "zeros")
            worst = f"{int(ulp_dist(got, ref).max())} ulp"
            ok &= ulp_dist(got, cpu) <= 1 if cmp == "sqrt" else vs_cpu
        elif cmp == "bound":
            exact, bound, fin = exact_sum_bound(prog, x)
            err = np.abs(got.astype(np.float64) - exact)
            ok = np.where(fin, err <= bound, True) & same_bits(got, ref)  # (ref: the index-order chain)
            special = ~np.isfinite(x).all(axis=1)
            ok &= np.where(special, special_class(got) == special_class(ref), True)
            with np.errstate(all="ignore"):
                worst = f"{float(np.max(err[fin] / bound[fin])):.3f} of the bound"
        else:
            err = ulp_error_vs_float64(got, exact64(name, x))
            ok = (special_class(got) == special_class(ref)) & (err <= cmp[1])
            worst = f"{float(err.max()):.3f} ulp"
        print(f"EDGE-OP {name:24s} max_vs_float64={worst} torch_cpu_exact={int(vs_cpu.sum())}/{len(x)}"
              f"{'' if ok.all() else f'  MISMATCH {int((~ok).sum())} rows'}")
        if not ok.all():
            failed.append((name, x[~ok][:3, :4], got[~ok][:3], ref[~ok][:3], cpu[~ok][:3]))
    assert not failed, failed


def test_terminations_at_edge_values(cuda_device, monkeypatch):
    """GFB_T_USER: `terminated` is the OR of the table's user terminations (last_actions 0 after reset)."""
    terms = {name: {"fn": fn} for name, fn in TERMINATIONS}
    terms.update(TIMEOUT_ONLY)
    env = _env(_spec({"x": {"fn": lambda e: e.actions[:, 0], "weight": WEIGHT}}, terms, contacts=False),
               len(x := edge_inputs()), cuda_device, monkeypatch)
    x[:, D:] = 0.0
    _, _, terminated, truncated, _ = _step_checked(env, torch.from_numpy(x[:, :D]).to(cuda_device).contiguous())
    want = np.zeros(len(x), dtype=bool)
    for name, fn in TERMINATIONS:
        prog = env._fused.user_terms[("termination", name)][0]
        ref = reference(prog, sources_of(x))
        assert (ref == torch_cpu(fn, x)).all(), name
        want |= ref
    assert 0 < want.sum() < len(x)
    assert (terminated.cpu().numpy() == want).all() and not truncated.any()


# ------------------------------------------------------------------------------------------------
# sources, at several tiles and sizes: identity and sum terms against the getters
# ------------------------------------------------------------------------------------------------
def _source_terms(contacts: bool) -> dict:
    getters = {
        "pos": lambda e: e.robot.get_pos(), "quat": lambda e: e.robot.get_quat(),
        "vel": lambda e: e.robot.get_vel(), "ang": lambda e: e.robot.get_ang(),
        "lin_b": lambda e: e.robot_manager.get_linear_velocity(),
        "ang_b": lambda e: e.robot_manager.get_angular_velocity(),
        "grav_b": lambda e: e.robot_manager.get_projected_gravity(),
        "dof_pos": lambda e: e.action_manager.get_dofs_position(),
        "dof_vel": lambda e: e.action_manager.get_dofs_velocity(),
        "targets": lambda e: e.action_manager.get_actions(),
        "actions": lambda e: e.actions, "last_actions": lambda e: e.last_actions,
        "command": lambda e: e.velocity_command.command,
    }
    if contacts:
        getters["contacts_z"] = lambda e: e.foot_contact_manager.contacts[:, :, 2]
        getters["air"] = lambda e: e.foot_contact_manager.last_air_time
    terms = {"episode_length": (lambda e: e.episode_length.float(), None)}
    for name, g in getters.items():
        terms[f"{name}_last"] = (lambda e, g=g: g(e)[:, -1], g)
        terms[f"{name}_sum"] = (lambda e, g=g: g(e).sum(dim=1), g)
    return terms


@pytest.mark.parametrize("contacts", [False, True], ids=["no_contacts", "contacts"])
@pytest.mark.parametrize("tile", [32, 64, 128])
@pytest.mark.parametrize("num_envs", [36, 260, 65536 + 4])
def test_sources_by_tile_and_tail(contacts, tile, num_envs, cuda_device, monkeypatch):
    terms = _source_terms(contacts)
    # without contacts, stock terms make the plan compute the body-frame registers; with contacts (and no
    # stock rewards) the user code rotates the vectors itself
    stock = () if contacts else ("tracking_lin_vel", "tracking_ang_vel")
    rewards = {name: {"fn": fn, "weight": WEIGHT} for name, (fn, _) in terms.items()}
    if not contacts:
        rewards["flat"] = {"fn": "flat_orientation_l2", "weight": -2.5}
    env = _env(_spec(rewards, TIMEOUT_ONLY, contacts, stock_rewards=stock), num_envs, cuda_device, monkeypatch,
               tile=tile)
    gen = torch.Generator(device=cuda_device).manual_seed(5)
    _step_checked(env, torch.randn(num_envs, D, device=cuda_device, generator=gen))
    env.reward_manager._episode_sums.fill_(-0.0)
    _step_checked(env, torch.randn(num_envs, D, device=cuda_device, generator=gen))
    sums = env.reward_manager._episode_sums.cpu().numpy()
    names = list(terms)
    for (name, (fn, getter)), r in zip(terms.items(), _rows(env, names)):
        got = sums[r]
        if getter is None:
            want = env.episode_length.float().cpu().numpy()
        else:
            v = getter(env).float().cpu().numpy().reshape(num_envs, -1)
            want = v[:, -1] if name.endswith("_last") else _chain_sum([v[:, k] for k in range(v.shape[1])])
        bad = ~same_bits(got, want)
        assert not bad.any(), (name, tile, num_envs, np.nonzero(bad)[0][:8], got[bad][:4], want[bad][:4])
