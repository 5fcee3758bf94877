"""
User terms that call stock mdp terms (configs/stock_calls.py) lowered with ManagedEnvironment.fuse_stock_calls,
on the GPU.  The identity wrappers equal their stock rows bit for bit every step; the lowered workloads match
the same functions run as host callbacks (fuse_stock_calls off: split execution, each stock call a one-term
launch) -- terminations, reset lists and observations bit-exact, rewards within 1e-5 rel + 1e-6 because the host
path of action_rate_l2 sums on the host (DESIGN.md section 1).  At 65536 envs the contacts workload is checked
against the Python functions on the fused environment's own state (split execution of a contacts table is not
run-to-run deterministic there, DESIGN.md section 9).
"""
import pytest
import torch

from configs import specs, stock_calls

pytestmark = pytest.mark.gpu

SWITCHES = ("fuse_user_terms", "fuse_stateful_terms")


def _build(spec, num_envs, cuda_device, seed, monkeypatch, stock):
    import genesis_forge_b200 as gfb
    from configs.env_builder import build_env, dropin_namespace
    from genesis_forge_b200.managed_env import ManagedEnvironment

    for name in SWITCHES:
        monkeypatch.setattr(ManagedEnvironment, name, True)
    monkeypatch.setattr(ManagedEnvironment, "fuse_stock_calls", stock)
    gfb.set_device(cuda_device)
    env = build_env(spec, dropin_namespace(), num_envs, cuda_device, pool=4, seed=seed, n_contacts=8)
    env.build()
    env.reset()
    return env


def _inject(envs, num_envs, cuda_device, gen):
    f = envs[0]._fused
    draws = {"max_len": torch.rand(num_envs, device=cuda_device, generator=gen) * 2 - 1}
    for k, mgr in enumerate(f.commands):
        for key in (f"cmd_step{k}", f"cmd_reset{k}"):
            draws[key] = torch.rand(mgr._command.shape, device=cuda_device, generator=gen) * 2 - 1
    for g, om in enumerate(f.observations):
        draws[f"obs_noise{g}"] = torch.rand((num_envs, om.frame_size), device=cuda_device, generator=gen) * 2 - 1
    for env in envs:
        env._fused.inject({k: v.clone() for k, v in draws.items()})


def _close(got, want, what):
    both_nan = got.isnan() & want.isnan()
    err = torch.where(both_nan, 0.0, (got - want).abs())
    assert bool((both_nan | (err <= 1e-6 + 1e-5 * want.abs())).all()), (what, float(err.max()))
    return float(err.max())


def test_identity_wrappers_equal_their_stock_rows_every_step(cuda_device, monkeypatch):
    env = _build(stock_calls.stock_calls_a(), 4096, cuda_device, 7, monkeypatch, True)
    f = env._fused
    assert not f.split_mode and not f.user_term_refusals
    gen = torch.Generator(device=cuda_device).manual_seed(3)
    _inject([env], 4096, cuda_device, gen)
    sums = env.managers["reward"]._episode_data
    t_names = list(env.managers["termination"].term_cfg)
    rows = {n: f.n_reward + t_names.index(n) for n in ("fall_over", "fall_over_wrap")}
    resets = fired = 0
    for i in range(48):
        out = env.step(torch.randn(4096, 12, device=cuda_device, generator=gen))
        assert torch.equal(sums["lin_vel_z_wrap"], sums["lin_vel_z"]), i
        log = env._log_snapshot()
        assert float(log[rows["fall_over_wrap"]]) == float(log[rows["fall_over"]]), i
        fired += round(float(log[rows["fall_over"]]) * 4096)
        resets += int((out[2] | out[3]).sum())
    assert resets > 0 and fired > 0
    print(f"STOCK-CALLS identity wrappers: 48 steps, resets={resets}, fall_over fired={fired}")


@pytest.mark.parametrize("workload,num_envs", [("stock_calls_a", 4096), ("stock_calls_b", 4096),
                                               ("stock_calls_a", 65536)])
def test_lowered_stock_calls_match_the_host_callbacks(workload, num_envs, cuda_device, monkeypatch):
    spec = getattr(stock_calls, workload)
    host = _build(spec(), num_envs, cuda_device, 7, monkeypatch, False)
    fused = _build(spec(), num_envs, cuda_device, 7, monkeypatch, True)
    stock = _build(specs.command_direction() if workload == "stock_calls_a" else specs.contacts(), num_envs,
                   cuda_device, 7, monkeypatch, True)
    f = fused._fused
    assert host._fused.split_mode and not host._fused.user_terms
    assert not f.split_mode and not f.user_term_refusals and not stock._fused.split_mode
    gen = torch.Generator(device=cuda_device).manual_seed(5)
    _inject([host, fused, stock], num_envs, cuda_device, gen)
    spec_before, launches = f.spec_stats()["specialised_launches"], f.launch_count()
    stock_launches = stock._fused.launch_count()
    worst, resets, steps = 0.0, 0, 40
    for i in range(steps):
        actions = torch.randn(num_envs, 12, device=cuda_device, generator=gen)
        a, b = host.step(actions), fused.step(actions.clone())
        stock.step(actions.clone())
        assert torch.equal(a[2], b[2]) and torch.equal(a[3], b[3]), i
        assert torch.equal(host._fused.reset_idx, fused._fused.reset_idx), i
        assert torch.equal(a[0], b[0]), i
        worst = max(worst, _close(b[1], a[1], (i, "rewards")))
        resets += int((a[2] | a[3]).sum())
    assert resets > 0
    assert f.spec_stats()["specialised_launches"] - spec_before == steps  # the specialised library, once a step
    assert f.launch_count() - launches == stock._fused.launch_count() - stock_launches
    assert f._eval_handle is None  # no one-term launch during lowered steps
    print(f"STOCK-CALLS {workload} N={num_envs} resets={resets} rewards max_abs={worst:.3e} {f.spec_stats()}")


def test_contacts_workload_at_65536_matches_the_functions_on_the_fused_state(cuda_device, monkeypatch):
    """The lowered contact rewards against the same Python functions evaluated on the fused environment's own
    state after the step (pool states, engine-side resets not applied), envs that reset this step left out (the
    reset clears their air-time state)."""
    fused = _build(stock_calls.stock_calls_b(), 65536, cuda_device, 7, monkeypatch, True)
    f = fused._fused
    assert not f.split_mode and not f.user_term_refusals
    gen = torch.Generator(device=cuda_device).manual_seed(11)
    _inject([fused], 65536, cuda_device, gen)
    cfg = fused.managers["reward"].cfg
    sums = fused.managers["reward"]._episode_data
    worst = 0.0
    for i in range(20):
        before = {n: sums[n].clone() for n in ("air_when_moving", "contact_mix", "slide")}
        out = fused.step(torch.randn(65536, 12, device=cuda_device, generator=gen))
        keep = ~(out[2] | out[3])
        for name in before:
            item = cfg[name]
            want = item.fn(fused, **item.params).float() * torch.tensor(item.weight * fused.dt, dtype=torch.float32)
            got = sums[name] - before[name]
            worst = max(worst, _close(got[keep], want[keep], (i, name)))
    print(f"STOCK-CALLS contacts N=65536 max_abs={worst:.3e}")
