"""
Class-style user terms lowered into the specialised post-physics kernel (ManagedEnvironment.fuse_stateful_terms,
configs/stateful_terms.py workload A) against the same instances run as host callbacks on the drop-in, on the
same seeded states with production Philox draws.  Bar: masks, counters and int / bool state bit-exact; fp32
rewards, observations, episode sums and state within 1e-5 rel + 1e-6.
"""
import pytest
import torch

from configs import stateful_terms

pytestmark = pytest.mark.gpu

STATE = {"joint_accel": ("prev_vel", "gain"), "action_jerk": ("prev1", "prev2"), "speed_ema": ("ema",),
         "tilt_latch": ("tilted",)}


def _pair(num_envs, cuda_device, seed, monkeypatch):
    import genesis_forge_b200 as gfb
    from configs.env_builder import build_env, dropin_namespace
    from genesis_forge_b200.managed_env import ManagedEnvironment

    envs = []
    for fuse in (False, True):
        monkeypatch.setattr(ManagedEnvironment, "fuse_stateful_terms", fuse)
        gfb.set_device(cuda_device)
        env = build_env(stateful_terms.stateful_terms(), dropin_namespace(), num_envs, cuda_device, pool=4, seed=seed,
                        n_contacts=0, apply_setters=False)
        env.build()
        env.reset()
        envs.append(env)
    split, fused = envs
    assert split._fused.split_mode and not fused._fused.split_mode and not fused._fused.user_term_refusals
    return split, fused


def _close(got, want, what):
    if got.dtype in (torch.bool, torch.int32, torch.int64):
        assert torch.equal(got, want), what
        return 0.0
    both_nan = got.isnan() & want.isnan()
    err = torch.where(both_nan, 0.0, (got - want).abs())
    assert bool((both_nan | (err <= 1e-6 + 1e-5 * want.abs())).all()), (what, float(err.max()))
    return float(err.max())


def _state(env, name):
    cfg = env.reward_manager.cfg if name in STATE else env.termination_manager.term_cfg
    attrs = STATE.get(name, ("count",))
    return [getattr(cfg[name].fn, a) for a in attrs]


def _compare_state(split, fused, rows=slice(None)):
    for name in list(STATE) + ["stuck"]:
        for a, b in zip(_state(split, name), _state(fused, name)):
            if a is None or b is None:
                assert a is None and b is None, name
                continue
            _close(b[rows], a[rows], name)


def _run(split, fused, steps, gen, nan_step=None, edit=None):
    N = fused.num_envs
    worst, resets = 0.0, 0
    for i in range(steps):
        if edit is not None:
            edit(i, split, fused)
        actions = torch.randn(N, 12, device=fused.episode_length.device, generator=gen)
        if nan_step is not None and i == nan_step:
            actions[3, 1] = float("nan")
        a, b = split.step(actions), fused.step(actions.clone())
        assert torch.equal(a[2], b[2]) and torch.equal(a[3], b[3]), i
        resets += int((a[2] | a[3]).sum())
        for got, want, what in ((b[1], a[1], "rewards"), (b[0], a[0], "obs"),
                                (fused.reward_manager._episode_sums, split.reward_manager._episode_sums, "sums")):
            worst = max(worst, _close(got, want, (i, what)))
        _compare_state(split, fused)
    return worst, resets


@pytest.mark.parametrize("num_envs,steps,nan_step", [(256, 120, 7), (65536, 20, None), (4100, 30, None)])
def test_lowered_class_terms_match_the_callbacks(num_envs, steps, nan_step, cuda_device, monkeypatch):
    split, fused = _pair(num_envs, cuda_device, 11, monkeypatch)
    gen = torch.Generator(device=cuda_device).manual_seed(3)
    worst, resets = _run(split, fused, steps, gen, nan_step)
    _compare_state(split, fused, rows=slice(num_envs - 1, num_envs))  # env N-1: shadowed by a tail slab's lanes
    stats = fused._fused.spec_stats()
    assert stats["specialised_launches"] == steps and stats["generic_launches"] == 2, stats
    assert resets > 0
    print(f"STATEFUL N={num_envs} steps={steps} resets={resets} max_abs={worst:.3e}")


def test_weight_zero_and_a_disabled_reward_manager_leave_the_state(cuda_device, monkeypatch):
    split, fused = _pair(256, cuda_device, 5, monkeypatch)
    for env in (split, fused):
        env.reward_manager.cfg["speed_ema"].weight = 0.0
    gen = torch.Generator(device=cuda_device).manual_seed(4)
    _run(split, fused, 6, gen)
    assert not bool(fused.reward_manager.cfg["speed_ema"].fn.ema.any())  # never evaluated
    assert fused.reward_manager.cfg["action_jerk"].fn.prev1 is not None

    def edit(i, *envs):
        for env in envs:
            if i == 3:
                env.reward_manager.cfg["speed_ema"].weight = 0.3
            if i == 6:
                env.reward_manager.enabled = False
            if i == 9:
                env.reward_manager.enabled = True

    frozen = {}

    def edit_and_watch(i, s, f):
        edit(i, s, f)
        if i == 7:
            frozen["ema"] = f.reward_manager.cfg["speed_ema"].fn.ema.clone()
        if i == 9:  # the reward phase did not run for two steps: the state did not advance
            assert torch.equal(f.reward_manager.cfg["speed_ema"].fn.ema, frozen["ema"])

    _run(split, fused, 14, gen, edit=edit_and_watch)


def test_host_edits_between_steps(cuda_device, monkeypatch):
    split, fused = _pair(256, cuda_device, 7, monkeypatch)
    gen = torch.Generator(device=cuda_device).manual_seed(5)

    def edit(i, *envs):
        for env in envs:
            inst = env.reward_manager.cfg
            if i == 4:  # a manual reset of some rows, in place
                inst["speed_ema"].fn.ema[:10] = 0.0
                env.termination_manager.term_cfg["stuck"].fn.count[5:9] = 30
            if i == 8:  # a compatible rebinding
                inst["joint_accel"].fn.prev_vel = torch.zeros_like(inst["joint_accel"].fn.prev_vel)
            if i == 12:  # an incompatible one: the lowered terms become callbacks from here on
                inst["speed_ema"].fn.ema = inst["speed_ema"].fn.ema.to(torch.float64)

    _run(split, fused, 20, gen, edit=edit)
    f = fused._fused
    assert f.split_mode and not f.stateful and "speed_ema" in f.user_term_refusals[("reward", "speed_ema")]


def test_without_specialisation_the_class_terms_stay_callbacks(cuda_device, monkeypatch):
    import genesis_forge_b200 as gfb
    from configs.env_builder import build_env, dropin_namespace
    from genesis_forge_b200.managed_env import ManagedEnvironment

    monkeypatch.setenv("GFB_NO_SPEC", "1")
    monkeypatch.setattr(ManagedEnvironment, "fuse_stateful_terms", True)
    gfb.set_device(cuda_device)
    env = build_env(stateful_terms.stateful_terms(), dropin_namespace(), 256, cuda_device, pool=4, seed=1,
                    n_contacts=0, apply_setters=False)
    env.build()
    env.reset()
    f = env._fused
    assert f.split_mode and not f.stateful and len(f.external_rows) == 5
    gen = torch.Generator(device=cuda_device).manual_seed(1)
    for _ in range(5):
        env.step(torch.randn(256, 12, device=cuda_device, generator=gen))
    assert env.reward_manager.cfg["action_jerk"].fn.prev1 is not None
    assert f.spec_stats()["specialised_launches"] == 0


def _port_instance(cls):
    """The oracle port calls a user term as fn(env, **params): stand in a callable that creates the class-style
    term once, with the port environment, and calls that instance every step (config_item.py:46-77)."""
    held = {}

    def fn(env, **params):
        if "inst" not in held:
            held["inst"] = cls(env, **params)
            held["inst"].build()
        return held["inst"](env, **params)

    fn.held = held
    return fn


def test_contact_term_matches_the_oracle_port(cuda_device, monkeypatch):
    """Workload B: the contacts table with a lazily initialised contact-streak term, lowered, against the port."""
    from genesis_forge_b200.managed_env import ManagedEnvironment
    from oracle.parity import ParityRun

    monkeypatch.setattr(ManagedEnvironment, "fuse_stateful_terms", True)
    run = ParityRun("contacts", num_envs=256, device=cuda_device, seed=1234,
                    spec_override=stateful_terms.contacts_override())
    rewards = run.port.spec["rewards"]
    port_fn = _port_instance(stateful_terms.contact_streak)
    rewards["contact_streak"] = dict(rewards["contact_streak"], fn=port_fn)
    fused = run.env._fused
    assert not fused.split_mode and not fused.external_rows and not fused.user_term_refusals
    stats = run.run(steps=120, nan_step=7)
    assert stats["resets"] > 0
    streak = run.env.reward_manager.cfg["contact_streak"].fn.streak
    assert streak is not None and bool((streak > 0).any())
    want = port_fn.held["inst"].streak
    assert torch.allclose(streak.cpu(), want, rtol=1e-5, atol=1e-6), float((streak.cpu() - want).abs().max())
    assert fused.spec_stats()["specialised_launches"] == 120
    print(f"STATEFUL-PORT max_abs={stats['max_abs']:.3e} max_rel={stats['max_rel']:.3e} inexact={stats['inexact']}")
