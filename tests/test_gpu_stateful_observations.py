"""
Class-style user observation terms lowered into the specialised post-physics kernel and its reset-path kernel
(ManagedEnvironment.fuse_stateful_terms, configs/stateful_observations.py).  Workloads A and A-split against the
same instances run as host columns on the drop-in, same seeds, production Philox draws; workload B against the
oracle port.  Bar: masks, counters and int32 state bit-exact; fp32 observations and state within
1e-5 rel + 1e-6.  The state of every env advances exactly once per observation, as on the host path: a reset
env's rows are compared after every step.
"""
import pytest
import torch

from configs import stateful_observations as so

pytestmark = pytest.mark.gpu


def _pair(num_envs, cuda_device, seed, monkeypatch, spec=so.stateful_observations):
    import genesis_forge_b200 as gfb
    from configs.env_builder import build_env, dropin_namespace
    from genesis_forge_b200.managed_env import ManagedEnvironment

    envs = []
    for fuse in (False, True):
        monkeypatch.setattr(ManagedEnvironment, "fuse_stateful_terms", fuse)
        gfb.set_device(cuda_device)
        env = build_env(spec(), dropin_namespace(), num_envs, cuda_device, pool=4, seed=seed, n_contacts=0,
                        apply_setters=False)
        env.build()
        env.reset()
        envs.append(env)
    host, fused = envs
    assert host._fused.split_mode and len(host._fused.external_obs) == 5
    assert not fused._fused.external_obs and not fused._fused.user_term_refusals and len(fused._fused.stateful) == 5
    return host, fused


def _close(got, want, what):
    if got.dtype in (torch.bool, torch.int32, torch.int64):
        assert torch.equal(got, want), what
        return 0.0
    both_nan = got.isnan() & want.isnan()
    err = torch.where(both_nan, 0.0, (got - want).abs())
    assert bool((both_nan | (err <= 1e-6 + 1e-5 * want.abs())).all()), (what, float(err.max()))
    return float(err.max())


def _state(env):
    groups = {om.name: om for om in env.managers["observation"]}
    return {(g, n, a): getattr(groups[g].cfg[n].fn, a) for (g, n), attrs in so.STATE.items() for a in attrs}


def _compare_state(host, fused, rows=slice(None), what=None):
    a, b = _state(host), _state(fused)
    for key in a:
        _close(b[key][rows], a[key][rows], (what, key))


def _compare_obs(host, fused, what, extras=None):
    worst = 0.0
    for om_h, om_f in zip(host.managers["observation"], fused.managers["observation"]):
        worst = max(worst, _close(om_f.get_observations(), om_h.get_observations(), (what, om_h.name)))
    return worst


def _run(host, fused, steps, gen, nan_step=None, edit=None):
    N = fused.num_envs
    worst, resets = 0.0, 0
    for i in range(steps):
        if edit is not None:
            edit(i, host, fused)
        actions = torch.randn(N, 12, device=fused.episode_length.device, generator=gen)
        if nan_step is not None and i == nan_step:
            actions[3, 1] = float("nan")
        a, b = host.step(actions), fused.step(actions.clone())
        assert torch.equal(a[2], b[2]) and torch.equal(a[3], b[3]), i
        done = a[2] | a[3]
        resets += int(done.sum())
        worst = max(worst, _close(b[1], a[1], (i, "rewards")), _compare_obs(host, fused, (i, "obs")))
        _compare_state(host, fused, what=i)
        if bool(done.any()):  # the envs this step reset: observed (and advanced) once, after the reset
            _compare_state(host, fused, rows=done, what=(i, "reset envs"))
    return worst, resets


@pytest.mark.parametrize("num_envs,steps,nan_step", [(256, 120, 7), (4100, 30, None), (65536, 20, None)])
def test_workload_a_matches_the_host_columns_in_one_launch(num_envs, steps, nan_step, cuda_device, monkeypatch):
    host, fused = _pair(num_envs, cuda_device, 11, monkeypatch)
    assert not fused._fused.split_mode
    _compare_state(host, fused, what="after reset")
    observed = fused._fused.spec_stats()["user_observe_launches"]
    gen = torch.Generator(device=cuda_device).manual_seed(3)
    worst, resets = _run(host, fused, steps, gen, nan_step)
    _compare_state(host, fused, rows=slice(num_envs - 1, num_envs))  # env N-1: shadowed by a tail slab's lanes
    stats = fused._fused.spec_stats()
    assert stats["specialised_launches"] == steps, stats  # one launch per step (the reset launches run generic)
    assert stats["user_observe_launches"] > observed, stats
    assert resets > 0
    print(f"STATEFUL-OBS A N={num_envs} steps={steps} resets={resets} max_abs={worst:.3e} {stats}")


@pytest.mark.parametrize("num_envs,steps", [(256, 60), (4100, 20)])
def test_workload_a_split_matches_the_host_columns(num_envs, steps, cuda_device, monkeypatch):
    host, fused = _pair(num_envs, cuda_device, 13, monkeypatch, spec=so.stateful_observations_split)
    assert fused._fused.split_mode and len(fused._fused.user_obs) == 5
    gen = torch.Generator(device=cuda_device).manual_seed(4)
    worst, resets = _run(host, fused, steps, gen, nan_step=5)
    assert resets > 0 and fused._fused.spec_stats()["specialised_launches"] > 0
    print(f"STATEFUL-OBS A-split N={num_envs} resets={resets} max_abs={worst:.3e}")


def test_between_steps(cuda_device, monkeypatch):
    """get_observations on a fresh extras, reset(subset), reset(), host edits: both envs stay equal."""
    host, fused = _pair(256, cuda_device, 7, monkeypatch)
    gen = torch.Generator(device=cuda_device).manual_seed(5)

    def edit(i, *envs):
        for env in envs:
            om = env.managers["observation"][0]
            if i == 3:
                env.extras.pop("observations", None)
                env.get_observations()  # evaluates (and advances) every env once more
            if i == 5:
                env.reset(torch.arange(0, 256, 7, device=cuda_device))
            if i == 8:
                env.reset()
            if i == 10:  # a manual reset of some rows, in place, and a compatible rebinding
                om.cfg["still_steps"].fn.count[:10] = 3
                om.cfg["gait_clock"].fn.phase = torch.zeros_like(om.cfg["gait_clock"].fn.phase)
            if i == 14:  # incompatible: the lowered terms become host columns from here on
                om.cfg["action_history"].fn.prev1 = om.cfg["action_history"].fn.prev1.to(torch.float64)
        if i in (3, 8):
            _compare_obs(envs[0], envs[1], (i, "observe"))
            _compare_state(envs[0], envs[1], what=(i, "observe"))

    _run(host, fused, 20, gen, edit=edit)
    f = fused._fused
    assert f.split_mode and not f.stateful and "action_history" in f.user_term_refusals[("observation", "action_history")]


def test_without_specialisation_the_terms_stay_host_columns(cuda_device, monkeypatch):
    import genesis_forge_b200 as gfb
    from configs.env_builder import build_env, dropin_namespace
    from genesis_forge_b200.managed_env import ManagedEnvironment

    monkeypatch.setenv("GFB_NO_SPEC", "1")
    envs = []
    for fuse in (True, False):
        monkeypatch.setattr(ManagedEnvironment, "fuse_stateful_terms", fuse)
        gfb.set_device(cuda_device)
        env = build_env(so.stateful_observations(), dropin_namespace(), 256, cuda_device, pool=4, seed=1,
                        n_contacts=0, apply_setters=False)
        env.build()
        env.reset()
        envs.append(env)
    off, ref = envs  # the switch on without a specialisation; the switch off
    f = off._fused
    assert f.split_mode and not f.stateful and not f.user_obs and len(f.external_obs) == 5
    gen = torch.Generator(device=cuda_device).manual_seed(1)
    for i in range(10):
        actions = torch.randn(256, 12, device=cuda_device, generator=gen)
        a, b = ref.step(actions), off.step(actions.clone())
        assert torch.equal(a[1], b[1]) and torch.equal(a[2], b[2]), i
        for om_r, om_o in zip(ref.managers["observation"], off.managers["observation"]):
            assert torch.equal(om_r.get_observations(), om_o.get_observations()), (i, om_r.name)
    a, b = _state(ref), _state(off)
    assert all(torch.equal(a[k], b[k]) for k in a)
    assert f.spec_stats()["specialised_launches"] == 0


def _port_instances(monkeypatch):
    """The oracle port calls a user observation term as fn(env=env): a class-style one is instantiated once, with
    the port environment, and that instance is called every time, as the ObservationManager does."""
    from genesis_forge_b200.managers.config import MdpFnClass
    from oracle import manager_port, parity

    held = {}
    plain, plain_width = manager_port.PortEnv._obs_value, parity.ParityRun._term_width

    def obs_value(self, term):
        cls = term["fn"]
        if isinstance(cls, type) and issubclass(cls, MdpFnClass):
            if cls not in held:
                held[cls] = cls(self)
                held[cls].build()
            return held[cls](env=self)
        return plain(self, term)

    def term_width(self, term):  # (the column layout: from a throw-away instance, the held one's state stays)
        cls = term["fn"]
        if isinstance(cls, type) and issubclass(cls, MdpFnClass):
            return int(cls(self.port)(env=self.port).reshape(self.N, -1).shape[1])
        return plain_width(self, term)

    monkeypatch.setattr(manager_port.PortEnv, "_obs_value", obs_value)
    monkeypatch.setattr(parity.ParityRun, "_term_width", term_width)
    return held


@pytest.mark.parametrize("num_envs,steps,philox", [(4096, 40, False), (65536, 6, True)])
def test_workload_b_matches_the_oracle_port(num_envs, steps, philox, cuda_device, monkeypatch):
    from genesis_forge_b200.managed_env import ManagedEnvironment
    from oracle.parity import ParityRun

    monkeypatch.setattr(ManagedEnvironment, "fuse_stateful_terms", True)
    held = _port_instances(monkeypatch)
    run = ParityRun("contacts", num_envs=num_envs, device=cuda_device, seed=1234 if not philox else 11,
                    spec_override=so.contacts_override(), philox=philox)
    fused = run.env._fused
    assert not fused.split_mode and not fused.external_obs and not fused.user_term_refusals
    assert len(fused.stateful) == 1
    stats = run.run(steps=steps, nan_step=3 if not philox else None)
    assert stats["resets"] > 0
    since = run.env.managers["observation"][0].cfg["touchdown_clock"].fn.since
    assert bool((since > 0).any())
    want = held[so.touchdown_clock].since
    assert torch.allclose(since.cpu(), want.cpu(), rtol=1e-5, atol=1e-6), float((since.cpu() - want.cpu()).abs().max())
    assert fused.spec_stats()["specialised_launches"] == steps
    print(f"STATEFUL-OBS B N={num_envs} max_abs={stats['max_abs']:.3e} max_rel={stats['max_rel']:.3e}")
