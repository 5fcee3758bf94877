"""
User terms that read per-link state (configs/link_terms.py) lowered into the specialised post-physics kernel and
its reset-path kernel, against the same functions run as host callbacks / host columns on the drop-in (every
lowering switch off), same seeds.  Bar: masks, counters, reset lists and observations bit-exact (foot speeds,
3-norms, within the reward bar); rewards within 1e-5 rel + 1e-6 -- at 65536 envs against the Python functions on
the fused environment's own state, because split execution of a contacts table is not run-to-run deterministic
there.  The reset path is checked with an engine whose reset moves the links of the reset envs.
"""
import pytest
import torch

from configs import link_terms

pytestmark = pytest.mark.gpu

SWITCHES = ("fuse_user_terms", "fuse_user_observations", "fuse_stateful_terms")
FEET = [4, 8, 12, 16]


def _build(spec, num_envs, cuda_device, seed, monkeypatch, fuse, apply_setters=False):
    import genesis_forge_b200 as gfb
    from configs.env_builder import build_env, dropin_namespace
    from genesis_forge_b200.managed_env import ManagedEnvironment

    for name in SWITCHES:
        monkeypatch.setattr(ManagedEnvironment, name, fuse)
    gfb.set_device(cuda_device)
    env = build_env(spec, dropin_namespace(), num_envs, cuda_device, pool=4, seed=seed, n_contacts=8,
                    apply_setters=apply_setters)
    env.build()
    env.reset()
    return env


def _pair(spec_fn, num_envs, cuda_device, seed, monkeypatch, apply_setters=False):
    host = _build(spec_fn(), num_envs, cuda_device, seed, monkeypatch, False, apply_setters)
    fused = _build(spec_fn(), num_envs, cuda_device, seed, monkeypatch, True, apply_setters)
    return host, fused


def _inject(envs, num_envs, cuda_device, gen):
    """The same dense draws for both environments (the injected mode of the kernel)."""
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


def _feet_rel_base(env):
    robot = env.robot
    return (robot.get_links_pos(links_idx_local=FEET) - robot.get_pos().unsqueeze(1)).flatten(1)


def _run(host, fused, steps, gen, check_reset_path=False, contact_rewards=True):
    """`contact_rewards=False`: rewards and the swing-peak state (both read contact forces) are not compared --
    split execution of a contacts table is not run-to-run deterministic at 65536 envs and above (DESIGN.md
    section 9), so the host-callback reference is no reference for them there."""
    N = fused.num_envs
    worst, resets = 0.0, 0
    for i in range(steps):
        actions = torch.randn(N, 12, device=fused.episode_length.device, generator=gen)
        a, b = host.step(actions), fused.step(actions.clone())
        assert torch.equal(a[2], b[2]) and torch.equal(a[3], b[3]), i
        assert torch.equal(host.episode_length, fused.episode_length), i
        assert torch.equal(host._fused.reset_idx, fused._fused.reset_idx), i
        obs_h, obs_f = host.managers["observation"][0].get_observations(), fused.managers["observation"][0].get_observations()
        # stock columns and feet_rel_base (a difference) bit-exact; foot_speed is a 3-norm, which torch's CUDA
        # reduction may round differently from the kernel's (torch-CPU's) sum order
        assert torch.equal(obs_f[:, :60], obs_h[:, :60]), i
        worst = max(worst, _close(obs_f[:, 60:], obs_h[:, 60:], (i, "foot_speed")))
        if contact_rewards:
            worst = max(worst, _close(b[1], a[1], (i, "rewards")))
            peak_h = host.managers["reward"].cfg["swing_peak"].fn.peak
            peak_f = fused.managers["reward"].cfg["swing_peak"].fn.peak
            worst = max(worst, _close(peak_f, peak_h, (i, "swing_peak state")))
        done = a[2] | a[3]
        resets += int(done.sum())
        if check_reset_path and bool(done.any()):
            # a reset env's lowered link observation reads the links after the reset fan-out, as the getter does
            obs = fused.managers["observation"][0].get_observations()
            assert torch.equal(obs[done, 48:60], _feet_rel_base(fused)[done]), i
    return worst, resets


@pytest.mark.parametrize("num_envs,steps,injected", [(4096, 48, True), (4096, 40, False), (65536, 40, False),
                                                     (65536, 40, True)])
def test_lowered_link_terms_match_the_host_callbacks(num_envs, steps, injected, cuda_device, monkeypatch):
    host, fused = _pair(link_terms.link_terms, num_envs, cuda_device, 7, monkeypatch)
    f = fused._fused
    assert host._fused.split_mode and not host._fused.user_terms and not host._fused.user_obs
    assert not f.split_mode and not f.user_term_refusals and f._link_layout
    gen = torch.Generator(device=cuda_device).manual_seed(3)
    if injected:
        _inject([host, fused], num_envs, cuda_device, gen)
    before = f.spec_stats()["specialised_launches"]
    # (rewards at 65536: test_rewards_at_65536_match_the_functions_on_the_fused_state)
    worst, resets = _run(host, fused, steps, gen, contact_rewards=num_envs <= 4096)
    stats = f.spec_stats()
    assert stats["specialised_launches"] - before == steps, stats  # one post-physics launch a step
    assert resets > 0
    print(f"LINK-TERMS N={num_envs} injected={injected} resets={resets} max_abs={worst:.3e} {stats}")


def _moving_reset(monkeypatch):
    """An engine whose base reset also moves the links of the reset envs (links around the new base)."""
    from genesis_forge_b200.synthetic import SyntheticRobot

    plain = SyntheticRobot.set_pos

    def set_pos(self, pos, envs_idx=None, zero_velocity=True, relative=False):
        plain(self, pos, envs_idx, zero_velocity, relative)
        if self._scene.apply_setters:
            offset = torch.linspace(-0.5, 0.5, self._scene.state["links_pos"].shape[1], device=pos.device)
            self._scene.state["links_pos"][envs_idx] = pos.unsqueeze(1) + offset[None, :, None]

    monkeypatch.setattr(SyntheticRobot, "set_pos", set_pos)


def test_reset_path_reads_post_reset_links(cuda_device, monkeypatch):
    _moving_reset(monkeypatch)
    host, fused = _pair(link_terms.link_terms, 4096, cuda_device, 9, monkeypatch, apply_setters=True)
    assert not fused._fused.split_mode and fused._fused._obs_reads_links
    observed = fused._fused.spec_stats()["user_observe_launches"]
    gen = torch.Generator(device=cuda_device).manual_seed(5)
    worst, resets = _run(host, fused, 40, gen, check_reset_path=True)
    assert resets > 0 and fused._fused.spec_stats()["user_observe_launches"] > observed
    print(f"LINK-TERMS reset path resets={resets} max_abs={worst:.3e}")


def _split_spec():
    s = link_terms.link_terms()
    # a callback the tracer refuses (cumsum): the step runs split, the lowered terms in their launches
    s["rewards"] = dict(s["rewards"], host_only={"fn": lambda env: env.robot.get_vel()[:, :2].cumsum(1)[:, 1],
                                                 "weight": 0.1})
    return s


def test_split_step_observes_post_reset_links(cuda_device, monkeypatch):
    _moving_reset(monkeypatch)
    host, fused = _pair(_split_spec, 4096, cuda_device, 9, monkeypatch, apply_setters=True)
    f = fused._fused
    assert f.split_mode and [n for _, n, _ in f.external_rows] == ["host_only"] and len(f.user_obs) == 2
    gen = torch.Generator(device=cuda_device).manual_seed(6)
    worst, resets = _run(host, fused, 40, gen, check_reset_path=True)
    assert resets > 0 and f.spec_stats()["specialised_launches"] > 0
    print(f"LINK-TERMS split resets={resets} max_abs={worst:.3e}")


def _one_link(env, link=4):  # (an int param used as an index: traced with params as constants)
    return env.robot.get_links_pos(links_idx_local=[link])[:, 0, 2]


def _one_link_spec():
    s = link_terms.link_terms()
    s["rewards"] = dict(s["rewards"], one_link={"fn": _one_link, "weight": 0.2, "params": {"link": 4}})
    return s


def test_a_specialisation_that_cannot_be_attached_demotes_the_terms(cuda_device, monkeypatch):
    """Mid-run, an edit traces a term again and no specialised kernel can be attached for the new table: the
    step's launch is refused before anything runs, the lowered terms become callbacks, the results hold and the
    class-style term continues from the state the kernel left."""
    from genesis_forge_b200 import spec

    host, fused = _pair(_one_link_spec, 4096, cuda_device, 7, monkeypatch)
    f = fused._fused
    assert not f.split_mode and ("reward", "one_link") in f.user_terms
    gen = torch.Generator(device=cuda_device).manual_seed(8)
    _run(host, fused, 10, gen)  # lowered: swing_peak's state advances in the kernel

    def no_compiler(*args, **kwargs):
        raise RuntimeError("nvcc failed (simulated)")

    monkeypatch.setattr(spec, "ensure", no_compiler)
    for env in (host, fused):
        env.managers["reward"].cfg["one_link"].params["link"] = 8
    worst, resets = _run(host, fused, 30, gen)
    assert f.split_mode and not f.user_terms and not f._link_layout
    assert "no specialised kernel" in f.user_term_refusals[("reward", "swing_peak")], f.user_term_refusals
    assert resets > 0
    print(f"LINK-TERMS demoted resets={resets} max_abs={worst:.3e}")


def _rewards_only():
    s = link_terms.link_terms()
    s["rewards"] = {k: v for k, v in s["rewards"].items() if k in link_terms.LINK_REWARDS}
    return s


@pytest.mark.parametrize("injected", [False, True])
def test_rewards_at_65536_match_the_functions_on_the_fused_state(injected, cuda_device, monkeypatch):
    """The lowered rewards at 65536 envs against the Python functions evaluated on the fused environment's own
    state (pool states, engine-side resets not applied: after the step it is the state the kernel read), the
    class-style term from a twin holding the state of before the step -- no split execution involved."""
    fused = _build(_rewards_only(), 65536, cuda_device, 7, monkeypatch, True)
    f = fused._fused
    assert not f.split_mode and not f.user_term_refusals and len(f.user_terms) == 6
    gen = torch.Generator(device=cuda_device).manual_seed(11)
    if injected:
        _inject([fused], 65536, cuda_device, gen)
    cfg = fused.managers["reward"].cfg
    inst = cfg["swing_peak"].fn
    worst = 0.0
    for i in range(20):
        twin = type(inst).__new__(type(inst))
        twin.__dict__.update({k: v.clone() if torch.is_tensor(v) else v for k, v in vars(inst).items()})
        out = fused.step(torch.randn(65536, 12, device=cuda_device, generator=gen))
        want = torch.zeros(65536, device=cuda_device)
        for name, item in cfg.items():
            fn = item.fn
            value = type(fn).__call__(twin, fused, **item.params) if fn is inst else fn(fused, **item.params)
            want = want + value.float() * torch.tensor(item.weight * fused.dt, dtype=torch.float32)
        worst = max(worst, _close(out[1], want, (i, "rewards")), _close(inst.peak, twin.peak, (i, "swing_peak")))
    print(f"LINK-TERMS rewards N=65536 injected={injected} max_abs={worst:.3e}")


def test_without_an_attachable_specialisation_the_terms_stay_callbacks(cuda_device, monkeypatch):
    from genesis_forge_b200 import spec

    def no_compiler(*args, **kwargs):
        raise RuntimeError("nvcc failed (simulated)")

    monkeypatch.setattr(spec, "ensure", no_compiler)
    host, fused = _pair(link_terms.link_terms, 4096, cuda_device, 7, monkeypatch)
    gen = torch.Generator(device=cuda_device).manual_seed(9)
    worst, resets = _run(host, fused, 20, gen)
    f = fused._fused
    assert f.split_mode and not f.user_terms and not f._link_layout and resets > 0
    assert f.spec_stats()["specialised_launches"] == 0
