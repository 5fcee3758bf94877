"""
User-defined reward / termination terms lowered into the specialised post-physics kernel
(ManagedEnvironment.fuse_user_terms, genesis_forge_b200/expr.py) against the oracle port, which calls
the same Python functions on CPU tensors.  Bar: masks / counters / reset indices bit-exact; fp32
within 1e-5 rel + 1e-6 (exp / sin / log / tanh may differ in the last ulp between Sleef and CUDA).
"""
import pytest

from configs import user_terms

pytestmark = pytest.mark.gpu


@pytest.fixture()
def fused_user_terms(monkeypatch):
    from genesis_forge_b200.managed_env import ManagedEnvironment

    monkeypatch.setattr(ManagedEnvironment, "fuse_user_terms", True)


def _user_library(fused):
    """Library file of the specialised one-launch kernel carrying this table's user-term code."""
    from genesis_forge_b200 import _native as nat
    from genesis_forge_b200 import spec

    phases = nat.K["GFB_PHASE_ALL"]
    canon, plan, tile = spec.describe(fused, phases)
    text = spec.header_text(canon, plan, tile, phases, fused.user_code)
    assert "GFB_SPEC_USER_TERMS" in text
    return spec.library_path(spec.key_of(text)).name


@pytest.mark.parametrize("num_envs,steps,nan_step,philox", [(256, 120, 7, False), (65536, 4, 1, False),
                                                            (65536, 4, None, True)])
def test_user_terms_run_in_one_launch(num_envs, steps, nan_step, philox, cuda_device, fused_user_terms):
    from oracle.parity import ParityRun

    run = ParityRun("contacts", num_envs=num_envs, device=cuda_device, seed=1234 if num_envs == 256 else 11,
                    spec_override=user_terms.override(), philox=philox)
    fused = run.env._fused
    assert not fused.split_mode and not fused.external_rows and not fused.user_term_refusals
    stats = run.run(steps=steps, nan_step=nan_step)
    assert stats["resets"] > 0
    spec_stats = fused.spec_stats()
    assert spec_stats["specialised_launches"] == steps and spec_stats["generic_launches"] == 2, spec_stats
    assert _user_library(fused) in spec_stats["libraries"], spec_stats
    print(f"USER-TERMS N={num_envs} philox={philox} max_abs={stats['max_abs']:.3e} max_rel={stats['max_rel']:.3e} "
          f"inexact={stats['inexact']}")


def _launches_per_step(name, cuda_device, steps=20):
    from oracle.parity import ParityRun

    run = ParityRun(name, num_envs=256, device=cuda_device, seed=1234)
    run.reset()
    before = run.env._fused.launch_count()
    for _ in range(steps):
        run.step()
    return (run.env._fused.launch_count() - before) / steps, run


def test_custom_terms_keep_only_their_callbacks(cuda_device, monkeypatch):
    from genesis_forge_b200.managed_env import ManagedEnvironment

    split, _ = _launches_per_step("custom_terms", cuda_device)
    monkeypatch.setattr(ManagedEnvironment, "fuse_user_terms", True)
    fused_rate, run = _launches_per_step("custom_terms", cuda_device)
    fused = run.env._fused
    assert fused.split_mode and not fused.external_rows  # the user-level command manager and observation remain
    assert fused_rate < split, (fused_rate, split)
    print(f"custom_terms launches per step: split {split}, with lowered user terms {fused_rate}")


def test_live_param_mutation_keeps_the_library(cuda_device, fused_user_terms):
    from oracle.parity import ParityRun

    run = ParityRun("contacts", num_envs=256, device=cuda_device, seed=3, spec_override=user_terms.override())
    run.reset()
    for _ in range(8):
        run.step()
    for kind, name, key, value in (("rewards", "level_speed", "scale", 0.75), ("rewards", "action_excess", "lim", 0.5),
                                   ("terminations", "wandered_off", "limit", 8.0)):
        mgr = run.env.reward_manager.cfg if kind == "rewards" else run.env.termination_manager.term_cfg
        mgr[name].params[key] = value
        run.port.spec[kind][name]["params"][key] = value
    for _ in range(12):
        run.step()
    stats = run.env._fused.spec_stats()
    assert stats["specialised_launches"] == 20 and len(stats["libraries"]) == 1, stats


def test_without_specialisation_the_terms_stay_callbacks(cuda_device, fused_user_terms, monkeypatch):
    from oracle.parity import ParityRun

    monkeypatch.setenv("GFB_NO_SPEC", "1")
    run = ParityRun("contacts", num_envs=256, device=cuda_device, seed=1234, spec_override=user_terms.override())
    fused = run.env._fused
    assert fused.split_mode and not fused.user_terms and len(fused.external_rows) == 11
    stats = run.run(steps=30, nan_step=7)
    assert stats["resets"] > 0 and fused.spec_stats()["specialised_launches"] == 0


def _pair(num_envs, cuda_device, seed):
    """The entity workload twice on the same seeded states: user terms as host callbacks / lowered."""
    import genesis_forge_b200 as gfb
    from configs.env_builder import build_env, dropin_namespace
    from genesis_forge_b200.managed_env import ManagedEnvironment

    envs = []
    for fuse in (False, True):
        ManagedEnvironment.fuse_user_terms = fuse
        gfb.set_device(cuda_device)
        env = build_env(user_terms.user_terms_entity(), dropin_namespace(), num_envs, cuda_device, pool=4, seed=seed,
                        n_contacts=0, apply_setters=False)
        env.build()
        env.reset()
        envs.append(env)
    return envs


@pytest.mark.parametrize("num_envs,steps,nan_step", [(256, 120, 7), (65536, 4, 1), (65536, 20, None)])
def test_manager_getter_terms_match_the_callback_path(num_envs, steps, nan_step, cuda_device, monkeypatch):
    """
    The EntityManager / action-manager sources (body-frame vectors, cached pose, joint state, targets) and
    the ops the first workload does not use, against the same functions run as host callbacks on the
    drop-in (the oracle port has no manager objects for user terms to call).  Production Philox draws.
    """
    import torch

    from genesis_forge_b200.managed_env import ManagedEnvironment

    monkeypatch.setattr(ManagedEnvironment, "fuse_user_terms", ManagedEnvironment.fuse_user_terms)
    split, fused = _pair(num_envs, cuda_device, seed=11)
    assert split._fused.split_mode and not fused._fused.split_mode and not fused._fused.user_term_refusals
    gen = torch.Generator(device=cuda_device).manual_seed(3)
    names = list(fused.reward_manager.cfg)
    worst, resets = 0.0, 0
    for i in range(steps):
        actions = torch.randn(num_envs, 12, device=cuda_device, generator=gen)
        if nan_step is not None and i == nan_step:
            actions[3, 1] = float("nan")
        a, b = split.step(actions), fused.step(actions.clone())
        assert torch.equal(a[2], b[2]) and torch.equal(a[3], b[3]), i
        resets += int((a[2] | a[3]).sum())
        for got, want, what in ((b[1], a[1], "rewards"), (b[0], a[0], "obs"),
                                (fused.reward_manager._episode_sums, split.reward_manager._episode_sums, "sums")):
            both_nan = got.isnan() & want.isnan()  # (the NaN action reaches the observed raw actions)
            err = torch.where(both_nan, 0.0, (got - want).abs())
            ok = both_nan | (err <= 1e-6 + 1e-5 * want.abs())
            assert bool(ok.all()), (i, what, float(err.max()),
                                                                   names if what == "sums" else None)
            worst = max(worst, float(err.max()))
    stats = fused._fused.spec_stats()
    assert stats["specialised_launches"] == steps, stats
    assert resets > 0
    print(f"USER-TERMS-ENTITY N={num_envs} steps={steps} resets={resets} max_abs={worst:.3e}")


def test_a_specialisation_that_cannot_be_attached_falls_back_to_callbacks(cuda_device, fused_user_terms,
                                                                           monkeypatch):
    """The first step finds no specialised kernel for the lowered terms: they become host callbacks, results hold."""
    from genesis_forge_b200 import spec
    from oracle.parity import ParityRun

    def no_compiler(*args, **kwargs):
        raise RuntimeError("nvcc failed (simulated)")

    monkeypatch.setattr(spec, "ensure", no_compiler)
    run = ParityRun("contacts", num_envs=256, device=cuda_device, seed=1234, spec_override=user_terms.override())
    fused = run.env._fused
    assert not fused.split_mode and len(fused.user_terms) == 11
    stats = run.run(steps=20, nan_step=7)
    assert fused.split_mode and not fused.user_terms and len(fused.external_rows) == 11
    assert "no specialised kernel" in fused.user_term_refusals[("reward", "contact_z")]
    assert stats["resets"] > 0 and fused.spec_stats()["specialised_launches"] == 0
