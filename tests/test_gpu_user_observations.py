"""
User-defined observation terms lowered into the specialised post-physics kernel and its reset-path kernel
(ManagedEnvironment.fuse_user_observations, configs/user_observations.py).  Workload A against the oracle
port, workload B against the same functions run as host columns.  Bar: masks / counters / reset indices
bit-exact; fp32 within 1e-5 rel + 1e-6 (sin / cos may differ in the last ulp between Sleef and CUDA).
"""
import pytest

from configs import user_observations as uo

pytestmark = pytest.mark.gpu


@pytest.fixture()
def fused_user_obs(monkeypatch):
    from genesis_forge_b200.managed_env import ManagedEnvironment

    monkeypatch.setattr(ManagedEnvironment, "fuse_user_observations", True)


@pytest.mark.parametrize("num_envs,steps,nan_step,philox", [(256, 120, 7, False), (65536, 4, None, True)])
def test_workload_a_matches_the_port_in_one_launch(num_envs, steps, nan_step, philox, cuda_device, fused_user_obs):
    from oracle.parity import ParityRun

    run = ParityRun("contacts", num_envs=num_envs, device=cuda_device, seed=1234 if num_envs == 256 else 11,
                    spec_override=uo.override(noise=not philox), philox=philox)
    fused = run.env._fused
    assert not fused.split_mode and not fused.external_obs and not fused.user_term_refusals
    assert len(fused.user_obs) == 8
    stats = run.run(steps=steps, nan_step=nan_step)
    assert stats["resets"] > 0
    spec_stats = fused.spec_stats()
    # one specialised post launch per step (the reset launch runs the generic kernel); the reset path's kernel
    # ran for the initial observation and for every step with resets
    assert spec_stats["specialised_launches"] == steps, spec_stats
    assert spec_stats["user_observe_launches"] >= 2, spec_stats
    print(f"USER-OBS A N={num_envs} philox={philox} resets={stats['resets']} max_abs={stats['max_abs']:.3e} "
          f"max_rel={stats['max_rel']:.3e} {spec_stats}")


def _pair(num_envs, cuda_device, seed, spec=uo.user_observations_entity):
    """The same seeded workload twice: user observation terms as host columns / lowered."""
    import genesis_forge_b200 as gfb
    from configs.env_builder import build_env, dropin_namespace
    from genesis_forge_b200.managed_env import ManagedEnvironment

    envs = []
    for fuse in (False, True):
        ManagedEnvironment.fuse_user_observations = fuse
        gfb.set_device(cuda_device)
        env = build_env(spec(), dropin_namespace(), num_envs, cuda_device, pool=4, seed=seed, n_contacts=0,
                        apply_setters=False)
        env.build()
        env.reset()
        envs.append(env)
    return envs


def _close(got, want):
    import torch

    both_nan = got.isnan() & want.isnan()
    err = torch.where(both_nan, 0.0, (got - want).abs())
    return bool((both_nan | (err <= 1e-6 + 1e-5 * want.abs())).all()), float(err.max())


@pytest.mark.parametrize("num_envs,steps,nan_step", [(256, 120, 7), (65536, 20, None)])
def test_workload_b_matches_the_host_columns(num_envs, steps, nan_step, cuda_device, monkeypatch):
    import torch

    from genesis_forge_b200.managed_env import ManagedEnvironment

    monkeypatch.setattr(ManagedEnvironment, "fuse_user_observations", ManagedEnvironment.fuse_user_observations)
    host, fused = _pair(num_envs, cuda_device, seed=11)
    assert host._fused.split_mode and len(host._fused.external_obs) == 6
    assert not fused._fused.split_mode and not fused._fused.external_obs and not fused._fused.user_term_refusals
    ok, err = _close(fused.get_observations(), host.get_observations())
    assert ok, ("initial observation", err)
    gen = torch.Generator(device=cuda_device).manual_seed(3)
    worst, resets = 0.0, 0
    for i in range(steps):
        actions = torch.randn(num_envs, 12, device=cuda_device, generator=gen)
        if nan_step is not None and i == nan_step:
            actions[3, 1] = float("nan")
        a, b = host.step(actions), fused.step(actions.clone())
        assert torch.equal(a[2], b[2]) and torch.equal(a[3], b[3]), i
        resets += int((a[2] | a[3]).sum())
        for got, want, what in ((b[0], a[0], "obs"), (b[1], a[1], "rewards")):
            ok, err = _close(got, want)
            assert ok, (i, what, err)
            worst = max(worst, err)
    stats = fused._fused.spec_stats()
    assert stats["specialised_launches"] == steps and stats["user_observe_launches"] >= 1, stats
    assert resets > 0
    print(f"USER-OBS B N={num_envs} steps={steps} resets={resets} max_abs={worst:.3e} {stats}")


def test_without_specialisation_the_terms_stay_host_columns(cuda_device, fused_user_obs, monkeypatch):
    from oracle.parity import ParityRun

    monkeypatch.setenv("GFB_NO_SPEC", "1")
    run = ParityRun("contacts", num_envs=256, device=cuda_device, seed=1234, spec_override=uo.override())
    fused = run.env._fused
    assert fused.split_mode and not fused.user_obs and len(fused.external_obs) == 8
    stats = run.run(steps=30, nan_step=7)
    assert stats["resets"] > 0 and fused.spec_stats()["specialised_launches"] == 0


def test_a_failed_specialisation_demotes_the_terms(cuda_device, fused_user_obs, monkeypatch):
    """No specialised library can be built: the lowered terms become host columns and the results hold."""
    from genesis_forge_b200 import spec
    from oracle.parity import ParityRun

    def no_compiler(*args, **kwargs):
        raise RuntimeError("nvcc failed (simulated)")

    monkeypatch.setattr(spec, "ensure", no_compiler)
    run = ParityRun("contacts", num_envs=256, device=cuda_device, seed=1234, spec_override=uo.override())
    fused = run.env._fused
    assert not fused.split_mode and len(fused.user_obs) == 8
    stats = run.run(steps=20, nan_step=7)
    assert fused.split_mode and not fused.user_obs and len(fused.external_obs) == 8
    assert ("observation", "gait_clock") in fused.user_term_refusals
    assert stats["resets"] > 0 and fused.spec_stats()["specialised_launches"] == 0


def test_a_closure_constant_is_part_of_the_library_identity(cuda_device, monkeypatch):
    """Two tables that differ only in an observation term's closure constant get different libraries, and a
    library attached to the other table's handle is not run there."""
    import torch

    from genesis_forge_b200 import spec
    from genesis_forge_b200.managed_env import ManagedEnvironment

    monkeypatch.setattr(ManagedEnvironment, "fuse_user_observations", ManagedEnvironment.fuse_user_observations)

    def with_gain(gain):
        def tilt(env):
            return env.robot_manager.get_projected_gravity()[:, :2] * gain

        def make():
            s = uo.user_observations_entity()
            s["observations"]["policy"]["terms"]["upright"] = {"fn": tilt}
            return s
        return make

    envs = []
    for gain in (2.0, 3.0):
        host, fused = _pair(256, cuda_device, seed=5, spec=with_gain(gain))
        envs.append((host, fused))
    (host2, fused2), (host3, fused3) = envs
    libs2, libs3 = set(fused2._fused.spec_stats()["libraries"]), set(fused3._fused.spec_stats()["libraries"])
    assert libs2 and libs3 and not libs2 & libs3
    for path in fused2._fused.spec_paths:  # the other table's library, attached to this handle as well
        spec.attach(fused3._fused, path)
    gen = torch.Generator(device=cuda_device).manual_seed(9)
    for i in range(12):
        actions = torch.randn(256, 12, device=cuda_device, generator=gen)
        for host, fused in envs:
            a, b = host.step(actions), fused.step(actions.clone())
            ok, err = _close(b[0], a[0])
            assert ok, (i, err)
    assert fused3._fused.spec_stats()["specialised_launches"] == 12
