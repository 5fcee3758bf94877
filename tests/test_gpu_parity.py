"""
GPU parity tests proper: the CUDA drop-in, called through the C ABI, against the oracle port on the
same seeded inputs, step by step with resets, resamples, a NaN-action step and (short-episode
variants) timeouts.  Bar: masks / counters / reset indices bit-exact; fp32 within 1e-5 rel + 1e-6.
"""
import pytest
import torch

pytestmark = pytest.mark.gpu

CONFIGS = ["simple", "command_direction", "contacts", "gait_trainer", "rough_terrain", "berkeley_humanoid",
           "kitchen_sink", "custom_terms"]
SPLIT = {"custom_terms", "gait_trainer"}  # user-defined Python terms / managers: kernel phases as separate launches


@pytest.mark.parametrize("name", CONFIGS)
def test_step_parity(name, cuda_device):
    """Default path: the specialised kernel for the config's table structure."""
    from oracle.parity import ParityRun

    run = ParityRun(name, num_envs=256, device=cuda_device, seed=1234)
    stats = run.run(steps=120, nan_step=7)
    assert stats["steps"] == 120
    assert stats["resets"] > 0
    spec_stats = run.env._fused.spec_stats()
    if name in SPLIT:
        # several launches per step with the Python callbacks in between, every one of them specialised
        assert run.env._fused.split_mode, spec_stats
        per_step = len(run.env._fused.split_plan)
        assert spec_stats["generic_launches"] == 2 and spec_stats["specialised_launches"] == per_step * 120, spec_stats
    else:
        # (the two generic launches are the build-time entity phase and the initial reset phase)
        assert spec_stats["specialised_launches"] == 120 and spec_stats["generic_launches"] == 2, spec_stats
    print(name, stats, spec_stats)


@pytest.mark.parametrize("name", CONFIGS)
def test_step_parity_generic_interpreter(name, cuda_device, monkeypatch):
    """Same run through the generic (interpreting) kernel: what runs when no specialisation exists."""
    from oracle.parity import ParityRun

    monkeypatch.setenv("GFB_NO_SPEC", "1")
    run = ParityRun(name, num_envs=256, device=cuda_device, seed=1234)
    stats = run.run(steps=60, nan_step=7)
    assert stats["resets"] > 0
    spec_stats = run.env._fused.spec_stats()
    assert spec_stats["specialised_launches"] == 0
    per_step = len(run.env._fused.split_plan) if name in SPLIT else 1
    assert spec_stats["generic_launches"] == 2 + per_step * 60


def _benchmark_library(fused):
    """(slab size, library file) of the specialised fused launch this environment's step uses."""
    from genesis_forge_b200 import _native as nat
    from genesis_forge_b200 import spec

    phases = nat.K["GFB_PHASE_ALL"]
    canon, plan, tile = spec.describe(fused, phases)
    return tile, spec.library_path(spec.key_of(spec.header_text(canon, plan, tile, phases))).name


BENCH_SIZES = [("command_direction", 32768), ("command_direction", 65536), ("contacts", 32768), ("contacts", 65536),
               ("rough_terrain", 32768), ("rough_terrain", 65536), ("berkeley_humanoid", 32768),
               ("berkeley_humanoid", 65536)]


@pytest.mark.parametrize("name,num_envs", BENCH_SIZES)
def test_step_parity_at_benchmark_slab_sizes(name, num_envs, cuda_device):
    """
    Default mode (no switches) at the batch sizes where the library picks the LARGE slabs (128 envs,
    or 64 with contact slots staged): the specialised one-launch kernels of the BASELINE configs, whose
    slab plan, row-assembly ownership and late-load overlay all depend on the slab size, against the
    oracle value by value.
    """
    from oracle.parity import ParityRun

    run = ParityRun(name, num_envs=num_envs, device=cuda_device, seed=2025)
    stats = run.run(steps=4, nan_step=1)
    fused = run.env._fused
    spec_stats = fused.spec_stats()
    tile, library = _benchmark_library(fused)
    assert tile in (64, 128), tile
    assert spec_stats["specialised_launches"] == 4 and library in spec_stats["libraries"], (spec_stats, library)
    assert stats["resets"] > 0
    print(f"PARITY-VARIANT {name} N={num_envs} slab={tile} draws=injected library={library} stats={stats}")


@pytest.mark.parametrize("name,num_envs,steps", [
    ("command_direction", 65536, 6), ("contacts", 65536, 4), ("rough_terrain", 262144, 3),
    ("berkeley_humanoid", 65536, 4), ("command_direction", 1 << 20, 2), ("berkeley_humanoid", 1 << 20, 2),
])
def test_production_kernel_parity(name, num_envs, steps, cuda_device):
    """
    The PRODUCTION binaries -- in-kernel Philox draws, large slabs: exactly the specialised libraries
    bench.py times (its `kernel_variant.libraries`) -- against the oracle at BASELINE batch sizes up
    to 1,048,576 envs.  The kernels' draws are transplanted into the oracle (oracle/parity.py,
    `philox=True`); every other value of the step is compared as in the injected-draw tests.
    """
    from oracle.parity import ParityRun

    n_contacts = 8 if name != "command_direction" else 0  # as bench.py builds the workload
    run = ParityRun(name, num_envs=num_envs, device=cuda_device, seed=11, n_contacts=n_contacts, philox=True)
    stats = run.run(steps=steps)
    fused = run.env._fused
    spec_stats = fused.spec_stats()
    tile, library = _benchmark_library(fused)
    assert fused.injected is None and tile in (64, 128)
    assert spec_stats["specialised_launches"] == steps and library in spec_stats["libraries"], (spec_stats, library)
    assert stats["resets"] > 0
    print(f"PARITY-VARIANT {name} N={num_envs} slab={tile} draws=philox library={library} stats={stats}")


def test_disabled_managers(cuda_device):
    """
    `manager.enabled = False` (action / termination / reward): the manager's step() returns before it
    touches anything in the reference (position_action_manager.py:383-384, termination_manager.py:159-160,
    reward_manager.py:172-173, :204) -- stale masks keep resetting the same envs, episode sums are neither
    advanced nor logged nor cleared, targets stay put and nothing is sent to the actuators.
    """
    from oracle.parity import ParityRun

    run = ParityRun("contacts", num_envs=256, device=cuda_device, seed=21)
    run.reset()
    toggles = {5: {"reward": False}, 12: {"reward": True, "termination": False},
               20: {"termination": True, "action": False}, 27: {"action": True}}
    for i in range(40):
        for kind, enabled in toggles.get(i, {}).items():
            getattr(run.env, f"{kind}_manager").enabled = enabled
            (run.port.disabled.discard if enabled else run.port.disabled.add)(kind)
        out_e, out_p = run.step()
        assert ("terminations" in out_e[4]) == ("terminations" in out_p[4]), i
    assert run.stats["resets"] > 0


def test_external_controller_feeds_the_fused_terms(cuda_device):
    """
    CommandManager.use_external_controller (command_manager.py:85-90, 176-180): while a controller is
    attached, every term that reads the manager's `command` -- the observation column, the tracking
    rewards -- sees the controller's tensor, the interval resample is skipped, and reset() still
    resamples the manager's own buffer.
    """
    import genesis_forge_b200 as gfb
    from configs import specs
    from configs.env_builder import build_env, dropin_namespace

    gfb.set_device(cuda_device)
    n = 512

    def make():
        env = build_env(specs.get("command_direction"), dropin_namespace(), n, cuda_device, seed=3, n_contacts=0)
        env.build()
        env.reset()
        return env

    env, twin = make(), make()
    ctrl = torch.rand(n, 3, device=cuda_device) * 2 - 1
    env.velocity_command.use_external_controller(lambda step_count: ctrl)
    twin.velocity_command._command.copy_(ctrl)  # same commands, the ordinary way
    own = env.velocity_command._command.clone()
    actions = torch.randn(n, 12, device=cuda_device)
    obs, rew, term, trunc, _ = env.step(actions)
    obs_t, rew_t, term_t, trunc_t, _ = twin.step(actions)
    done = term | trunc
    assert bool(done.any()) and torch.equal(done, term_t | trunc_t)
    assert torch.equal(obs[:, :3], ctrl)                       # every env observes the controller's command
    assert torch.equal(rew, rew_t)                             # rewards were computed from it
    assert torch.equal(obs[~done], obs_t[~done])
    mine = env.velocity_command._command
    assert torch.equal(mine[~done], own[~done])                # no interval resample ...
    assert not torch.equal(mine[done], own[done])              # ... but reset() resampled the manager's own buffer
    env.velocity_command.use_external_controller(None)        # detach: the manager's buffer is used again
    obs2, *_ = env.step(actions)
    done2 = env.termination_manager.terminated | env.termination_manager.truncated
    assert torch.equal(obs2[~done2][:, :3], env.velocity_command._command[~done2])


def test_live_mutation_keeps_the_specialised_kernel(cuda_device):
    """Weights / params / ranges are live values: mutating them must not need a new specialisation."""
    from oracle.parity import ParityRun

    run = ParityRun("command_direction", num_envs=64, device=cuda_device, seed=3)
    run.reset()
    for i in range(10):
        run.step()
    for env_like in (run.env,):
        env_like.reward_manager.cfg["lin_vel_z"].weight = -4.0
        env_like.reward_manager.cfg["base_height_target"].params["target_height"] = 0.33
        env_like.velocity_command.range = {"lin_vel_x": [0.0, 2.0], "lin_vel_y": [-0.5, 0.5], "ang_vel_z": [-1.0, 1.0]}
    run.port.spec["rewards"]["lin_vel_z"]["weight"] = -4.0
    run.port.spec["rewards"]["base_height_target"]["params"]["target_height"] = 0.33
    run.port.command["velocity_command"]["range"] = {"lin_vel_x": [0.0, 2.0], "lin_vel_y": [-0.5, 0.5], "ang_vel_z": [-1.0, 1.0]}
    for i in range(20):
        run.step()
    stats = run.env._fused.spec_stats()
    assert stats["generic_launches"] == 2 and stats["specialised_launches"] == 30 and len(stats["libraries"]) == 1, stats


@pytest.mark.parametrize("name", ["command_direction", "berkeley_humanoid"])
def test_short_episodes_exercise_timeouts(name, cuda_device):
    from oracle.parity import ParityRun

    run = ParityRun(name, num_envs=192, device=cuda_device, seed=99, spec_override={"max_episode_length_sec": 1})
    stats = run.run(steps=150)
    assert stats["resets"] > 192  # every env timed out at least once


@pytest.mark.parametrize("num_envs", [1, 31, 33, 130])
def test_ragged_sizes(num_envs, cuda_device):
    """Slab tails: env counts that are not multiples of the slab size or of 4 (non-TMA path)."""
    from oracle.parity import ParityRun

    run = ParityRun("contacts", num_envs=num_envs, device=cuda_device, seed=5)
    run.run(steps=40)


@pytest.mark.parametrize("name", CONFIGS + ["within_limits"])
def test_cuda_path_reproduces_reference_golden_trace(name, cuda_device):
    """
    The CUDA path against the committed traces of the UNMODIFIED reference (tests/golden/, generated
    in the build container by oracle/make_golden.py): same seeded inputs, the reference's random draws
    injected via the oracle port (which the CPU suite pins bit-exactly to the same traces).
    """
    from oracle import make_golden
    from oracle.parity import ParityRun, _close

    gold = make_golden.load(name)
    run = ParityRun(name, num_envs=gold["num_envs"], device=cuda_device, seed=gold["seed"], sanitize=False)
    run.reset()
    for i, g in enumerate(gold["step"]):
        out_e, out_p = run.step(nan_action=(i == gold["nan_step"]))
        assert torch.equal(out_e[2].cpu(), g["terminated"]), f"step {i} terminated"
        assert torch.equal(out_e[3].cpu(), g["truncated"]), f"step {i} truncated"
        n = int(g["reset_idx"].numel())
        assert torch.equal(run.env._fused.reset_idx[:n].cpu(), g["reset_idx"]), f"step {i} reset_idx"
        ok, abs_err, _ = _close(out_e[1], g["rewards"])
        assert ok, f"step {i} rewards err {abs_err}"
        for group, want in g["obs"].items():
            ok, abs_err, _ = _close(out_e[4]["observations"][group], want)
            assert ok, f"step {i} obs[{group}] err {abs_err}"
        for key, want in g["logging"].items():
            ok, abs_err, _ = _close(torch.as_tensor(out_e[4]["episode"][key]).reshape(()), want)
            assert ok, f"step {i} extras[{key}] err {abs_err}"


def test_million_env_properties(cuda_device):
    """
    Full-size (1,048,576 envs) run checked through size-independent properties: reset indices are
    exactly the ascending positions of (terminated | truncated); the logged termination fractions
    equal the mask means; episode length is zero exactly on reset envs; observations are finite and
    the command columns of the observation row equal the command buffer.
    """
    import genesis_forge_b200 as gfb
    from configs import specs
    from configs.env_builder import build_env, dropin_namespace

    gfb.set_device(cuda_device)
    n = 1 << 20
    env = build_env(specs.get("command_direction"), dropin_namespace(), n, cuda_device, pool=2, seed=7, n_contacts=0,
                    apply_setters=False)
    env.build()
    env.reset()
    for step in range(3):
        actions = torch.randn(n, 12, device=cuda_device)
        obs, rew, term, trunc, extras = env.step(actions)
        done = term | trunc
        idx = done.nonzero().reshape(-1)
        n_reset = env._fused.report.n_reset
        assert n_reset == idx.numel() > 0
        assert torch.equal(env._fused.reset_idx[:n_reset], idx)
        assert torch.equal(env.episode_length == 0, done)
        assert bool(torch.isfinite(obs).all()) and bool(torch.isfinite(rew).all())
        assert torch.equal(obs[:, :3], env.velocity_command.command)
        assert torch.equal(obs[:, 36:48], env.action_manager.get_actions())
        frac = extras["episode"]["Terminations / fall_over"]
        assert abs(float(frac) - float(term.float().mean())) < 1e-6
        assert torch.equal(env.actions[idx], torch.zeros(n_reset, 12, device=cuda_device))


def test_spawn_pose_matches_the_oracle(cuda_device):
    """
    Reset-side writer (gfb_spawn_pose): positions / quaternions handed to the engine setters and the
    managers' persistent spawn buffers, against the oracle's restatement of
    terrain_manager.py:168-279 and mdp/reset.py:172-195 fed with the same draws.  x / y are
    specified op by op (bit-exact); z goes through the bilinear height lookup (1e-5 relative, as for
    the base_height reward); the quaternion goes through cos/sin (1e-6 absolute).
    """
    from oracle.parity import ParityRun

    run = ParityRun("rough_terrain", num_envs=512, device=cuda_device, seed=4321)
    run.port.robot.record_calls = True
    run.env.robot.record_calls = True
    stats = run.run(steps=60)
    assert stats["resets"] > 40

    def poses(robot, name):
        return [(c[1].cpu(), c[2].cpu()) for c in robot.calls if c[0] == name]

    for name, exact in (("set_pos", True), ("set_quat", False)):
        want, got = poses(run.port.robot, name), poses(run.env.robot, name)
        assert len(want) == len(got) > 10
        for (w_val, w_idx), (g_val, g_idx) in zip(want, got):
            assert torch.equal(w_idx, g_idx)
            if exact:  # x, y: two specified roundings; z: bilinear lookup, the package's fp32 tolerance
                assert torch.equal(w_val[:, :2], g_val[:, :2])
                assert torch.allclose(w_val[:, 2], g_val[:, 2], rtol=1e-5, atol=1e-6)
            else:
                assert torch.allclose(w_val, g_val, rtol=0.0, atol=1e-6)
    terrain = run.env.managers["terrain"][0]
    assert torch.equal(terrain._env_pos_buffer.cpu()[:, :2], run.port.t_env_pos[:, :2])
    assert torch.allclose(terrain._env_pos_buffer.cpu()[:, 2], run.port.t_env_pos[:, 2], rtol=1e-5, atol=1e-6)
    item = next(i for i in run.port.reset_items if i["fn"] == "randomize_terrain_position")
    (cfg,) = [c for c in run.env.managers["entity"][0].on_reset.values() if hasattr(c.fn, "_rotation_buffer")]
    assert torch.equal(cfg.fn._rotation_buffer.cpu(), item["rotation_buffer"])
    assert torch.allclose(cfg.fn._quat_buffer.cpu(), item["quat_buffer"], rtol=0.0, atol=1e-6)


def test_spawn_pose_in_kernel_draws(cuda_device):
    """Production mode (no injected draws): Philox in the kernel; statistical and geometric properties."""
    import genesis_forge_b200 as gfb
    from configs import specs
    from configs.env_builder import build_env, dropin_namespace

    gfb.set_device(cuda_device)
    n = 1 << 16
    env = build_env(specs.get("rough_terrain"), dropin_namespace(), n, cuda_device, pool=2, seed=5, n_contacts=8)
    env.build()
    env.reset()
    terrain = env.managers["terrain"][0]
    launches = env._fused.launch_count()
    pos = terrain.generate_random_env_pos()
    assert env._fused.launch_count() == launches + 1  # one kernel, no torch op chain
    x_min, x_max, y_min, y_max = terrain.get_bounds()
    cx, cy, hx, hy = (x_min + x_max) / 2, (y_min + y_max) / 2, (x_max - x_min) / 4, (y_max - y_min) / 4
    assert bool(((pos[:, 0] >= cx - hx) & (pos[:, 0] <= cx + hx)).all())
    assert bool(((pos[:, 1] >= cy - hy) & (pos[:, 1] <= cy + hy)).all())
    assert abs(float(pos[:, 0].mean()) - cx) < 0.05 * hx and abs(float(pos[:, 1].mean()) - cy) < 0.05 * hy
    assert abs(float(pos[:, 0].std()) - 2 * hx / 12 ** 0.5) < 0.02 * hx
    height = terrain.get_terrain_height(pos[:, 0], pos[:, 1])  # torch grid_sample on the same field
    assert torch.allclose(pos[:, 2], height + 0.1e-3, rtol=1e-5, atol=1e-6)
    assert torch.equal(terrain._env_pos_buffer, pos)
    again = terrain.generate_random_env_pos()
    assert not torch.equal(again, pos)  # a new counter per call
    some = torch.tensor([5, 17, 4000], device=cuda_device)
    before = terrain._env_pos_buffer.clone()
    sub = terrain.generate_random_env_pos(envs_idx=some)
    changed = (terrain._env_pos_buffer != before).any(dim=1).nonzero().reshape(-1)
    assert torch.equal(changed, some) and torch.equal(terrain._env_pos_buffer[some], sub)


@pytest.mark.parametrize("name", ["kitchen_sink", "rough_terrain", "berkeley_humanoid"])
def test_direct_term_calls_match_the_oracle(name, cuda_device):
    """
    Stock mdp terms called directly (`rewards.x(env, **params)`, as user-defined terms and curricula
    do) return the unweighted per-env value, evaluated by the kernel on a one-term table, and leave
    no trace: the step-by-step parity run continues unchanged afterwards.
    """
    from oracle.parity import ParityRun, _close

    run = ParityRun(name, num_envs=200, device=cuda_device, seed=77)
    run.reset()
    for _ in range(12):
        run.step()
    env, port = run.env, run.port
    checked = 0
    for kind, cfg, spec_terms, oracle in (
        ("reward", env.reward_manager.cfg, port.spec["rewards"], port._reward_value),
        ("termination", env.termination_manager.term_cfg, port.spec["terminations"], port._termination_value),
    ):
        for tname, item in cfg.items():
            spec_item = spec_terms[tname]
            if callable(spec_item["fn"]) or spec_item["fn"] == "body_acceleration_exp":
                continue
            got = item.fn(env, **item.params)
            want = oracle(spec_item["fn"], spec_item.get("params") or {})
            assert got.shape == want.shape == (200,), (tname, got.shape)
            if kind == "termination":
                assert got.dtype == torch.bool and torch.equal(got.cpu(), want), tname
            else:
                ok, abs_err, rel_err = _close(got, want)
                assert ok, (tname, abs_err, rel_err)
            checked += 1
    assert checked >= 6
    for _ in range(5):
        run.step()


def test_within_limits_action_manager(cuda_device):
    """PositionWithinLimitsActionManager (position_within_limits.py:99-131): clamp to [-1, 1], then the joint-limit map."""
    from configs import specs
    from oracle.parity import ParityRun

    action = dict(specs.get("command_direction")["action"], type="within_limits")
    for key in ("scale", "use_default_offset"):
        action.pop(key, None)
    run = ParityRun("command_direction", num_envs=200, device=cuda_device, seed=31, spec_override={"action": action})
    assert run.env.action_manager.kernel_mode == 2
    run.reset()
    clamped = 0
    for i in range(40):
        run.step(nan_action=(i == 4))
        # clamp_ (:127) acts on the manager's own copy (base.py:76-82), never on the tensor the caller passed
        given_port, given_env = run.last_action_args
        assert torch.equal(given_env.cpu().nan_to_num(nan=7.0), given_port.nan_to_num(nan=7.0))
        clamped += int((given_port.abs() > 1.0).sum())
    assert clamped > 0 and run.stats["resets"] > 0


def test_base_height_with_a_per_env_target_tensor(cuda_device):
    """rewards.base_height(target_height=<(N,) tensor>) (rewards.py:54-90): GFB_RF_TARGET_FROM_TENSOR."""
    from configs import specs
    from oracle.parity import ParityRun

    n = 160
    rewards = specs.get("command_direction")["rewards"]
    name = next(k for k, v in rewards.items() if v["fn"] == "base_height")
    rewards[name]["params"] = dict(rewards[name]["params"],
                                   target_height=0.25 + 0.1 * torch.rand(n, generator=torch.Generator().manual_seed(3)))
    run = ParityRun("command_direction", num_envs=n, device=cuda_device, seed=57, spec_override={"rewards": rewards})
    stats = run.run(steps=30)
    assert stats["resets"] > 0


@pytest.mark.parametrize("switch", ["GFB_DISABLE_TMA=1", "GFB_NO_OVERLAY=1", "GFB_TILE=64", "GFB_TILE=64:persistent"])
def test_kernel_switches_keep_parity(switch, cuda_device, monkeypatch):
    """
    The alternative code paths behind the environment switches (cooperative loads instead of TMA, one
    load group, another slab size) give the same results, and so does the persistent loop of the
    GENERIC kernel when there are more slabs than resident blocks (every block draws several tickets).
    Generic kernels: no specialisation is pre-built for these plans and none is compiled here.
    """
    from oracle.parity import ParityRun

    switch, _, mode = switch.partition(":")
    key, value = switch.split("=")
    monkeypatch.setenv(key, value)
    monkeypatch.setenv("GFB_SPEC_JIT", "0")
    n, steps = (400_000, 3) if mode == "persistent" else (328, 40)
    if mode == "persistent":
        monkeypatch.setenv("GFB_NO_SPEC", "1")
    run = ParityRun("contacts", num_envs=n, device=cuda_device, seed=404)
    stats = run.run(steps=steps, nan_step=3)
    assert stats["resets"] > 0


def test_production_draws_philox(cuda_device):
    """
    Production mode (nothing injected): the draws made inside the kernels come from Philox4x32-10.
    Checked: command resample and episode-length draws stay inside their ranges with the moments of
    a uniform distribution, observation noise is bounded by its scale with uniform spread, the
    stream is reproducible for a seed and changes with it and with the step.
    """
    import copy

    import genesis_forge_b200 as gfb
    from configs import specs
    from configs.env_builder import build_env, dropin_namespace

    gfb.set_device(cuda_device)
    n = 1 << 16
    spec = specs.get("command_direction")
    spec["observations"]["policy"]["terms"]["dof_position"]["noise"] = 0.02

    def make(seed_offset=0):
        env = build_env(copy.deepcopy(spec), dropin_namespace(), n, cuda_device, pool=2, seed=9, n_contacts=0,
                        apply_setters=False)
        env.build()
        env._fused.rng_seed += seed_offset
        env.reset()
        return env

    env = make()
    cmd = env.velocity_command.command.clone()
    ranges = env.velocity_command.ranges_list()
    for k, (lo, hi) in enumerate(ranges):
        col = cmd[:, k]
        assert bool(((col >= lo) & (col <= hi)).all())
        assert abs(float(col.mean()) - (lo + hi) / 2) < 0.02 * (hi - lo)
        assert abs(float(col.std()) - (hi - lo) / 12 ** 0.5) < 0.02 * (hi - lo)
    assert abs(float(torch.corrcoef(cmd.T)[0, 1])) < 0.02  # columns are independent draws
    # genesis_env.py:246-252: max_episode_length = round(base + U(-1,1) * base * scaling)
    base, scale = env._base_max_episode_length, env._max_episode_random_scaling
    max_len = env.max_episode_length.float()
    assert float(max_len.min()) >= round(base * (1 - scale)) and float(max_len.max()) <= round(base * (1 + scale))
    assert abs(float(max_len.mean()) - base) < 0.01 * base * scale + 1
    assert abs(float(max_len.std()) - base * scale / 3 ** 0.5) < 0.05 * base * scale
    # observation noise on dof_position: obs = q + 0.02 * U(-1, 1)
    off = 0
    for name, _, width in env.observation_managers["policy"]._sources:
        if name == "dof_position":
            break
        off += width
    obs, *_ = env.step(torch.zeros(n, 12, device=cuda_device))
    q = env.robot.get_dofs_position(env.action_manager.dofs_idx)
    done = (env.episode_length == 0)
    noise = (obs[:, off:off + 12] - q)[~done]  # reset envs were re-observed from the reset pose
    assert float(noise.abs().max()) <= 0.02 * (1 + 1e-5) + 1e-6
    assert abs(float(noise.std()) - 0.02 / 3 ** 0.5) < 2e-4 and abs(float(noise.mean())) < 2e-4
    # same seed -> same stream; another seed or step -> another stream
    twin = make()
    assert torch.equal(twin.velocity_command.command, cmd)
    other = make(seed_offset=1)
    assert not torch.equal(other.velocity_command.command, cmd)
    obs_twin, *_ = twin.step(torch.zeros(n, 12, device=cuda_device))
    assert torch.equal(obs_twin, obs)
    obs2, *_ = env.step(torch.zeros(n, 12, device=cuda_device))
    q2 = env.robot.get_dofs_position(env.action_manager.dofs_idx)
    keep = ~(done | (env.episode_length == 0))
    assert not torch.equal((obs2[:, off:off + 12] - q2)[keep], (obs[:, off:off + 12] - q)[keep])
