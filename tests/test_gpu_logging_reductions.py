"""
The end-of-step reductions of the post-physics kernel on the GPU, driven to their edges: the logged episode
means of the reward terms (reward_manager.py:205-216), the termination fractions, the reset count and the
ordered reset list compact_kernel builds.

Harness: every reward term is `action_rate_l2` under its own name, and the actions are 0 in every step, so
each term's value is +-0 and the episode sum a term ends the step with is the one written here before it.
Each term's row of `_episode_sums` carries one family of values; `_episode_seconds` is set so that
E = fadd(E0, dt) is 1, and the quotient the kernel logs is q = fdiv(S0, E) (computed here with numpy fp32,
the same IEEE operations).  The resetting envs are chosen through the timeout: `episode_length` is set to
`max_episode_length` for them (the kernel tests ep_len > max_len after the increment) and 0 elsewhere.
The means are checked against the contract of tail.cuh (exact sum S of the reset envs' quotients, via
math.fsum) and against torch-CPU's fp32 mean within its own summation bound.
"""
import math

import numpy as np
import pytest
import torch

from test_logging_reductions import check_vs_torch

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def device():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda", 0)

DT = 1 / 50
SPECIAL_STEPS = (1, 5)  # steps whose special-value terms carry NaN / Inf on a reset env (the next step is clean)


def _families(n: int, rng) -> dict:
    """name -> (weight, episode sums S0 of every env), one family of quotients per term."""
    cyc = lambda vals: np.resize(np.asarray(vals, dtype=np.float32), n)  # noqa: E731
    normal = rng.uniform(-10, 10, n).astype(np.float32)
    return {
        "normal": (-0.5, normal),
        "tiny": (-1.0, cyc([1e-9, 1e-30, 2.0 ** -149, 7 * 2.0 ** -149, -1e-9, 2.0 ** -130, 3.7e-6])),
        "large_40000": (1.0, cyc([40000.0])),
        "large_mixed": (2.0, cyc([2.0 ** 20 - 2.0 ** -4, 2.0 ** 20, 1e10, 1e30, -1e10, 40000.0])),
        "cancel": (1.5, cyc([2.0 ** 100, -(2.0 ** 100), 1e-30, -3e-30])),
        "nan_one": (-2.0, normal.copy()),
        "inf_one": (0.25, normal.copy()),
        "inf_both": (-0.25, normal.copy()),
        "big_3e38": (1.0, cyc([3e38])),
        "minus_zero": (-3.0, cyc([-0.0])),
        "unlogged": (0.0, cyc([math.nan, 1.0])),
    }


def _patterns(n: int, tile: int, seed: int = 3) -> list:
    idx = np.arange(n)
    slab = 1 if n > tile else 0
    return [
        ("none", np.zeros(n, bool)),
        ("all", np.ones(n, bool)),
        ("first", idx == 0),
        ("last", idx == n - 1),
        ("slab_last", (idx % tile == tile - 1) | (idx == n - 1)),
        ("every_32nd", idx % 32 == 0),
        ("alternate_words", (idx // 32) % 2 == 0),
        ("one_slab", idx // tile == slab),
        ("all_but_one", idx != n // 2),
        ("random_half", np.random.default_rng(seed).random(n) < 0.5),
    ]


def _spec(families: dict, user_term=False) -> dict:
    from configs import specs

    s = specs.command_direction()
    assert s["dt"] == DT
    s.update(name="logging_reductions", max_episode_length_sec=10000, max_episode_random_scaling=0.0)
    s["rewards"] = {name: {"fn": "action_rate_l2", "weight": w} for name, (w, _) in families.items()}
    if user_term:  # a Python reward term: split execution
        s["rewards"]["user_zero"] = {"fn": lambda e: torch.zeros(e.num_envs, device=e.actions.device), "weight": 1.0}
    s["terminations"] = {"timeout": {"fn": "timeout", "time_out": True}}
    return s


def _env(spec, n, device, monkeypatch, tile, generic, debug):
    import genesis_forge_b200 as gfb
    from configs.env_builder import build_env, dropin_namespace
    from genesis_forge_b200.managed_env import ManagedEnvironment

    monkeypatch.setattr(ManagedEnvironment, "fuse_user_terms", False)
    if tile is not None:
        monkeypatch.setenv("GFB_TILE", str(tile))
    if generic:
        monkeypatch.setenv("GFB_NO_SPEC", "1")
    if debug:
        monkeypatch.setenv("GFB_DEBUG", str(debug))
    gfb.set_device(device)
    env = build_env(spec, dropin_namespace(), n, device, pool=4, seed=11, n_contacts=0, apply_setters=False)
    env.build()
    env.reset()
    return env


def _seconds_to_one() -> np.float32:
    """E0 with fadd(E0, fp32(dt)) == 1 exactly."""
    dt, e0 = np.float32(DT), np.float32(1) - np.float32(DT)
    for _ in range(8):
        e = e0 + dt
        if e == np.float32(1):
            return e0
        e0 = np.nextafter(e0, np.float32(0) if e > 1 else np.float32(2))
    raise AssertionError("no E0 with E0 + dt == 1")


def _check_mean(got: float, q: np.ndarray, name: str):
    """The contract of a logged mean (tail.cuh) over the reset envs' quotients q."""
    got = np.float32(got)
    n = len(q)
    if np.isnan(q).any() or (np.isposinf(q).any() and np.isneginf(q).any()):
        assert np.isnan(got), (name, got)
        return
    if np.isinf(q).any():
        assert got == q[np.isinf(q)][0], (name, got)
        return
    s = math.fsum(q.astype(np.float64))  # the exact sum rounded to double
    if abs(s) >= 2.0 ** 128 - 2.0 ** 103:
        assert got == np.float32(math.copysign(math.inf, s)), (name, got, s)
        return
    if s == 0.0:
        assert got == 0 and not np.signbit(got), (name, got)
        return
    exact = s / n
    ulp = float(np.spacing(np.float32(abs(exact))))
    assert abs(float(got) - exact) <= ulp, (name, float(got), exact, ulp)


def _run_steps(env, tile, generic, split=False):
    fused = env._fused
    n = env.num_envs
    dev = fused.device
    fam = _families(n, np.random.default_rng(0))
    if split:  # the host-callback term (+0 values) logs +0 from its -0 sums
        fam["user_zero"] = (1.0, np.full(n, -0.0, dtype=np.float32))
    names = list(fam)
    cfg = list(env.reward_manager.cfg)
    rows = [cfg.index(k) for k in names]
    rew_tag, term_tag = env.reward_manager.logging_tag, env.termination_manager.logging_tag
    e0 = _seconds_to_one()
    actions = torch.zeros(n, fused.D, device=dev)
    env.step(actions)  # (last_actions == actions == 0 from here on)
    max_len = env.max_episode_length.clone()
    for step, (pname, mask) in enumerate(_patterns(n, tile)):
        where = f"{pname} (step {step}, N={n}, tile={tile}, generic={generic}, split={split})"
        s0 = {k: v.copy() for k, (_, v) in fam.items()}
        reset_ids = np.nonzero(mask)[0]
        if step in SPECIAL_STEPS and len(reset_ids):
            mid = reset_ids[len(reset_ids) // 2]
            s0["nan_one"][mid] = np.nan
            s0["inf_one"][mid] = np.inf
            s0["inf_both"][mid] = np.inf
            s0["inf_both"][reset_ids[0] if reset_ids[0] != mid else reset_ids[-1]] = -np.inf
        sums = env.reward_manager._episode_sums
        for k, r in zip(names, rows):
            sums[r].copy_(torch.from_numpy(s0[k]))
        env.reward_manager._episode_seconds.fill_(float(e0))
        m = torch.from_numpy(mask).to(dev)
        env.episode_length.zero_()
        env.episode_length[m] = max_len[m]

        stats0 = fused.spec_stats()
        _, _, terminated, truncated, extras = env.step(actions)
        stats = fused.spec_stats()
        if generic:
            assert stats["specialised_launches"] == stats0["specialised_launches"], (where, stats)
            assert stats["generic_launches"] > stats0["generic_launches"], (where, stats)
        else:
            assert stats["generic_launches"] == stats0["generic_launches"], (where, stats)
            launched = stats["specialised_launches"] - stats0["specialised_launches"]
            assert launched == 1 or (split and launched > 1), (where, stats)

        # resets, the reset count and the ordered list compact_kernel built
        assert not terminated.any() and torch.equal(truncated.cpu(), torch.from_numpy(mask)), where
        n_reset = int(mask.sum())
        assert fused.report.n_reset == n_reset and fused.report.global_n_reset == n_reset, where
        want_idx = (terminated | truncated).nonzero().flatten()
        assert torch.equal(fused.reset_idx[:n_reset], want_idx), where

        # the reset envs' sums are +0 and their seconds 1e-10; the others keep theirs (+ a +-0 value)
        after = env.reward_manager._episode_sums.cpu().numpy()
        secs = env.reward_manager._episode_seconds.cpu().numpy()
        for k, r in zip(names, rows):
            assert (after[r][mask].view(np.int32) == 0).all(), (where, k)
            kept = after[r][~mask]
            assert np.array_equal(kept, s0[k][~mask], equal_nan=True), (where, k)
        assert (secs[mask] == np.float32(1e-10)).all() and (secs[~mask] == np.float32(1)).all(), where

        # the published keys and values
        episode = extras["episode"]
        want_keys = set()
        if n_reset:
            want_keys.add(f"{term_tag} / timeout")
            want_keys |= {f"{rew_tag} / {k}" for k in names if fam[k][0] != 0}
        assert set(episode) == want_keys, (where, sorted(episode), sorted(want_keys))
        if not n_reset:
            continue
        frac = float(episode[f"{term_tag} / timeout"])
        want_frac = truncated.cpu().float().mean().item()
        assert np.float32(frac).view(np.int32) == np.float32(want_frac).view(np.int32), (where, frac, want_frac)
        for k in names:
            if fam[k][0] == 0:
                continue
            q = s0[k][mask] / (e0 + np.float32(DT))  # fdiv(S0, fadd(E0, dt)) in fp32
            got = float(episode[f"{rew_tag} / {k}"])
            _check_mean(got, q, f"{k} at {where}")
            check_vs_torch(np.float32(got), q)


# (num_envs, tile, generic, GFB_DEBUG): sizes with a tail slab, several slabs per block at 1M envs, and the
# compact geometry of 1,048,580 and 1,572,864 envs (blocks that used to start past the mask words)
CASES = [
    *[(n, t, False, 0) for n in (36, 260, 4096 + 4, 65536 + 4) for t in (32, 64, 128)],
    *[(n, 32, True, 8) for n in (36, 4096 + 4, 65536 + 4)],
    *[(n, t, True, 0) for n in (260, 65536 + 4) for t in (64, 128)],
    (1 << 20, 128, False, 0),
    (1 << 20, 32, True, 8),
    (1_048_580, 128, False, 0),
    (1_572_864, 128, False, 0),
]


@pytest.mark.parametrize("num_envs,tile,generic,debug", CASES,
                         ids=[f"{n}-t{t}-{'generic' if g else 'spec'}{'-dbg' + str(d) if d else ''}"
                              for n, t, g, d in CASES])
def test_logged_means_counts_and_reset_list(num_envs, tile, generic, debug, device, monkeypatch):
    env = _env(_spec(_families(num_envs, np.random.default_rng(0))), num_envs, device, monkeypatch, tile,
               generic, debug)
    fused = env._fused
    assert not fused.split_mode
    _run_steps(env, tile, generic)


@pytest.mark.parametrize("generic", [False, True], ids=["spec", "generic"])
def test_split_execution_reset_launch_carries_the_tail(generic, device, monkeypatch):
    """A host-callback reward term: the RESET-phase launch of split execution does the reductions."""
    n = 4096 + 4
    env = _env(_spec(_families(n, np.random.default_rng(0)), user_term=True), n, device, monkeypatch, 64,
               generic, 0)
    assert env._fused.split_mode
    _run_steps(env, 64, generic, split=True)
