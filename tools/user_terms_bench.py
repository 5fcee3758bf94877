"""
env.step of the user-terms workload (configs/user_terms.py) with its user-defined rewards / terminations
as host callbacks (split execution, fuse_user_terms off) and lowered into the specialised post-physics
kernel (fuse_user_terms on), at 65,536 and 1,048,576 envs.  `--workload user_observations` does the same
for workload A of configs/user_observations.py (fuse_user_observations), adds the stock `contacts` table
as a third, reference environment for the post-physics kernel's time, and reports the reset-path kernel
of the lowered observation terms.  `--workload stateful_terms` compares workload A of configs/stateful_terms.py
(class-style terms with per-env state) as callbacks and lowered (fuse_stateful_terms), and
`--workload stateful_observations` workload A of configs/stateful_observations.py (class-style observation
terms: host columns against lowered, fuse_stateful_terms), and `--workload link_terms` configs/link_terms.py (user
terms that read per-link state: callbacks / host columns against lowered, every lowering switch on), and
`--workload stock_calls` both workloads of configs/stock_calls.py (user terms that call stock mdp terms: callbacks
against lowered with fuse_user_terms, fuse_stateful_terms and fuse_stock_calls on).  The two modes are built side by side and
timed alternately in one process (CUDA events around `steps` steps, in-kernel Philox draws as bench.py
runs them, on bench.py's pool of pre-generated state sets); the post-physics kernel's device time comes
from the library's own event brackets.  The outputs of one more step of both modes (same states, same
actions, same draws) are compared.

    python tools/user_terms_bench.py [--workload user_terms|user_observations|stateful_terms|stateful_observations|
                                                 link_terms|stock_calls]
                                     [--sizes 65536 1048576]
                                     [--steps 50] [--warmup 10] [--rounds 3]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def gpu_info() -> dict:
    import torch

    info = {"name": torch.cuda.get_device_name(0)}
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit_and_max_sm_clock"] = out
    except Exception as e:  # noqa: BLE001
        info["power_limit_and_max_sm_clock"] = f"unavailable ({e})"
    return info


def make_env(n: int, mode: str, dev, workload: str = "user_terms"):
    import genesis_forge_b200 as gfb
    from configs import (link_terms, specs, stateful_observations, stateful_terms, stock_calls, user_observations,
                         user_terms)
    from configs.env_builder import build_env, dropin_namespace
    from genesis_forge_b200.managed_env import ManagedEnvironment

    obs = workload == "user_observations"
    stateful = workload in ("stateful_terms", "stateful_observations")
    links = workload == "link_terms"
    calls = workload.startswith("stock_calls")
    ManagedEnvironment.fuse_user_terms = mode == "fused" and (links or calls or not (obs or stateful))
    ManagedEnvironment.fuse_user_observations = mode == "fused" and (obs or links)
    ManagedEnvironment.fuse_stateful_terms = mode == "fused" and (stateful or links or calls)
    ManagedEnvironment.fuse_stock_calls = mode == "fused" and calls
    gfb.set_device(dev)
    spec = specs.contacts() if mode == "stock" else (link_terms.link_terms() if links
                                                     else getattr(stock_calls, workload)() if calls
                                                     else user_observations.user_observations() if obs
                                                     else stateful_terms.stateful_terms() if workload == "stateful_terms"
                                                     else stateful_observations.stateful_observations() if stateful
                                                     else user_terms.user_terms())
    # as bench.py: a pool of pre-generated state sets rotated by scene.step() (the same states for both modes),
    # engine-side reset writes accepted but not applied
    env = build_env(spec, dropin_namespace(), n, dev, pool=4, seed=7, n_contacts=8, apply_setters=False)
    env.build()
    env.reset()
    return env


def timed(env, actions, steps: int) -> tuple[float, float, int, float]:
    """(ms per step, post-physics kernel ms per step, post-physics launches per step, reset-path kernel us per
    launch of the lowered observation terms or 0)"""
    import torch

    fused = env._fused
    fused.profile(True)
    before = fused.profile_read()
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for i in range(steps):
        env.step(actions[i % len(actions)])
    end.record()
    end.synchronize()
    after = fused.profile_read()
    user_us = fused.profile_read_aux().get("user_observe_kernel", {}).get("kernel_us", 0.0)
    fused.profile(False)
    launches = after["post_launches"] - before["post_launches"]
    return (start.elapsed_time(end) / steps, (after["post_ms"] - before["post_ms"]) / steps, launches // steps,
            user_us)


def main():
    import torch

    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", type=int, nargs="+", default=[65536, 1 << 20])
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--workload", choices=["user_terms", "user_observations", "stateful_terms",
                                                       "stateful_observations", "link_terms", "stock_calls"],
                    default="user_terms")
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    print(json.dumps({"gpu": gpu_info()}), flush=True)
    workloads = ["stock_calls_a", "stock_calls_b"] if args.workload == "stock_calls" else [args.workload]
    for n, workload in ((n, w) for n in args.sizes for w in workloads):
        modes = ("split", "fused") + (("stock",) if workload == "user_observations" else ())
        envs = {mode: make_env(n, mode, dev, workload) for mode in modes}
        print(f"# N={n}: both environments built", flush=True)
        assert envs["split"]._fused.split_mode and not envs["fused"]._fused.split_mode
        gen = torch.Generator(device=dev).manual_seed(5)
        actions = [torch.randn(n, 12, device=dev, generator=gen) for _ in range(8)]
        for env in envs.values():
            for i in range(args.warmup):
                env.step(actions[i % len(actions)])
        rows = {mode: [] for mode in envs}
        for r in range(args.rounds):  # alternate the two modes
            for mode, env in envs.items():
                rows[mode].append(timed(env, actions, args.steps))
                print(f"# N={n} round {r} {mode}: {rows[mode][-1]}", flush=True)
        # same seeded state and actions through both modes: compare one more step's outputs
        outs = {mode: envs[mode].step(actions[0]) for mode in ("split", "fused")}
        a, b = outs["split"], outs["fused"]
        diff = {
            "rewards_max_abs": float((a[1] - b[1]).abs().max()),
            "terminated_equal": bool(torch.equal(a[2], b[2])),
            "truncated_equal": bool(torch.equal(a[3], b[3])),
            "obs_max_abs": float((a[0] - b[0]).abs().max()),
        }
        result = {"workload": workload, "num_envs": n, "steps": args.steps, "rounds": args.rounds,
                  "compare": diff}
        for mode, r in rows.items():
            ms = sorted(x[0] for x in r)[len(r) // 2]
            post = sorted(x[1] for x in r)[len(r) // 2]
            result[mode] = {"ms_per_step_median": round(ms, 4), "env_steps_per_s": round(n / ms * 1e3),
                            "post_kernel_ms_per_step_median": round(post, 4), "post_launches_per_step": r[0][2],
                            "ms_per_step_all": [round(x[0], 4) for x in r]}
            if workload in ("user_observations", "stateful_observations", "link_terms", "stock_calls_a",
                            "stock_calls_b") and mode == "fused":
                result[mode]["user_observe_kernel_us_median"] = round(sorted(x[3] for x in r)[len(r) // 2], 2)
                result[mode]["spec_stats"] = envs[mode]._fused.spec_stats()
        print(json.dumps(result), flush=True)
        del envs
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
