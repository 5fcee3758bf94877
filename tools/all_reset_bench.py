"""
Worst case of the end-of-step reductions: config 2 (command_direction) at 1,048,576 envs with EVERY env
timing out in every step, so every env adds its episode quotients to the slabs' shared accumulators and
compact_kernel lists all envs.  Before each step the episode lengths are set to the episode limit; the
post-physics kernel's device time comes from the library's own event brackets, the step time from CUDA
events around `steps` steps.  Prints one JSON line.

    python tools/all_reset_bench.py [--num-envs 1048576] [--steps 50] [--warmup 10]
"""
from __future__ import annotations

import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def main():
    import torch

    import genesis_forge_b200 as gfb
    from configs import specs
    from configs.env_builder import build_env, dropin_namespace
    from tools.user_terms_bench import gpu_info

    ap = argparse.ArgumentParser()
    ap.add_argument("--num-envs", type=int, default=1 << 20)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=10)
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    gfb.set_device(dev)
    env = build_env(specs.command_direction(), dropin_namespace(), args.num_envs, dev, pool=4, seed=7,
                    apply_setters=False)
    env.build()
    env.reset()
    fused = env._fused
    gen = torch.Generator(device=dev).manual_seed(3)
    actions = [torch.randn(args.num_envs, fused.D, device=dev, generator=gen) for _ in range(4)]

    def run(steps: int) -> tuple[float, float, int, float]:
        """(ms per step, post-physics kernel ms per step, reset envs per step, compact_kernel us)"""
        start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        fused.profile(True)
        before = fused.profile_read()
        resets = 0
        start.record()
        for i in range(steps):
            env.episode_length.copy_(env.max_episode_length)
            env.step(actions[i % len(actions)])
            resets += fused.report.n_reset
        end.record()
        end.synchronize()
        after = fused.profile_read()
        compact_us = fused.profile_read_aux()["compact_kernel"]["kernel_us"]
        fused.profile(False)
        return (start.elapsed_time(end) / steps, (after["post_ms"] - before["post_ms"]) / steps, resets // steps,
                compact_us)

    run(args.warmup)
    step_ms, post_ms, resets, compact_us = run(args.steps)
    assert resets == args.num_envs, resets
    print(json.dumps({"workload": "command_direction, every env resets in every step", "num_envs": args.num_envs,
                      "steps": args.steps, "step_ms": round(step_ms, 4), "post_kernel_us": round(post_ms * 1e3, 2),
                      "compact_kernel_us": round(compact_us, 2),
                      "resets_per_step": resets, "gpu": gpu_info()}))


if __name__ == "__main__":
    main()
