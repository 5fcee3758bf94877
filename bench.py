#!/usr/bin/env python
"""
bench.py -- manager env-steps/s of the fused B200 manager step, on synthetic physics state.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference]
                    [--config command_direction] [--num-envs 1048576] [--no-sweep] [--dump-outputs DIR]

One "step" = one full `env.step(actions)` of the drop-in ManagedEnvironment through its public API
(gfb_action_step -> synthetic scene.step() -> gfb_post_physics -> report read-back -> host reset
fan-out -> gfb_observe), on a pool of pre-generated synthetic state sets that is larger than L2.
Every timed loop (headline, per-kernel pass, e2e, sweep, configs, CPU baseline) runs K steps after W
warm-up steps.  Prints ONE JSON line (rank 0).  See DESIGN.md "Measurement" for what each key means.

--dump-outputs DIR writes what the last timed step of the headline run returned (rank 0) as
DIR/<name>.npy, float32 / float64, at most 64 MB in all, plus DIR/outputs.json describing them; the
inputs are seeded, so two builds run with the same arguments can be compared array for array.

  value      whole-job env-steps/s, inputs resident in HBM, device-timed (CUDA events), max over ranks
  roofline   the post-physics kernel: its algorithmic bytes / its CUDA-event time / measured HBM peak
  e2e        same metric with HOST state + action buffers: H2D of the step's inputs and D2H of
             obs/reward/masks inside the timed region
  cpu_baseline   the oracle port (torch-CPU restatement of the reference managers, bit-identical to
             the reference) timed on this box's host cores on the same workload
  --impl reference   times only that CPU path and prints the same line shape
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np
import torch

sys.dont_write_bytecode = True  # the tree may be read-only; nothing is cached in it
ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "manager env-steps/sec"
UNIT = "env-steps/s"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="command_direction")
    ap.add_argument("--num-envs", type=int, default=1 << 20, help="envs per GPU (weak scaling)")
    ap.add_argument("--pool", type=int, default=4, help="pre-generated state sets rotated by scene.step()")
    ap.add_argument("--no-sweep", action="store_true", help="skip the 4096 / 65536 env points")
    ap.add_argument("--no-configs", action="store_true", help="skip the BASELINE configs 3 / 4 / 5 block")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--cpu-envs", type=int, default=0,
                    help="envs for the CPU baseline (0 = --num-envs, bounded to a few minutes of host work)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs to DIR/<name>.npy")
    return ap.parse_args()


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


# --------------------------------------------------------------------------------------------------
# clocks sampler
# --------------------------------------------------------------------------------------------------
_SAMPLER_SRC = r"""
import sys, time
import pynvml as N
N.nvmlInit()
key = sys.argv[1]
if key.startswith('GPU-'):
    try:
        h = N.nvmlDeviceGetHandleByUUID(key)
    except Exception:
        h = N.nvmlDeviceGetHandleByUUID(key.encode())
else:
    h = N.nvmlDeviceGetHandleByIndex(int(key))
reasons_fn = getattr(N, 'nvmlDeviceGetCurrentClocksEventReasons', None) or N.nvmlDeviceGetCurrentClocksThrottleReasons
mx = N.nvmlDeviceGetMaxClockInfo(h, N.NVML_CLOCK_SM)
print('ready', flush=True)
while True:
    print(time.time(), N.nvmlDeviceGetClockInfo(h, N.NVML_CLOCK_SM), mx, int(reasons_fn(h)), flush=True)
    time.sleep(0.002)
"""


class ClockSampler:
    """
    SM clock + throttle reasons every ~2 ms from a side process (NVML), time-stamped so that the
    samples INSIDE the timed region can be picked out afterwards (`window`); the step loop itself
    is host-bound at small env counts, so nothing is sampled from this process.
    """
    REASONS = {0x4: "sw_power_cap", 0x8: "hw_slowdown", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown"}

    def __init__(self, index: int):
        self.proc = None
        try:
            key = str(index)
            uuid = getattr(torch.cuda.get_device_properties(index), "uuid", None)
            if uuid is not None:
                key = f"GPU-{uuid}"
            self.proc = subprocess.Popen([sys.executable, "-c", _SAMPLER_SRC, key], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            if self.proc.stdout.readline().strip() != "ready":  # NVML is up: samples flow from here on
                raise RuntimeError("sampler did not start")
        except Exception:
            if self.proc is not None:
                self.proc.kill()
            self.proc = None

    def stop(self, window: tuple[float, float] | None = None) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "samples": 0, "reasons": ["NVML sampler unavailable"]}
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except Exception:
            self.proc.kill()
            out = ""
        rows = []
        for line in out.strip().splitlines():
            parts = line.split()
            if len(parts) == 4:
                try:
                    rows.append((float(parts[0]), float(parts[1]), float(parts[2]), int(parts[3])))
                except ValueError:
                    pass
        inside = [r for r in rows if window is None or window[0] <= r[0] <= window[1]]
        where = "timed region"
        if not inside and rows and window is not None:  # region shorter than the sampling period: nearest samples
            mid = 0.5 * (window[0] + window[1])
            inside = sorted(rows, key=lambda r: abs(r[0] - mid))[:3]
            where = "nearest to the timed region"
        bits = 0
        for r in inside:
            bits |= r[3]
        return {
            "sm_mhz": statistics.median(r[1] for r in inside) if inside else None,
            "sm_max_mhz": max(r[2] for r in inside) if inside else None,
            "samples": len(inside),
            "sampled": where,
            "reasons": sorted(name for bit, name in self.REASONS.items() if bits & bit),
        }


def measured_traffic(config: str, num_envs: int):
    """
    DRAM bytes (read + write) of ONE post_kernel launch of this workload, measured with
    `ncu --metrics dram__bytes_read.sum,dram__bytes_write.sum` by tools/measure_traffic.py and kept in
    profiles/traffic.json TOGETHER WITH the hash of the kernel sources it was measured on.  An entry
    whose hash is not the hash of the sources in this tree is stale and refused (None).
    """
    from genesis_forge_b200 import spec

    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "profiles", "traffic.json")
    try:
        with open(path) as f:
            entry = json.load(f).get(f"{config}:{num_envs}")
        if entry is None or entry.get("kernel_source_hash") != spec.source_hash():
            return None
        return entry["dram_bytes"]
    except (OSError, ValueError):
        return None


# --------------------------------------------------------------------------------------------------
# environments
# --------------------------------------------------------------------------------------------------
def make_dropin_env(spec, num_envs, device, pool, seed):
    import genesis_forge_b200 as gfb
    from configs.env_builder import build_env, dropin_namespace

    gfb.set_device(device)
    # apply_setters=False: see SyntheticScene -- the pool's state sets are reused, so engine-side
    # reset writes are accepted but not applied (keeps the reset rate stationary over the run)
    env = build_env(spec, dropin_namespace(), num_envs, device, pool=pool, seed=seed,
                    n_contacts=8 if spec["contacts"] else 0, apply_setters=False)
    env.build()
    env.reset()
    return env


def time_dropin(env, actions, steps, warmup, dist_on, keep_outputs=False):
    """
    CUDA-event time of `steps` full env.step() calls; returns ms per step (max over ranks).
    keep_outputs: env.timed_outputs = step_outputs() of the last timed step.
    """
    import torch.distributed as dist

    dev = env._fused.device
    for i in range(warmup):
        env.step(actions[i % len(actions)])
    torch.cuda.synchronize(dev)
    if dist_on:
        dist.barrier()
    torch.cuda.synchronize(dev)
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n_reset = 0
    launches0 = env._fused.launch_count()
    wall0 = time.time()
    start.record()
    for i in range(steps):
        out = env.step(actions[i % len(actions)])
        n_reset += env._fused.report.n_reset
    end.record()
    torch.cuda.synchronize(dev)
    env.timed_window = (wall0, time.time())
    env.timed_launches = env._fused.launch_count() - launches0
    if keep_outputs:  # before the next step overwrites the buffers
        env.timed_outputs = step_outputs(out, env.extras_logging_key)
    if dist_on:
        dist.barrier()
    ms = start.elapsed_time(end) / steps
    if dist_on:
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    # per-kernel device times (roofline block): the same steps once more, now with a CUDA-event pair
    # around every launch -- kept out of the timed region above, where the ~10 extra event records per
    # step would cost host time
    env._fused.profile(True)
    for i in range(steps):
        env.step(actions[i % len(actions)])
    torch.cuda.synchronize(dev)
    return ms, n_reset / max(steps, 1)


DUMP_BYTES = 64_000_000
DUMP_SAMPLE_SEED = 2024


def step_outputs(out, logging_key: str) -> dict:
    """
    What one env.step() returned, as float32 / float64 numpy arrays: every observation group, rewards,
    terminated / truncated (0 / 1) and the logged scalars (float64, in the order of `logging_keys`).
    When the per-env arrays together exceed DUMP_BYTES, all of them are cut to the same fixed, seeded
    sample of env rows, stored as `env_index` (float64).
    """
    _, rewards, terminated, truncated, extras = out
    per_env = {f"obs_{group}": t for group, t in extras["observations"].items()}
    per_env.update(rewards=rewards, terminated=terminated, truncated=truncated)
    n = rewards.shape[0]
    row_bytes = sum(4 * (t.numel() // n) for t in per_env.values()) + 8  # + env_index
    keep = min(n, (DUMP_BYTES - 1_000_000) // row_bytes)  # (1 MB left for the logged scalars and file headers)
    arrays = {}
    if keep < n:
        rows = torch.randperm(n, generator=torch.Generator().manual_seed(DUMP_SAMPLE_SEED))[:keep].sort().values
        arrays["env_index"] = rows.double().numpy()
        per_env = {name: t.index_select(0, rows.to(t.device)) for name, t in per_env.items()}
    for name, t in per_env.items():
        arrays[name] = t.float().cpu().numpy()
    logging = extras.get(logging_key, {})
    keys = sorted(logging)
    arrays["logging"] = np.array([float(logging[k]) for k in keys], dtype=np.float64)
    return {"arrays": arrays, "num_envs": n, "logging_keys": keys}


def dump_outputs(directory: str, outputs: dict, meta: dict) -> None:
    os.makedirs(directory, exist_ok=True)
    for name, a in outputs["arrays"].items():
        np.save(os.path.join(directory, f"{name}.npy"), a)
    index = {
        **meta, "num_envs": outputs["num_envs"], "logging_keys": outputs["logging_keys"],
        "arrays": {name: {"shape": list(a.shape), "dtype": str(a.dtype)} for name, a in outputs["arrays"].items()},
    }
    with open(os.path.join(directory, "outputs.json"), "w") as f:
        json.dump(index, f, indent=1)


def pin_to_gpu_numa_node(index: int) -> dict:
    """
    Keep this process (and therefore the pinned host buffers it allocates next: first-touch / local
    allocation policy) on the NUMA node the GPU hangs off, so that host<->device copies do not cross
    the socket interconnect.  Returns what was done, for the `e2e` block.
    """
    info = {"gpu_numa_node": None, "cpus": None}
    try:
        p = torch.cuda.get_device_properties(index)
        bdf = f"{p.pci_domain_id:04x}:{p.pci_bus_id:02x}:{p.pci_device_id:02x}.0"
        with open(f"/sys/bus/pci/devices/{bdf}/numa_node") as f:
            node = int(f.read().strip())
        info["gpu_numa_node"] = node
        if node < 0:
            return info
        with open(f"/sys/devices/system/node/node{node}/cpulist") as f:
            cpus = set()
            for part in f.read().strip().split(","):
                lo, _, hi = part.partition("-")
                cpus.update(range(int(lo), int(hi or lo) + 1))
        allowed = cpus & os.sched_getaffinity(0)
        if allowed:
            os.sched_setaffinity(0, allowed)
            info["cpus"] = len(allowed)
    except Exception as e:  # pragma: no cover - depends on the box
        info["note"] = f"{type(e).__name__}: {e}"[:80]
    return info


def time_e2e(env, actions_host, steps, warmup, dist_on):
    """
    Same step with HOST buffers: every step copies that step's engine state (the arrays the step
    reads) and actions from pinned host memory to the device (inside scene.step(), i.e. where the
    physics engine would produce them) and reads obs / reward / masks back to pinned host memory.
    The observation read-back (the bulk of the D2H bytes) runs on a copy stream so that it overlaps
    the next step's H2D copies (PCIe is full duplex); the host waits for step i-1's read-back before
    it starts step i+1, and the timed region ends when the last read-back has landed.
    """
    import torch.distributed as dist

    fused = env._fused
    dev = fused.device
    scene = env.scene
    # which state arrays does one step read?
    used: set[str] = set()
    original_get = scene._get

    def recording_get(key):
        used.add(key)
        return original_get(key)

    scene._get = recording_get
    env.step(actions_host[0].to(dev))
    scene._get = original_get
    keys = sorted(used)
    host_pool = [{k: st[k].cpu().pin_memory() for k in keys} for st in scene._pool]
    dev_state = {k: (torch.empty_like(v) if k in used else v) for k, v in scene._pool[0].items()}
    h2d_state = sum(dev_state[k].numel() * dev_state[k].element_size() for k in keys)
    counter = {"i": 0}

    def host_fed_step():
        counter["i"] += 1
        src = host_pool[counter["i"] % len(host_pool)]
        for k, v in src.items():
            dev_state[k].copy_(v, non_blocking=True)
        scene.state = dev_state

    original_step = scene.step
    scene.step = host_fed_step
    obs_dev = env.managers["observation"][0]._buffers[0]
    out_host = {
        "obs": [torch.empty_like(obs_dev, device="cpu").pin_memory() for _ in range(2)],
        "rew": torch.empty(env.num_envs, dtype=torch.float32).pin_memory(),
        "term": torch.empty(env.num_envs, dtype=torch.bool).pin_memory(),
        "trunc": torch.empty(env.num_envs, dtype=torch.bool).pin_memory(),
    }
    act_dev = torch.empty((env.num_envs, fused.D), device=dev)
    h2d = h2d_state + act_dev.numel() * 4
    d2h = out_host["obs"][0].numel() * 4 + sum(v.numel() * v.element_size() for k, v in out_host.items() if k != "obs")
    main = torch.cuda.current_stream(dev)
    copy_out = torch.cuda.Stream(dev)
    stepped = [torch.cuda.Event() for _ in range(2)]
    landed = [torch.cuda.Event() for _ in range(2)]

    def one(i):
        act_dev.copy_(actions_host[i % len(actions_host)], non_blocking=True)
        obs, rew, term, trunc, _ = env.step(act_dev)
        out_host["rew"].copy_(rew, non_blocking=True)      # small, rewritten by the next step: in order
        out_host["term"].copy_(term, non_blocking=True)
        out_host["trunc"].copy_(trunc, non_blocking=True)
        stepped[i % 2].record(main)
        with torch.cuda.stream(copy_out):                   # ping-pong observation buffer: safe to overlap
            copy_out.wait_event(stepped[i % 2])
            out_host["obs"][i % 2].copy_(obs, non_blocking=True)
            landed[i % 2].record(copy_out)
        if i > 0:
            landed[(i - 1) % 2].synchronize()               # step i-1's results are on the host

    try:
        for i in range(warmup):
            one(i)
        torch.cuda.synchronize(dev)
        if dist_on:
            dist.barrier()
        start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        start.record(main)
        for i in range(steps):
            one(i)
        main.wait_stream(copy_out)
        end.record(main)
        torch.cuda.synchronize(dev)
        ms = start.elapsed_time(end) / steps
        if dist_on:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
    finally:
        scene.step = original_step
    return ms, h2d, d2h


def time_cpu_reference(spec, num_envs, pool, steps, warmup, seed):
    """
    The reference's own CPU implementation of the path on the host cores, all threads:
    the UNMODIFIED reference package (from /root/reference, or its verbatim copy oracle/_ref made by
    oracle/make_ref.py, which travels to the GPU box) driving the same synthetic engine -- kind
    "reference" -- or, if neither is present, the oracle port (bit-identical to it) -- kind "port".
    Returns (env-steps/s, threads, ms per step, kind).
    """
    from configs.env_builder import make_scene

    threads = os.cpu_count() or 1
    torch.set_num_threads(threads)
    n_contacts = 8 if spec["contacts"] else 0
    kind = "port"
    env = None
    try:
        from oracle import ref_harness

        if ref_harness.reference_available():
            env = ref_harness.make_reference_env(spec, num_envs, n_contacts=n_contacts, seed=seed, pool=pool,
                                                 apply_setters=False)
            kind = "reference"
    except Exception as e:  # pragma: no cover - depends on the box
        print(f"[bench] unmodified reference unavailable ({e}); timing the oracle port", file=sys.stderr)
        env = None
    if env is None:
        from oracle.manager_port import PortEnv

        scene, terrain, robot = make_scene(spec, torch.device("cpu"), copy_on_get=True, pool=pool, seed=seed,
                                           n_contacts=n_contacts, apply_setters=False)
        env = PortEnv(spec, num_envs, scene, terrain, robot)
    import contextlib
    import io

    env.build()
    env.reset()
    gen = torch.Generator().manual_seed(seed)
    n_act = env.action_space.shape[0] if kind == "reference" else env.num_actions
    actions = [torch.randn(num_envs, n_act, generator=gen) for _ in range(2)]
    with contextlib.redirect_stdout(io.StringIO()):  # (the reference prints per-step warnings)
        for i in range(warmup):
            env.step(actions[i % 2])
        t0 = time.perf_counter()
        for i in range(steps):
            env.step(actions[i % 2])
        dt = (time.perf_counter() - t0) / steps
    return num_envs / dt, threads, dt * 1e3, kind


def workload_name(config: str, num_envs: int) -> str:
    return f"{config} manager step (full reward/termination/observation table), num_envs={num_envs} per GPU"


def cpu_sample_envs(num_envs: int, steps: int, warmup: int) -> int:
    """
    Envs per step of the CPU arm: the workload's own batch when the whole run fits in a few minutes,
    otherwise a bounded sample (the metric, env-steps/s, does not depend on the batch beyond cache
    effects; ~1e7 env-steps/s on 16 cores -> 1.2e9 env-steps is about two minutes).
    """
    budget = int(1.2e9 // max(steps + warmup, 1))
    return max(4096, min(num_envs, (budget // 4096) * 4096))


def cpu_model() -> str:
    try:
        with open("/proc/cpuinfo") as f:
            for line in f:
                if line.startswith("model name"):
                    return line.split(":", 1)[1].strip()
    except Exception:
        pass
    return "unknown"


# the BASELINE.json configs 3 / 4 / 5 at the batch sizes it names (config 2 is the headline workload)
EXTRA_CONFIGS = [
    ("contacts", 65536), ("contacts", 1 << 20), ("gait_trainer", 65536), ("rough_terrain", 262144),
    ("berkeley_humanoid", 4096), ("berkeley_humanoid", 65536), ("berkeley_humanoid", 262144),
    ("berkeley_humanoid", 1 << 20),
]


def measure_config(name, n, dev, pool, seed, steps, warmup, peak, dist_on=False, shard=False):
    """One workload through the public API: step time, step / kernel roofline fractions, kernel variant."""
    from configs import specs
    from genesis_forge_b200 import roofline

    env = make_dropin_env(specs.get(name), n, dev, pool, seed)
    fused = env._fused
    if shard:
        env.shard()
    acts = [torch.randn(n, fused.D, device=dev) for _ in range(4)]
    ms, resets = time_dropin(env, acts, steps, warmup, dist_on)
    prof = fused.profile_read()
    fused.profile(False)
    per_step = len(fused.split_plan) if fused.split_mode else 1
    post_us = 1e3 * prof["post_ms"] / max(prof["post_launches"], 1) * per_step
    step_bytes, post_bytes = roofline.step_bytes(fused), roofline.post_kernel_bytes(fused)
    state_mb = sum(v.numel() * v.element_size() for v in env.scene._pool[0].values()) / 1e6
    out = {
        "num_envs": n, "ms_per_step": ms, "value": n / (ms / 1e3), "resets_per_step": resets,
        "step_bytes_per_env": step_bytes, "step_roofline_frac": step_bytes * n / (ms / 1e3) / 1e9 / peak,
        "post_kernel_us": post_us, "post_kernel_launches_per_step": per_step, "post_kernel_bytes_per_env": post_bytes,
        "post_kernel_frac": post_bytes * n / (post_us / 1e6) / 1e9 / peak if post_us > 0 else 0.0,
        "action_kernel_us": 1e3 * prof["action_ms"] / max(prof["action_launches"], 1),
        "traffic": measured_traffic(name, n),
        "l2": f"{pool} state sets of {state_mb:.0f} MB rotated" + ("" if pool * state_mb > 2 * 126 else " (L2-resident: latency point)"),
        "step_mode": "split execution around user-level Python terms" if fused.split_mode else "fused",
        "libraries": fused.spec_stats()["libraries"],
    }
    del env
    torch.cuda.empty_cache()
    return out


# --------------------------------------------------------------------------------------------------
def run_reference(args, rank, world):
    """
    `--impl reference`: the reference's CPU implementation of the same workload, same metric / unit /
    config as the GPU arm, honouring --steps / --warmup; rank 0 only (the other ranks exit).
    """
    from configs import specs

    if rank != 0:
        return
    spec = specs.get(args.config)
    N = args.num_envs
    n = args.cpu_envs or cpu_sample_envs(N, args.steps, args.warmup)
    value, threads, ms, kind = time_cpu_reference(spec, n, args.pool, args.steps, args.warmup, 1234)
    sample = (f"{args.steps} steps of {n} envs ({args.config} term table) on torch-CPU, {threads} threads, "
              f"{cpu_model()}; " + ("the unmodified reference package" if kind == "reference" else "oracle port"))
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name(args.config, N), "pool": args.pool},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def run_b200(args, rank, local_rank, world):
    import torch.distributed as dist

    from genesis_forge_b200 import roofline
    from configs import specs

    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    all_cpus = os.sched_getaffinity(0)
    numa = pin_to_gpu_numa_node(local_rank)  # before any pinned host buffer is allocated
    dist_on = world > 1
    if dist_on:
        dist.init_process_group("nccl", device_id=dev)
    spec = specs.get(args.config)
    N = args.num_envs
    seed = 1234 + rank

    env = make_dropin_env(spec, N, dev, args.pool, seed)
    fused = env._fused
    if dist_on:
        env.shard()  # logging becomes global over WORLD (in-kernel peer-memory exchange)
    gen = torch.Generator().manual_seed(seed)
    actions_host = [torch.randn(N, fused.D, generator=gen).pin_memory() for _ in range(4)]
    actions = [a.to(dev) for a in actions_host]

    sampler = ClockSampler(local_rank) if rank == 0 else None
    dump = args.dump_outputs is not None and rank == 0
    ms, resets_per_step = time_dropin(env, actions, args.steps, args.warmup, dist_on, keep_outputs=dump)
    prof = fused.profile_read()
    aux_prof = fused.profile_read_aux()
    fused.profile(False)
    launches = env.timed_launches
    clocks = sampler.stop(env.timed_window) if sampler else None
    if dump:
        dump_outputs(args.dump_outputs, env.timed_outputs,
                     {"config": args.config, "num_envs_per_gpu": N, "n_gpus": world, "rank": rank, "seed": seed,
                      "steps": args.steps, "warmup": args.warmup, "pool": args.pool})

    value = N * world / (ms / 1e3)
    peak, peak_src = peaks()
    post_ms = prof["post_ms"] / max(prof["post_launches"], 1)
    act_ms = prof["action_ms"] / max(prof["action_launches"], 1)
    post_bytes = roofline.post_kernel_bytes(fused)
    achieved = post_bytes * N / (post_ms / 1e3) / 1e9 if post_ms > 0 else 0.0
    step_bytes = roofline.step_bytes(fused)

    e2e = None
    if not args.no_e2e:
        e2e_ms, h2d, d2h = time_e2e(env, actions_host, args.steps, args.warmup, dist_on)
        e2e = {"value": N * world / (e2e_ms / 1e3), "unit": UNIT, "h2d_bytes_per_step": h2d,
               "d2h_bytes_per_step": d2h, "ms_per_step": e2e_ms, "steps": args.steps, "numa": numa,
               "overlap": "observation read-back of step i on a copy stream, overlapping step i+1's H2D copies"}

    sweep = {}
    if not args.no_sweep and not dist_on:
        for n_small in (4096, 65536):
            if n_small >= N:
                continue
            m = measure_config(args.config, n_small, dev, max(args.pool, 4), seed, args.steps, args.warmup, peak)
            sweep[str(n_small)] = {k: m[k] for k in ("value", "ms_per_step", "post_kernel_us", "action_kernel_us",
                                                       "step_roofline_frac", "l2")}

    # BASELINE configs 3 / 4 / 5 at their named batch sizes (single GPU); under torchrun the
    # strong-scaling point of config 4 instead: 262,144 rough_terrain envs in total, sharded over the ranks
    configs = {}
    strong = None
    if dist_on:
        total = 262144
        if total % world == 0:
            m = measure_config("rough_terrain", total // world, dev, args.pool, seed, args.steps, args.warmup, peak,
                               dist_on=True, shard=True)
            strong = {"config": "rough_terrain", "total_envs": total, "envs_per_gpu": total // world, "scaling": "strong",
                      "ms_per_step": m["ms_per_step"], "value": total / (m["ms_per_step"] / 1e3),
                      "post_kernel_us": m["post_kernel_us"]}
    elif not args.no_configs:
        for name, n_cfg in EXTRA_CONFIGS:
            configs[f"{name}:{n_cfg}"] = measure_config(name, n_cfg, dev, 4, seed, args.steps, args.warmup, peak)

    cpu = None
    os.sched_setaffinity(0, all_cpus)  # the CPU baseline uses every core of the box
    if rank == 0 and not dist_on and not args.no_cpu:
        n_cpu = args.cpu_envs or cpu_sample_envs(N, args.steps, args.warmup)
        v, threads, cpu_ms, kind = time_cpu_reference(spec, n_cpu, args.pool, args.steps, args.warmup, 1234)
        cpu = {"value": v, "unit": UNIT, "cores": threads, "kind": kind, "ms_per_step": cpu_ms,
               "sample": f"{args.steps} steps of {n_cpu} envs ({args.config} term table) on torch-CPU, {cpu_model()}; "
                         + ("the unmodified reference package" if kind == "reference" else "oracle port")}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {
                "workload": workload_name(args.config, N), "pool": args.pool,
                "step_mode": "action kernel, one persistent post-physics kernel (compaction + report inside), "
                             "sparse re-observation of the reset envs",
                "l2_policy": f"{args.pool} pre-generated state sets rotated per step, each set > L2 at this size",
                "resets_per_step": resets_per_step,
                "step_algorithmic_bytes_per_env": step_bytes,
                "step_roofline_frac": step_bytes * N / (ms / 1e3) / 1e9 / peak,
            },
            "roofline": {
                # whole step first (SURVEY.md 8(d): B_alg * N / t_step), then the dominant kernel
                "scope": "whole manager step: algorithmic bytes of the step / device time per step (CUDA events)",
                "bound": "hbm", "achieved": step_bytes * N / (ms / 1e3) / 1e9, "peak": peak, "unit": "GB/s",
                "frac": step_bytes * N / (ms / 1e3) / 1e9 / peak, "bytes_per_env": step_bytes,
                "peak_source": peak_src,
                "traffic": measured_traffic(args.config, N),  # DRAM bytes of one post_kernel launch (ncu), or null if stale
                "kernel": {
                    "name": "post_kernel (gfb_post_physics)", "bytes_per_env": post_bytes, "kernel_us": post_ms * 1e3,
                    "achieved": achieved, "frac": achieved / peak,
                    # sharded envs: the kernel's last block waits inside the launch for the slowest peer's
                    # logging partials (csrc/tail.cuh), so this duration includes the ranks' skew
                    **({"includes_peer_wait": True} if world > 1 else {}),
                },
                "action_kernel": {"bytes_per_env": roofline.action_kernel_bytes(fused), "kernel_us": act_ms * 1e3,
                                  "achieved": roofline.action_kernel_bytes(fused) * N / max(act_ms, 1e-9) / 1e6,
                                  "frac": roofline.action_kernel_bytes(fused) * N / max(act_ms, 1e-9) / 1e6 / peak},
                "small_kernels": aux_prof,  # CUDA-event time per launch: reset rows, re-observation, spawn
            },
            "cpu_baseline": cpu,
            "e2e": e2e,
            "gpu_launches": launches,
            "kernel_variant": fused.spec_stats(),
            "clocks": clocks,
            "sweep": sweep,
            "configs": configs,
            "strong_scaling": strong,
        }
        print(json.dumps(line), flush=True)
    if dist_on:
        dist.destroy_process_group()


def main():
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl b200 needs a CUDA device (the manager step has no CPU fallback)")
    run_b200(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
