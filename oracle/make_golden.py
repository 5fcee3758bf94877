"""
TEST INFRASTRUCTURE (oracle).  Regenerates tests/golden/<config>.pt.xz from the UNMODIFIED reference.

    python -m oracle.make_golden            (needs /root/reference; run in the build container)

For every spec in configs/specs.py the reference's own ManagedEnvironment + managers (imported from
/root/reference under oracle/shim.py, Taichi contact kernel replaced by the ordered restatement) is
built against the seeded synthetic engine and stepped; the trace records, per step, the actions
fed in and everything the step returned (obs per group, rewards, terminated, truncated, logged
extras, reset indices), plus a full snapshot of every manager buffer at the end and a float64
checksum of each step's synthetic physics state (so a test can tell "the input stream drifted"
from "the implementation is wrong").  The torch build string is stored with the trace because the
last-ulp behaviour of the CPU reference depends on ATen's dispatch level (SURVEY.md 7-1d).
"""
from __future__ import annotations

import io
import lzma
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN_DIR = os.path.join(ROOT, "tests", "golden")
NUM_ENVS, STEPS, SEED, NAN_STEP = 16, 48, 2024, 5


def save(trace: dict, name: str) -> str:
    """tests/golden/<name>.pt.xz: the torch.save of `trace`, xz-compressed (a trace with a few hundred
    observation columns is 1.5 MB raw, 0.2 MB compressed); replaces an uncompressed <name>.pt."""
    buf = io.BytesIO()
    torch.save(trace, buf)
    path = os.path.join(GOLDEN_DIR, f"{name}.pt.xz")
    with open(path, "wb") as f:
        f.write(lzma.compress(buf.getvalue(), preset=9 | lzma.PRESET_EXTREME))
    stale = os.path.join(GOLDEN_DIR, f"{name}.pt")
    if os.path.exists(stale):
        os.remove(stale)
    return path


def load(name: str) -> dict:
    """The golden trace `name`: tests/golden/<name>.pt.xz, or the uncompressed tests/golden/<name>.pt."""
    path = os.path.join(GOLDEN_DIR, f"{name}.pt.xz")
    if os.path.exists(path):
        with open(path, "rb") as f:
            return torch.load(io.BytesIO(lzma.decompress(f.read())), weights_only=False)
    path = os.path.join(GOLDEN_DIR, f"{name}.pt")
    assert os.path.exists(path), f"missing golden fixture {path} (python -m oracle.make_golden)"
    return torch.load(path, weights_only=False)


def state_checksum(scene) -> float:
    return float(sum(v.double().sum() for k, v in sorted(scene.state.items()) if v.is_floating_point()))


def trace_of(env, spec, num_envs: int, steps: int, seed: int, nan_step: int | None, logging_of, snapshot_of,
             extra_of=None):
    """Drive `env` (any implementation with the reference API) and record the golden trace."""
    torch.manual_seed(seed)
    env.build()
    obs, extras = env.reset()
    trace = {
        "spec_name": spec["name"], "num_envs": num_envs, "steps": steps, "seed": seed, "nan_step": nan_step,
        "torch": torch.__version__, "torch_config": torch.__config__.show(),
        "reset": {"obs": {g: t.clone() for g, t in extras["observations"].items()}, "logging": logging_of(extras)},
        "step": [],
    }
    gen = torch.Generator().manual_seed(seed + 77)
    n_act = env.action_space.shape[0] if hasattr(env, "action_space") else env.num_actions
    for i in range(steps):
        actions = torch.randn(num_envs, n_act, generator=gen)
        if nan_step is not None and i == nan_step:
            actions[min(3, num_envs - 1), 1] = float("nan")
        out = env.step(actions.clone())
        trace["step"].append({
            "obs": {g: t.clone() for g, t in out[4]["observations"].items()},
            "rewards": out[1].clone(), "terminated": out[2].clone(), "truncated": out[3].clone(),
            "reset_idx": (out[2] | out[3]).nonzero().reshape(-1).clone(),
            "logging": logging_of(out[4]),
            "state_checksum": state_checksum(env.scene),
        })
        if extra_of is not None:
            trace["step"][-1]["extra"] = extra_of(env)
    trace["final"] = snapshot_of(env)
    return trace


def main(names=None):
    from configs import specs

    from . import compare, ref_harness

    if not ref_harness.reference_available():
        raise SystemExit("needs /root/reference")
    os.makedirs(GOLDEN_DIR, exist_ok=True)
    for name in (n for n in names if not n.startswith("second_entity")) if names else list(specs.ALL) + list(specs.VARIANTS):
        spec = specs.get(name)
        env = ref_harness.make_reference_env(spec, NUM_ENVS, seed=SEED)
        trace = trace_of(env, spec, NUM_ENVS, STEPS, SEED, NAN_STEP, compare.extras_to_cpu, compare.reference_snapshot)
        path = save(trace, name)
        n_reset = sum(int(s["reset_idx"].numel()) for s in trace["step"])
        print(f"{path}: {os.path.getsize(path) / 1024:.0f} KiB, {n_reset} resets in {STEPS} steps")
    for stock_terms in (False, True):
        name = "second_entity_terms" if stock_terms else "second_entity"
        if not names or name in names:
            second_entity_trace(stock_terms)


def second_entity_trace(stock_terms: bool = False):
    """Two EntityManagers (configs/second_entity.py): the reference's trace incl. the prop manager's cache."""
    from configs import second_entity
    from configs.env_builder import reference_namespace

    from . import compare, ref_harness

    spec = second_entity.spec(stock_terms)
    env = second_entity.add_prop(ref_harness.make_reference_env(spec, NUM_ENVS, seed=SEED), reference_namespace())
    trace = trace_of(env, spec, NUM_ENVS, STEPS, SEED, None, compare.extras_to_cpu, lambda env: {},
                     extra_of=second_entity.prop_cache)
    path = save(trace, spec["name"])
    n_reset = sum(int(s["reset_idx"].numel()) for s in trace["step"])
    print(f"{path}: {os.path.getsize(path) / 1024:.0f} KiB, {n_reset} resets in {STEPS} steps")


if __name__ == "__main__":
    main(sys.argv[1:] or None)
