"""
Workloads of the lowered class-style user observation terms (ManagedEnvironment.fuse_stateful_terms):
MdpFnClass observation terms that keep per-env state from one observation to the next.

A -- `override()`: the `command_direction` table (no contact managers) plus, in the policy group,
    gait_clock      a gait-phase clock: fp32 (N,) phase advanced by dt * freq and wrapped with where, where
                    freq is a read-only per-env tensor drawn in __init__; cleared at episode_length == 0 and
                    observed as stack([sin, cos]);
    joint_vel_filt  low-pass-filtered joint velocities, (N, 12), initialised lazily from the first velocity
                    (the build's dry run makes that first call);
    action_history  the last two actions, two (N, 12) tensors rebound every call, observed as cat;
    still_steps     an int32 "steps without moving" counter written with [:] =, observed as a clamped float.
                    It is exact, so a state that advanced twice in one step shows;
  and a second group ("history", history_len=3) with another instance of the clock under the same name.
  A uses exactly the 8 state slots of the ABI: 2 per clock, 1 for the filter, 2 for the history, 1 for the
  counter.  The port has no manager objects for these to call, so they are checked against the drop-in's own
  host-column path (fuse_stateful_terms off).

A-split -- `split_override()`: A plus one plain user reward, which stays a host callback (fuse_user_terms
  off): the step runs split, and the lowered observation terms run in its observe-only launch.

B -- `contacts_override()`: the `contacts` table plus a per-foot "seconds since touchdown" observation,
  (N, Lc) fp32 state initialised lazily, which reads nothing but what the oracle port exposes too.

User observation terms are called with their default arguments (as the port calls them).  Kept out of specs.ALL / VARIANTS (which the golden-trace tests walk), like configs/user_terms.py.
"""
from __future__ import annotations

import math

import torch

from genesis_forge_b200.managers.config import MdpFnClass

from . import specs


def _rows(env, *shape, dtype=torch.float32):
    return torch.zeros((env.num_envs,) + shape, device=env.episode_length.device, dtype=dtype)


class gait_clock(MdpFnClass):
    def __init__(self, env, seed=5):
        super().__init__(env)
        dev = env.episode_length.device
        gen = torch.Generator(device=dev).manual_seed(seed)
        self.freq = torch.rand(env.num_envs, generator=gen, device=dev) + 1.5  # read-only per-env state
        self.phase = _rows(env)

    def __call__(self, env, seed=5):
        phase = torch.where(env.episode_length == 0, 0.0, self.phase + env.dt * self.freq)
        self.phase = torch.where(phase >= 1.0, phase - 1.0, phase)
        angle = self.phase * (2.0 * math.pi)
        return torch.stack([torch.sin(angle), torch.cos(angle)], dim=1)


class joint_vel_filt(MdpFnClass):
    def __init__(self, env, alpha=0.3):
        super().__init__(env)
        self.alpha = alpha  # a Python-scalar attribute: a trace constant
        self.filt = None

    def __call__(self, env, alpha=0.3):
        v = env.action_manager.get_dofs_velocity()
        if self.filt is None:
            self.filt = v.clone()
        self.filt = self.filt + (v - self.filt) * self.alpha
        return self.filt * 0.05


class action_history(MdpFnClass):
    def __init__(self, env):
        super().__init__(env)
        self.prev1 = _rows(env, 12)
        self.prev2 = _rows(env, 12)

    def __call__(self, env):
        out = torch.cat([self.prev1, self.prev2], dim=1)
        self.prev2 = self.prev1
        self.prev1 = env.action_manager.get_actions().clone()
        return out


class still_steps(MdpFnClass):
    def __init__(self, env, min_speed=0.2, cap=50):
        super().__init__(env)
        self.count = _rows(env, dtype=torch.int32)

    def __call__(self, env, min_speed=0.2, cap=50):
        moving = env.robot_manager.get_linear_velocity()[:, :2].norm(dim=1) > min_speed
        self.count[:] = torch.where(moving | (env.episode_length == 0), 0, self.count + 1)
        return self.count.clamp(max=cap).float()


class touchdown_clock(MdpFnClass):
    """Seconds each tracked foot has been on the ground since its last touchdown (0 in the air), capped at 1 s."""

    def __init__(self, env, threshold=1.0):
        super().__init__(env)
        self.since = None

    def __call__(self, env, threshold=1.0):
        forces = env.foot_contact_manager.contacts
        if self.since is None:
            self.since = torch.zeros_like(forces[:, :, 0])
        on = forces[:, :, 2].abs() > threshold
        self.since = torch.where(on, self.since + env.dt, 0.0)
        return self.since.clamp(max=1.0)


# the A terms that keep state: name -> (group, state attributes)
STATE = {("policy", "gait_clock"): ("phase", "freq"), ("policy", "joint_vel_filt"): ("filt",),
         ("policy", "action_history"): ("prev1", "prev2"), ("policy", "still_steps"): ("count",),
         ("history", "gait_clock"): ("phase", "freq")}


def override() -> dict:
    """`spec_override` turning the command_direction spec into workload A."""
    s = specs.command_direction()
    policy = dict(s["observations"]["policy"]["terms"])
    policy.update({
        "gait_clock": {"fn": gait_clock},
        "joint_vel_filt": {"fn": joint_vel_filt},
        "action_history": {"fn": action_history},
        "still_steps": {"fn": still_steps, "scale": 0.02},
    })
    history = {"gait_clock": {"fn": gait_clock}}
    return {"name": "stateful_observations",
            "observations": {"policy": {"terms": policy}, "history": {"terms": history, "history_len": 3}}}


def stateful_observations() -> dict:
    s = specs.command_direction()
    s.update(override())
    return s


def upright_bonus(env):
    return -env.robot_manager.get_projected_gravity()[:, 2]


def split_override() -> dict:
    """`spec_override` turning the command_direction spec into workload A-split."""
    out = override()
    rewards = dict(specs.command_direction()["rewards"])
    rewards["upright_bonus"] = {"fn": upright_bonus, "weight": 0.1}
    return dict(out, name="stateful_observations_split", rewards=rewards)


def stateful_observations_split() -> dict:
    s = specs.command_direction()
    s.update(split_override())
    return s


def contacts_override() -> dict:
    """`spec_override` turning the contacts spec into workload B."""
    s = specs.contacts()
    policy = dict(s["observations"]["policy"]["terms"])
    policy["touchdown_clock"] = {"fn": touchdown_clock}
    return {"name": "stateful_contact_observations", "observations": {"policy": {"terms": policy}}}


def stateful_contact_observations() -> dict:
    s = specs.contacts()
    s.update(contacts_override())
    return s
