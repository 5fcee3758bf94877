"""
Workloads of the lowered class-style user terms (ManagedEnvironment.fuse_stateful_terms): MdpFnClass terms
that keep per-env state from one step to the next, the usual legged-RL kind.

A -- `override()`: the `command_direction` table (no contact managers) plus
    joint_accel   joint acceleration from the previous joint velocity (fp32 (N,12) state, rebound), scaled by
                  a read-only per-env gain drawn in __init__;
    action_jerk   action jerk over two steps of action history, initialised lazily (the first call sees
                  zeros);
    speed_ema     an exponential moving average of the forward velocity (fp32 (N,) state; the rate is a
                  Python-scalar attribute, a trace constant);
    tilt_latch    a bool "was tilted this episode" latch, written with copy_;
    stuck         a termination after `limit` steps without moving (int32 (N,) counter written with
                  [:] =, cleared at episode_length == 1).
The port has no manager objects for these to call, so they are checked against the drop-in's own
host-callback path (fuse_stateful_terms off).

B -- `contacts_override()`: the `contacts` table plus one lazily initialised contact-streak reward, which
reads nothing but what the oracle port exposes too.

Kept out of specs.ALL / VARIANTS (which the golden-trace tests walk), like configs/user_terms.py.
"""
from __future__ import annotations

import torch

from genesis_forge_b200.managers.config import MdpFnClass

from . import specs


def _rows(env, *shape, dtype=torch.float32):
    return torch.zeros((env.num_envs,) + shape, device=env.episode_length.device, dtype=dtype)


class joint_accel(MdpFnClass):
    def __init__(self, env, scale=1.0e-4, seed=3):
        super().__init__(env)
        self.prev_vel = _rows(env, 12)
        dev = env.episode_length.device
        gen = torch.Generator(device=dev).manual_seed(seed)
        self.gain = torch.rand(env.num_envs, generator=gen, device=dev) + 0.5  # read-only per-env state

    def __call__(self, env, scale=1.0e-4, seed=3):
        vel = env.action_manager.get_dofs_velocity()
        acc = (vel - self.prev_vel) / env.dt
        self.prev_vel = vel.clone()
        return acc.square().sum(dim=1) * scale * self.gain


class action_jerk(MdpFnClass):
    def __init__(self, env):
        super().__init__(env)
        self.prev1 = None
        self.prev2 = None

    def __call__(self, env):
        a = env.actions
        if self.prev1 is None:
            self.prev1 = torch.zeros_like(a)
            self.prev2 = torch.zeros_like(a)
        jerk = a - 2.0 * self.prev1 + self.prev2
        self.prev2 = self.prev1
        self.prev1 = a.clone()
        return jerk.square().sum(dim=1)


class speed_ema(MdpFnClass):
    def __init__(self, env, rate=0.1):
        super().__init__(env)
        self.rate = rate
        self.ema = _rows(env)

    def __call__(self, env, rate=0.1):
        v = env.robot_manager.get_linear_velocity()[:, 0]
        self.ema = self.ema * (1.0 - self.rate) + v * self.rate
        err = self.ema - env.velocity_command.command[:, 0]
        return torch.exp(-err.square() / 0.25)


class tilt_latch(MdpFnClass):
    def __init__(self, env, limit=-0.98):
        super().__init__(env)
        self.tilted = _rows(env, dtype=torch.bool)

    def __call__(self, env, limit=-0.98):
        g = env.robot_manager.get_projected_gravity()
        self.tilted.copy_((self.tilted | (g[:, 2] > limit)) & (env.episode_length > 1))
        return self.tilted.float()


class stuck(MdpFnClass):
    def __init__(self, env, min_speed=0.05, limit=40):
        super().__init__(env)
        self.count = _rows(env, dtype=torch.int32)

    def __call__(self, env, min_speed=0.05, limit=40):
        moving = env.robot_manager.get_linear_velocity()[:, :2].norm(dim=1) > min_speed
        self.count[:] = torch.where(moving | (env.episode_length == 1), 0, self.count + 1)
        return self.count >= limit


class contact_streak(MdpFnClass):
    """Seconds each tracked foot has been in contact (reset when it lifts), capped at 0.5 s and summed."""

    def __init__(self, env, threshold=1.0):
        super().__init__(env)
        self.streak = None

    def __call__(self, env, threshold=1.0):
        forces = env.foot_contact_manager.contacts
        if self.streak is None:
            self.streak = torch.zeros_like(forces[:, :, 0])
        on = forces[:, :, 2].abs() > threshold
        self.streak = torch.where(on, self.streak + env.dt, 0.0)
        return self.streak.clamp(max=0.5).sum(dim=1)


def override() -> dict:
    """`spec_override` turning the command_direction spec into workload A."""
    s = specs.command_direction()
    rewards = dict(s["rewards"])
    rewards.update({
        "joint_accel": {"fn": joint_accel, "weight": -0.5, "params": {"scale": 1.0e-4}},
        "action_jerk": {"fn": action_jerk, "weight": -0.01},
        "speed_ema": {"fn": speed_ema, "weight": 0.3, "params": {"rate": 0.1}},
        "tilt_latch": {"fn": tilt_latch, "weight": -0.2},
    })
    terminations = dict(s["terminations"])
    terminations["stuck"] = {"fn": stuck, "params": {"min_speed": 0.05, "limit": 40}}
    return {"name": "stateful_terms", "rewards": rewards, "terminations": terminations}


def stateful_terms() -> dict:
    s = specs.command_direction()
    s.update(override())
    return s


def contacts_override() -> dict:
    """`spec_override` turning the contacts spec into workload B."""
    s = specs.contacts()
    rewards = dict(s["rewards"])
    rewards["contact_streak"] = {"fn": contact_streak, "weight": 0.2, "params": {"threshold": 1.0}}
    return {"name": "stateful_contacts", "rewards": rewards}


def stateful_contacts() -> dict:
    s = specs.contacts()
    s.update(contacts_override())
    return s
