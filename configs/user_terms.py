"""
Workload of the lowered user-defined terms (ManagedEnvironment.fuse_user_terms): the `contacts` table
(configs/specs.py) plus user-defined rewards and terminations that together read every source the
expression IR supports on the oracle port's side as well -- the robot's getters, contact forces and
air time, the velocity command, env.actions / last_actions, episode_length / max_episode_length and,
in rewards, extras["terminations"] / ["time_outs"] -- with every op class of genesis_forge_b200/expr.py.

Kept out of specs.ALL / VARIANTS (which the golden-trace tests walk): it is run through
`ParityRun("contacts", ..., spec_override=override())`.  Termination thresholds only compare values
the kernel reproduces bit for bit (raw engine state, counters, raw actions), so the masks stay exact
without guard-band knowledge of user thresholds.
"""
from __future__ import annotations

import torch

from . import specs

CLOCK_RATE = 0.05  # a closure constant: folded into the kernel


def contact_z(env, gain=0.01):
    return env.foot_contact_manager.contacts[:, :, 2].sum(dim=1) * gain + env.extras["terminations"].float()


def level_speed(env, scale=0.25):
    return torch.exp(-env.robot.get_vel()[:, :2].square().sum(1) / scale)


def action_excess(env, lim=1.5):
    a = env.actions.abs()
    return torch.where(a > lim, a - lim, 0.0).sum(1)


def clock(env):
    return torch.sin(env.episode_length.float() * CLOCK_RATE) * env.velocity_command.command[:, 0]


def air_time(env, lo=0.1):
    return torch.clamp(env.foot_contact_manager.last_air_time - lo, min=0.0, max=0.5).mean(1)


def smoothness(env):
    delta = (env.actions - env.last_actions).norm(dim=-1)
    spin = env.robot.get_ang()[..., 2].abs().sqrt()
    every4 = (env.episode_length % 4 == 0).float()
    return torch.tanh(delta * 0.1) + torch.cos(spin) * every4 - torch.log(1.0 + delta)


def progress(env):
    frac = env.episode_length.float() / env.max_episode_length.float()
    peak = env.robot.get_quat().amax(dim=1) - env.robot.get_quat().amin(dim=-1)
    return torch.minimum(frac, torch.tensor(0.5)) + torch.maximum(peak, env.robot.get_pos()[:, 2]) ** 2


def outcome(env):
    alive = ~env.extras["terminations"]
    return env.extras["time_outs"].float() * 0.5 - alive.float() * 0.01 + (alive & (env.episode_length > 10)).float()


def wandered_off(env, limit=9.6):
    return env.robot.get_pos()[:, 0] > limit


def slow_start(env, min_speed=-1.2):
    return (env.episode_length > 50) & (env.robot.get_vel()[:, 0] < min_speed)


def dropped(env):
    low = env.robot.get_pos()[:, 2] < 0.1
    return low | ((env.episode_length % 97) == 96) | (env.actions.abs() > 3.5).any(dim=1)


# ---- second workload: the first EntityManager's and the action manager's getters ---------------------
# The oracle port has no manager objects for user terms to call, so these are checked against the drop-in's
# own host-callback path (fuse_user_terms off), which evaluates them with the library's rotation kernel
# and the engine getters.  Based on command_direction (no contact managers).
JOINT_CENTER = torch.tensor([0.0, 0.8, -1.5, 0.0, 0.8, -1.5, 0.0, 1.0, -1.5, 0.0, 1.0, -1.5])  # folded in


def upright(env, scale=0.25):
    g = env.robot_manager.get_projected_gravity()
    return torch.exp(-g[:, :2].square().sum(1) / scale)


def joint_limit(env, lim=0.6):
    q = env.action_manager.get_dofs_position()
    dev = (q - JOINT_CENTER.to(q.device)).abs()
    return torch.where(dev > lim, dev - lim, 0.0).sum(1)


def body_rates(env):
    v = env.robot_manager.get_linear_velocity()
    w = env.robot_manager.get_angular_velocity()
    calm = (w.abs() <= 2.0).all(dim=1).float()
    return torch.clip(v[:, 0], -1.0, 1.0) * calm + (v[:, 1] >= 0.0).float() * 0.1 + (w[:, 2] != 0.0).float() * 0.01


def joint_effort(env):
    am = env.action_manager
    return am.get_dofs_velocity().square().mean(1) * 0.01 + (am.get_actions() - am.get_dofs_position()).abs().amax(dim=1)


def cached_height(env, target=0.3):
    em = env.robot_manager
    return (em.base_pos[:, 2] - target).square() + em.base_quat[:, 0].abs()


def tipped(env, limit=-0.2):
    return (env.robot_manager.get_projected_gravity()[:, 2] >= limit) & (env.episode_length > 5)


def joint_out(env):
    return (env.action_manager.get_dofs_position().abs() > 2.5).any(dim=1)


def entity_override() -> dict:
    """`spec_override` turning the command_direction spec into the second workload."""
    s = specs.command_direction()
    rewards = dict(s["rewards"])
    rewards.update({
        "upright": {"fn": upright, "weight": 0.5, "params": {"scale": 0.25}},
        "joint_limit": {"fn": joint_limit, "weight": -0.1, "params": {"lim": 0.6}},
        "body_rates": {"fn": body_rates, "weight": 0.2},
        "joint_effort": {"fn": joint_effort, "weight": -0.05},
        "cached_height": {"fn": cached_height, "weight": -1.0, "params": {"target": 0.3}},
    })
    terminations = dict(s["terminations"])
    terminations.update({
        "tipped": {"fn": tipped, "params": {"limit": -0.2}},
        "joint_out": {"fn": joint_out},
    })
    return {"name": "user_terms_entity", "rewards": rewards, "terminations": terminations}


def user_terms_entity() -> dict:
    s = specs.command_direction()
    s.update(entity_override())
    return s


def override() -> dict:
    """`spec_override` turning the contacts spec into this workload."""
    s = specs.contacts()
    rewards = dict(s["rewards"])
    rewards.update({
        "contact_z": {"fn": contact_z, "weight": -0.2, "params": {"gain": 0.02}},
        "level_speed": {"fn": level_speed, "weight": 0.3, "params": {"scale": 0.5}},
        "action_excess": {"fn": action_excess, "weight": -0.05, "params": {"lim": 1.5}},
        "clock": {"fn": clock, "weight": 0.1},
        "air_time": {"fn": air_time, "weight": 1.0, "params": {"lo": 0.1}},
        "smoothness": {"fn": smoothness, "weight": -0.02},
        "progress": {"fn": progress, "weight": 0.05},
        "outcome": {"fn": outcome, "weight": 1.0},
    })
    terminations = dict(s["terminations"])
    terminations.update({
        "wandered_off": {"fn": wandered_off, "params": {"limit": 9.6}},
        "slow_start": {"fn": slow_start, "params": {"min_speed": -1.2}},
        "dropped": {"fn": dropped},
    })
    return {"name": "user_terms", "rewards": rewards, "terminations": terminations}


def user_terms() -> dict:
    s = specs.contacts()
    s.update(override())
    return s
