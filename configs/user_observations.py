"""
Workloads of the lowered user-defined observation terms (ManagedEnvironment.fuse_user_observations).

A -- `override()`: the `contacts` table (configs/specs.py) with user observation functions over the sources
the oracle port exposes too: the robot's getters, episode_length, the velocity command, contact forces and
air time (not env.actions: it is still None when the reference sizes its observation space).  They use the layout ops (a two-column torch.stack clock,
torch.cat, unsqueeze, None in an index, view / reshape / flatten), carry scale and noise, and fill a second
group with history_len=3.  The policy group is 62 columns wide (not a multiple of 4), the history group 4.
Run through `ParityRun("contacts", ..., spec_override=override())` against the port.

B -- `entity_override()`: the `command_direction` table with user observation functions over the first
EntityManager's body-frame getters and cached pose and the action manager's getters (joint state,
targets).  The port has no manager objects, so these are checked against the drop-in's own host-column
path (fuse_user_observations off).

Kept out of specs.ALL / VARIANTS (which the golden-trace tests walk), like configs/user_terms.py.  Terms that
carry scale or noise return fresh tensors: the reference scales and perturbs a term's value in place.
"""
from __future__ import annotations

import torch

from . import specs

CLOCK_RATE = 0.1  # a closure constant: folded into the kernel
CMD_GAIN = torch.tensor([2.0, 2.0, 0.25])  # a constant vector: folded in


def gait_clock(env):
    phase = env.episode_length.float() * CLOCK_RATE
    return torch.stack([torch.sin(phase), torch.cos(phase)], 1)


def base_height(env):
    return env.robot.get_pos()[:, 2:3]


def command_scaled(env):
    return env.velocity_command.command * CMD_GAIN.to(env.velocity_command.command.device)


def feet_down(env, threshold=1.0):
    return (env.foot_contact_manager.contacts[..., 2] > threshold).float()


def planar_motion(env):
    return torch.cat([env.robot.get_vel()[:, :2], env.robot.get_ang()[:, None, 2]], dim=-1)


def quat_tail(env):
    return env.robot.get_quat().view(-1, 2, 2)[:, 1].reshape(env.num_envs, -1)


def air_clock(env):
    air = env.foot_contact_manager.last_air_time
    return (air.sum(1).unsqueeze(1) + env.episode_length.unsqueeze(-1)).flatten(1)


def override(noise: bool = True) -> dict:
    """`spec_override` turning the contacts spec into workload A (`noise=False`: without observation noise, for
    the port's production-mode comparison, which takes the kernels' draws and has none for noise)."""
    s = specs.contacts()
    policy = dict(s["observations"]["policy"]["terms"])
    policy.update({
        "gait_clock": {"fn": gait_clock},
        "base_height": {"fn": base_height},
        "command_scaled": {"fn": command_scaled, **({"noise": 0.05} if noise else {})},
        "feet_down": {"fn": feet_down, "scale": 0.5},
        "planar_motion": {"fn": planar_motion, "scale": 0.25, **({"noise": 0.01} if noise else {})},
        "air_clock": {"fn": air_clock, "scale": 0.01},
    })
    history = {"clock": {"fn": gait_clock}, "quat_tail": {"fn": quat_tail}}
    return {"name": "user_observations",
            "observations": {"policy": {"terms": policy}, "history": {"terms": history, "history_len": 3}}}


def user_observations() -> dict:
    s = specs.contacts()
    s.update(override())
    return s


# ---- workload B: the first EntityManager's and the action manager's getters --------------------------
def upright(env):
    return env.robot_manager.get_projected_gravity()[:, :2] * 2.0


def cached_pose(env):
    em = env.robot_manager
    return torch.cat([em.base_pos[:, 2:3], em.base_quat], dim=1)


def joint_error(env):
    am = env.action_manager
    return (am.get_actions() - am.get_dofs_position()) * 0.5


def body_speed(env):
    return env.robot_manager.get_linear_velocity().norm(dim=-1).unsqueeze(1)


def yaw_rate(env):
    return env.robot_manager.get_angular_velocity()[:, None, 2]


def joint_speed(env):
    return env.action_manager.get_dofs_velocity().view(-1, 4, 3).flatten(1)


def entity_override() -> dict:
    """`spec_override` turning the command_direction spec into workload B."""
    s = specs.command_direction()
    policy = dict(s["observations"]["policy"]["terms"])
    policy.update({
        "upright": {"fn": upright},
        "cached_pose": {"fn": cached_pose, "noise": 0.01},
        "joint_error": {"fn": joint_error},
        "body_speed": {"fn": body_speed, "scale": 0.5},
        "yaw_rate": {"fn": yaw_rate},
        "joint_speed": {"fn": joint_speed, "scale": 0.05},
    })
    return {"name": "user_observations_entity", "observations": {"policy": {"terms": policy}}}


def user_observations_entity() -> dict:
    s = specs.command_direction()
    s.update(entity_override())
    return s
