"""
Workloads of user terms that call stock mdp terms (ManagedEnvironment.fuse_stock_calls): the usual way of
gating, mixing or rescaling a stock reward or termination in user code.

A -- `stock_calls_a()`: the `command_direction` table plus
    gated_tracking  command_tracking_lin_vel with a live `sensitivity`, gated by the command's xy norm
    upright         1 - flat_orientation_l2, clamped at 0
    smooth          action_rate_l2 + 0.5 * lin_vel_z_l2
    alive_yaw       is_alive * command_tracking_ang_vel
    posture_ema     class-style: an exponential moving average of dof_similar_to_default
    lin_vel_z_wrap  an identity wrapper of the stock `lin_vel_z` row (same params, same weight)
  terminations
    fell            bad_orientation | base_height_below_minimum
    fall_over_wrap  an identity wrapper of the stock `fall_over` row (it fires with it: the step is unchanged)
B -- `stock_calls_b()`: the `contacts` table plus
    air_when_moving feet_air_time, credited only while the base moves forward
    contact_mix     has_contact(min_contacts=2) - 0.01 * contact_force(threshold=50)
    slide           feet_slide times a live user factor
  termination
    hard_hit        contact_force_with_grace_period | base below 0.1

Lowering everything needs fuse_user_terms, fuse_stateful_terms and fuse_stock_calls.  Kept out of specs.ALL /
VARIANTS (which the golden-trace tests walk), like configs/user_terms.py.
"""
from __future__ import annotations

import torch

from genesis_forge_b200.managers.config import MdpFnClass
from genesis_forge_b200.mdp import rewards, terminations

from . import specs


def gated_tracking(env, sensitivity=0.25):
    cmd = env.velocity_command.command
    tracking = rewards.command_tracking_lin_vel(env, vel_cmd_manager=env.velocity_command, sensitivity=sensitivity,
                                                entity_manager=env.robot_manager)
    return tracking * (cmd[:, :2].norm(dim=-1) > 0.1)


def upright(env):
    return (1.0 - rewards.flat_orientation_l2(env, entity_manager=env.robot_manager)).clamp(min=0.0)


def smooth(env):
    return rewards.action_rate_l2(env) + 0.5 * rewards.lin_vel_z_l2(env, entity_manager=env.robot_manager)


def alive_yaw(env):
    return rewards.is_alive(env) * rewards.command_tracking_ang_vel(env, vel_cmd_manager=env.velocity_command,
                                                                    entity_manager=env.robot_manager)


class posture_ema(MdpFnClass):
    def __init__(self, env, rate=0.2):
        super().__init__(env)
        self.rate = rate
        self.ema = torch.zeros(env.num_envs, device=env.episode_length.device)

    def __call__(self, env, rate=0.2):
        deviation = rewards.dof_similar_to_default(env, action_manager=env.action_manager)
        self.ema = self.ema * (1.0 - self.rate) + deviation * self.rate
        return self.ema


def lin_vel_z_wrap(env):
    return rewards.lin_vel_z_l2(env, entity_manager=env.robot_manager)


def fell(env):
    return (terminations.bad_orientation(env, limit_angle=35.0, entity_manager=env.robot_manager)
            | terminations.base_height_below_minimum(env, minimum_height=0.15, entity_manager=env.robot_manager))


def fall_over_wrap(env):
    return terminations.bad_orientation(env, limit_angle=10.0, entity_manager=env.robot_manager)


def air_when_moving(env, time_threshold=0.5):
    air = rewards.feet_air_time(env, contact_manager=env.foot_contact_manager, time_threshold=time_threshold)
    return air * (env.robot_manager.get_linear_velocity()[:, 0].abs() > 0.2)


def contact_mix(env):
    fcm = env.foot_contact_manager
    return (rewards.has_contact(env, fcm, threshold=1.0, min_contacts=2)
            - 0.01 * rewards.contact_force(env, fcm, threshold=50.0))


def slide(env, factor=0.5):
    return rewards.feet_slide(env, contact_manager=env.foot_contact_manager) * factor


def hard_hit(env):
    hit = terminations.contact_force_with_grace_period(env, contact_manager=env.foot_contact_manager,
                                                       threshold=400.0, grace_steps=10)
    return hit | (env.robot.get_pos()[:, 2] < 0.1)


# the wrapped stock rows' names next to the wrappers' (the GPU tests compare them step by step)
WRAPPED = {"lin_vel_z_wrap": "lin_vel_z", "fall_over_wrap": "fall_over"}


def stock_calls_a() -> dict:
    s = specs.command_direction()
    stock = s["rewards"]["lin_vel_z"]
    rewards_ = dict(s["rewards"])
    rewards_.update({
        "gated_tracking": {"fn": gated_tracking, "weight": 0.5, "params": {"sensitivity": 0.25}},
        "upright": {"fn": upright, "weight": 0.2},
        "smooth": {"fn": smooth, "weight": -0.01},
        "alive_yaw": {"fn": alive_yaw, "weight": 0.3},
        "posture_ema": {"fn": posture_ema, "weight": -0.05},
        "lin_vel_z_wrap": {"fn": lin_vel_z_wrap, "weight": stock["weight"]},
    })
    terms = dict(s["terminations"], fell={"fn": fell}, fall_over_wrap={"fn": fall_over_wrap})
    s.update({"name": "stock_calls_a", "rewards": rewards_, "terminations": terms})
    return s


def stock_calls_b() -> dict:
    s = specs.contacts()
    rewards_ = dict(s["rewards"])
    rewards_.update({
        "air_when_moving": {"fn": air_when_moving, "weight": 1.0, "params": {"time_threshold": 0.5}},
        "contact_mix": {"fn": contact_mix, "weight": 0.1},
        "slide": {"fn": slide, "weight": -0.1, "params": {"factor": 0.5}},
    })
    s.update({"name": "stock_calls_b", "rewards": rewards_,
              "terminations": dict(s["terminations"], hard_hit={"fn": hard_hit})})
    return s
