"""
Workload of lowered user terms that read per-link state (foot positions and velocities): the `contacts` table
(configs/specs.py) plus hand-written legged-locomotion terms of the kind most user code contains.

Rewards
    foot_clearance  squared height error of the four feet weighted by their xy speed (get_links_pos /
                    get_links_vel, norm over [:, :, :2])
    foot_slip       calf speed while the calf is in contact: link.get_vel() times a contact flag from
                    foot_contact_manager.get_contact_forces(link.idx) (a one-element index tensor)
    feet_spacing    xy distance of every foot to the front-left one: broadcasting against pos[:, 0:1, :2], the
                    links given as an integer tensor
    front_foot      the front-left foot's height, clamped, through a link object captured at build time
    swing_peak      class-style: the peak height of each foot's swing, (N, 4) state, rewarded at touchdown
Termination
    feet_below      a foot more than 2.5 below the ground plane (raw link z: the mask stays exact)
Observations
    feet_rel_base   feet relative to the base, (pos - robot.get_pos().unsqueeze(1)).flatten(1), 12 columns
    foot_speed      foot speeds, 4 columns

Lowering everything needs fuse_user_terms, fuse_user_observations and fuse_stateful_terms.  The synthetic engine
carries per-link state only for tables with contact slots, hence the contacts table.  Kept out of specs.ALL /
VARIANTS (which the golden-trace tests walk), like configs/user_terms.py.
"""
from __future__ import annotations

import torch

from genesis_forge_b200.managers.config import MdpFnClass

from . import specs

FEET = ("FL_foot", "FR_foot", "RL_foot", "RR_foot")
LINK_REWARDS = ("foot_clearance", "foot_slip", "feet_spacing", "front_foot", "swing_peak")
CALVES = ("FL_calf", "FR_calf", "RL_calf", "RR_calf")


def _feet(env) -> list[int]:
    return [env.robot.get_link(n).idx_local for n in FEET]


def foot_clearance(env, target=0.08):
    ids = _feet(env)
    pos = env.robot.get_links_pos(links_idx_local=ids)
    speed = env.robot.get_links_vel(links_idx_local=ids)[:, :, :2].norm(dim=-1)
    return ((pos[:, :, 2] - target).square() * speed).sum(dim=1)


def foot_slip(env, threshold=1.0):
    out = None
    for name in CALVES:
        link = env.robot.get_link(name)
        on = env.foot_contact_manager.get_contact_forces(link.idx)[:, 0, :].norm(dim=-1) > threshold
        slip = link.get_vel()[:, :2].norm(dim=1) * on
        out = slip if out is None else out + slip
    return out


def feet_spacing(env, width=0.3):
    ids = torch.tensor(_feet(env), device=env.episode_length.device)
    pos = env.robot.get_links_pos(links_idx_local=ids)[:, :, :2]
    return ((pos - pos[:, 0:1, :]).norm(dim=2)[:, 1:] - width).abs().mean(dim=1)


class front_foot(MdpFnClass):
    def __init__(self, env):
        super().__init__(env)
        self.foot = None

    def build(self):
        self.foot = self.env.robot.get_link("FL_foot")

    def __call__(self, env):
        return self.foot.get_pos()[:, 2].clamp(max=0.3)


class swing_peak(MdpFnClass):
    def __init__(self, env, threshold=1.0):
        super().__init__(env)
        self.feet = [env.robot.get_link(n) for n in FEET]
        self.peak = torch.zeros((env.num_envs, len(FEET)), device=env.episode_length.device)

    def __call__(self, env, threshold=1.0):
        z = env.robot.get_links_pos(links_idx_local=[link.idx_local for link in self.feet])[:, :, 2]
        on = env.foot_contact_manager.contacts[:, :, 2].abs() > threshold
        reward = torch.where(on, self.peak, 0.0).sum(dim=1)
        self.peak = torch.where(on, 0.0, torch.maximum(self.peak, z))
        return reward


def feet_below(env, depth=-2.5):
    return (env.robot.get_links_pos(links_idx_local=_feet(env))[:, :, 2] < depth).any(dim=1)


def feet_rel_base(env):
    return (env.robot.get_links_pos(links_idx_local=_feet(env)) - env.robot.get_pos().unsqueeze(1)).flatten(1)


def foot_speed(env):
    return env.robot.get_links_vel(links_idx_local=range(4, 17, 4)).norm(dim=2)


def override() -> dict:
    """`spec_override` turning the contacts spec into the link-terms workload."""
    s = specs.contacts()
    rewards = dict(s["rewards"])
    rewards.update({
        "foot_clearance": {"fn": foot_clearance, "weight": -0.5, "params": {"target": 0.08}},
        "foot_slip": {"fn": foot_slip, "weight": -0.1},
        "feet_spacing": {"fn": feet_spacing, "weight": -0.2},
        "front_foot": {"fn": front_foot, "weight": 0.05},
        "swing_peak": {"fn": swing_peak, "weight": 0.3},
    })
    terminations = dict(s["terminations"], feet_below={"fn": feet_below})
    policy = dict(s["observations"]["policy"]["terms"])
    policy.update({"feet_rel_base": {"fn": feet_rel_base}, "foot_speed": {"fn": foot_speed}})
    return {"name": "link_terms", "rewards": rewards, "terminations": terminations,
            "observations": {"policy": {"terms": policy}}}


def link_terms() -> dict:
    s = specs.contacts()
    s.update(override())
    return s
