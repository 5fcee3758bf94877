"""
Algorithmic bytes per environment-step, computed from the compiled term table.

Rule (SURVEY.md section 8(d)): every distinct per-env array is counted once when read and once
when written; persistent state counts read + write; parameters and the terrain height field are
O(1) and excluded; sparse reset traffic (command rewrite, 8 B per reset index, the re-observation of
reset envs) amortises to ~0 and is excluded.

`step_bytes(fused)`  -> whole manager step (what BASELINE.md's 710 B for config 2 refers to)
`post_kernel_bytes(fused)` / `action_kernel_bytes(fused)` -> the arrays each kernel itself must
touch (used for the per-kernel roofline in bench.py).  The sum of the two exceeds step_bytes by the
arrays that have to cross the physics substep through HBM (targets, action-rate scratch,
episode_length), which is stated, not hidden.
"""
from __future__ import annotations

from . import _native as nat


def _program_facts(fused):
    P = fused.program.head
    K = nat.K
    D = P.num_dofs
    n_reward = P.n_reward
    cmd_words = sum(P.command[k].n_dims for k in range(P.n_command))
    obs_out = sum(P.obs_group[g].n_cols * P.obs_group[g].history for g in range(P.n_obs_groups))
    obs_hist = sum(P.obs_group[g].n_cols * (P.obs_group[g].history - 1) for g in range(P.n_obs_groups))
    srcs = set()
    noise_words = 0
    for g in range(P.n_obs_groups):
        og = P.obs_group[g]
        for c in range(og.n_cols):
            oc = fused.program.obs_cols[og.col_begin + c]
            srcs.add(oc.src)
            if oc.noise != 0.0 and P.rng_mode == 0:
                noise_words += 1
    ops = {P.reward[r].op for r in range(n_reward) if P.reward[r].weight != 0.0}
    tops = {P.termination[t].op for t in range(P.n_termination)}
    uses = {
        "pos": bool(ops & {K["GFB_R_BASE_HEIGHT"]}) or bool(tops & {K["GFB_T_BASE_HEIGHT_MIN"], K["GFB_T_OUT_OF_BOUNDS"]})
        or fused.entity_manager is not None,
        "vel": bool(ops & {K["GFB_R_LIN_VEL_Z"], K["GFB_R_TRACK_LIN_VEL"]}) or K["GFB_O_LIN_VEL_B"] in srcs,
        "ang": bool(ops & {K["GFB_R_ANG_VEL_XY"], K["GFB_R_TRACK_ANG_VEL"]}) or K["GFB_O_ANG_VEL_B"] in srcs,
        "dof_pos": bool(ops & {K["GFB_R_DOF_SIMILAR"], K["GFB_R_STAND_STILL"]}) or K["GFB_O_DOF_POS"] in srcs,
        "dof_vel": K["GFB_O_DOF_VEL"] in srcs,
        "dof_force": K["GFB_O_DOF_FORCE"] in srcs,
        "targets": K["GFB_O_TARGETS"] in srcs,
        "action_rate": K["GFB_R_ACTION_RATE"] in ops,
    }
    # lowered user-defined terms (expr.py): each distinct array they read counts once, like the stock
    # terms' (contact forces / air time are this kernel's own outputs, actions and commands always counted)
    user = {"vel": "vel", "lin_vel_b": "vel", "ang": "ang", "ang_vel_b": "ang", "pos": "pos",
            "dof_pos": "dof_pos", "dof_vel": "dof_vel", "targets": "targets"}
    for (kind, name), entry in getattr(fused, "user_terms", {}).items():
        if kind == "reward" and fused.reward.cfg[name].weight == 0.0:
            continue
        for key in entry[0].sources():
            if key[0] in user:
                uses[user[key[0]]] = True
    contact_in = contact_out = air = 0
    if P.n_contact > 0:
        C, L = P.n_contact_slots, P.n_links_total
        contact_in = C * (3 + 3 + 1 + 1) + 4 * L  # shared by all contact managers
        for m in range(P.n_contact):
            cm = P.contact[m]
            contact_out += 6 * cm.n_links
            if cm.track_air_time:
                air += 4 * cm.n_links
    feet_slide = sum(
        P.contact[P.reward[r].mgr].n_links * 3 for r in range(n_reward)
        if P.reward[r].op == K["GFB_R_FEET_SLIDE"] and P.reward[r].weight != 0.0
    )
    return dict(D=D, n_reward=n_reward, cmd=cmd_words, obs_out=obs_out, obs_hist=obs_hist, uses=uses,
                contact_in=contact_in, contact_out=contact_out, air=air, noise=noise_words,
                entity=fused.entity_manager is not None, has_max=int(P.base_max_episode_length > 0),
                feet_slide=feet_slide)


def step_bytes(fused) -> int:
    """B_alg of the whole manager step, bytes per env-step."""
    f = _program_facts(fused)
    u, D = f["uses"], f["D"]
    read = 4 + 3 * u["pos"] + 3 * u["vel"] + 3 * u["ang"]           # quat + base vectors
    read += D * (u["dof_pos"] + u["dof_vel"] + u["dof_force"])
    read += 2 * D                                                    # raw actions + previous actions
    read += f["cmd"] + 1 + f["has_max"] + (1 + f["n_reward"] if f["n_reward"] else 0)
    read += f["contact_in"] + f["air"] + f["obs_hist"] + f["noise"] + f["feet_slide"]
    write = 3 * D + f["obs_out"] + 1 + 1                             # targets, actions, last_actions, obs, reward, ep_len
    write += (1 + f["n_reward"]) if f["n_reward"] else 0
    write += 11 * f["entity"] + f["contact_out"] + f["air"]
    return 4 * (read + write) + 2                                    # + two 1-byte masks


def post_kernel_bytes(fused) -> int:
    """Bytes the post-physics kernel itself has to move per env (its own roofline numerator)."""
    f = _program_facts(fused)
    u, D = f["uses"], f["D"]
    read = 4 + 3 * u["pos"] + 3 * u["vel"] + 3 * u["ang"]
    read += D * (u["dof_pos"] + u["dof_vel"] + u["dof_force"] + u["targets"])
    read += f["cmd"] + 1 + f["has_max"] + u["action_rate"] + (1 + f["n_reward"] if f["n_reward"] else 0)
    read += f["contact_in"] + f["air"] + f["obs_hist"] + f["noise"] + f["feet_slide"]
    write = f["obs_out"] + 1 + ((1 + f["n_reward"]) if f["n_reward"] else 0)
    write += 11 * f["entity"] + f["contact_out"] + f["air"]
    return 4 * (read + write) + 2


def action_kernel_bytes(fused) -> int:
    """Bytes the pre-physics kernel moves per env.  env.actions / env.last_actions are a ring
    (gfb_action_step_ring): the copy last_actions <- actions of the reference is a buffer exchange, so
    the kernel writes 2*D words, not the 3*D the whole-step model (`step_bytes`, the reference's
    semantics) counts."""
    D = fused.program.head.num_dofs
    return 4 * (2 * D + 1 + 2 * D + 1 + 1)  # raw, prev, ep_len | actions, targets, ep_len, action_rate
