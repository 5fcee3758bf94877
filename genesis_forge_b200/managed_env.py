"""
ManagedEnvironment: the reference's manager-driven environment
(genesis_forge/managed_env.py:32-398) with its step pipeline executed by the fused CUDA step.

Public surface kept: constructor arguments, `managers` registry and add_manager(), config(),
build() (manager build order terrain, action, contact, termination, reward, command, entity,
observation -- managed_env.py:257-272), step() returning
(obs, rewards, terminated, truncated, extras), reset(env_ids), get_observations(), the
action_space / observation_space properties, and the `extras` keys "episode", "observations",
"terminations", "time_outs".

What differs is who does the work.  The reference's step() walks the managers and issues a few
hundred eager torch ops with 6+ host syncs; here step() is
    gfb_action_step -> control_dofs_position -> scene.step() -> gfb_post_physics -> one report
    read-back -> host reset fan-out for the compacted reset indices -> gfb_observe on those envs.
Ordering facts of the reference that are preserved are listed in DESIGN.md (rewards see the
pre-resample command; timeout sees the incremented episode length; reset envs are observed after
the engine reset but with the pre-reset cached quaternion; ...).
"""
from __future__ import annotations

import os
from typing import Any

import torch

from . import _native as nat
from ._gs import gs
from .expr import is_class_term
from .fused import FusedStep, UnsupportedTermError, UserTermsDemoted, combine_logging, make_obs_dict
from .genesis_env import GenesisEnv
from .managers.base import BaseManager, ManagerType


class ManagedEnvironment(GenesisEnv):
    # The observation tensors returned by step() / get_observations() are the manager's own
    # double-buffered storage: the tensor handed out by step t is rewritten in place by step t+2 (the
    # reference returns a fresh torch.cat every step).  Callers that keep observations across more
    # than one step without copying them (rollout lists of raw references) set this to True -- or
    # GFB_COPY_OBSERVATIONS=1 in the environment -- to get a private copy per step (one extra
    # (N, O*H) device copy).
    copy_observations = os.environ.get("GFB_COPY_OBSERVATIONS", "0") == "1"
    # User-defined reward / termination functions are host callbacks between separate kernel launches
    # (split execution).  With this set to True -- or GFB_FUSE_USER_TERMS=1 in the environment -- build()
    # traces them into a small expression IR (expr.py) and the ones that lower run inside the specialised
    # post-physics kernel next to the stock terms; a table without other host callbacks is then one launch
    # per step again.  Terms the IR does not cover stay callbacks (FusedStep.user_term_refusals says why).
    fuse_user_terms = os.environ.get("GFB_FUSE_USER_TERMS", "0") == "1"
    # The same for user-defined observation functions (independent of fuse_user_terms): with this set to True
    # -- or GFB_FUSE_USER_OBS=1 in the environment -- the ones that lower are evaluated by the specialised
    # kernel instead of the host, and re-observed reset envs by a small kernel of the same library
    # (FusedStep.user_term_refusals[("observation", name)] says why a term stays a host column).
    fuse_user_observations = os.environ.get("GFB_FUSE_USER_OBS", "0") == "1"
    # Class-style (MdpFnClass) user reward / termination / observation terms, which keep per-env state from one
    # step to the next (independent of the two switches above, same preconditions): with this set to True -- or
    # GFB_FUSE_STATEFUL_TERMS=1 in the environment -- the ones that lower are evaluated by the specialised
    # kernel, which updates the instance's state tensors in place (FusedStep.user_term_refusals says why not).
    fuse_stateful_terms = os.environ.get("GFB_FUSE_STATEFUL_TERMS", "0") == "1"

    def __init__(
        self,
        num_envs: int = 1,
        dt: float = 1 / 100,
        max_episode_length_sec: int | None = 10,
        max_episode_random_scaling: float = 0.0,
        extras_logging_key: str = "episode",
    ):
        super().__init__(
            num_envs=num_envs,
            dt=dt,
            max_episode_length_sec=max_episode_length_sec,
            max_episode_random_scaling=max_episode_random_scaling,
            extras_logging_key=extras_logging_key,
        )
        self.managers: dict[str, Any] = {
            "contact": [], "entity": [], "command": [], "terrain": [],
            "action": None, "observation": [], "reward": None, "termination": None,
        }
        self._action_space = None
        self._observation_space = None
        self._reward_buf = torch.zeros((num_envs,), device=gs.device, dtype=gs.tc_float)
        self._terminated_buf = torch.zeros((num_envs,), device=gs.device, dtype=gs.tc_bool)
        self._truncated_buf = torch.zeros((num_envs,), device=gs.device, dtype=gs.tc_bool)
        # terminated | truncated of the last step, written by the post-physics kernel (wrapper glue:
        # RslRlWrapper hands it out as `dones` instead of launching an elementwise OR)
        self.dones = torch.zeros((num_envs,), device=gs.device, dtype=gs.tc_bool)
        self._fused: FusedStep | None = None
        self._tracing: dict | None = None
        self._log_key_cache: dict = {}
        self._reward_log_cache = None

    # -- spaces ---------------------------------------------------------------------------------
    @property
    def action_space(self):
        if self.managers["action"] is not None:
            return self.managers["action"].action_space
        return self._action_space

    @action_space.setter
    def action_space(self, space):
        self._action_space = space

    @property
    def observation_space(self):
        if self.managers["observation"]:
            for obs in self.managers["observation"]:
                if obs.name == "policy":
                    return obs.observation_space
            return self.managers["observation"][0].observation_space
        return self._observation_space

    @observation_space.setter
    def observation_space(self, space):
        self._observation_space = space

    # -- manager registry -----------------------------------------------------------------------
    def add_manager(self, manager_type: ManagerType, manager: BaseManager):
        if manager_type not in self.managers:
            raise ValueError(f"'{manager_type}' is not a valid manager type.")
        slot = self.managers[manager_type]
        if isinstance(slot, list):
            slot.append(manager)
        elif slot is None:
            self.managers[manager_type] = manager
        else:
            raise ValueError(
                f"Manager type '{manager_type}' already has a manager, and an environment cannot have "
                f"multiple {manager_type} managers."
            )

    def config(self):
        """Override and create the managers here."""

    # -- tracing of observation term functions ----------------------------------------------------
    def _trace_width(self, key) -> int:
        if isinstance(key, tuple):
            kind, mgr = key
            if kind == "command":
                return mgr._command.shape[1]
            if kind == "contact_norm":
                return mgr._link_ids.shape[0]
            if kind.startswith("entity_"):  # body-frame vector of a further EntityManager
                return 3
        if key in ("lin_vel_b", "ang_vel_b", "gravity_b", "lin_vel_uncached", "ang_vel_uncached", "gravity_uncached"):
            return 3
        return self.managers["action"].num_actions

    def _trace_or(self, key, compute):
        """Manager getters call this: a tagged placeholder while tracing, the real value otherwise."""
        if self._tracing is None:
            return compute()
        if not isinstance(self._tracing, dict):  # a user term traced into the expression IR (expr.py)
            return self._tracing.source(key, compute)
        if key not in self._tracing:
            self._tracing[key] = torch.empty((0, self._trace_width(key)))
        return self._tracing[key]

    def _trace_term(self, fn, params: dict, what: str):
        """Run an observation term once under tracing and identify which manager value it returns."""
        self._tracing = {}
        # a class-style term keeps state: this call on placeholders must not advance (or break) it -- the
        # reference calls the term once at build, the dry run of ObservationManager.resolve_external
        saved = dict(vars(fn)) if is_class_term(fn) and hasattr(fn, "__dict__") else None
        data = {k: v.clone() for k, v in saved.items() if torch.is_tensor(v)} if saved is not None else {}
        try:
            try:
                result = fn(env=self, **params)
            except Exception as e:
                if saved is None or isinstance(e, UnsupportedTermError):
                    raise
                raise UnsupportedTermError(f"{what}: a class-style term that does not run on placeholders") from e
            for key, sentinel in self._tracing.items():
                if result is sentinel:
                    if isinstance(key, str) and key.endswith("_uncached"):
                        # without an entity_manager the term inverts the CURRENT (post-reset) quaternion
                        # (utils.py:13-55); it runs as a host-evaluated term through the rotation kernel
                        err = UnsupportedTermError(f"{what}: body-frame term without an entity_manager")
                        err.width = 3
                        raise err
                    if isinstance(key, tuple) and key[0].startswith("entity_"):
                        # the kernel holds the pose of the first EntityManager's entity only
                        err = UnsupportedTermError(f"{what}: body-frame term of a further EntityManager")
                        err.width = 3
                        raise err
                    return key, sentinel.shape[1]
        finally:
            self._tracing = None
            if saved is not None:
                vars(fn).clear()
                vars(fn).update(saved)
                for k, t in data.items():
                    saved[k].copy_(t)
        raise UnsupportedTermError(
            f"{what}: the term function does not return a manager value the fused step recognises "
            "(EntityManager.get_*, action manager getters, CommandManager.observation, "
            "mdp.observations.*); user-defined observation terms are not supported yet"
        )

    # -- build ------------------------------------------------------------------------------------
    def build(self):
        super().build()
        try:
            self.scene._env = self
        except Exception:
            pass
        self.config()
        M = self.managers
        for terrain_manager in M["terrain"]:
            terrain_manager.build()
        if M["action"] is not None:
            M["action"].build()
        for contact_manager in M["contact"]:
            contact_manager.build()
        if M["termination"] is not None:
            M["termination"].build()
        if M["reward"] is not None:
            M["reward"].build()
        for command_manager in M["command"]:
            command_manager.build()
        for entity_manager in M["entity"]:
            entity_manager.build()
        for obs in M["observation"]:
            obs.build()
        self._fused = FusedStep(self, dry_run=getattr(self, "_dry_run", False), compile_now=False)
        for obs in M["observation"]:
            obs.resolve_external()  # user-defined terms are evaluated once for their width (may use the library)
        self._fused._compile()
        # EntityManager.build() caches the base pose once (entity_manager.py:157-167)
        if not self._fused.dry_run:
            self._fused.cache_entity()

    # -- multi-GPU ----------------------------------------------------------------------------------
    def shard(self, group=None, global_num_envs: int | None = None, peer: bool | None = None):
        """
        Declare this environment one shard of a job that runs one process per GPU (torch.distributed
        initialised, after build()): logged episode means / termination fractions and the decision
        which keys are published become global over `group` (default: WORLD).  Nothing else is
        exchanged -- envs are independent rows.  See FusedStep.shard for `peer`.
        """
        import torch.distributed as dist

        if self._fused is None:
            raise RuntimeError("build() the environment before sharding it")
        group = group if group is not None else dist.group.WORLD
        if global_num_envs is None:
            global_num_envs = self.num_envs * dist.get_world_size(group)
        self._fused.shard(group, global_num_envs, peer=peer)

    # -- step -------------------------------------------------------------------------------------
    def step(self, actions: torch.Tensor):
        fused = self._fused
        if fused is None:
            raise RuntimeError("build() the environment before stepping it")
        self._begin_step()
        fused.begin_step()
        if self._actions is None:
            self._allocate_action_buffers(actions.shape[1])
            fused.bind_action_buffers()
        self.extras["observations"] = make_obs_dict(gs.device)

        fused.action_step(actions)
        self.scene.step()
        for entity_manager in fused.secondary_entities:  # (the first one's step is the kernel's entity phase)
            entity_manager.step()
        # lowered user terms are checked before the first post-physics launch; if their specialised kernel
        # cannot run, they become host callbacks and the step runs split (FusedStep._demote_user_terms)
        fused.first_launch_of_step = True
        try:
            if fused.split_mode:
                return self._finish_step_split()
            # two-stage report: the rank's own reset count first -- on a sharded env the kernel's last block
            # then still waits for the slowest peer's logging partials, and that wait now overlaps the reset
            # fan-out and the re-observation launch below instead of preceding them
            n_reset = fused.post_physics_local(fused.step_phases)
        except UserTermsDemoted:
            return self._finish_step_split()
        if n_reset > 0:
            reset_idx = fused.reset_idx[:n_reset]
            self._host_reset(reset_idx)
            fused.observe(reset_idx, n_reset)
        report = fused.finish_report()  # status bits, per-term counts (global when sharded)
        fused.finish_logging()  # sharded envs: joins the logging all-reduce issued on a side stream
        self._publish(report, step=True)

        return self._step_outputs()

    def _finish_step_split(self):
        """
        Post-physics part of a step when the configuration contains user-defined (Python) terms or
        user-level command managers.  The kernel phases run as separate launches with the Python
        callbacks in between, in the reference's order (managed_env.py:294-326); which phases share
        a launch is decided once (FusedStep._make_split_plan).  User-level command managers step
        BEFORE the in-library reset, so that their interval test sees the episode lengths the
        reference's does (command_manager.py:152-162 runs ahead of managed_env.py:322-323).
        """
        fused = self._fused
        term = self.managers["termination"]
        report = None
        for callback, phases, reads_report in fused.split_plan:
            if callback == "observe":
                n_reset = report.n_reset
                if n_reset > 0:
                    reset_idx = fused.reset_idx[:n_reset]
                    self._host_reset(reset_idx)
                    for mgr in fused.python_commands:
                        mgr.reset(reset_idx)
                fused.evaluate_external_obs()
            elif callback == "commands":
                for mgr in fused.python_commands:
                    mgr.step()
            elif callback is not None:
                if callback == "reward" and term is not None and term.enabled:
                    self.extras["terminations"] = term._terminated_buf  # user rewards may read them
                    self.extras["time_outs"] = term._truncated_buf
                fused.evaluate_external(callback)
            out = fused.post_physics(phases, read_report=reads_report)
            if reads_report:
                report = out
        fused.finish_logging()
        self._publish(report, step=True)
        return self._step_outputs()

    def _step_outputs(self):
        obs = None
        obs_dict = self.extras["observations"]
        for om in self.managers["observation"]:
            om._current = 1 - om._current
            value = om.get_observations()
            if self.copy_observations:  # see the class attribute
                value = value.clone()
            obs_dict[om.name] = value
            if om.name == "policy":
                obs = value
        term = self.managers["termination"]
        terminated = term._terminated_buf if term is not None else self._terminated_buf
        truncated = term._truncated_buf if term is not None else self._truncated_buf
        rew = self.managers["reward"]
        rewards = rew._reward_buf if rew is not None else self._reward_buf
        return obs, rewards, terminated, truncated, self.extras

    def _publish(self, report, step: bool):
        """Logging entries of `extras` (termination_manager.py:178-189, reward_manager.py:205-216)."""
        fused = self._fused
        logging = self.extras[self.extras_logging_key]
        term, rew = self.managers["termination"], self.managers["reward"]
        status = report.status
        if status:
            action = self.managers["action"]
            quiet = action is not None and action._quiet_action_errors
            if not quiet and status & nat.K["GFB_STATUS_NAN_ACTION"]:
                print("ERROR: NaN actions received!")
            if not quiet and status & nat.K["GFB_STATUS_INF_ACTION"]:
                print("ERROR: Infinite actions received!")
            if status & nat.K["GFB_STATUS_BAD_CONTACT"]:
                print("Warning: Invalid contact forces detected (NaN/inf) and sanitized")
        snapshot = None  # tuple of 0-dim views of this step's logging vector
        n_r = fused.n_reward
        # sharded over ranks: keys are published when ANY rank saw the event (global counts)
        # (single rank / peer-memory exchange: the kernel's report carries the global counts)
        acc = fused.global_acc
        n_t = fused.n_termination
        counts = acc[n_r:n_r + n_t] if acc is not None else report.global_termination_count[:n_t]
        n_reset_logged = acc[-1] if acc is not None else report.global_n_reset
        if step and term is not None and term.enabled:  # (a disabled manager publishes nothing, :159-160)
            self.extras["terminations"] = term._terminated_buf
            self.extras["time_outs"] = term._truncated_buf
            if term.logging_enabled:
                for i, key in self._log_keys(term, fused.termination_terms):
                    if counts[i] > 0:
                        if snapshot is None:
                            snapshot = self._log_snapshot()
                        logging[key] = snapshot[n_r + i]
        if rew is not None and rew.enabled and rew.logging_enabled and n_reset_logged > 0:
            rows, keys, index = self._reward_log_plan(rew, fused)
            if rows:
                if snapshot is None:
                    snapshot = self._log_snapshot()
                for i, key in zip(rows, keys):
                    logging[key] = snapshot[i]
                rew._last_log = (snapshot[0]._base, index)

    def _reward_log_plan(self, rew, fused):
        """(rows, keys, {name: row}) of the reward terms that are logged (weight != 0); rebuilt when a weight changes."""
        weights = [item.weight for _, item, _ in fused.reward_terms]
        cached = self._reward_log_cache
        if cached is None or cached[0] != weights or cached[1] != rew.logging_tag:
            pairs = self._log_keys(rew, fused.reward_terms)
            rows = [i for (i, _), w in zip(pairs, weights) if w != 0]
            keys = [pairs[i][1] for i in rows]
            index = {fused.reward_terms[i][0]: i for i in rows}
            cached = self._reward_log_cache = (weights, rew.logging_tag, rows, keys, index)
        return cached[2], cached[3], cached[4]

    def _log_keys(self, manager, terms) -> list:
        """[(row, "<tag> / <term>")] of one manager's logged entries (built once per logging tag)."""
        cached = self._log_key_cache.get(manager.type)
        if cached is None or cached[0] != manager.logging_tag or len(cached[1]) != len(terms):
            cached = (manager.logging_tag, [(i, f"{manager.logging_tag} / {name}") for i, (name, _, _) in enumerate(terms)])
            self._log_key_cache[manager.type] = cached
        return cached[1]

    def _log_snapshot(self) -> tuple:
        """The kernel's logging vector of this step as 0-dim views."""
        fused = self._fused
        if fused.dist is None or fused.peer_mode:
            return fused.log_views()  # (the next step gets fresh storage, FusedStep.begin_step)
        return fused.global_log_snapshot().unbind(0)

    def _host_reset(self, env_ids: torch.Tensor | None):
        """Engine-side part of reset(): action manager gains / joint positions, entity on_reset items."""
        if self.managers["action"] is not None:
            self.managers["action"].reset(env_ids)
        for entity_manager in self.managers["entity"]:
            entity_manager.reset(env_ids)
        if self._fused.any_controller:
            for mgr in self._fused.commands:
                # command_manager.py:164-170: reset() resamples `_command` even while an external controller
                # supplies `command`; the kernel skips such managers, so it is done here (rare: teleoperation)
                if mgr._external_controller is not None and mgr.enabled and mgr not in self._fused.python_commands:
                    mgr.resample_command(
                        env_ids if env_ids is not None else torch.arange(self.num_envs, device=gs.device))

    # -- reset ------------------------------------------------------------------------------------
    def reset(self, env_ids=None):
        """
        Reset some (or, with None, all) environments.  The in-library part (counters, action
        buffers, episode sums + their logged means, air-time state, command resample) is one launch
        of the post-physics kernel restricted to the reset phase; engine writes follow on the host.
        """
        fused = self._fused
        if fused is None:
            raise RuntimeError("build() the environment before resetting it")
        if self.step_count == 0 and self._actions is None and self.action_space is not None:
            self._allocate_action_buffers(self.action_space.shape[0])
            fused.bind_action_buffers()
        K = nat.K
        fused.begin_step()
        mask = None
        if env_ids is not None:
            env_ids = torch.as_tensor(env_ids, device=gs.device, dtype=torch.int64)
            mask = torch.zeros(self.num_envs, device=gs.device, dtype=torch.bool)
            mask[env_ids] = True
        fused._set(K["GFB_B_FORCE_RESET"], mask)
        self._reset_mask_keep = mask
        if env_ids is None or env_ids.numel() > 0:
            report = fused.post_physics(K["GFB_PHASE_RESET"] | K["GFB_PHASE_FORCED_RESET"])
            fused.finish_logging()
            self._publish(report, step=False)
            self._host_reset(env_ids)
            for mgr in fused.python_commands:
                mgr.reset(env_ids)
        obs = None
        if env_ids is None:
            self.extras.pop("observations", None)
            obs = self.get_observations()
        return obs, self.extras

    # -- observations -------------------------------------------------------------------------------
    def get_observations(self) -> torch.Tensor:
        if not self.managers["observation"]:
            return super().get_observations()
        if "observations" in self.extras and "policy" in self.extras["observations"]:
            return self.extras["observations"]["policy"]
        if "observations" not in self.extras:
            self.extras["observations"] = make_obs_dict(gs.device)
        fused = self._fused
        fused.begin_step()
        # shift history (observation_manager.py:223-226), then frame 0 for every env
        for om in self.managers["observation"]:
            cur, nxt = om._buffers[om._current], om._buffers[1 - om._current]
            single = om.frame_size
            if om._history_len > 1:
                nxt[:, single:] = cur[:, : single * (om._history_len - 1)]
        fused.evaluate_external_obs()
        fused.observe(None, self.num_envs)
        policy = None
        for om in self.managers["observation"]:
            om._current = 1 - om._current
            obs = om.get_observations()
            self.extras["observations"][om.name] = obs
            if om.name == "policy":
                policy = obs
        return policy
