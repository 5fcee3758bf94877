"""
The fused manager step: term compiler + per-step driver on top of libgfb200 (include/gfb200.h).

`FusedStep` is created by ManagedEnvironment.build().  It
  * compiles the manager objects (their live config items) into the packed term table
    (`gfb_program`): one opcode per recognised mdp function, one column descriptor per observation
    column, per-DOF action parameters, command ranges, contact link ids;
  * owns the small auxiliary tensors the kernels need (action-rate scratch, reset index list,
    logging vectors, injected-draw buffers);
  * drives the launches of one environment step:
        gfb_action_step -> engine PD target write -> scene.step() -> gfb_post_physics
        -> gfb_read_report (the single host sync) -> host-side reset fan-out for the compacted
        reset indices -> gfb_observe for those envs.

Random draws made inside the kernels come either from Philox (default) or from dense injected
buffers (`inject()`), which is how the parity harness feeds the reference's own draws through.
"""
from __future__ import annotations

import ctypes as C
import logging
import math
import os

import numpy as np
import torch

from . import _native as nat
from ._gs import gs

try:  # pragma: no cover - depends on the environment
    from tensordict import TensorDict as _TensorDict  # type: ignore

    def make_obs_dict(device):
        return _TensorDict({}, device=device)

except Exception:

    def make_obs_dict(device):
        return {}


_F32 = np.float32
_log = logging.getLogger(__name__)
_TORCH_DTYPE = {"f32": torch.float32, "i32": torch.int32, "bool": torch.bool}  # (expr.F32, I32, BOOL)


def _check_width(prog, name: str, width: int):
    """An observation term's traced columns must be the width its dry run returned."""
    if prog.nodes[prog.out].shape != (width,):
        raise UnsupportedTermError(f"observation '{name}': traced {prog.nodes[prog.out].shape[0]} columns, "
                                   f"the function returned {width}")


def _f32(x) -> float:
    """Python float -> the fp32 value torch uses when a Python scalar meets a float32 tensor."""
    return float(_F32(x))


def asin_tilt_threshold(limit_angle_deg: float) -> float:
    """
    Smallest fp32 tilt t in [0, 0.99] for which the reference's test
        torch.asin(torch.clamp(tilt, max=0.99)) > math.radians(limit_angle)
    (mdp/terminations.py:63-71) is true under THIS host's torch-CPU asin; +inf if none.

    The kernel then evaluates `min(tilt, 0.99) >= threshold`, which is the same predicate without
    depending on device asin bits (asin is monotonic).  Bisection over the fp32 bit patterns.
    """
    limit = math.radians(limit_angle_deg)

    def fires(bits: int) -> bool:
        t = torch.tensor([bits], dtype=torch.int32).view(torch.float32)
        return bool((torch.asin(torch.clamp(t, max=0.99)) > limit).item())

    hi = int(np.array([0.99], dtype=np.float32).view(np.int32)[0])
    if not fires(hi):
        return float("inf")
    if fires(0):
        return 0.0
    lo = 0  # fires(lo) False, fires(hi) True
    while hi - lo > 1:
        mid = (lo + hi) // 2
        if fires(mid):
            hi = mid
        else:
            lo = mid
    return float(np.array([hi], dtype=np.int32).view(np.float32)[0])


from .managers.observation import UnsupportedTermError  # noqa: E402  (one class, importable from here too)


class UserTermsDemoted(Exception):
    """Raised before a step's first post-physics launch when its lowered user terms became host callbacks."""


def combine_logging(acc: torch.Tensor, n_reward: int, n_termination: int, global_num_envs: int) -> torch.Tensor:
    """
    Logging vector from the (all-reduced) accumulator written by the finalize kernel.

    acc = [sum over reset envs of (episode sum / episode seconds) per reward term,
           fire count per termination term, number of reset envs]          (float64)
    ->    [mean per reward term (reward_manager.py:211-216), fired fraction per termination term
           (termination_manager.py:178-182)]                               (float32)
    With envs sharded over ranks the accumulator is summed over ranks first, so the means are the
    same numbers a single process over all envs would log.
    """
    out = torch.empty(n_reward + n_termination, device=acc.device, dtype=torch.float32)
    n_reset = acc[n_reward + n_termination].clamp(min=1.0)
    s = acc[:n_reward].float()  # a sum past the fp32 range is logged as +-Inf, as in tail.cuh (xs_mean)
    out[:n_reward] = torch.where(torch.isfinite(s), (acc[:n_reward] / n_reset).float(), s)
    out[n_reward:] = (acc[n_reward:n_reward + n_termination] / float(global_num_envs)).float()
    return out


class FusedStep:
    def __init__(self, env, dry_run: bool = False, compile_now: bool = True):
        """`dry_run` compiles and packs the term table without a device (host-logic tests only)."""
        self.env = env
        self.device = torch.device(gs.device)
        self.N = env.num_envs
        self.dry_run = dry_run
        if dry_run:
            # host-only handle: packs the term table and describes specialisations, cannot launch
            self.lib = nat.lib()
            self.handle = nat.Handle(self.N, -1)
            self.index = -1  # Tensor.get_device() of host tensors
        else:
            if self.device.type != "cuda":
                raise nat.NativeLibraryError(
                    f"the fused manager step runs on a CUDA device (gs.device is {self.device}); "
                    "there is no CPU implementation in this package"
                )
            self.index = self.device.index if self.device.index is not None else torch.cuda.current_device()
            self.lib = nat.lib()
            self.handle = nat.Handle(self.N, self.index)
        self.program = nat.Program()
        self.buffers = nat.Buffers()
        self.report = nat.Report()
        self._fingerprint = None
        self._threshold_cache: dict[float, float] = {}
        self._keepalive: list = []
        self.injected: dict[str, torch.Tensor] | None = None
        self.rng_seed = 0x5EED
        self.dist = None  # (process group) when envs are sharded over ranks
        self.peer_mode = False  # True: the logging exchange runs inside the finalize kernel (peer memory)
        self._contact_dims = None
        self._feet_slide_manager = None
        self._dof_force_used = None
        self.global_acc = None
        self._acc_host = None
        self._log_stream = None
        self._log_event = None
        self._log_out_host = None
        self._log_pending = False
        self._stream_ptr = None
        self._program_pushed = False
        self._program_ever_pushed = False
        self._injected_bound = object()
        self._spec_tried: set = set()
        self._spec_ok: dict = {}  # _spec_tag -> a specialised library was attached for it
        self.first_launch_of_step = False  # set by ManagedEnvironment.step: check lowered user terms first
        self._spec_checked: set = set()  # phase sets looked at since the last re-pack
        self._eval_handle = None  # second library handle for directly called mdp terms
        self._obs_ptrs = None
        self._log_views = None
        self._log_spare = None
        self._fp_items = None
        self._log_out_handed_out = False
        K = nat.K
        self._spec_phases = {K["GFB_PHASE_ALL"], K["GFB_PHASE_OBSERVE"]}
        self.step_phases = K["GFB_PHASE_ALL"]  # minus the phases of disabled managers (pack)
        self._buffers_ref = C.byref(self.buffers)
        self._report_ref = C.byref(self.report)
        self._local_n = C.c_int32(0)
        self._local_n_ref = C.byref(self._local_n)
        self._h = self.handle.ptr
        self._engine_cache: dict = {}  # buffer id -> (tensor, data_ptr) of the last bound engine tensor
        self._action_enabled_packed = True
        self._PHASE_REWARD = K["GFB_PHASE_REWARD"]
        self._B = {name: value for name, value in K.items() if name.startswith("GFB_B_")}
        self._phase_mask = 0xFFFFFFFF  # phases of disabled managers are dropped from every launch (pack)
        self.spec_paths: list = []
        self._body_acc_prev = None
        self._body_acc_started: dict[str, bool] = {}
        self._after_launch_started: list = []
        self._body_acc_terms: set = set()
        self._lazy_started: dict = {}  # (kind, name) -> the lazily initialised state of a lowered class term exists
        self._after_launch_lazy: set = set()
        self.entities = list(env.managers["entity"])
        self.entity_manager = self.entities[0] if self.entities else None
        self.secondary_entities = self.entities[1:]
        if self.entity_manager is None:
            self._inv_base_quat = torch.zeros((self.N, 4), device=self.device)
        self.global_num_envs = self.N
        # set by ObservationManager.resolve_external around a dry run's evaluation of a user observation term for
        # its width: body-frame rotations return zeros of the right shape (a dry run has no device)
        self.width_probe = False
        if compile_now:
            self._compile()

    # ------------------------------------------------------------------------------------------
    # compile: static structure
    # ------------------------------------------------------------------------------------------
    def _compile(self):
        env, M = self.env, self.env.managers
        self.action = M["action"]
        self.commands = list(M["command"])
        self.contacts = list(M["contact"])
        self.entities = list(M["entity"])
        self.reward = M["reward"]
        self.termination = M["termination"]
        self.observations = list(M["observation"])
        self.terrains = list(M["terrain"])
        if len(self.commands) > nat.MAX_COMMANDS:
            raise UnsupportedTermError(f"at most {nat.MAX_COMMANDS} command managers are supported")
        if len(self.contacts) > nat.MAX_CONTACT:
            raise UnsupportedTermError(f"at most {nat.MAX_CONTACT} contact managers are supported")
        if len(self.observations) > nat.MAX_OBS_GROUPS:
            raise UnsupportedTermError(f"at most {nat.MAX_OBS_GROUPS} observation managers are supported")
        self.primary_entity = self.entities[0].entity if self.entities else getattr(env, "robot", None)
        self._dof_entity = self.primary_entity
        self.entity_manager = self.entities[0] if self.entities else None
        # Further EntityManagers (the registry is a list, managed_env.py:200-220): a prop, a second robot.
        # The kernel caches the pose of the FIRST manager's entity and lowers the mdp terms of that
        # entity; the others keep their cache on the host side of the step (EntityManager._cached_calcs,
        # device copies) and their body-frame getters go through the rotation entry point, so terms
        # reading them run as host-evaluated columns / rows (split execution, `_other_entity`).
        self.secondary_entities = self.entities[1:]
        self.D = self.action.num_actions if self.action is not None else 0
        if self.D > nat.MAX_DOFS:
            raise UnsupportedTermError(f"at most {nat.MAX_DOFS} controlled DOFs are supported")

        dev = self.device
        N = self.N
        self.action_rate = torch.zeros(N, device=dev)
        self.reset_idx = torch.zeros(N, device=dev, dtype=torch.int64)
        n_r = len(self.reward.cfg) if self.reward is not None else 0
        n_t = len(self.termination.term_cfg) if self.termination is not None else 0
        self.n_reward, self.n_termination = n_r, n_t
        self.log_out = torch.zeros(max(n_r + n_t, 1), device=dev)
        self.log_acc = torch.zeros(n_r + n_t + 1, device=dev, dtype=torch.float64)
        self._fixed_command = None
        self._fixed_command_parts = None
        # command managers with overridden behaviour are stepped / reset in Python
        from .managers.command import CommandManager, VelocityCommandManager

        def stock(mgr) -> bool:
            cls = type(mgr)
            for attr in ("step", "reset", "resample_command"):
                if getattr(cls, attr) is not getattr(CommandManager, attr) and getattr(cls, attr) is not getattr(VelocityCommandManager, attr):
                    return False
            return True

        self.python_commands = [m for m in self.commands if not stock(m)]
        # terms.  Functions that are not mdp descriptors are user-defined: they stay Python callbacks
        # whose (N,) result is handed to the kernel as a row of the external-values buffer, and the step
        # runs in split mode (see ManagedEnvironment._step_split).
        # With ManagedEnvironment.fuse_user_terms they are first traced into the expression IR (expr.py) and,
        # where that succeeds, evaluated inside the kernel (GFB_R_USER / GFB_T_USER).
        self.reward_terms = []
        self.external_rows: list[tuple[str, str, object]] = []  # (kind, name, config item)
        self.user_terms: dict = {}  # (kind, name) -> [Program, params live, params traced as constants]
        self.user_term_refusals: dict = {}  # (kind, name) -> why the term stays a host callback
        self._user_code = None
        self._lower_user = bool(getattr(env, "fuse_user_terms", False)) and self._can_specialise_user_terms()
        # class-style terms (ManagedEnvironment.fuse_stateful_terms): their per-env tensors are bound to the
        # GFB_B_USER_STATE slots and updated in place by the kernel
        self._lower_stateful = bool(getattr(env, "fuse_stateful_terms", False)) and self._can_specialise_user_terms()
        # (kind, name), for an observation term ("observation", name, group) -> {"inst", "attrs": {attr: (slot,
        # shape, dtype, lazy)}, "tensors", "constants"}
        self.stateful: dict = {}
        self._state_refusal = None  # why a class-style observation term could not be traced again (demotes)
        if self.reward is not None:
            for name, item in self.reward.cfg.items():
                opcode = self._opcode_of(item.fn, "reward")
                if opcode is None and self._lower_user_term("reward", name, item):
                    opcode = nat.K["GFB_R_USER"]
                if opcode is None or self._other_entity(item, f"reward '{name}'") is not None:
                    opcode = nat.K["GFB_R_EXTERNAL"]
                    self.external_rows.append(("reward", name, item))
                self.reward_terms.append((name, item, opcode))
        self.termination_terms = []
        if self.termination is not None:
            for name, item in self.termination.term_cfg.items():
                opcode = self._opcode_of(item.fn, "termination")
                if opcode is None and self._lower_user_term("termination", name, item):
                    opcode = nat.K["GFB_T_USER"]
                if opcode is None or self._other_entity(item, f"termination '{name}'") is not None:
                    opcode = nat.K["GFB_T_EXTERNAL"]
                    self.external_rows.append(("termination", name, item))
                self.termination_terms.append((name, item, opcode))
        self._external_values()
        self._has_command_override = any(m._external_controller is not None for m in self.commands)
        self._controller_bound = [False] * len(self.commands)  # GFB_B_COMMAND0+k points at a controller's tensor
        self.any_controller = False
        self._has_command_override = False  # set by CommandManager.use_external_controller / use_gamepad
        # user-defined observation terms: one (N, W) array filled on the host; with
        # ManagedEnvironment.fuse_user_observations the ones that lower are evaluated in the kernel instead
        self.user_obs: dict = {}  # (group, name) -> [Program, params it was traced with, first word, width]
        self._lower_obs = bool(getattr(env, "fuse_user_observations", False)) and self._can_specialise_user_terms()
        self._observation_columns()
        self._plan_launches()
        self._static_buffers()

    def _observation_columns(self):
        """
        Columns of the user-defined observation terms: lowered ones are words of the (N, user_obs_width)
        user-observation row (GFB_O_USER: the kernel's stash, GFB_B_OBS_EXT1 on the reset path), the rest
        columns of the host-filled (N, ext_obs_width) array (GFB_O_EXTERNAL).
        """
        self.external_obs: list[tuple[object, str, object, int, int]] = []  # (manager, name, item, col0, width)
        width = words = 0
        for g, om in enumerate(self.observations):
            for name, key, w in om._sources:
                if not (isinstance(key, tuple) and key[0] == "external"):
                    continue
                item = om.cfg[name]
                if name not in om._host_columns and self._lower_user_obs(g, name, item, w):
                    self.user_obs[(g, name)][2] = words
                    words += w
                    continue
                self.external_obs.append((om, name, item, width, w))
                om._external_col0[name] = width
                width += w
        self.ext_obs_width = width
        self.ext_obs = torch.zeros((self.N, width), device=self.device) if width else None
        self.user_obs_width = words
        self.user_obs_values = torch.zeros((self.N, words), device=self.device) if words else None
        self._obs_user_id = 0
        self._obs_reads_pose = any(n.op == "src" and n.attr[0] in ("pos", "quat")
                                   for prog, *_ in self.user_obs.values() for n in prog.nodes)

    def _lower_user_obs(self, g: int, name: str, item, width: int) -> bool:
        """Trace a user-defined observation term into the expression IR; False (reason kept) when it stays a host column."""
        from . import expr

        stateful = self._lower_stateful and expr.is_class_term(item.fn)
        if not (self._lower_obs or stateful):
            return False
        try:
            if stateful:
                prog = self._trace_stateful("observation", name, item, (g, width))
            else:
                prog, _ = expr.lower_term(self, "observation", name, item)
                _check_width(prog, name, width)
        except Exception as e:  # noqa: BLE001 - whatever the function does on symbolic inputs, it stays a host column
            why = str(e) if isinstance(e, UnsupportedTermError) else f"{type(e).__name__} while tracing: {e}"
            self.user_term_refusals[("observation", name)] = why
            _log.debug("observation '%s' stays a host column: %s", name, why)
            return False
        self.user_obs[(g, name)] = [prog, dict(item.params or {}), 0, width]
        return True

    def _user_obs_program(self, g: int, name: str, item):
        """The term's Program for its current params (folded as constants: traced again when they change)."""
        from . import expr

        entry = self.user_obs[(g, name)]
        bound = self.stateful.get(("observation", name, g))
        if bound is not None:
            # a new instance (params edited) or an edited scalar attribute: traced again.  If that fails, the
            # table keeps the old program until _check_state demotes the lowered terms (before any launch that
            # evaluates this one)
            if self._state_refusal is None and (item.fn is not bound["inst"] or dict(item.params or {}) != entry[1]
                                                or expr.instance_constants(item.fn) != bound["constants"]):
                try:
                    entry[0] = self._trace_stateful("observation", name, item, (g, entry[3]))
                except Exception as e:  # noqa: BLE001 - as at build: the term becomes a host column
                    self._state_refusal = str(e) if isinstance(e, UnsupportedTermError) else \
                        f"{type(e).__name__} while tracing: {e}"
                    return entry[0]
                entry[1] = dict(item.params or {})
                self._user_code = None
            return entry[0]
        if dict(item.params or {}) != entry[1]:
            prog, _ = expr.lower_term(self, "observation", name, item)
            if prog.nodes[prog.out].shape != (entry[3],):
                raise UnsupportedTermError(f"observation '{name}': its width changed with its params")
            entry[0], entry[1] = prog, dict(item.params or {})
            self._user_code = None
        return entry[0]

    @property
    def lowered_user_terms(self) -> bool:
        return bool(self.user_terms or self.user_obs)

    def _external_values(self):
        """The (J, N) buffer of host-evaluated term values, one row per external reward / termination."""
        self.ext_values = None
        if self.external_rows:
            self.ext_values = torch.zeros((len(self.external_rows), self.N), device=self.device)
        self.ext_row = {(kind, name): j for j, (kind, name, _) in enumerate(self.external_rows)}

    def _plan_launches(self):
        self.split_mode = bool(self.external_rows or self.python_commands or self.external_obs)
        self.split_plan = self._make_split_plan() if self.split_mode else []
        for _, phases, _ in self.split_plan:
            self._spec_phases.add(phases)

    def _can_specialise_user_terms(self) -> bool:
        """
        Lowered user terms run in the specialised kernel only, and the library selects a specialisation only
        for launches that can use TMA: it must exist or be compilable, and the batch must be TMA-eligible.
        """
        from . import spec

        return (not spec.disabled() and spec.jit_allowed() and self.N % 4 == 0
                and os.environ.get("GFB_DISABLE_TMA", "0") != "1")

    # buffers the slab plan may stage or store with TMA (gfb200.cu tma_eligible): 16-byte aligned
    _TMA_BUFFERS = ("GFB_B_POS", "GFB_B_QUAT", "GFB_B_VEL", "GFB_B_ANG", "GFB_B_DOF_POS", "GFB_B_DOF_VEL",
                    "GFB_B_DOF_FORCE", "GFB_B_TARGETS", "GFB_B_ENV_ACTIONS", "GFB_B_C_FORCE", "GFB_B_C_POS",
                    "GFB_B_C_LINK_A", "GFB_B_C_LINK_B", "GFB_B_OBS_EXT0", "GFB_B_EP_SUMS", "GFB_B_BASE_POS",
                    "GFB_B_BASE_QUAT") + tuple(f"GFB_B_{a}{k}" for a in ("COMMAND", "CONTACTS", "CONTACT_POS")
                                               for k in range(4))

    def _user_terms_blocked(self) -> str | None:
        """
        Why a launch of this split step that evaluates lowered user terms could not run their specialised
        kernel (None: every one can) -- the library's own conditions (gfb200.cu), checked before the step's
        first post-physics launch with the step's buffers bound: no specialisation attached for a phase set
        (compile failure, no JIT), or a buffer the slab plan transfers with TMA that is not 16-byte aligned.
        (The one launch of a fused step needs no such check: the library refuses it before anything runs.)
        """
        if self.dry_run:
            return None
        if not self._can_specialise_user_terms():
            return "the specialised kernel cannot be used (GFB_NO_SPEC, no nvcc, GFB_DISABLE_TMA or num_envs % 4)"
        K = nat.K
        if self.user_obs and not self.buffers.buf[K["GFB_B_OBS_EXT1"]]:
            return "GFB_B_OBS_EXT1 (the user-observation rows of the reset path) is not bound"
        buf = self.buffers.buf
        for name in self._TMA_BUFFERS:
            ptr = buf[K[name]]
            if ptr and ptr % 16:
                return f"{name} is not 16-byte aligned (the specialised kernel's TMA transfers need it)"
        sets = [p for _, p, _ in self.split_plan] if self.split_mode else [self.step_phases]
        lowered = K["GFB_PHASE_REWARD"] | K["GFB_PHASE_TERMINATION"] | (K["GFB_PHASE_OBSERVE"] if self.user_obs else 0)
        for phases in sets:
            phases &= self._phase_mask
            if not phases & lowered:
                continue
            self._maybe_specialise(phases)
            if not self._spec_ok.get(self._spec_tag(phases)):
                return f"no specialised kernel could be attached for phases {phases:#x}"
        return None

    def _demote_user_terms(self, why: str):
        """Every lowered user term becomes a host callback again (split execution), for the rest of the run."""
        K = nat.K
        _log.warning("lowered user terms run as host callbacks from now on: %s", why)
        for key in self.user_terms:
            self.user_term_refusals[key] = why
        for _, name in self.user_obs:
            self.user_term_refusals[("observation", name)] = why
        self.user_terms = {}
        self.user_obs = {}
        self._user_code = None
        self._lower_user = False
        self._lower_obs = False
        self._lower_stateful = False
        # the instances already hold their state (updated in place; a lazily initialised attribute is None until
        # the kernel's first evaluation has filled it): the Python __call__ continues from there
        for slot in range(K["GFB_B_COUNT"] - K["GFB_B_USER_STATE0"]):
            self._set(K["GFB_B_USER_STATE0"] + slot, None)
        self.stateful = {}
        self._state_refusal = None
        self._lazy_started = {}
        self._after_launch_lazy = set()
        self._observation_columns()
        self._set(K["GFB_B_OBS_EXT0"], self.ext_obs)
        self._set(K["GFB_B_OBS_EXT1"], None)
        self.reward_terms = [(n, i, K["GFB_R_EXTERNAL"] if op == K["GFB_R_USER"] else op) for n, i, op in self.reward_terms]
        self.termination_terms = [(n, i, K["GFB_T_EXTERNAL"] if op == K["GFB_T_USER"] else op)
                                  for n, i, op in self.termination_terms]
        self.external_rows = (
            [("reward", n, i) for n, i, op in self.reward_terms if op == K["GFB_R_EXTERNAL"]]
            + [("termination", n, i) for n, i, op in self.termination_terms if op == K["GFB_T_EXTERNAL"]])
        self._external_values()
        self._set(K["GFB_B_EXT_VALUES"], self.ext_values)
        self._plan_launches()
        self._fingerprint = None
        self._fp_items = None
        self._program_pushed = False
        self._spec_checked = set()

    def _lower_user_term(self, kind: str, name: str, item) -> bool:
        """Trace a user-defined term into the expression IR; False (and the reason kept) when it stays a callback."""
        from . import expr

        stateful = self._lower_stateful and expr.is_class_term(item.fn)
        if not (self._lower_user or stateful):
            return False
        try:
            if stateful:
                prog, live = self._trace_stateful(kind, name, item), False
            else:
                prog, live = expr.lower_term(self, kind, name, item)
        except Exception as e:  # noqa: BLE001 - whatever the function does on symbolic inputs, it stays a callback
            why = str(e) if isinstance(e, UnsupportedTermError) else f"{type(e).__name__} while tracing: {e}"
            self.user_term_refusals[(kind, name)] = why
            _log.debug("%s '%s' stays a host callback: %s", kind, name, why)
            return False
        self.user_terms[(kind, name)] = [prog, live, None if live else dict(item.params or {}),
                                         expr.param_kinds(item.params)]
        return True

    def _trace_stateful(self, kind: str, name: str, item, obs: tuple | None = None):
        """
        Trace a class-style term and bind its state: the instance's own per-env tensors, and for a lazily
        initialised attribute a zeroed tensor that the instance gets once the kernel has evaluated the term
        (`_after_report`).  The kernel updates them in place -- the one difference from the host path, where the
        term rebinds its attributes: a reference kept to a state tensor sees the new values.  `obs`: (group,
        width) of an observation term (keyed by group too: the same class in two groups is two instances).
        """
        from . import expr

        key = (kind, name) if obs is None else (kind, name, obs[0])
        old = self.stateful.get(key)
        own = {a: b[0] for a, b in old["attrs"].items()} if old else {}
        taken = {slot for k, b in self.stateful.items() if k != key for slot in b["tensors"]}
        prog = expr.trace_stateful(self, kind, name, item,
                                   expr.StateSlots(own, [s for s in range(expr.MAX_STATE_SLOTS)
                                                         if s not in taken and s not in own.values()]))
        if obs is not None:
            _check_width(prog, name, obs[1])
        inst, tensors = item.fn, {}
        for attr, (slot, shape, dtype, lazy) in prog.bindings.items():
            tensors[slot] = (torch.zeros((self.N,) + tuple(shape), device=self.device, dtype=_TORCH_DTYPE[dtype])
                             if lazy else vars(inst)[attr])
        others = {t.untyped_storage().data_ptr(): k for k, b in self.stateful.items() if k != key
                  for t in b["tensors"].values()}
        for t in tensors.values():
            if t.untyped_storage().data_ptr() in others:
                raise UnsupportedTermError(f"{kind} '{name}': a state tensor shares storage with the state of "
                                           f"{others[t.untyped_storage().data_ptr()][0]} "
                                           f"'{others[t.untyped_storage().data_ptr()][1]}'")
        K = nat.K
        for slot in (old["tensors"] if old else {}):
            self._set(K["GFB_B_USER_STATE0"] + slot, None)
        for slot, t in tensors.items():
            self._set(K["GFB_B_USER_STATE0"] + slot, t)
        self.stateful[key] = {"inst": inst, "attrs": prog.bindings, "tensors": tensors,
                              "constants": expr.instance_constants(inst)}
        if prog.first is not None:
            self._lazy_started[key] = False
        else:
            self._lazy_started.pop(key, None)
        return prog

    def _check_state(self) -> str | None:
        """
        Before a step's first post-physics launch and before the host columns of an observation are evaluated
        (evaluate_external_obs, which precedes every other launch that evaluates a lowered class-style
        observation term): every state attribute of a lowered class-style term must still be the tensor bound to
        its slot.  A compatible tensor the user assigned (a manual reset, a direct call of the term) is bound
        instead; anything else -- another shape, dtype or device, a non-contiguous tensor, None -- is returned
        as the reason to demote the lowered terms to callbacks, as is a class-style observation term that
        could not be traced again after an edit.
        """
        for key in [k for k in self.stateful if len(k) == 3]:  # (a new instance or constants: traced again)
            self._user_obs_program(key[2], key[1], self.observations[key[2]].cfg[key[1]])
        if self._state_refusal is not None:
            return self._state_refusal
        K = nat.K
        for key, b in self.stateful.items():
            d = vars(b["inst"])
            started = self._lazy_started.get(key, True)
            for attr, (slot, shape, dtype, lazy) in b["attrs"].items():
                cur, want = d.get(attr), b["tensors"][slot]
                if cur is (want if started or not lazy else None):
                    continue
                if not (torch.is_tensor(cur) and tuple(cur.shape) == (self.N,) + tuple(shape)
                        and cur.dtype == _TORCH_DTYPE[dtype] and cur.device == self.device and cur.is_contiguous()):
                    return (f"{key[0]} '{key[1]}': self.{attr} is no longer a contiguous "
                            f"{_TORCH_DTYPE[dtype]} tensor of shape {(self.N,) + tuple(shape)} on {self.device}")
                b["tensors"][slot] = cur
                self._set(K["GFB_B_USER_STATE0"] + slot, cur)
                if lazy and not started:  # assigned by the user before the first evaluation: it is the state now
                    self._lazy_started[key] = started = True
                    for a, (s2, _, _, lz) in b["attrs"].items():
                        if lz and a != attr and d.get(a) is None:
                            d[a] = b["tensors"][s2]
        return None

    @property
    def user_code(self) -> str:
        """Device functions of the lowered user terms for the specialised kernel's header ('' if none)."""
        if self._user_code is None:
            from . import expr

            rows = {"reward": {}, "termination": {}}
            for kind, terms in (("reward", self.reward_terms), ("termination", self.termination_terms)):
                for row, (name, _, _) in enumerate(terms):
                    if (kind, name) in self.user_terms:
                        rows[kind][row] = self.user_terms[(kind, name)][0]
            obs = sorted((entry[2], entry[0]) for entry in self.user_obs.values())
            self._user_code = (expr.device_code(rows["reward"], rows["termination"], obs, self.user_obs_width)
                               if self.lowered_user_terms else "")
        return self._user_code

    def _user_program(self, kind: str, name: str, item):
        """The term's Program for its current params (a term traced with constant params is traced again
        when they change: its expression, and with it the specialised kernel, changes)."""
        from . import expr

        entry = self.user_terms[(kind, name)]
        bound = self.stateful.get((kind, name))
        if bound is not None:
            # a new instance (params edited: ConfigItem._rebuild) or an edited scalar attribute: traced again,
            # with the new instance's tensors bound
            if (item.fn is not bound["inst"] or dict(item.params or {}) != entry[2]
                    or expr.instance_constants(item.fn) != bound["constants"]):
                entry[0], entry[2] = self._trace_stateful(kind, name, item), dict(item.params or {})
                self._user_code = None
            return entry[0]
        # traced with constant params and they changed, or a live param changed between int and float (its
        # kernel type, int32 or fp32, was fixed by the trace)
        changed = entry[2] is not None and dict(item.params or {}) != entry[2]
        if changed or expr.param_kinds(item.params) != entry[3]:
            entry[0], live = expr.lower_term(self, kind, name, item)
            entry[2] = None if live else dict(item.params or {})
            entry[3] = expr.param_kinds(item.params)
            self._user_code = None
        return entry[0]

    def _make_split_plan(self) -> list:
        """
        Split execution: the kernel phases as separate launches with the host callbacks of the
        configuration in between, in the reference's order (managed_env.py:294-326):
            entity, contacts | user terminations | terminations | user rewards | rewards, stock command
            resample | user-level command managers' step() | in-library reset (+ report) |
            engine reset, user-level command managers' reset(idx) | user observation terms | observations
        Neighbouring phases with no callback between them share a launch.  Returns
        [(callback name or None, phases, reads_report)].
        """
        K = nat.K
        ext_term = any(kind == "termination" for kind, _, _ in self.external_rows)
        ext_rew = any(kind == "reward" for kind, _, _ in self.external_rows)
        stages = [
            (None, K["GFB_PHASE_ENTITY"] | K["GFB_PHASE_CONTACT"]),
            ("termination" if ext_term else None, K["GFB_PHASE_TERMINATION"]),
            ("reward" if ext_rew else None, K["GFB_PHASE_REWARD"] | K["GFB_PHASE_COMMAND"]),
            ("commands" if self.python_commands else None, K["GFB_PHASE_RESET"]),
        ]
        plan: list = []
        for callback, phases in stages:
            if callback is None and plan:
                plan[-1][1] |= phases
            else:
                plan.append([callback, phases, False])
        plan[-1][2] = True  # the launch with the reset phase delivers the report
        plan.append(["observe", K["GFB_PHASE_OBSERVE"], False])
        return [tuple(p) for p in plan]

    def split_phase_sets(self) -> list[int]:
        return [phases for _, phases, _ in self.split_plan]

    @staticmethod
    def _opcode_of(fn, kind: str) -> int | None:
        """Kernel opcode of an mdp descriptor, None for a user-defined function."""
        target = getattr(fn, "__func__", fn)
        if not hasattr(target, "gfb_opcode") and hasattr(type(target), "gfb_opcode"):
            target = type(target)  # instance of a class-style term (MdpFnClass)
        opcode = getattr(target, "gfb_opcode", None)
        if opcode is None or getattr(target, "gfb_kind", None) != kind:
            return None
        return nat.K[opcode]

    def _set(self, buf_id: int, tensor: torch.Tensor | None, dtype=None, keep: bool = False):
        if tensor is None:
            self.buffers.buf[buf_id] = None
            return
        if tensor.device != self.device:
            raise ValueError(f"buffer {buf_id}: tensor on {tensor.device}, expected {self.device}")
        if dtype is not None and tensor.dtype != dtype:
            tensor = tensor.to(dtype)
            keep = True
        if not tensor.is_contiguous():
            tensor = tensor.contiguous()
            keep = True
        if keep:
            self._keepalive.append(tensor)
        self.buffers.buf[buf_id] = tensor.data_ptr()

    def _set_engine(self, buf_id: int, tensor: torch.Tensor, dtype):
        """Pointer of an engine getter's tensor (kept alive until the next launch group)."""
        seen = self._engine_cache.get(buf_id)
        if seen is None:
            seen = self._engine_cache[buf_id] = {}
        hit = seen.get(id(tensor))
        if hit is not None:  # a tensor object validated before (engines that hand out views of solver state)
            self.buffers.buf[buf_id] = hit[1]
            return
        given = tensor
        if tensor.dtype is not dtype or not tensor.is_contiguous() or tensor.get_device() != self.index:
            tensor = tensor.to(self.device, dtype).contiguous()
        ptr = tensor.data_ptr()
        if tensor is given:
            if len(seen) >= 8:  # engines that return fresh tensors every call: nothing to remember
                seen.clear()
            seen[id(tensor)] = (tensor, ptr)  # (the reference held here keeps the id unique)
        else:
            self._keepalive.append(tensor)
        self.buffers.buf[buf_id] = ptr

    def _static_buffers(self):
        """Pointers that never change: tensors owned by the env / managers / this object."""
        env, K = self.env, nat.K
        s = self._set
        s(K["GFB_B_EPISODE_LENGTH"], env.episode_length)
        s(K["GFB_B_MAX_EPISODE_LENGTH"], env.max_episode_length)
        s(K["GFB_B_ACTION_RATE"], self.action_rate)
        s(K["GFB_B_RESET_IDX"], self.reset_idx)
        s(K["GFB_B_LOG_OUT"], self.log_out)
        self._log_out_id = K["GFB_B_LOG_OUT"]
        s(K["GFB_B_LOG_ACC"], self.log_acc)
        for k, mgr in enumerate(self.commands):
            s(K["GFB_B_COMMAND0"] + k, mgr._command)
        if self.entity_manager is not None:
            s(K["GFB_B_BASE_POS"], self.entity_manager._base_pos)
            s(K["GFB_B_BASE_QUAT"], self.entity_manager._base_quat)
            s(K["GFB_B_INV_BASE_QUAT"], self.entity_manager._inv_base_quat)
        else:
            s(K["GFB_B_INV_BASE_QUAT"], self._inv_base_quat)
        for m, mgr in enumerate(self.contacts):
            s(K["GFB_B_CONTACTS0"] + m, mgr.contacts)
            s(K["GFB_B_CONTACT_POS0"] + m, mgr.contact_positions)
            s(K["GFB_B_AIR0"] + m, mgr._air)
        if self.termination is not None:
            # torch.bool is one byte per element, 0/1
            s(K["GFB_B_TERMINATED"], self.termination._terminated_buf)
            s(K["GFB_B_TRUNCATED"], self.termination._truncated_buf)
        else:
            s(K["GFB_B_TERMINATED"], env._terminated_buf)
            s(K["GFB_B_TRUNCATED"], env._truncated_buf)
        if self.reward is not None:
            s(K["GFB_B_REWARD"], self.reward._reward_buf)
            s(K["GFB_B_EP_SECONDS"], self.reward._episode_seconds)
            s(K["GFB_B_EP_SUMS"], self.reward._episode_sums)
        else:
            s(K["GFB_B_REWARD"], env._reward_buf)
        for t in self.terrains:
            if t.height_field is not None:
                s(K["GFB_B_HEIGHT_FIELD"], t.height_field)
        s(K["GFB_B_DONES"], getattr(env, "dones", None))
        s(K["GFB_B_EXT_VALUES"], self.ext_values)
        s(K["GFB_B_OBS_EXT0"], self.ext_obs)
        s(K["GFB_B_OBS_EXT1"], self.user_obs_values)

    def bind_action_buffers(self):
        K = nat.K
        self._set(K["GFB_B_ENV_ACTIONS"], self.env._actions)
        self._set(K["GFB_B_ENV_LAST_ACTIONS"], self.env._last_actions)
        if self.action is not None:
            self._set(K["GFB_B_TARGETS"], self.action._actions)

    # ------------------------------------------------------------------------------------------
    # pack: live config -> gfb_program
    # ------------------------------------------------------------------------------------------
    def _live_fingerprint(self):
        """Every live value the packed table depends on (one tuple compare per step decides on a re-pack)."""
        env = self.env
        items = self._fp_items
        if items is None:  # the item lists are fixed after _compile()
            items = self._fp_items = (
                [item for _, item, _ in self.reward_terms],
                [item for _, item, _ in self.termination_terms],
                [item for om in self.observations for item in om.cfg.values()],
            )
        rewards, terminations, obs_items = items
        return (
            env.dt, env._base_max_episode_length, env._max_episode_random_scaling, self.injected is not None,
            self.rng_seed, tuple(sorted(self._body_acc_started.items())) if self._body_acc_started else (),
            [(i.weight, i.version) for i in rewards],
            [(i.time_out, i.version) for i in terminations],
            # (range values may be lists the user mutates in place: copied into tuples, never referenced)
            [(tuple(map(tuple, m.ranges_list())), m._resample_steps, m._external_controller is None)
             for m in self.commands],
            [(m._air_time_contact_threshold, m.enabled) for m in self.contacts],
            (self.reward is None or self.reward.enabled, self.termination is None or self.termination.enabled,
             self.action is None or self.action.enabled, [m.enabled for m in self.commands]),
            [(om.noise, om.enabled) for om in self.observations],
            [(i.scale, i.noise) for i in obs_items],
            # lowered user observation terms fold their params in: a change traces them again (pack)
            [repr(sorted(dict(self.observations[g].cfg[n].params or {}).items())) for g, n in self.user_obs],
            # lowered class-style terms: a new instance or an edited scalar attribute traces them again (pack)
            self._stateful_fingerprint() if self.stateful else (),
        )

    def _stateful_fingerprint(self) -> list:
        from .expr import instance_constants

        cfg = {"reward": self.reward.cfg if self.reward is not None else {},
               "termination": self.termination.term_cfg if self.termination is not None else {}}
        out = []
        for key in self.stateful:
            fn = (self.observations[key[2]].cfg if len(key) == 3 else cfg[key[0]])[key[1]].fn
            out.append((id(fn), instance_constants(fn), self._lazy_started.get(key)))
        return out

    def _entity_of(self, params: dict):
        """The entity a term's (bound) parameters refer to, or None when the term takes no entity."""
        em = params.get("entity_manager")
        if em is not None:
            return em.entity
        if "entity_attr" in params:
            return getattr(self.env, params["entity_attr"], None)
        return None

    def _other_entity(self, item, what: str):
        """
        A stock mdp term that refers to an entity other than the kernel's (a further EntityManager, another
        `entity_attr`): the step's kernel holds one entity's state, so the term is evaluated like a
        user-defined one -- a host callback between the kernel phases -- through the one-term path of
        `evaluate_single_term`, bound to that entity's state and to its manager's cache.
        """
        sig = getattr(item.fn, "gfb_signature", None)
        if sig is None or getattr(item.fn, "__self__", None) is not None:  # user function / a manager's own term
            return None
        entity = self._entity_of(sig(self.env, **(item.params or {})))
        if entity is None or entity is self.primary_entity:
            return None
        if item.fn.gfb_opcode == "GFB_R_BODY_ACC_EXP":
            raise UnsupportedTermError(f"{what}: body_acceleration_exp keeps per-term state in the kernel and is "
                                       "lowered for the first EntityManager's entity only")
        return entity

    def _entity_ok(self, params: dict, what: str):
        em = params.get("entity_manager")
        if em is not None:
            if em.entity is not self.primary_entity:
                raise UnsupportedTermError(
                    f"{what}: stock mdp terms are lowered for the first EntityManager's entity only; wrap a term "
                    "of another entity in a user-defined function around that manager's getters"
                )
            return
        attr = params.get("entity_attr", "robot")
        if getattr(self.env, attr, None) is not self.primary_entity:
            raise UnsupportedTermError(f"{what}: entity_attr '{attr}' is not the fused step's entity")

    def _command_index(self, mgr, what: str) -> int:
        for k, m in enumerate(self.commands):
            if m is mgr:
                return k
        raise UnsupportedTermError(f"{what}: command manager is not registered with this environment")

    def _contact_index(self, mgr, what: str) -> int:
        for k, m in enumerate(self.contacts):
            if m is mgr:
                return k
        raise UnsupportedTermError(f"{what}: contact manager is not registered with this environment")

    def _pack_user_term(self, t, kind: str, name: str, item):
        prog = self._user_program(kind, name, item)
        t.i0 = prog.digest()  # structural: part of what a specialised kernel is matched on
        params = item.params or {}
        for k, pname in enumerate(prog.params):
            t.p[k] = params[pname]  # live: a curriculum may change them without a new kernel
        if prog.first is not None:  # class-style terms have no live params: p[0] selects the steady program
            t.p[0] = 1.0 if self._lazy_started.get((kind, name), False) else 0.0

    def _tilt_threshold(self, limit_angle: float) -> float:
        key = float(limit_angle)
        if key not in self._threshold_cache:
            self._threshold_cache[key] = asin_tilt_threshold(key)
        return self._threshold_cache[key]

    def pack(self):
        fp = self._live_fingerprint()
        if fp == self._fingerprint:
            return
        self._spec_checked = set()  # the structure may have changed with the values
        env, K, P = self.env, nat.K, self.program.head
        C.memset(C.byref(self.program), 0, C.sizeof(self.program))
        P.num_envs, P.num_dofs = self.N, self.D
        P.env_dt = env.dt
        P.base_max_episode_length = env._base_max_episode_length or 0
        if env._base_max_episode_length and env._max_episode_random_scaling > 0.0:
            P.max_len_random_span = env._base_max_episode_length * env._max_episode_random_scaling
        P.rng_mode = 0 if self.injected is not None else 1
        P.rng_seed = self.rng_seed

        # action
        if self.action is not None:
            # a disabled action manager returns before anything (position_action_manager.py:383-384):
            # targets stay as they are and nothing is sent to the actuators; GenesisEnv.step still runs
            P.action_mode = self.action.kernel_mode if self.action.enabled else 0
            self._action_enabled_packed = self.action.enabled
            kp = {k: v.detach().cpu().tolist() for k, v in self.action.kernel_params().items()}
            for d in range(self.D):
                P.action_scale[d] = kp["scale"][d]
                P.action_offset[d] = kp["offset"][d]
                P.action_clip_lo[d] = kp["clip_lo"][d]
                P.action_clip_hi[d] = kp["clip_hi"][d]
                P.default_dof_pos[d] = kp["default"][d]

        # commands
        P.n_command = len(self.commands)
        for k, mgr in enumerate(self.commands):
            cm = P.command[k]
            ranges = mgr.ranges_list()
            if len(ranges) > nat.MAX_COMMAND_DIMS:
                raise UnsupportedTermError("command manager with too many ranges")
            if not ranges and mgr not in self.python_commands:
                raise UnsupportedTermError("command manager without a range")
            cm.n_dims = len(ranges)
            cm.resample_steps = mgr._resample_steps
            cm.enabled = 1 if (mgr.enabled and mgr._external_controller is None and mgr not in self.python_commands) else 0
            for i, (lo, hi) in enumerate(ranges):
                cm.lo[i], cm.hi[i] = lo, hi

        # contacts
        P.n_contact = len(self.contacts)
        scene = env.scene
        for m, mgr in enumerate(self.contacts):
            cm = P.contact[m]
            ids = mgr._link_ids.tolist()
            local = mgr._local_link_ids.tolist()
            withs = [int(w) for w in mgr._with_link_ids.tolist()]
            if len(ids) > nat.MAX_CONTACT_LINKS or len(withs) > nat.MAX_WITH_LINKS:
                raise UnsupportedTermError("contact manager tracks too many links")
            cm.n_links, cm.n_with = len(ids), len(withs)
            cm.has_with_filter = 1 if mgr._has_with_filter else 0
            cm.track_air_time = 1 if mgr._track_air_time else 0
            cm.air_time_threshold = mgr._air_time_contact_threshold
            cm.scene_dt = scene.dt
            cm.disabled = 0 if mgr.enabled else 1  # contact_manager.py:331-336: nothing is recomputed
            for i, v in enumerate(ids):
                cm.link_ids[i] = v
                cm.local_link_ids[i] = local[i]
            for i, v in enumerate(withs):
                cm.with_ids[i] = v

        # phases of disabled managers are not launched: their step() returns before touching anything
        # (termination_manager.py:159-160, reward_manager.py:172-173)
        mask = 0xFFFFFFFF
        if self.termination is not None and not self.termination.enabled:
            mask &= ~K["GFB_PHASE_TERMINATION"]
        # rewards
        P.manager_flags = 0
        if self.reward is not None and not self.reward.enabled:
            mask &= ~K["GFB_PHASE_REWARD"]
            P.manager_flags |= K["GFB_MF_REWARD_DISABLED"]  # reward_manager.py:204: no logging, sums kept
        self._phase_mask = mask
        P.n_reward = len(self.reward_terms)
        if P.n_reward > nat.MAX_REWARD:
            raise UnsupportedTermError(f"at most {nat.MAX_REWARD} reward terms are supported")
        self._feet_slide_manager = None
        self._fixed_command_parts = None
        for r, (name, item, opcode) in enumerate(self.reward_terms):
            t = P.reward[r]
            t.op, t.mgr, t.i0 = opcode, -1, 0
            t.weight = item.weight * env.dt  # reward_manager.py:184
            if opcode == K["GFB_R_EXTERNAL"]:
                t.ext_col = self.ext_row[("reward", name)]
                continue
            if opcode == K["GFB_R_USER"]:
                self._pack_user_term(t, "reward", name, item)
                continue
            sig = getattr(item.fn, "gfb_signature", None) or item.fn.__func__.gfb_signature
            p = sig(env, **item.params)
            what = f"reward '{name}'"
            if opcode == K["GFB_R_BODY_ACC_EXP"]:
                self._entity_ok(p, what)
                t.p[0] = p["sensitivity"]
                t.p[1] = 1.0 if self._body_acc_started.get(name, False) else 0.0
                if self._body_acc_prev is None:
                    self._body_acc_prev = torch.zeros((self.N, 6), device=self.device)
                self._set(K["GFB_B_BODY_ACC_PREV"], self._body_acc_prev)
                self._body_acc_terms.add(name)
            if opcode in (K["GFB_R_LIN_VEL_Z"], K["GFB_R_ANG_VEL_XY"], K["GFB_R_FLAT_ORIENTATION"],
                          K["GFB_R_TRACK_LIN_VEL"], K["GFB_R_TRACK_ANG_VEL"], K["GFB_R_BASE_HEIGHT"]):
                self._entity_ok(p, what)
            if opcode == K["GFB_R_BASE_HEIGHT"]:
                if p["height_command"] is not None:
                    t.flags |= K["GFB_RF_TARGET_FROM_COMMAND"]
                    t.mgr = self._command_index(p["height_command"], what)
                elif torch.is_tensor(p["target_height"]):
                    t.flags |= K["GFB_RF_TARGET_FROM_TENSOR"]
                    self._set(K["GFB_B_TARGET_HEIGHT"], p["target_height"].expand(self.N), torch.float32, keep=True)
                else:
                    t.p[0] = p["target_height"]
                tm = p["terrain_manager"]
                if tm is not None:
                    if tm.height_field is None:
                        t.flags |= K["GFB_RF_TERRAIN_FLAT"]
                        t.p[1] = float(tm._origin[2])
                    else:
                        t.flags |= K["GFB_RF_TERRAIN_HEIGHT"]
                        P.height_field_rows, P.height_field_cols = tm.height_field.shape
                        for i, b in enumerate(tm.get_bounds()):
                            P.terrain_bounds[i] = b
                        self._set(K["GFB_B_HEIGHT_FIELD"], tm.height_field)
            elif opcode in (K["GFB_R_TRACK_LIN_VEL"], K["GFB_R_TRACK_ANG_VEL"]):
                t.p[0] = p["sensitivity"]
                if p["vel_cmd_manager"] is not None:
                    t.mgr = self._command_index(p["vel_cmd_manager"], what)
                else:
                    t.flags |= K["GFB_RF_FIXED_COMMAND"]
                    parts = self._fixed_command_parts or {}
                    if opcode == K["GFB_R_TRACK_LIN_VEL"]:
                        parts["lin"] = p["command"]
                    else:
                        parts["ang"] = p["commanded_ang_vel"]
                    self._fixed_command_parts = parts
            elif opcode == K["GFB_R_STAND_STILL"]:
                t.p[0] = p["command_threshold"]
                t.mgr = self._command_index(p["vel_cmd_manager"], what)
            elif opcode == K["GFB_R_HAS_CONTACT"]:
                t.mgr = self._contact_index(p["contact_manager"], what)
                t.p[0], t.i0 = p["threshold"], int(p["min_contacts"])
            elif opcode == K["GFB_R_CONTACT_FORCE"]:
                t.mgr = self._contact_index(p["contact_manager"], what)
                t.p[0] = p["threshold"]
            elif opcode == K["GFB_R_FEET_AIR_TIME"]:
                t.mgr = self._contact_index(p["contact_manager"], what)
                t.p[0] = p["time_threshold"]
                if p["time_threshold_max"] is not None:
                    t.flags |= K["GFB_RF_HAS_MAX"]
                    t.p[1] = p["time_threshold_max"] - p["time_threshold"]
                t.p[2] = env.dt + 1.0e-8  # has_made_contact(env.dt), contact_manager.py:198-224
                t.i0 = self._command_index(p["vel_cmd_manager"], what) if p["vel_cmd_manager"] is not None else -1
            elif opcode == K["GFB_R_FEET_SLIDE"]:
                t.mgr = self._contact_index(p["contact_manager"], what)
                self._feet_slide_manager = (p["contact_manager"], p["entity_attr"])

        # terminations
        P.n_termination = len(self.termination_terms)
        if P.n_termination > nat.MAX_TERMINATION:
            raise UnsupportedTermError(f"at most {nat.MAX_TERMINATION} termination terms are supported")
        for i, (name, item, opcode) in enumerate(self.termination_terms):
            t = P.termination[i]
            t.op, t.mgr, t.time_out = opcode, -1, 1 if item.time_out else 0
            if opcode == K["GFB_T_EXTERNAL"]:
                t.i0 = self.ext_row[("termination", name)]
                continue
            if opcode == K["GFB_T_USER"]:
                self._pack_user_term(t, "termination", name, item)
                continue
            sig = getattr(item.fn, "gfb_signature", None) or item.fn.__func__.gfb_signature
            p = sig(env, **item.params)
            what = f"termination '{name}'"
            if opcode == K["GFB_T_BAD_ORIENTATION"]:
                self._entity_ok(p, what)
                t.p[0] = self._tilt_threshold(p["limit_angle"])
                t.i0 = int(p["grace_steps"])
            elif opcode == K["GFB_T_BASE_HEIGHT_MIN"]:
                self._entity_ok(p, what)
                t.p[0] = p["minimum_height"]
            elif opcode == K["GFB_T_OUT_OF_BOUNDS"]:
                self._entity_ok(p, what)
                x_min, x_max, y_min, y_max = p["terrain_manager"].get_bounds(p["subterrain"])
                margin = p["border_margin"]
                t.p[0], t.p[1] = x_min + margin, x_max - margin
                t.p[2], t.p[3] = y_min + margin, y_max - margin
            elif opcode == K["GFB_T_HAS_CONTACT"]:
                t.mgr = self._contact_index(p["contact_manager"], what)
                t.p[0], t.i0 = p["threshold"], int(p["min_contacts"])
            elif opcode == K["GFB_T_CONTACT_FORCE"]:
                t.mgr = self._contact_index(p["contact_manager"], what)
                t.p[0] = p["threshold"]
            elif opcode == K["GFB_T_CONTACT_FORCE_GRACE"]:
                t.mgr = self._contact_index(p["contact_manager"], what)
                t.p[0], t.i0 = p["threshold"], int(p["grace_steps"])

        # observations
        P.n_obs_groups = len(self.observations)
        if self.user_obs:
            import hashlib

            progs = {key: self._user_obs_program(*key, self.observations[key[0]].cfg[key[1]]) for key in self.user_obs}
            text = "".join(f"{self.user_obs[k][2]}:{self.user_obs[k][3]}:{progs[k].digest()};" for k in sorted(progs))
            uid = int.from_bytes(hashlib.sha1(text.encode()).digest()[:4], "little") & 0x7FFFFFFF
            self._obs_user_id = uid or 1  # structural: the specialised kernels are matched on it
        col = 0
        src_of = {
            "targets": K["GFB_O_TARGETS"], "dof_pos": K["GFB_O_DOF_POS"], "dof_vel": K["GFB_O_DOF_VEL"],
            "dof_force": K["GFB_O_DOF_FORCE"], "lin_vel_b": K["GFB_O_LIN_VEL_B"], "ang_vel_b": K["GFB_O_ANG_VEL_B"],
            "gravity_b": K["GFB_O_GRAVITY_B"], "env_actions": K["GFB_O_ENV_ACTIONS"],
        }
        for g, om in enumerate(self.observations):
            og = P.obs_group[g]
            cols = om.columns() if om.enabled else []
            og.n_cols, og.history, og.col_begin = len(cols), om._history_len, col
            og.user_id = self._obs_user_id
            if col + len(cols) > nat.MAX_OBS_COLS:
                raise UnsupportedTermError(f"more than {nat.MAX_OBS_COLS} observation columns")
            for c in cols:
                oc = self.program.obs_cols[col]
                key = c["key"]
                oc.col, oc.scale, oc.noise, oc.mgr = c["col"], c["scale"], c["noise"], -1
                if isinstance(key, tuple) and key[0] == "command":
                    oc.src, oc.mgr = K["GFB_O_COMMAND"], self._command_index(key[1], "observation")
                elif isinstance(key, tuple) and key[0] == "contact_norm":
                    oc.src, oc.mgr = K["GFB_O_CONTACT_NORM"], self._contact_index(key[1], "observation")
                elif isinstance(key, tuple) and key[0] == "external" and (g, key[1]) in self.user_obs:
                    oc.src, oc.mgr = K["GFB_O_USER"], self.user_obs_width
                    oc.col = self.user_obs[(g, key[1])][2] + c["col"]
                elif isinstance(key, tuple) and key[0] == "external":
                    oc.src, oc.mgr = K["GFB_O_EXTERNAL"], self.ext_obs_width
                    oc.col = om._external_col0[key[1]] + c["col"]
                elif key in src_of:
                    oc.src = src_of[key]
                else:
                    raise UnsupportedTermError(f"observation source {key!r} is not supported by the fused step")
                col += 1
        self._fingerprint = fp

    # ------------------------------------------------------------------------------------------
    # per-step pointers
    # ------------------------------------------------------------------------------------------
    def _engine_buffers(self, post_reset: bool = False):
        """Pointers to the engine's state tensors (zero-copy; getters are called once per launch)."""
        s, B = self._set_engine, self._B
        self._keepalive = []
        robot = self.primary_entity
        f32 = torch.float32
        # the re-observation of reset envs reads the cached quaternion, not pos/quat -- except lowered user
        # observation terms that read the engine's pose
        if not post_reset or self._obs_reads_pose:
            s(B["GFB_B_POS"], robot.get_pos(), f32)
            s(B["GFB_B_QUAT"], robot.get_quat(), f32)
        s(B["GFB_B_VEL"], robot.get_vel(), f32)
        s(B["GFB_B_ANG"], robot.get_ang(), f32)
        if self.action is not None:
            idx = self.action.dofs_idx
            jointed = self._dof_entity  # (a one-term evaluation may point `primary_entity` at another entity)
            s(B["GFB_B_DOF_POS"], jointed.get_dofs_position(idx), f32)
            s(B["GFB_B_DOF_VEL"], jointed.get_dofs_velocity(idx), f32)
            if self._uses_dof_force:
                s(B["GFB_B_DOF_FORCE"], jointed.get_dofs_force(idx), f32)
        # a command manager driven by an external controller / gamepad: the terms read what its
        # `command` property returns -- the controller's tensor for this step (command_manager.py:85-90)
        if self._has_command_override:
            K = nat.K
            any_controller = False
            for k, mgr in enumerate(self.commands):
                if mgr._external_controller is not None:
                    s(K["GFB_B_COMMAND0"] + k, mgr._external_controller(self.env.step_count), f32)
                    self._controller_bound[k] = any_controller = True
                elif self._controller_bound[k]:
                    self._set(K["GFB_B_COMMAND0"] + k, mgr._command)
                    self._controller_bound[k] = False
            self.any_controller = any_controller
            self._has_command_override = any_controller
        K = nat.K
        if self.contacts and not post_reset:
            solver = self.env.scene.rigid_solver
            c = solver.collider.get_contacts(as_tensor=True, to_torch=True)
            s(K["GFB_B_C_FORCE"], c["force"], f32)
            s(K["GFB_B_C_POS"], c["position"], f32)
            s(K["GFB_B_C_LINK_A"], c["link_a"], torch.int32)
            s(K["GFB_B_C_LINK_B"], c["link_b"], torch.int32)
            lq = solver.get_links_quat()
            s(K["GFB_B_LINKS_QUAT"], lq, f32)
            dims = (c["link_a"].shape[-1], lq.shape[1])
            if dims != self._contact_dims:
                self._contact_dims = dims
                self._program_pushed = False
                self._spec_checked = set()
            if self._feet_slide_manager is not None:
                mgr, attr = self._feet_slide_manager
                vel = getattr(self.env, attr).get_links_vel(links_idx_local=mgr.local_link_ids)
                s(K["GFB_B_LINKS_VEL"], vel, f32)
        if self._fixed_command_parts:
            s(K["GFB_B_FIXED_COMMAND"], self._resolve_fixed_command(), f32)

    def _resolve_fixed_command(self) -> torch.Tensor:
        """(N,3) tensor [cmd_x, cmd_y, cmd_yaw] for tracking terms configured with fixed tensors."""
        parts = self._fixed_command_parts
        lin, ang = parts.get("lin"), parts.get("ang")
        base = None
        for t in (lin, ang):
            if t is not None and t._base is not None and tuple(t._base.shape) == (self.N, 3):
                base = t._base
        if base is not None and base.is_contiguous():
            ok_lin = lin is None or (lin._base is base and lin.data_ptr() == base.data_ptr() and lin.stride() == (3, 1))
            ok_ang = ang is None or (ang._base is base and ang.data_ptr() == base.data_ptr() + 8 and ang.stride() == (3,))
            if ok_lin and ok_ang:
                return base  # zero-copy: both are views of one (N,3) command tensor
        if self._fixed_command is None:
            self._fixed_command = torch.zeros((self.N, 3), device=self.device)
        if lin is not None:
            self._fixed_command[:, :2] = lin
        if ang is not None:
            self._fixed_command[:, 2] = ang.reshape(self.N)
        return self._fixed_command

    @property
    def _uses_dof_force(self) -> bool:
        if self._dof_force_used is None:
            self._dof_force_used = any(key == "dof_force" for om in self.observations for (_, key, _) in om._sources)
        return self._dof_force_used

    def _obs_buffers(self):
        """The two frame buffers of every observation group swap roles each step (fixed storage)."""
        table = self._obs_ptrs
        if table is None:
            K = nat.K
            table = self._obs_ptrs = [
                (om, K["GFB_B_OBS_PREV0"] + g, K["GFB_B_OBS_OUT0"] + g,
                 (om._buffers[0].data_ptr(), om._buffers[1].data_ptr()), (om._buffers[0], om._buffers[1]))
                for g, om in enumerate(self.observations)
            ]
        buf = self.buffers.buf
        for om, prev_id, out_id, ptrs, _ in table:
            cur = om._current
            buf[prev_id] = ptrs[cur]
            buf[out_id] = ptrs[1 - cur]

    def _injection_buffers(self):
        if self._injected_bound is self.injected:
            return
        self._injected_bound = self.injected
        K, s = nat.K, self._set
        inj = self.injected or {}
        for k in range(len(self.commands)):
            s(K["GFB_B_INJ_CMD_STEP0"] + k, inj.get(f"cmd_step{k}"))
            s(K["GFB_B_INJ_CMD_RESET0"] + k, inj.get(f"cmd_reset{k}"))
        s(K["GFB_B_INJ_MAX_LEN"], inj.get("max_len"))
        for g in range(len(self.observations)):
            s(K["GFB_B_OBS_NOISE0"] + g, inj.get(f"obs_noise{g}"))

    def inject(self, draws: dict[str, torch.Tensor] | None):
        """
        Parity mode: dense buffers holding the reference's own draws.
            cmd_step<k>, cmd_reset<k>   (N, K_k)  command values for resampled / reset envs
            max_len                     (N,)      U(-1,1) draws of genesis_env.py:249
            obs_noise<g>                (N, O_g)  U(-1,1) draws of observation_manager.py:249
        None returns to in-kernel Philox.
        """
        self.injected = draws
        self._program_pushed = False  # rng_mode is part of the packed table

    def _stream(self):
        if self._stream_ptr is None:
            self._stream_ptr = torch._C._cuda_getCurrentRawStream(self.index)
        return self._stream_ptr

    def begin_step(self):
        """Per-step caches: the caller's current stream; fresh logging storage once views were handed out."""
        self._stream_ptr = None
        self._program_pushed = False
        # logged means are handed out as views of this vector and may be kept by the caller (rsl_rl
        # collects extras["episode"] over a whole iteration): once views were handed out, the next
        # step writes into fresh storage
        if self._log_out_handed_out:
            if self._log_spare is not None:  # prepared while the GPU was busy (prepare_spare_log)
                self.log_out, self._log_views = self._log_spare
                self._log_spare = None
            else:
                self.log_out, self._log_views = torch.empty_like(self.log_out), None
            self.buffers.buf[self._log_out_id] = self.log_out.data_ptr()
            self._log_out_handed_out = False

    # ------------------------------------------------------------------------------------------
    # launches
    # ------------------------------------------------------------------------------------------
    def log_views(self) -> tuple:
        """0-dim views of the current logging vector, one per entry (what `extras` hands out)."""
        if self._log_views is None:
            self._log_views = self.log_out.unbind(0)
        self._log_out_handed_out = True  # the next step gets fresh storage
        return self._log_views

    def prepare_spare_log(self):
        """
        Next step's logging vector and its views.  Creating the ~10 view objects costs ~1 us each;
        called after the step's kernels are enqueued and before the host blocks on the report, i.e.
        while the GPU is busy, instead of on the critical path between the report and the next launch.
        """
        if self._log_spare is None:
            spare = torch.empty_like(self.log_out)
            self._log_spare = (spare, spare.unbind(0))

    def _set_program(self, force: bool = False):
        """Pack (if a live value changed) and hand the term table to the library; once per step."""
        if self._program_pushed and not force:
            return
        self.pack()
        P = self.program.head
        P.step_index = self.env.step_count
        if self.contacts:
            if self._contact_dims is None:
                solver = self.env.scene.rigid_solver
                c = solver.collider.get_contacts(as_tensor=True, to_torch=True)
                self._contact_dims = (c["link_a"].shape[-1], solver.get_links_quat().shape[1])
            P.n_contact_slots, P.n_links_total = self._contact_dims
        self.handle.check(self.lib.gfb_set_program(self.handle.ptr, C.byref(self.program)), "gfb_set_program")
        self._program_pushed = not self.dry_run
        self._program_ever_pushed = True

    def cache_entity(self):
        """Entity phase alone (EntityManager.build() caches the pose before the first reset)."""
        self._engine_buffers()
        self._set_program()
        self.handle.check(
            self.lib.gfb_post_physics(self.handle.ptr, C.byref(self.buffers), nat.K["GFB_PHASE_ENTITY"], self._stream()),
            "gfb_post_physics(entity)",
        )

    def action_step(self, actions: torch.Tensor):
        """
        Pre-physics launch + the engine's PD-target write.  This is on the host's critical path (the
        GPU idles until the launch is issued), so nothing that can wait is done here: the live-config
        check / re-pack happens in the shadow of this kernel (post_physics).  The launch only reads the
        action part of the table, which is fixed at build time -- except for `action.enabled`.
        """
        if actions.dtype is not torch.float32 or not actions.is_contiguous() or actions.device != self.device:
            actions = actions.to(self.device, torch.float32).contiguous()
        action = self.action
        enabled = action is None or action.enabled
        # (a disabled manager's step() returns before its delay FIFO moves, position_action_manager.py:383-384)
        raw_mgr = action._delayed(actions) if action is not None and enabled else actions
        if raw_mgr is not actions and (raw_mgr.dtype is not torch.float32 or not raw_mgr.is_contiguous()):
            raw_mgr = raw_mgr.to(self.device, torch.float32).contiguous()
        self._action_keep = (actions, raw_mgr)
        if not self._program_ever_pushed or enabled != self._action_enabled_packed:
            self._set_program()
        # env.actions / env.last_actions are a ring (genesis_env.py:202 `last_actions <- actions` as an
        # exchange of the two buffers instead of a copy: 4*D bytes per env less traffic per step)
        env = self.env
        env._actions, env._last_actions = env._last_actions, env._actions
        buf, ia, il = self.buffers.buf, self._B["GFB_B_ENV_ACTIONS"], self._B["GFB_B_ENV_LAST_ACTIONS"]
        buf[ia], buf[il] = buf[il], buf[ia]  # (both tensors were validated when they were first bound)
        rc = self.lib.gfb_action_step_ring(self._h, self._buffers_ref, actions.data_ptr(), raw_mgr.data_ptr(), self._stream())
        if rc:  # nothing was launched: undo the exchange before raising
            env._actions, env._last_actions = env._last_actions, env._actions
            buf[ia], buf[il] = buf[il], buf[ia]
            self.handle.check(rc, "gfb_action_step_ring")
        if action is not None and enabled:  # position_action_manager.py:383-384: a disabled manager sends nothing
            self.env.robot.control_dofs_position(action._actions, action.dofs_idx)

    # ------------------------------------------------------------------------------------------
    # specialised kernels (spec.py)
    # ------------------------------------------------------------------------------------------
    def prepare_describe(self, injected: bool):
        """Bind every buffer the way a real step does, so that the slab plan can be described."""
        if injected:
            draws = {"max_len": torch.zeros(self.N, device=self.device)}
            for k, mgr in enumerate(self.commands):
                draws[f"cmd_step{k}"] = torch.zeros_like(mgr._command)
                draws[f"cmd_reset{k}"] = torch.zeros_like(mgr._command)
            for g, om in enumerate(self.observations):
                draws[f"obs_noise{g}"] = torch.zeros((self.N, om.frame_size), device=self.device)
            self.inject(draws)
        else:
            self.inject(None)
        self._engine_buffers()
        self._obs_buffers()
        self._injection_buffers()
        self._set_program(force=True)

    def _maybe_specialise(self, phases: int):
        """Attach the specialised kernel for the current table structure (once per structure)."""
        if phases in self._spec_checked:  # nothing was re-packed since the last look
            return
        self._spec_checked.add(phases)
        from . import spec

        if spec.disabled() or self.dry_run:
            return
        tag = self._spec_tag(phases)
        if tag in self._spec_tried:
            return
        self._spec_tried.add(tag)
        try:
            path = spec.ensure(self, phases)
            if path is not None and path not in self.spec_paths:
                spec.attach(self, path)
                self.spec_paths.append(path)
            self._spec_ok[tag] = path is not None
        except Exception as e:  # a failed specialisation is not fatal: the generic kernel runs
            self._spec_ok[tag] = False
            print(f"[genesis_forge_b200] kernel specialisation skipped: {e}")

    def _spec_tag(self, phases: int):
        return (self._fingerprint_structure(), self.injected is not None, phases)

    def _fingerprint_structure(self):
        """Cheap proxy for 'the table structure may have changed' (exact matching is done in C)."""
        return (
            tuple(item.weight == 0 for _, item, _ in self.reward_terms),
            tuple(item.version for _, item, _ in self.reward_terms),
            tuple(item.version for _, item, _ in self.termination_terms),
            tuple(m._external_controller is None for m in self.commands),
            self._contact_dims,
            self._obs_user_id,
            tuple(self.user_terms[k][0].digest() for k in self.stateful if k in self.user_terms),
        )

    def spec_stats(self) -> dict:
        a, b, u = C.c_int64(), C.c_int64(), C.c_int64()
        self.lib.gfb_spec_stats(self.handle.ptr, C.byref(a), C.byref(b), C.byref(u))
        stats = {"specialised_launches": a.value, "generic_launches": b.value, "libraries": [p.name for p in self.spec_paths]}
        if self.user_obs:  # the reset path's kernel of the lowered observation terms (gfb_observe)
            stats["user_observe_launches"] = u.value
        return stats

    def evaluate_external(self, kind: str):
        """Run the user-defined reward / termination functions; their values become kernel inputs."""
        mgr = self.reward if kind == "reward" else self.termination
        if mgr is not None and not mgr.enabled:  # a disabled manager calls no term (a class-style term's state stays)
            return
        for j, (k, name, item) in enumerate(self.external_rows):
            if k != kind:
                continue
            if kind == "reward" and item.weight == 0:
                continue  # reward_manager.py:181-182: zero-weight terms are not evaluated
            value = item.fn(self.env, **item.params)
            self.ext_values[j].copy_(value.reshape(self.N))

    def evaluate_external_obs(self):
        if any(len(k) == 3 for k in self.stateful):
            # the lowered class-style observation terms are evaluated next (get_observations, the observation
            # launch of a split step): their state is checked first; demoted, they are host columns from here on
            why = self._check_state()
            if why is not None:
                self._demote_user_terms(why)
        for om, name, item, col0, width in self.external_obs:
            value = item.fn(env=self.env, **item.params)
            self.ext_obs[:, col0:col0 + width].copy_(value.reshape(self.N, width))

    def post_physics_local(self, phases: int) -> int:
        """
        The post-physics launch of the one-launch step; returns the rank's number of reset envs as soon as
        the FIRST stage of the report arrives (gfb_report.local_seq: before the kernel's last block waits
        for the peers' logging partials).  `finish_report()` completes the report before it is published.
        On a single rank the two stages arrive together.
        """
        self.post_physics(phases, read_report=False)
        if self.dist is not None and not self.peer_mode:
            self._allreduce_logging()
        self.prepare_spare_log()  # host work hidden behind the kernel just enqueued
        rc = self.lib.gfb_read_report_local(self._h, self._local_n_ref, self._stream())
        if rc:
            self.handle.check(rc, "gfb_read_report_local")
        return self._local_n.value

    def finish_report(self) -> nat.Report:
        rc = self.lib.gfb_read_report(self._h, self._report_ref, self._stream())
        if rc:
            self.handle.check(rc, "gfb_read_report")
        self._after_report()
        return self.report

    def post_physics(self, phases: int, read_report: bool = True) -> nat.Report | None:
        """
        The post-physics launch.  Everything up to the launch call runs in the shadow of the action
        kernel (which the GPU is still executing); the host then prepares the next step's logging
        storage while the kernel runs and finally spins on the report, which the kernel's last block
        writes into mapped host memory (include/gfb200.h).
        """
        self._engine_buffers()
        self._obs_buffers()
        self._injection_buffers()
        self._set_program()
        phases &= self._phase_mask
        first = self.first_launch_of_step
        self.first_launch_of_step = False
        if first and self.stateful:
            why = self._check_state()
            if why is not None:
                self._demote_user_terms(why)
                raise UserTermsDemoted(why)
            self._set_program()  # (a state tensor the user assigned may start a lazily initialised term)
        if first and self.lowered_user_terms and self.split_mode:
            # a later launch of the split step evaluates the lowered terms: check before anything is launched
            why = self._user_terms_blocked()
            if why is not None:
                self._demote_user_terms(why)
                raise UserTermsDemoted(why)
        if phases in self._spec_phases:
            self._maybe_specialise(phases)
        if phases & self._PHASE_REWARD:
            self._after_launch_started = [
                name for name in self._body_acc_terms
                if not self._body_acc_started.get(name, False) and self.reward.cfg[name].weight != 0
            ] if self._body_acc_terms else []
        for key, started in self._lazy_started.items():  # lowered class terms this launch evaluates
            if not started and phases & (self._PHASE_REWARD if key[0] == "reward" else nat.K["GFB_PHASE_TERMINATION"]):
                if key[0] == "termination" or self.reward.cfg[key[1]].weight != 0:
                    self._after_launch_lazy.add(key)
        stream = self._stream()
        rc = self.lib.gfb_post_physics(self._h, self._buffers_ref, phases, stream)
        if rc:
            if first and rc == nat.K["GFB_ERR_UNSUPPORTED"] and self.lowered_user_terms and not self.split_mode:
                # the one launch of the fused step was refused before anything ran: no specialised kernel
                # matched the table with its lowered terms (not attached, or the launch cannot use TMA)
                why = self.lib.gfb_last_error(self._h).decode()
                self._demote_user_terms(why)
                raise UserTermsDemoted(why)
            self.handle.check(rc, "gfb_post_physics")
        if not read_report:
            return None
        if self.dist is not None and not self.peer_mode:
            self._allreduce_logging()
        self.prepare_spare_log()  # host work hidden behind the kernel just enqueued
        rc = self.lib.gfb_read_report(self._h, self._report_ref, stream)
        if rc:
            self.handle.check(rc, "gfb_read_report")
        self._after_report()
        return self.report

    def _after_report(self):
        self.global_acc = None
        if self.report.status & nat.K["GFB_STATUS_PEER_TIMEOUT"]:
            raise nat.NativeLibraryError(
                "sharded logging: a peer rank did not take part in this step's exchange within 2 s "
                "(every rank must issue the same sequence of env.step / env.reset calls)"
            )
        if self.report.status & nat.K["GFB_STATUS_SCAN_TIMEOUT"]:
            raise nat.NativeLibraryError("post-physics kernel: the ordered reset-index scan stalled (internal error)")
        for name in self._after_launch_started:  # the term now has a previous velocity to difference
            self._body_acc_started[name] = True
        self._after_launch_started = []
        for key in self._after_launch_lazy:  # the kernel has initialised the state: the instance holds it now
            if key in self.stateful:
                b = self.stateful[key]
                self._lazy_started[key] = True
                for attr, (slot, _, _, lazy) in b["attrs"].items():
                    if lazy:
                        setattr(b["inst"], attr, b["tensors"][slot])
        self._after_launch_lazy = set()

    def observe(self, idx: torch.Tensor | None, n: int):
        self._engine_buffers(post_reset=True)
        self._obs_buffers()
        self._injection_buffers()
        self._set_program()
        if self.user_obs:  # the lowered observation terms' reset path is a kernel of the table's specialised library
            K = nat.K
            self._maybe_specialise(K["GFB_PHASE_OBSERVE"] if self.split_mode else self.step_phases & self._phase_mask)
        rc = self.lib.gfb_observe(self._h, self._buffers_ref, idx.data_ptr() if idx is not None else None, n, self._stream())
        if rc == nat.K["GFB_ERR_UNSUPPORTED"] and self.user_obs:
            # no specialised library for the lowered terms: they become host columns (split execution from now on)
            self._demote_user_terms(self.lib.gfb_last_error(self._h).decode())
            self.evaluate_external_obs()
            self._set_program()
            rc = self.lib.gfb_observe(self._h, self._buffers_ref, idx.data_ptr() if idx is not None else None, n,
                                      self._stream())
        if rc:
            self.handle.check(rc, "gfb_observe")

    def reset_rows(self, mode: str, tag: str, idx: torch.Tensor | None, n: int, width: int, a: float, b: float = 0.0,
                   base: torch.Tensor | None = None, out: torch.Tensor | None = None,
                   scatter: torch.Tensor | None = None) -> torch.Tensor:
        """
        Value rows for the engine setters of a reset, one launch of gfb_reset_rows (include/gfb200.h):
        mode "noise": base + U(-1,1) * a (position_action_manager.py:516-525); "uniform": U(a, b)
        (mdp/reset.py:229-284).  Draws come from the kernel's Philox stream unless the environment
        carries a replaying `rng` (parity harness), whose recorded draws for `tag` are passed through.
        """
        from .rng import HostRng

        if out is None:
            out = torch.empty((n, width), device=self.device)
        rng = getattr(self.env, "rng", None)
        draws = None
        if rng is not None and type(rng) is not HostRng:
            lo, hi = (-1.0, 1.0) if mode == "noise" else (a, b)
            like = out.reshape(-1) if (idx is None and n == 1) else out  # (a single row was drawn as a vector)
            draws = rng.uniform(tag, like, lo, hi).to(self.device, torch.float32).contiguous()
        code = nat.K["GFB_ROWS_NOISE"] if mode == "noise" else nat.K["GFB_ROWS_UNIFORM"]
        counter = (int(self.env.step_count) << 16) ^ (hash(tag) & 0xFFFF)
        ptr = lambda t: t.data_ptr() if t is not None else None  # noqa: E731
        rc = self.lib.gfb_reset_rows(self._h, ptr(idx), n, width, code, ptr(base), float(a), float(b), ptr(draws),
                                     (self.rng_seed << 4) ^ 0xD0, counter, ptr(out), ptr(scatter), self._stream())
        if rc:
            self.handle.check(rc, "gfb_reset_rows")
        return out

    def rotate_by_inv_base_quat(self, vec: torch.Tensor | None) -> torch.Tensor:
        quat = self.entity_manager._inv_base_quat if self.entity_manager is not None else self._inv_base_quat
        return self._rotate(vec, quat, conjugate=0)

    def rotate_by_inv_quat(self, vec: torch.Tensor | None, quat: torch.Tensor) -> torch.Tensor:
        return self._rotate(vec, quat, conjugate=1)

    def _rotate(self, vec, quat, conjugate: int) -> torch.Tensor:
        quat = quat.to(self.device, torch.float32).contiguous()
        n = quat.shape[0]
        if self.width_probe:  # a dry run's width probe of a user observation term: no device, the shape only
            return torch.zeros((n, 3), device=self.device)
        out = torch.empty((n, 3), device=self.device)
        vptr = None
        if vec is not None:
            vec = vec.to(self.device, torch.float32).contiguous()
            vptr = C.c_void_p(vec.data_ptr())
        self.handle.check(
            self.lib.gfb_rotate(self.handle.ptr, vptr, C.c_void_p(quat.data_ptr()), C.c_void_p(out.data_ptr()),
                                n, conjugate, self._stream()),
            "gfb_rotate",
        )
        return out

    def evaluate_single_term(self, kind, fn, params):
        """
        A stock mdp term called directly -- `rewards.lin_vel_z_l2(env, ...)` inside a user-defined term
        or from curriculum code -- is evaluated by the SAME kernel code as in the fused step: a
        one-term table goes to a second library handle and the reward (or termination) phase runs
        alone, with every array that phase writes redirected to scratch.  The value is the
        unweighted term, as in the reference (reward_manager.py:185, termination_manager.py:168);
        terms given an `entity_manager` use the base pose cached by the last step, the others the
        entity's current pose; contact terms read the last step's net forces.
        """
        from .expr import ExprMode

        if isinstance(self.env._tracing, ExprMode):
            raise UnsupportedTermError(f"user term: a direct call of the stock term {fn.__name__} is not inlined")
        if self.dry_run:
            raise nat.NativeLibraryError("direct evaluation of mdp terms needs a CUDA device (dry-run handle)")
        K = nat.K
        opcode = K[fn.gfb_opcode]
        if kind == "reward" and opcode == K["GFB_R_BODY_ACC_EXP"]:
            raise UnsupportedTermError("body_acceleration_exp keeps per-term state and cannot be evaluated on its own")
        if self._eval_handle is None:
            self._eval_handle = nat.Handle(self.N, self.index)

        class _Item:  # what pack() reads from a config item
            weight, time_out, version = 1.0, False, 0

        item = _Item()
        item.fn, item.params = fn, params
        saved = {k: getattr(self, k) for k in (
            "program", "buffers", "handle", "_fingerprint", "_program_pushed", "reward_terms", "termination_terms",
            "_feet_slide_manager", "_fixed_command_parts", "_keepalive", "_body_acc_terms", "_spec_checked",
            "primary_entity",
        )}
        N, dev = self.N, self.device
        try:
            self.program = nat.Program()
            self.buffers = nat.Buffers.from_buffer_copy(saved["buffers"])
            self.handle = self._eval_handle
            self._fingerprint = None
            self._program_pushed = False
            self._keepalive = []
            entity = self._entity_of(params)
            if entity is not None and entity is not self.primary_entity:
                # a term of another entity: that entity's state arrays, and its manager's cached pose
                self.primary_entity = entity
                other = params.get("entity_manager")
                if other is not None:
                    self._set(K["GFB_B_BASE_POS"], other._base_pos)
                    self._set(K["GFB_B_BASE_QUAT"], other._base_quat)
                    self._set(K["GFB_B_INV_BASE_QUAT"], other._inv_base_quat)
            if kind == "reward":
                self.reward_terms, self.termination_terms = [("direct", item, opcode)], []
                phase = K["GFB_PHASE_REWARD"]
                out = torch.empty(N, device=dev)
                scratch = [out, torch.zeros((1, N), device=dev), torch.zeros(N, device=dev)]
                self._set(K["GFB_B_REWARD"], out)
                self._set(K["GFB_B_EP_SUMS"], scratch[1])
                self._set(K["GFB_B_EP_SECONDS"], scratch[2])
            else:
                self.reward_terms, self.termination_terms = [], [("direct", item, opcode)]
                phase = K["GFB_PHASE_TERMINATION"]
                out = torch.empty(N, device=dev, dtype=torch.bool)
                scratch = [out, torch.empty(N, device=dev, dtype=torch.bool)]
                self._set(K["GFB_B_TERMINATED"], out)
                self._set(K["GFB_B_TRUNCATED"], scratch[1])
            if params.get("entity_manager") is None and "entity_attr" in params:
                # the uncached variant (utils.py:13-55) rotates by the entity's CURRENT quaternion: run the
                # entity phase as well, its cache outputs going to scratch
                phase |= K["GFB_PHASE_ENTITY"]
                scratch += [torch.empty((N, 3), device=dev), torch.empty((N, 4), device=dev), torch.empty((N, 4), device=dev)]
                self._set(K["GFB_B_BASE_POS"], scratch[-3])
                self._set(K["GFB_B_BASE_QUAT"], scratch[-2])
                self._set(K["GFB_B_INV_BASE_QUAT"], scratch[-1])
            if kind == "reward" and opcode == K["GFB_R_ACTION_RATE"]:
                # in the step this sum is produced by the action kernel before the reset; a direct call
                # sees the env's current action buffers (rewards.py:257-271)
                env = self.env
                scratch.append(torch.square(env.last_actions - env.actions).sum(dim=1).contiguous())
                self._set(K["GFB_B_ACTION_RATE"], scratch[-1])
            self._set(K["GFB_B_RESET_IDX"], None)  # nothing of the step's bookkeeping is touched
            self._set(K["GFB_B_LOG_OUT"], None)
            self._set(K["GFB_B_LOG_ACC"], None)
            self.pack()
            if kind == "reward":
                self.program.head.reward[0].weight = 1.0  # value * fp32(1.0): the unweighted term
            self._engine_buffers()
            em = params.get("entity_manager")
            if kind == "termination" and opcode == K["GFB_T_BASE_HEIGHT_MIN"] and em is not None:
                self._set(K["GFB_B_POS"], em._base_pos)  # the cached position (terminations.py:74-99)
            P = self.program.head
            P.step_index = self.env.step_count
            if self.contacts and self._contact_dims is not None:
                P.n_contact_slots, P.n_links_total = self._contact_dims
            self.handle.check(self.lib.gfb_set_program(self.handle.ptr, C.byref(self.program)), "gfb_set_program")
            self.handle.check(
                self.lib.gfb_post_physics(self.handle.ptr, C.byref(self.buffers), phase, self._stream()),
                f"gfb_post_physics({kind} term)",
            )
        finally:
            for k, v in saved.items():
                setattr(self, k, v)
        return out

    # ------------------------------------------------------------------------------------------
    # multi-GPU logging
    # ------------------------------------------------------------------------------------------
    def shard(self, group, global_num_envs: int, peer: bool | None = None):
        """
        Envs sharded over the ranks of `group` (this object holds one shard): logged means and
        publish decisions become global.  With `peer` (default on for NCCL groups, GFB_PEER_LOGGING=0
        turns it off) the exchange of the per-term partials runs INSIDE the finalize kernel over
        NVLink peer memory (gfb_peer_connect) and the step keeps its single host sync; otherwise one
        NCCL all-reduce per step runs on a side stream.
        """
        import os

        import torch.distributed as dist

        self.dist = group
        self.global_num_envs = int(global_num_envs)
        # every shard draws from its own Philox stream (the counters are local env indices)
        base_seed = getattr(self, "_unsharded_seed", self.rng_seed)
        self._unsharded_seed = base_seed
        self.rng_seed = (base_seed ^ ((dist.get_rank(group) + 1) << 40)) & 0xFFFFFFFFFFFFFFFF
        if peer is None:
            peer = os.environ.get("GFB_PEER_LOGGING", "1") != "0" and dist.get_backend(group) == "nccl"
        self.peer_mode = False
        if not peer or self.dry_run:
            return
        world, rank = dist.get_world_size(group), dist.get_rank(group)
        mine = (C.c_ubyte * nat.K["GFB_IPC_HANDLE_BYTES"])()
        self.handle.check(self.lib.gfb_peer_export(self.handle.ptr, mine), "gfb_peer_export")
        local = torch.tensor(list(bytes(mine)), dtype=torch.uint8, device=self.device)
        gathered = [torch.empty_like(local) for _ in range(world)]
        dist.all_gather(gathered, local, group=group)
        handles = b"".join(bytes(g.cpu().tolist()) for g in gathered)
        rc = self.lib.gfb_peer_connect(self.handle.ptr, rank, world, handles, self.global_num_envs)
        # the decision is collective: if any rank cannot map its peers (ranks on another node, no P2P
        # path), every rank falls back to the NCCL all-reduce
        ok = torch.tensor([1 if rc == 0 else 0], device=self.device, dtype=torch.int32)
        dist.all_reduce(ok, op=dist.ReduceOp.MIN, group=group)
        if int(ok.item()) == 0:
            why = self.lib.gfb_last_error(self.handle.ptr).decode() if rc != 0 else "a peer rank could not connect"
            self.lib.gfb_peer_disconnect(self.handle.ptr)
            if rank == 0:
                print(f"[genesis_forge_b200] peer-memory logging exchange unavailable ({why}); using NCCL all-reduce")
            return
        self.peer_mode = True

    def _allreduce_logging(self):
        """
        Sum per-term partials over ranks so that logged means are global (SURVEY.md 8(e)).  The
        collective and its read-back run on a side stream: nothing on the step's critical path (the
        local reset count, the reset fan-out, the re-observation) depends on them, so their latency
        overlaps that work; `finish_logging()` joins before the extras are published.
        """
        import torch.distributed as dist

        main = torch.cuda.current_stream(self.device)
        if self._log_stream is None:
            self._log_stream = torch.cuda.Stream(self.device)
            self._log_event = torch.cuda.Event()
            self._acc_host = torch.empty_like(self.log_acc, device="cpu").pin_memory()
        self._log_stream.wait_stream(main)
        with torch.cuda.stream(self._log_stream):
            dist.all_reduce(self.log_acc, op=dist.ReduceOp.SUM, group=self.dist)
            self._acc_host.copy_(self.log_acc, non_blocking=True)
            self._log_event.record(self._log_stream)
        self._log_pending = True

    def global_log_snapshot(self) -> torch.Tensor:
        """
        Logging vector of the all-reduced accumulator (same arithmetic as `combine_logging`), computed
        on the host from the pinned read-back that `finish_logging` already waited for, and sent to the
        device with one small async copy (a handful of eager device ops here cost ~80 us of host time).
        """
        n_r, n_t = self.n_reward, self.n_termination
        acc = self._acc_host.numpy()
        if self._log_out_host is None:
            self._log_out_host = torch.empty(n_r + n_t, dtype=torch.float32).pin_memory()
        out = self._log_out_host.numpy()
        n_reset = max(float(acc[n_r + n_t]), 1.0)
        with np.errstate(over="ignore", invalid="ignore"):
            s = acc[:n_r].astype(np.float32)  # a sum past the fp32 range is logged as +-Inf (tail.cuh xs_mean)
        out[:n_r] = np.where(np.isfinite(s), acc[:n_r] / n_reset, s)
        out[n_r:] = acc[n_r:n_r + n_t] / float(self.global_num_envs)
        snap = torch.empty(n_r + n_t, device=self.device, dtype=torch.float32)
        snap.copy_(self._log_out_host, non_blocking=True)
        return snap

    def finish_logging(self):
        """Join the side-stream all-reduce of this step (no-op when envs are not sharded)."""
        if self._log_pending:
            self._log_event.synchronize()
            torch.cuda.current_stream(self.device).wait_stream(self._log_stream)  # log_acc is rewritten next step
            self.global_acc = self._acc_host.tolist()
            self._log_pending = False

    def launch_count(self) -> int:
        return int(self.lib.gfb_launch_count(self.handle.ptr))

    def profile(self, enabled: bool):
        self.handle.check(self.lib.gfb_profile_enable(self.handle.ptr, 1 if enabled else 0), "gfb_profile_enable")

    def profile_read_aux(self) -> dict:
        """Average device time (us) of the small kernels since profiling was enabled (the reset path of lowered
        user observation terms only for tables that have them)."""
        ms, n = (C.c_float * 4)(), (C.c_int32 * 4)()
        self.handle.check(self.lib.gfb_profile_read_aux(self.handle.ptr, ms, n), "gfb_profile_read_aux")
        names = ("compact_kernel", "observe_kernel", "spawn_kernel") + (("user_observe_kernel",) if self.user_obs else ())
        return {name: {"kernel_us": ms[k] / max(n[k], 1) * 1e3, "launches": n[k]} for k, name in enumerate(names)}

    def profile_read(self) -> dict:
        post_ms, act_ms = C.c_float(), C.c_float()
        n_post, n_act = C.c_int32(), C.c_int32()
        self.handle.check(
            self.lib.gfb_profile_read(self.handle.ptr, C.byref(post_ms), C.byref(n_post), C.byref(act_ms), C.byref(n_act)),
            "gfb_profile_read",
        )
        return {"post_ms": post_ms.value, "post_launches": n_post.value,
                "action_ms": act_ms.value, "action_launches": n_act.value}
