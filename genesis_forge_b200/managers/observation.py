"""
ObservationManager: concatenation of observation terms (value * scale + U(-1,1) * noise), optional
history of the last H frames newest-first, named groups for asymmetric actor/critic.

API of genesis_forge/managers/observation_manager.py.  At build() each term function is *traced*
once: the manager getters it may call (EntityManager.get_*, action manager getters,
CommandManager.observation, mdp.observations.*) hand out tagged placeholder tensors while tracing is
active, and a term is accepted when it returns exactly one of those placeholders -- which covers
both direct function references and the `lambda env: self.robot_manager.get_angular_velocity()`
style of every reference example.  The resulting column table is what the kernels assemble rows
from (observation_manager.py:232-256); history frames are shifted inside the same kernel
(:223-226).  As in the reference, history is not cleared on reset.
"""
from __future__ import annotations

import numpy as np
import torch

from .._gs import gs
from ..spaces import Box
from .base import BaseManager
from .config import ObservationConfigItem


class UnsupportedTermError(NotImplementedError):
    """A term configuration the fused step cannot execute."""


class ObservationManager(BaseManager):
    def __init__(self, env, cfg: dict[str, dict], name: str = "policy", history_len: int | None = None, noise=None):
        super().__init__(env, "observation")
        self._name = name
        self.noise = noise
        self._observation_size = 1
        self._observation_space = None
        if history_len is not None and history_len < 1:
            raise ValueError("history_len must be greater than 0")
        self._history_len = history_len if history_len is not None else 1
        self.cfg: dict[str, ObservationConfigItem] = {k: ObservationConfigItem(c, env) for k, c in cfg.items()}
        self._sources: list[tuple[str, tuple, int]] = []  # per term: (name, source key, width)
        self._buffers: list[torch.Tensor] = []            # ping-pong (N, O*H) rows
        self._current = 0
        self._external_col0: dict[str, int] = {}          # user-defined terms: first column in the host-filled array
        # host-evaluated terms that are not user functions (body-frame terms without an entity_manager, terms of
        # a further EntityManager): never lowered into the kernel (FusedStep, fuse_user_observations)
        self._host_columns: set[str] = set()

    @property
    def name(self) -> str:
        return self._name

    @property
    def observation_space(self):
        return self._observation_space

    @property
    def frame_size(self) -> int:
        return sum(w for _, _, w in self._sources)

    def build(self):
        self._sources = []
        self._pending: list[str] = []
        self._host_columns = set()
        for name, cfg in self.cfg.items():
            cfg.build()
            assert callable(cfg.fn), f"Observation function {name} is not callable"
            try:
                key, width = self.env._trace_term(cfg.fn, dict(cfg.params), what=f"observation '{name}'")
            except UnsupportedTermError as e:
                # user-defined term: stays a Python callback, handed to the kernel as extra columns
                key, width = ("external", name), getattr(e, "width", None)
                if width is None:
                    self._pending.append(name)
                else:
                    self._host_columns.add(name)
            self._sources.append((name, key, width))
        if not self._pending:
            self._allocate()

    def resolve_external(self):
        """Evaluate pending user-defined terms once for their width (the reference's dry run,
        observation_manager.py:202-210), after the fused step's library handle exists."""
        if not self._pending:
            return
        for i, (name, key, width) in enumerate(self._sources):
            if name in self._pending:
                fused = self.env._fused
                fused.width_probe = fused.dry_run  # (a dry run cannot launch: shapes only)
                try:
                    value = self.cfg[name].fn(env=self.env, **self.cfg[name].params)
                finally:
                    fused.width_probe = False
                self._sources[i] = (name, key, int(value.reshape(self.env.num_envs, -1).shape[1]))
        self._pending = []
        self._allocate()

    def _allocate(self):
        single = self.frame_size
        self._observation_size = single * self._history_len
        self._observation_space = Box(low=-np.inf, high=np.inf, shape=(self._observation_size,), dtype=np.float32)
        shape = (self.env.num_envs, self._observation_size)
        self._buffers = [torch.zeros(shape, device=gs.device, dtype=gs.tc_float) for _ in range(2)]
        self._current = 0

    def columns(self) -> list[dict]:
        """One entry per output column of a frame: source key, column, live scale and noise."""
        cols = []
        for (name, key, width) in self._sources:
            cfg = self.cfg[name]
            scale = cfg.scale
            scale = 1.0 if scale is None else float(scale)
            noise = cfg.noise or self.noise  # observation_manager.py:247 (term noise 0.0 is falsy)
            noise = 0.0 if noise is None else float(noise)
            for c in range(width):
                cols.append({"key": key, "col": c, "scale": scale, "noise": noise})
        return cols

    def get_observations(self) -> torch.Tensor:
        """The rows assembled by the most recent fused step / reset."""
        return self._buffers[self._current]
