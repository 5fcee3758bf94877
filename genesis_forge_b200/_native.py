"""
ctypes binding of libgfb200.so (the C ABI declared in include/gfb200.h).

There is no CPU fallback: if the shared library is missing or was built for another ABI version,
importing this module's `lib()` raises with the build command to run.  Enum values and #define
constants are read from the header itself so the Python side cannot drift from the C side; struct
layouts are written out below and checked against `gfb_abi_sizeof()` when the library loads.
"""
from __future__ import annotations

import ctypes as C
import os
import re
from pathlib import Path

_PKG = Path(__file__).resolve().parent
HEADER = _PKG.parent / "include" / "gfb200.h"
LIB_PATH = _PKG / "libgfb200.so"


class NativeLibraryError(RuntimeError):
    pass


# ----------------------------------------------------------------------------------------------
# constants from the header
# ----------------------------------------------------------------------------------------------
def _parse_header(path: Path) -> dict[str, int]:
    text = path.read_text()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    consts: dict[str, int] = {}
    for name, value in re.findall(r"#define\s+(GFB_[A-Z0-9_]+)\s+([0-9]+)u?\b", text):
        consts[name] = int(value)
    for body in re.findall(r"typedef\s+enum\s*\{(.*?)\}\s*\w+\s*;", text, flags=re.S):
        nxt = 0
        for item in body.split(","):
            item = item.strip()
            if not item:
                continue
            if "=" in item:
                name, value = (x.strip() for x in item.split("="))
                nxt = int(value, 0)
            else:
                name = item
            consts[name] = nxt
            nxt += 1
    return consts


K = _parse_header(HEADER)
globals().update(K)  # GFB_B_POS, GFB_R_BASE_HEIGHT, GFB_PHASE_ALL, ...

MAX_DOFS = K["GFB_MAX_DOFS"]
MAX_REWARD = K["GFB_MAX_REWARD_TERMS"]
MAX_TERMINATION = K["GFB_MAX_TERMINATION_TERMS"]
MAX_COMMANDS = K["GFB_MAX_COMMANDS"]
MAX_COMMAND_DIMS = K["GFB_MAX_COMMAND_DIMS"]
MAX_CONTACT = K["GFB_MAX_CONTACT_MANAGERS"]
MAX_CONTACT_LINKS = K["GFB_MAX_CONTACT_LINKS"]
MAX_WITH_LINKS = K["GFB_MAX_WITH_LINKS"]
MAX_OBS_GROUPS = K["GFB_MAX_OBS_GROUPS"]
MAX_OBS_COLS = K["GFB_MAX_OBS_COLS"]
B_COUNT = K["GFB_B_COUNT"]


# ----------------------------------------------------------------------------------------------
# struct layouts (must match include/gfb200.h; verified against gfb_abi_sizeof at load)
# ----------------------------------------------------------------------------------------------
class RewardTerm(C.Structure):
    _fields_ = [
        ("op", C.c_int32), ("mgr", C.c_int32), ("flags", C.c_uint32), ("i0", C.c_int32),
        ("weight", C.c_float), ("p", C.c_float * 4), ("ext_col", C.c_int32),
    ]


class TerminationTerm(C.Structure):
    _fields_ = [
        ("op", C.c_int32), ("mgr", C.c_int32), ("time_out", C.c_int32), ("i0", C.c_int32),
        ("p", C.c_float * 4),
    ]


class CommandManagerDesc(C.Structure):
    _fields_ = [
        ("n_dims", C.c_int32), ("resample_steps", C.c_int32), ("enabled", C.c_int32), ("_pad", C.c_int32),
        ("lo", C.c_float * MAX_COMMAND_DIMS), ("hi", C.c_float * MAX_COMMAND_DIMS),
    ]


class ContactManagerDesc(C.Structure):
    _fields_ = [
        ("n_links", C.c_int32), ("n_with", C.c_int32), ("has_with_filter", C.c_int32),
        ("track_air_time", C.c_int32), ("air_time_threshold", C.c_float), ("scene_dt", C.c_float),
        ("disabled", C.c_int32), ("_pad", C.c_int32),
        ("link_ids", C.c_int32 * MAX_CONTACT_LINKS), ("local_link_ids", C.c_int32 * MAX_CONTACT_LINKS),
        ("with_ids", C.c_int32 * MAX_WITH_LINKS),
    ]


class ObsCol(C.Structure):
    _fields_ = [
        ("src", C.c_int32), ("mgr", C.c_int32), ("col", C.c_int32), ("scale", C.c_float), ("noise", C.c_float),
    ]


class ObsGroup(C.Structure):
    _fields_ = [("n_cols", C.c_int32), ("history", C.c_int32), ("col_begin", C.c_int32), ("user_id", C.c_int32)]


class ProgramHead(C.Structure):
    _fields_ = [
        ("num_envs", C.c_int32), ("num_dofs", C.c_int32), ("n_contact_slots", C.c_int32),
        ("n_links_total", C.c_int32), ("env_dt", C.c_float), ("base_max_episode_length", C.c_int32),
        ("max_len_random_span", C.c_float), ("rng_mode", C.c_int32),
        ("rng_seed", C.c_uint64), ("step_index", C.c_uint64),
        ("n_reward", C.c_int32), ("n_termination", C.c_int32), ("n_command", C.c_int32),
        ("n_contact", C.c_int32), ("n_obs_groups", C.c_int32), ("manager_flags", C.c_uint32),
        ("height_field_rows", C.c_int32), ("height_field_cols", C.c_int32),
        ("terrain_bounds", C.c_float * 4),
        ("action_mode", C.c_int32), ("_pad1", C.c_int32),
        ("action_scale", C.c_float * MAX_DOFS), ("action_offset", C.c_float * MAX_DOFS),
        ("action_clip_lo", C.c_float * MAX_DOFS), ("action_clip_hi", C.c_float * MAX_DOFS),
        ("default_dof_pos", C.c_float * MAX_DOFS),
        ("reward", RewardTerm * MAX_REWARD),
        ("termination", TerminationTerm * MAX_TERMINATION),
        ("command", CommandManagerDesc * MAX_COMMANDS),
        ("contact", ContactManagerDesc * MAX_CONTACT),
        ("obs_group", ObsGroup * MAX_OBS_GROUPS),
    ]


class Program(C.Structure):
    _fields_ = [("head", ProgramHead), ("obs_cols", ObsCol * MAX_OBS_COLS)]


class Buffers(C.Structure):
    _fields_ = [("buf", C.c_void_p * B_COUNT)]


class Spawn(C.Structure):
    _fields_ = [
        ("x_lo", C.c_float), ("x_span", C.c_float), ("y_lo", C.c_float), ("y_span", C.c_float),
        ("height_offset", C.c_float), ("flat_height", C.c_float), ("terrain_bounds", C.c_float * 4),
        ("height_field_rows", C.c_int32), ("height_field_cols", C.c_int32), ("with_rotation", C.c_int32),
        ("rot_mode", C.c_int32 * 3), ("rot_lo", C.c_float * 3), ("rot_hi", C.c_float * 3),
        ("rng_seed", C.c_uint64), ("rng_counter", C.c_uint64),
    ]


class Report(C.Structure):
    _fields_ = [
        ("n_reset", C.c_int32), ("status", C.c_uint32),
        ("termination_count", C.c_int32 * MAX_TERMINATION),
        ("global_n_reset", C.c_int64), ("global_termination_count", C.c_int64 * MAX_TERMINATION),
        ("seq", C.c_uint64), ("local_seq", C.c_uint64),
    ]


# ----------------------------------------------------------------------------------------------
# loading
# ----------------------------------------------------------------------------------------------
_LIB = None

EXPORTS = [
    "gfb_abi_version", "gfb_abi_sizeof", "gfb_create", "gfb_destroy", "gfb_last_error", "gfb_set_program",
    "gfb_action_step", "gfb_action_step_ring", "gfb_post_physics", "gfb_read_report", "gfb_read_report_local", "gfb_observe", "gfb_contact_forces",
    "gfb_rotate", "gfb_spawn_pose", "gfb_peer_export", "gfb_peer_connect", "gfb_peer_disconnect", "gfb_spec_describe", "gfb_spec_attach", "gfb_spec_stats",
    "gfb_profile_enable", "gfb_profile_read", "gfb_profile_read_aux", "gfb_launch_count",
    "gfb_post_physics_report", "gfb_reset_rows",
]


def build_command() -> str:
    return "python -m genesis_forge_b200.build_native"


def lib() -> C.CDLL:
    """Load libgfb200.so (once), set prototypes, verify the ABI.  Raises if it is not there."""
    global _LIB
    if _LIB is not None:
        return _LIB
    if not LIB_PATH.exists():
        raise NativeLibraryError(
            f"{LIB_PATH} not found. The manager step has no CPU fallback; build the CUDA library with "
            f"`{build_command()}` (needs nvcc)."
        )
    try:
        L = C.CDLL(str(LIB_PATH))
    except OSError as e:
        raise NativeLibraryError(f"cannot load {LIB_PATH}: {e}") from e

    vp, i32, u32, i64 = C.c_void_p, C.c_int32, C.c_uint32, C.c_int64
    fp = C.POINTER(C.c_float)
    L.gfb_abi_version.restype = C.c_int
    L.gfb_abi_sizeof.restype = i64
    L.gfb_abi_sizeof.argtypes = [i32]
    L.gfb_create.restype = C.c_int
    L.gfb_create.argtypes = [i32, i32, C.POINTER(vp)]
    L.gfb_destroy.restype = None
    L.gfb_destroy.argtypes = [vp]
    L.gfb_last_error.restype = C.c_char_p
    L.gfb_last_error.argtypes = [vp]
    L.gfb_set_program.restype = C.c_int
    L.gfb_set_program.argtypes = [vp, C.POINTER(Program)]
    L.gfb_action_step.restype = C.c_int
    L.gfb_action_step.argtypes = [vp, C.POINTER(Buffers), vp, vp, vp]
    L.gfb_action_step_ring.restype = C.c_int
    L.gfb_action_step_ring.argtypes = [vp, C.POINTER(Buffers), vp, vp, vp]
    L.gfb_post_physics.restype = C.c_int
    L.gfb_post_physics.argtypes = [vp, C.POINTER(Buffers), u32, vp]
    L.gfb_read_report.restype = C.c_int
    L.gfb_read_report.argtypes = [vp, C.POINTER(Report), vp]
    L.gfb_read_report_local.restype = C.c_int
    L.gfb_read_report_local.argtypes = [vp, C.POINTER(C.c_int32), vp]
    L.gfb_observe.restype = C.c_int
    L.gfb_observe.argtypes = [vp, C.POINTER(Buffers), vp, i32, vp]
    L.gfb_contact_forces.restype = C.c_int
    L.gfb_contact_forces.argtypes = [vp] + [vp] * 10 + [i32] * 6 + [vp]
    L.gfb_rotate.restype = C.c_int
    L.gfb_rotate.argtypes = [vp, vp, vp, vp, i32, i32, vp]
    L.gfb_spawn_pose.restype = C.c_int
    L.gfb_spawn_pose.argtypes = [vp, C.POINTER(Spawn), vp, i32, i32] + [vp] * 11 + [vp]
    L.gfb_peer_export.restype = C.c_int
    L.gfb_peer_export.argtypes = [vp, vp]
    L.gfb_peer_connect.restype = C.c_int
    L.gfb_peer_connect.argtypes = [vp, i32, i32, vp, i64]
    L.gfb_peer_disconnect.restype = C.c_int
    L.gfb_peer_disconnect.argtypes = [vp]
    L.gfb_spec_describe.restype = C.c_int
    L.gfb_spec_describe.argtypes = [vp, C.POINTER(Buffers), u32, vp, C.POINTER(i32), i32, C.POINTER(i32), C.POINTER(i32)]
    L.gfb_spec_attach.restype = C.c_int
    L.gfb_spec_attach.argtypes = [vp, C.c_char_p]
    L.gfb_spec_stats.restype = C.c_int
    L.gfb_spec_stats.argtypes = [vp, C.POINTER(i64), C.POINTER(i64), C.POINTER(i64)]
    L.gfb_profile_enable.restype = C.c_int
    L.gfb_profile_enable.argtypes = [vp, i32]
    L.gfb_profile_read.restype = C.c_int
    L.gfb_profile_read.argtypes = [vp, fp, C.POINTER(i32), fp, C.POINTER(i32)]
    L.gfb_profile_read_aux.restype = C.c_int
    L.gfb_profile_read_aux.argtypes = [vp, fp, C.POINTER(i32)]
    L.gfb_post_physics_report.restype = C.c_int
    L.gfb_post_physics_report.argtypes = [vp, C.POINTER(Buffers), u32, C.POINTER(Report), vp]
    L.gfb_reset_rows.restype = C.c_int
    L.gfb_reset_rows.argtypes = [vp, vp, i32, i32, i32, vp, C.c_float, C.c_float, vp, C.c_uint64, C.c_uint64, vp, vp, vp]
    L.gfb_launch_count.restype = i64
    L.gfb_launch_count.argtypes = [vp]

    if L.gfb_abi_version() != K["GFB_ABI_VERSION"]:
        raise NativeLibraryError(
            f"{LIB_PATH} has ABI version {L.gfb_abi_version()}, header says {K['GFB_ABI_VERSION']}; "
            f"rebuild with `{build_command()}`"
        )
    checks = [(0, Program), (1, Buffers), (2, Report), (3, ProgramHead), (5, Spawn)]
    for which, struct in checks:
        if L.gfb_abi_sizeof(which) != C.sizeof(struct):
            raise NativeLibraryError(
                f"ABI layout mismatch for {struct.__name__}: library {L.gfb_abi_sizeof(which)} bytes, "
                f"binding {C.sizeof(struct)} bytes"
            )
    if L.gfb_abi_sizeof(4) != B_COUNT:
        raise NativeLibraryError("ABI mismatch: GFB_B_COUNT")
    _LIB = L
    return L


def available() -> bool:
    return LIB_PATH.exists()


class Handle:
    """Owner of one gfb_handle; raises `NativeLibraryError` with the library's message on failure."""

    def __init__(self, num_envs: int, device_index: int):
        self._lib = lib()
        self._h = C.c_void_p()
        rc = self._lib.gfb_create(num_envs, device_index, C.byref(self._h))
        if rc != 0:
            msg = self._lib.gfb_last_error(self._h).decode() if self._h else f"status {rc}"
            if self._h:
                self._lib.gfb_destroy(self._h)
                self._h = C.c_void_p()
            raise NativeLibraryError(f"gfb_create failed: {msg}")

    def check(self, rc: int, what: str):
        if rc != 0:
            raise NativeLibraryError(f"{what} failed ({rc}): {self._lib.gfb_last_error(self._h).decode()}")

    @property
    def ptr(self):
        return self._h

    def close(self):
        if self._h:
            self._lib.gfb_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
