// libgfb200: C ABI + launch logic (see include/gfb200.h).
#include <cuda_runtime.h>
#include <dlfcn.h>

#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/gfb200.h"
#include "aux_kernels.cuh"
#include "plan.h"
#include "post_kernel.cuh"

using namespace gfb;

namespace {

constexpr int kMaxSmemBytes = 227 * 1024;
constexpr int kPlanSlots = 6;
constexpr int kEventPairs = 2048;
constexpr int kObserveTile = 32;  // (only sizes the unused slab of the observe-only plan)

inline int align4(int w) { return (w + 3) & ~3; }

struct PlanSlot {
  bool used = false;
  uint32_t phases = 0;
  int tile = 0;
  std::vector<int32_t> table_host;
  int32_t* table_dev = nullptr;
};

}  // namespace

// Host-side result of planning one launch.  The plan is a pure function of the term table, the
// phase set and, per buffer, whether it is present and 16-byte aligned -- so it is computed once
// and looked up by that key on every later step (planning costs 10-20 us, a launch 3-4 us).
struct BufferKey {
  uint64_t w[(2 * GFB_B_COUNT + 63) / 64];
  bool operator==(const BufferKey& o) const { return memcmp(w, o.w, sizeof(w)) == 0; }
};

inline BufferKey buffer_key(const gfb_buffers& b) {
  BufferKey k{};
  for (int i = 0; i < GFB_B_COUNT; ++i) {
    const uintptr_t p = reinterpret_cast<uintptr_t>(b.buf[i]);
    const uint64_t bits = (p ? 1u : 0u) | ((p & 15) == 0 ? 2u : 0u);
    k.w[(2 * i) >> 6] |= bits << ((2 * i) & 63);
  }
  return k;
}

struct LaunchCache {
  bool valid = false;
  uint64_t prog_epoch = 0, spec_gen = 0;
  uint32_t phases = 0;
  BufferKey key{};
  Plan plan;
  std::vector<int32_t> table;
  int tile = 0, n_stages = 1;
  int tma_ok = 0;
  int spec_index = -1;  // index into gfb_handle::specs, -1 = generic kernel
  int resident_blocks = 0;  // blocks of this kernel / shared-memory size that fit on the device at once
};
constexpr int kLaunchCaches = 8;

struct AttachedSpec {
  void* dl = nullptr;
  int (*launch)(const KParams*, int, unsigned, void*) = nullptr;
  int (*blocks_per_sm)(unsigned) = nullptr;
  // reset path of the lowered user-defined observation terms (spec_kernel.cu), if the library has them
  int (*user_observe)(const gfb_buffers*, int, const int64_t*, int, int, void*) = nullptr;
  uint32_t state_slots = 0;  // GFB_B_USER_STATE slots its lowered class-style terms use (bit i: slot i)
  int tile = 0;
  uint32_t phases = 0;
  gfb_program_head canon;
  Plan plan;
};

struct gfb_handle {
  std::vector<AttachedSpec> specs;
  int64_t n_spec_launches = 0, n_generic_launches = 0, n_user_observe_launches = 0;
  bool host_only = false;
  int device = 0;
  int num_envs = 0;
  std::string err;
  gfb_program prog;
  bool has_prog = false;
  Scratch scratch{};
  int scratch_tiles = 0;
  gfb_report* report_host = nullptr;  // pinned + mapped: the post-physics kernel writes the report into it
  uint32_t epoch = 0;                 // launches of the post-physics kernel so far
  uint64_t report_seq = 0;            // launches with the reset phase so far (= seq of the latest report)
  PlanSlot slots[kPlanSlots];
  PlanSlot observe_slot;
  uint64_t prog_epoch = 0;  // bumped when anything but the step index of the term table changes
  uint64_t spec_gen = 0;    // bumped by gfb_spec_attach
  LaunchCache post_cache[kLaunchCaches];
  int post_cache_next = 0;
  LaunchCache observe_cache;
  // logging exchange over peer memory (gfb_peer_*)
  PeerInbox* inbox_own = nullptr;
  PeerInbox* inbox[GFB_MAX_PEERS] = {};
  int peer_rank = 0, peer_world = 0;
  uint64_t peer_seq = 0;
  int64_t global_num_envs = 0;
  bool disable_tma = false;
  bool disable_overlay = false;  // GFB_NO_OVERLAY=1: load every staged array up front
  int force_tile = 0;
  uint32_t debug = 0;
  int num_sms = 0;
  int64_t launches = 0;
  // profiling
  bool profiling = false;
  std::vector<cudaEvent_t> ev_post, ev_action;
  std::vector<uint8_t> ev_post_obs_only;  // per event pair: the launch ran the observation phase alone
  int n_post = 0, n_action = 0;
  float post_ms = 0.f, action_ms = 0.f, post_obs_ms = 0.f;
  int post_count = 0, action_count = 0, post_obs_count = 0;
  // the small kernels: 0 index compaction, 1 observe (reset envs), 2 spawn, 3 lowered user observation terms
  std::vector<cudaEvent_t> ev_aux;
  std::vector<uint8_t> ev_aux_kind;
  int n_aux = 0;
  float aux_ms[4] = {0.f, 0.f, 0.f, 0.f};
  int aux_count[4] = {0, 0, 0, 0};
  int smem_attr_post[4] = {0, 0, 0, 0};
  int smem_attr_action[4] = {0, 0, 0, 0};
};

namespace {

int fail(gfb_handle* h, int code, const std::string& msg) {
  if (h) h->err = msg;
  return code;
}

#define CUDA_TRY(expr)                                                                                     \
  do {                                                                                                     \
    cudaError_t _e = (expr);                                                                               \
    if (_e != cudaSuccess)                                                                                 \
      return fail(h, GFB_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(_e));                    \
  } while (0)

// The structural part of a program head: every live value zeroed (see gfb_spec_describe).
void canonicalize(gfb_program_head& c) {
  c.num_envs = 0;
  c.env_dt = 0.f;
  c.base_max_episode_length = 0;
  c.max_len_random_span = 0.f;
  c.rng_seed = 0;
  c.step_index = 0;
  c.height_field_rows = c.height_field_cols = 0;
  memset(c.terrain_bounds, 0, sizeof(c.terrain_bounds));
  memset(c.action_scale, 0, sizeof(c.action_scale));
  memset(c.action_offset, 0, sizeof(c.action_offset));
  memset(c.action_clip_lo, 0, sizeof(c.action_clip_lo));
  memset(c.action_clip_hi, 0, sizeof(c.action_clip_hi));
  memset(c.default_dof_pos, 0, sizeof(c.default_dof_pos));
  for (auto& r : c.reward) {
    r.weight = 0.f;
    memset(r.p, 0, sizeof(r.p));
  }
  for (auto& t : c.termination) memset(t.p, 0, sizeof(t.p));
  for (auto& k : c.command) {
    k.resample_steps = 0;
    memset(k.lo, 0, sizeof(k.lo));
    memset(k.hi, 0, sizeof(k.hi));
  }
  for (auto& m : c.contact) {
    m.air_time_threshold = 0.f;
    m.scene_dt = 0.f;
  }
}

bool has_user_observations(const gfb_program_head& P) {
  for (int g = 0; g < P.n_obs_groups; ++g)
    if (P.obs_group[g].user_id != 0) return true;
  return false;
}

bool uses_user_terms(const gfb_program_head& P, uint32_t phases) {
  if ((phases & GFB_PHASE_OBSERVE) && has_user_observations(P)) return true;
  if (phases & GFB_PHASE_REWARD)
    for (int r = 0; r < P.n_reward; ++r)
      if (P.reward[r].op == GFB_R_USER && P.reward[r].weight != 0.0f) return true;
  if (phases & GFB_PHASE_TERMINATION)
    for (int t = 0; t < P.n_termination; ++t)
      if (P.termination[t].op == GFB_T_USER) return true;
  return false;
}

bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

int tile_index(int tile) { return tile == 32 ? 0 : (tile == 64 ? 1 : (tile == 128 ? 2 : 3)); }

// ---------------------------------------------------------------------------------------------
// term-table analysis: which derived vectors / staged slabs does the program need
// ---------------------------------------------------------------------------------------------
uint32_t compute_needs(const gfb_program& prog, uint32_t phases) {
  const gfb_program_head& P = prog.head;
  uint32_t needs = 0;
  if (phases & GFB_PHASE_REWARD)
    for (int r = 0; r < P.n_reward; ++r) {
      const gfb_reward_term& t = P.reward[r];
      if (t.weight == 0.0f) continue;
      switch (t.op) {
        case GFB_R_LIN_VEL_Z:
        case GFB_R_TRACK_LIN_VEL:
          needs |= NEED_LIN;
          break;
        case GFB_R_ANG_VEL_XY:
        case GFB_R_TRACK_ANG_VEL:
          needs |= NEED_ANG;
          break;
        case GFB_R_FLAT_ORIENTATION:
          needs |= NEED_GRAV;
          break;
        case GFB_R_BODY_ACC_EXP:
          needs |= NEED_LIN | NEED_ANG;
          break;
        case GFB_R_BASE_HEIGHT:
          needs |= NEED_POS;
          break;
        case GFB_R_DOF_SIMILAR:
        case GFB_R_STAND_STILL:
          needs |= NEED_DOF_POS;
          break;
        default:
          break;
      }
    }
  if (phases & GFB_PHASE_TERMINATION)
    for (int t = 0; t < P.n_termination; ++t) {
      switch (P.termination[t].op) {
        case GFB_T_BAD_ORIENTATION:
          needs |= NEED_GRAV;
          break;
        case GFB_T_BASE_HEIGHT_MIN:
        case GFB_T_OUT_OF_BOUNDS:
          needs |= NEED_POS;
          break;
        default:
          break;
      }
    }
  if (phases & GFB_PHASE_OBSERVE)
    for (int g = 0; g < P.n_obs_groups; ++g)
      for (int c = 0; c < P.obs_group[g].n_cols; ++c) {
        switch (prog.obs_cols[P.obs_group[g].col_begin + c].src) {
          case GFB_O_LIN_VEL_B:
            needs |= NEED_LIN;
            break;
          case GFB_O_ANG_VEL_B:
            needs |= NEED_ANG;
            break;
          case GFB_O_GRAVITY_B:
            needs |= NEED_GRAV;
            break;
          default:
            break;
        }
      }
  return needs;
}

// Lay out the shared-memory slab for one (program, phases, tile) combination and lower the
// observation columns to device descriptors.
// observe_only: the plan of gfb_observe, whose observe_kernel reads every column from global memory
int build_plan(gfb_handle* h, const gfb_buffers& b, uint32_t phases, int tile, int n_stages, Plan& plan,
               std::vector<int32_t>& table, bool observe_only = false) {
  std::vector<DevObsCol> cols;
  const gfb_program& prog = h->prog;
  const gfb_program_head& P = prog.head;
  memset(&plan, 0, sizeof(plan));
  plan.tile = tile;
  plan.needs = compute_needs(prog, phases);
  plan.off_pos = plan.off_quat = plan.off_vel = plan.off_ang = plan.off_dof_pos = -1;
  plan.off_cforce = plan.off_cpos = plan.off_cla = plan.off_clb = -1;
  for (int k = 0; k < GFB_MAX_COMMANDS; ++k) plan.off_cmd[k] = -1;
  int cursor = 0;
  auto stage = [&](int buf, int words, int store) -> int {
    if (plan.n_staged >= GFB_MAX_STAGED) return -1;
    const int i = plan.n_staged++;
    plan.staged_buf[i] = buf;
    plan.staged_words[i] = words;
    plan.staged_off[i] = cursor;
    plan.staged_store[i] = store;
    const int off = cursor;
    cursor = align4(cursor + words * tile);
    return off;
  };
  const bool entity = phases & GFB_PHASE_ENTITY;
  const bool contact = (phases & GFB_PHASE_CONTACT) && P.n_contact > 0;
  // ---- early group: what the entity and contact phases read ---------------------------------------
  if (entity) {
    if (!b.buf[GFB_B_QUAT]) return fail(h, GFB_ERR_INVALID, "GFB_B_QUAT is required for the entity phase");
    plan.off_quat = stage(GFB_B_QUAT, 4, GFB_B_BASE_QUAT);
  }
  if ((plan.needs & NEED_POS) || (entity && b.buf[GFB_B_BASE_POS])) {
    if (!b.buf[GFB_B_POS]) return fail(h, GFB_ERR_INVALID, "GFB_B_POS missing");
    plan.off_pos = stage(GFB_B_POS, 3, entity ? GFB_B_BASE_POS : -1);
  }
  if (plan.needs & NEED_LIN) {
    if (!b.buf[GFB_B_VEL]) return fail(h, GFB_ERR_INVALID, "GFB_B_VEL missing");
    plan.off_vel = stage(GFB_B_VEL, 3, -1);
  }
  if (plan.needs & NEED_ANG) {
    if (!b.buf[GFB_B_ANG]) return fail(h, GFB_ERR_INVALID, "GFB_B_ANG missing");
    plan.off_ang = stage(GFB_B_ANG, 3, -1);
  }
  plan.n_prefetch = plan.n_staged;  // everything staged so far: quat, pos, vel, ang
  int contact_begin = cursor, contact_end = cursor;
  if (contact) {
    for (int id : {GFB_B_C_FORCE, GFB_B_C_POS, GFB_B_C_LINK_A, GFB_B_C_LINK_B, GFB_B_LINKS_QUAT})
      if (!b.buf[id]) return fail(h, GFB_ERR_INVALID, "contact input buffer missing");
    const int C = P.n_contact_slots;
    plan.off_cforce = stage(GFB_B_C_FORCE, 3 * C, -1);
    plan.off_cpos = stage(GFB_B_C_POS, 3 * C, -1);
    plan.off_cla = stage(GFB_B_C_LINK_A, C, -1);
    plan.off_clb = stage(GFB_B_C_LINK_B, C, -1);
    contact_end = cursor;
  }
  // ---- late group: read by rewards / command resample / reset / observations only.  With contact
  // slots staged (single-stage kernel) these arrays are loaded after the contact phase into the
  // contact slots' shared memory; otherwise they simply follow the early arrays.
  const bool overlay = contact && n_stages == 1 && !h->disable_overlay;
  plan.n_early = plan.n_staged;
  if (overlay) cursor = contact_begin;
  if (plan.needs & NEED_DOF_POS) {
    if (!b.buf[GFB_B_DOF_POS]) return fail(h, GFB_ERR_INVALID, "GFB_B_DOF_POS missing");
    plan.off_dof_pos = stage(GFB_B_DOF_POS, P.num_dofs, -1);
  }
  if (phases & (GFB_PHASE_REWARD | GFB_PHASE_COMMAND | GFB_PHASE_RESET | GFB_PHASE_OBSERVE))
    for (int k = 0; k < P.n_command; ++k) {
      if (P.command[k].n_dims == 0) continue;  // a user-level manager without a command vector of its own
      if (!b.buf[GFB_B_COMMAND0 + k]) return fail(h, GFB_ERR_INVALID, "command buffer missing");
      plan.off_cmd[k] = stage(GFB_B_COMMAND0 + k, P.command[k].n_dims, -1);
    }
  // arrays that only the observation rows read (dof velocity / force, targets, raw actions) are
  // staged as well, so that the row assembly reads nothing but shared memory and every HBM read of
  // the slab is issued by the TMA engine
  int off_obs_src[GFB_B_COUNT];
  for (int i = 0; i < GFB_B_COUNT; ++i) off_obs_src[i] = -1;
  if (phases & GFB_PHASE_OBSERVE) {
    for (int g = 0; g < P.n_obs_groups; ++g)
      for (int c = 0; c < P.obs_group[g].n_cols; ++c) {
        int buf = -1;
        switch (prog.obs_cols[P.obs_group[g].col_begin + c].src) {
          case GFB_O_DOF_VEL: buf = GFB_B_DOF_VEL; break;
          case GFB_O_DOF_FORCE: buf = GFB_B_DOF_FORCE; break;
          case GFB_O_TARGETS: buf = GFB_B_TARGETS; break;
          case GFB_O_ENV_ACTIONS: buf = GFB_B_ENV_ACTIONS; break;
          case GFB_O_DOF_POS: buf = GFB_B_DOF_POS; break;
          case GFB_O_EXTERNAL: buf = GFB_B_OBS_EXT0; break;
          default: break;
        }
        if (buf < 0 || off_obs_src[buf] >= 0 || !b.buf[buf]) continue;
        if (buf == GFB_B_DOF_POS && plan.off_dof_pos >= 0) {
          off_obs_src[buf] = plan.off_dof_pos;
          continue;
        }
        // ENV_ACTIONS rows are zeroed for reset envs inside this kernel; staged copies would be stale
        if (buf == GFB_B_ENV_ACTIONS && (phases & GFB_PHASE_RESET)) continue;
        const int row_words = buf == GFB_B_OBS_EXT0 ? prog.obs_cols[P.obs_group[g].col_begin + c].mgr : P.num_dofs;
        off_obs_src[buf] = stage(buf, row_words, -1);
        if (buf == GFB_B_DOF_POS) plan.off_dof_pos = off_obs_src[buf];
      }
  }
  const bool stage_sums = (phases & (GFB_PHASE_REWARD | GFB_PHASE_RESET)) && P.n_reward > 0;
  if (overlay) {
    plan.sums_off = cursor;
    if (stage_sums) cursor = align4(cursor + P.n_reward * tile);
    plan.sums_late = stage_sums ? 1 : 0;
    if (plan.n_early == plan.n_staged && !stage_sums) plan.sums_late = 0;  // nothing is late
    cursor = std::max(cursor, contact_end);
  } else {
    plan.n_early = plan.n_staged;  // one group
  }
  // stash
  int stride = 9;
  for (int m = 0; m < P.n_contact; ++m) {
    plan.st_cnorm[m] = stride;
    stride += P.contact[m].n_links;
    plan.st_air[m] = stride;
    if (P.contact[m].track_air_time) stride += 4 * P.contact[m].n_links;
  }
  // the lowered user-defined observation terms' values (GFB_O_USER), written by the owner threads
  // (post_kernel.cuh: user_stash_base); `mgr` of such a column is the terms' total width
  const int st_user = stride;
  int user_words = 0;
  if ((phases & GFB_PHASE_OBSERVE) && !observe_only)
    for (int g = 0; g < P.n_obs_groups; ++g)
      for (int c = 0; c < P.obs_group[g].n_cols; ++c) {
        const gfb_obs_col& oc = prog.obs_cols[P.obs_group[g].col_begin + c];
        if (oc.src == GFB_O_USER) user_words = std::max(user_words, (int)oc.mgr);
      }
  stride += user_words;
  if ((stride & 1) == 0) ++stride;  // odd stride: conflict-free per-thread rows
  plan.stash_stride = stride;
  plan.stash_off = cursor;
  cursor = align4(cursor + stride * tile);
  if (!overlay) {
    plan.sums_off = cursor;
    if (stage_sums) cursor = align4(cursor + P.n_reward * tile);
  }
  for (int m = 0; m < P.n_contact; ++m) plan.cout_off[m] = plan.cposout_off[m] = -1;  // outputs are not staged

  // observation columns
  cols.clear();
  int n_cols_total = 0;
  for (int g = 0; g < P.n_obs_groups; ++g) n_cols_total = std::max(n_cols_total, P.obs_group[g].col_begin + P.obs_group[g].n_cols);
  if (n_cols_total > GFB_MAX_OBS_COLS) return fail(h, GFB_ERR_INVALID, "too many observation columns");
  cols.resize(n_cols_total);
  for (int i = 0; i < n_cols_total; ++i) {
    const gfb_obs_col& oc = prog.obs_cols[i];
    DevObsCol d{};
    d.scale = oc.scale;
    d.noise = oc.noise;
    d.col = oc.col;
    auto global_src = [&](int buf, int row_words) {
      d.kind = 2;
      d.gbuf = buf;
      d.row_words = row_words;
      if (off_obs_src[buf] >= 0) {
        d.kind = 1;
        d.a = off_obs_src[buf];
      }
    };
    switch (oc.src) {
      case GFB_O_COMMAND:
        if (oc.mgr < 0 || oc.mgr >= P.n_command) return fail(h, GFB_ERR_INVALID, "obs: bad command manager");
        global_src(GFB_B_COMMAND0 + oc.mgr, P.command[oc.mgr].n_dims);
        if (plan.off_cmd[oc.mgr] >= 0) {
          d.kind = 1;
          d.a = plan.off_cmd[oc.mgr];
        }
        break;
      case GFB_O_ANG_VEL_B:
        d.kind = 3; d.a = 0 + oc.col;
        break;
      case GFB_O_LIN_VEL_B:
        d.kind = 3; d.a = 3 + oc.col;
        break;
      case GFB_O_GRAVITY_B:
        d.kind = 3; d.a = 6 + oc.col;
        break;
      case GFB_O_DOF_POS:
        global_src(GFB_B_DOF_POS, P.num_dofs);
        if (plan.off_dof_pos >= 0) {
          d.kind = 1;
          d.a = plan.off_dof_pos;
        }
        break;
      case GFB_O_DOF_VEL:
        global_src(GFB_B_DOF_VEL, P.num_dofs);
        break;
      case GFB_O_DOF_FORCE:
        global_src(GFB_B_DOF_FORCE, P.num_dofs);
        break;
      case GFB_O_TARGETS:
        global_src(GFB_B_TARGETS, P.num_dofs);
        break;
      case GFB_O_ENV_ACTIONS:
        global_src(GFB_B_ENV_ACTIONS, P.num_dofs);
        break;
      case GFB_O_CONTACT_NORM:
        if (oc.mgr < 0 || oc.mgr >= P.n_contact) return fail(h, GFB_ERR_INVALID, "obs: bad contact manager");
        d.kind = 3;
        d.a = plan.st_cnorm[oc.mgr] + oc.col;
        break;
      case GFB_O_EXTERNAL:
        if (oc.mgr <= 0) return fail(h, GFB_ERR_INVALID, "obs: external column needs its array width in mgr");
        global_src(GFB_B_OBS_EXT0, oc.mgr);
        break;
      case GFB_O_USER:
        if (oc.mgr <= 0 || oc.col < 0 || oc.col >= oc.mgr)
          return fail(h, GFB_ERR_INVALID, "obs: user column needs the terms' width in mgr and col < mgr");
        if (observe_only) {
          global_src(GFB_B_OBS_EXT1, oc.mgr);  // written by the specialised library's user_observe
        } else {
          d.kind = 3;
          d.a = st_user + oc.col;
        }
        break;
      case GFB_O_ZERO:
        d.kind = 0;
        break;
      default:
        return fail(h, GFB_ERR_UNSUPPORTED, "obs: unsupported column source");
    }
    if ((d.kind == 2 || d.kind == 1) && (phases & GFB_PHASE_OBSERVE) && !b.buf[d.gbuf])
      return fail(h, GFB_ERR_INVALID, "obs: source buffer " + std::to_string(d.gbuf) + " is NULL");
    cols[i] = d;
  }
  // mark 4-aligned runs that can move as one 16-byte piece
  for (int g = 0; g < P.n_obs_groups; ++g) {
    const gfb_obs_group& og = P.obs_group[g];
    if (og.n_cols & 3) continue;
    for (int c = 0; c + 3 < og.n_cols; c += 4) {
      DevObsCol* d = &cols[og.col_begin + c];
      bool ok = (d[0].kind == 1 || d[0].kind == 2) && (d[0].col & 3) == 0 && (d[0].row_words & 3) == 0;
      if (d[0].kind == 1) ok = ok && (d[0].a & 3) == 0;
      for (int j = 1; j < 4 && ok; ++j)
        ok = d[j].kind == d[0].kind && d[j].a == d[0].a && d[j].gbuf == d[0].gbuf &&
             d[j].row_words == d[0].row_words && d[j].col == d[0].col + j && d[j].scale == d[0].scale &&
             d[j].noise == d[0].noise;
      if (ok && d[0].kind == 2) ok = aligned16(b.buf[d[0].gbuf]);
      d[0].vec = ok ? 1 : 0;
    }
  }
  plan.n_cols_total = n_cols_total;

  // 16-byte group path.  Each frame-0 group of 4 columns is either an aligned contiguous run of one
  // staged array ("run": one 16-byte shared load) or 4 independent shared sources ("mixed").  The
  // two kinds are assembled in separate, warp-uniform passes; history pieces are a third pass.
  struct Group { int32_t off[4], stride[4]; float scale[4], noise[4]; int32_t c4; };
  std::vector<Group> runs, mixed;
  for (int g = 0; g < P.n_obs_groups; ++g) {
    const gfb_obs_group& og = P.obs_group[g];
    plan.grp_run_begin[g] = plan.grp_mixed_begin[g] = -1;
    plan.grp_run_count[g] = plan.grp_mixed_count[g] = 0;
    if ((og.n_cols & 3) || !(phases & GFB_PHASE_OBSERVE)) continue;
    if ((og.n_cols >> 2) > tile) continue;  // a sweep needs at least one whole row per pass
    bool all_shared = true;
    for (int c = 0; c < og.n_cols; ++c) all_shared = all_shared && cols[og.col_begin + c].kind != 2;
    if (!all_shared) continue;  // some source lives in global memory: per-element path
    plan.grp_run_begin[g] = (int)runs.size();
    plan.grp_mixed_begin[g] = (int)mixed.size();
    for (int c = 0; c < og.n_cols; c += 4) {
      const DevObsCol* d = &cols[og.col_begin + c];
      Group G{};
      G.c4 = c >> 2;
      for (int j = 0; j < 4; ++j) {
        G.scale[j] = d[j].scale;
        G.noise[j] = d[j].noise;
        if (d[j].kind == 1) {
          G.off[j] = d[j].a + d[j].col;
          G.stride[j] = d[j].row_words;
        } else if (d[j].kind == 3) {
          G.off[j] = plan.stash_off + d[j].a;
          G.stride[j] = plan.stash_stride;
        } else {  // constant zero column
          G.off[j] = plan.stash_off;
          G.stride[j] = 0;
          G.scale[j] = 0.0f;
        }
      }
      (d[0].vec ? runs : mixed).push_back(G);
    }
    plan.grp_run_count[g] = (int)runs.size() - plan.grp_run_begin[g];
    plan.grp_mixed_count[g] = (int)mixed.size() - plan.grp_mixed_begin[g];
  }

  // descriptor table: [DevObsCol x n_cols][runs: off stride scale noise[4] c4][mixed SoA], 16-byte padded
  table.clear();
  auto push_words = [&](const void* p, size_t bytes) {
    const int32_t* w = static_cast<const int32_t*>(p);
    table.insert(table.end(), w, w + bytes / 4);
  };
  auto push_f = [&](float f) { int32_t w; memcpy(&w, &f, 4); table.push_back(w); };
  auto pad4 = [&]() { while (table.size() & 3) table.push_back(0); };
  bool need_cols = false;  // the per-column table is only read by the per-element path
  for (int g = 0; g < P.n_obs_groups; ++g) need_cols = need_cols || plan.grp_run_begin[g] < 0;
  if (!(phases & GFB_PHASE_OBSERVE)) need_cols = false;
  if (phases == GFB_PHASE_OBSERVE) need_cols = true;  // observe_kernel reads it
  if (need_cols && !cols.empty()) push_words(cols.data(), cols.size() * sizeof(DevObsCol));
  pad4();
  // runs: per group {off, stride, c4, scale} as int4, then noise float4
  plan.run_off = (int)table.size();
  plan.n_runs = (int)runs.size();
  for (const auto& G : runs) {
    table.push_back(G.off[0]);
    table.push_back(G.stride[0]);
    table.push_back(G.c4);
    push_f(G.scale[0]);
  }
  for (const auto& G : runs) for (int j = 0; j < 4; ++j) push_f(G.noise[j]);
  // mixed: off int4, stride int4, scale float4, noise float4, c4
  plan.mixed_off = (int)table.size();
  plan.n_mixed = (int)mixed.size();
  for (const auto& G : mixed) for (int j = 0; j < 4; ++j) table.push_back(G.off[j]);
  for (const auto& G : mixed) for (int j = 0; j < 4; ++j) table.push_back(G.stride[j]);
  for (const auto& G : mixed) for (int j = 0; j < 4; ++j) push_f(G.scale[j]);
  for (const auto& G : mixed) for (int j = 0; j < 4; ++j) push_f(G.noise[j]);
  for (const auto& G : mixed) table.push_back(G.c4);
  pad4();
  plan.table_words = (int)table.size();
  // ring layout: [stage 0][stage 1][descriptor table]; offsets above are relative to a stage base
  plan.stage_words = (cursor + 31) & ~31;
  plan.n_stages = n_stages;
  plan.cols_off = plan.stage_words * n_stages;
  // behind the table: the reward terms' exact sums of a RESET launch, 160 bytes a term (post_kernel.cuh)
  plan.rew_acc_off = plan.cols_off + align4(plan.table_words);
  const bool reward_log = h->prog.head.n_reward > 0 && !(h->prog.head.manager_flags & GFB_MF_REWARD_DISABLED);
  const int acc_words = (phases & GFB_PHASE_RESET) && reward_log ? h->prog.head.n_reward * XS_WORDS * 4 : 0;
  plan.smem_words = plan.rew_acc_off + acc_words;
  if (const char* pad = getenv("GFB_PAD_SMEM_KB"))  // occupancy experiments: unused shared memory per block
    plan.smem_words += atoi(pad) * 256;
  return GFB_OK;
}

bool tma_eligible(const gfb_handle* h, const gfb_buffers& b, const Plan& plan, uint32_t phases) {
  if (h->disable_tma) return false;
  const gfb_program_head& P = h->prog.head;
  if (P.num_envs & 3) return false;
  for (int i = 0; i < plan.n_staged; ++i) {
    if (!aligned16(b.buf[plan.staged_buf[i]])) return false;
    if ((phases & GFB_PHASE_ENTITY) && plan.staged_store[i] >= 0 && b.buf[plan.staged_store[i]] &&
        !aligned16(b.buf[plan.staged_store[i]]))
      return false;
  }
  if ((phases & (GFB_PHASE_REWARD | GFB_PHASE_RESET)) && P.n_reward > 0 && !aligned16(b.buf[GFB_B_EP_SUMS])) return false;
  if ((phases & GFB_PHASE_CONTACT))
    for (int m = 0; m < P.n_contact; ++m)
      if (!aligned16(b.buf[GFB_B_CONTACTS0 + m]) || !aligned16(b.buf[GFB_B_CONTACT_POS0 + m])) return false;
  return true;
}

// profiling bracket of an auxiliary kernel: records the start event, returns the end event (or null)
cudaEvent_t aux_begin(gfb_handle* h, int kind, cudaStream_t stream) {
  if (!h->profiling || h->n_aux + 2 > (int)h->ev_aux.size()) return nullptr;
  h->ev_aux_kind[h->n_aux / 2] = (uint8_t)kind;
  cudaEvent_t e0 = h->ev_aux[h->n_aux++];
  cudaEvent_t e1 = h->ev_aux[h->n_aux++];
  cudaEventRecord(e0, stream);
  return e1;
}

int choose_tile(const gfb_handle* h) {
  if (h->force_tile == 32 || h->force_tile == 64 || h->force_tile == 128 || h->force_tile == 256) return h->force_tile;
  return h->num_envs >= 32768 ? 128 : 32;
}

// Slab size for a launch: shrink the slab until it fits comfortably.  (n_stages stays 1: the two-stage
// ring of round 1 was measured slower on B200 -- only 3 blocks fit per SM -- and has been removed from
// the kernel; the plan keeps the field for the layout arithmetic.)
int plan_for_launch(gfb_handle* h, const gfb_buffers& b, uint32_t phases, Plan& plan, std::vector<int32_t>& table,
                    int& tile, int& n_stages) {
  tile = choose_tile(h);
  n_stages = 1;
  if (h->force_tile == 0 && tile == 128 && n_stages == 1) {
    // big slabs (contact slots staged): pick the slab size that keeps the most warps resident
    // (shared memory per block vs. the 80-register limit of 6 x 128 threads).  Ties go to the larger
    // slab, except between 128 and 64 when contact slots are staged: those kernels run longer per
    // slab and the finer grain balances the SMs better at mid batch sizes (config 5 at 262144 envs:
    // 78 vs 86 us; no difference at 1M)
    const bool contact_slots = (phases & GFB_PHASE_CONTACT) && h->prog.head.n_contact > 0;
    int best_tile = 128, best_warps = -1;
    for (int t : {128, 64, 32}) {
      int rc = build_plan(h, b, phases, t, 1, plan, table);
      if (rc != GFB_OK) return rc;
      const size_t bytes = (size_t)plan.smem_words * 4 + 2048;
      if (bytes > (size_t)kMaxSmemBytes) continue;
      const int by_smem = (int)((size_t)(228 * 1024) / bytes);
      const int by_regs = 768 / t;
      const int warps = std::min(std::min(by_smem, by_regs), 32) * (t / 32);
      if (warps > best_warps || (warps == best_warps && t == 64 && best_tile == 128 && contact_slots)) {
        best_warps = warps;
        best_tile = t;
      }
    }
    tile = best_tile;
  }
  for (;;) {
    int rc = build_plan(h, b, phases, tile, n_stages, plan, table);
    if (rc != GFB_OK) return rc;
    if ((size_t)plan.smem_words * 4 <= (size_t)kMaxSmemBytes / 2) break;
    if (tile > 32) tile /= 2;
    else if (n_stages == 2) n_stages = 1;
    else break;
  }
  if ((size_t)plan.smem_words * 4 > (size_t)kMaxSmemBytes)
    return fail(h, GFB_ERR_UNSUPPORTED, "slab does not fit in shared memory");
  return GFB_OK;
}

template <int TILE>
int launch_post(gfb_handle* h, const KParams& kp, size_t smem, cudaStream_t stream, int grid) {
  int& cur = h->smem_attr_post[tile_index(TILE)];
  if ((int)smem > 44 * 1024 /* static shared memory counts towards the 48 KB default */ && (int)smem > cur) {
    CUDA_TRY(cudaFuncSetAttribute(post_kernel<TILE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    cur = (int)smem;
  }
  post_kernel<TILE><<<grid, TILE, smem, stream>>>(kp);
  CUDA_TRY(cudaGetLastError());
  return GFB_OK;
}

template <int TILE>
int blocks_per_sm(gfb_handle* h, size_t smem) {
  int& cur = h->smem_attr_post[tile_index(TILE)];
  if ((int)smem > 44 * 1024 /* static shared memory counts towards the 48 KB default */ && (int)smem > cur) {
    if (cudaFuncSetAttribute(post_kernel<TILE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) == cudaSuccess)
      cur = (int)smem;
  }
  int n = 0;
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, post_kernel<TILE>, TILE, smem) != cudaSuccess) n = 0;
  return n;
}

template <int TILE>
int launch_action(gfb_handle* h, const ActionParams& ap, size_t smem, cudaStream_t stream, int grid) {
  int& cur = h->smem_attr_action[tile_index(TILE)];
  if ((int)smem > 44 * 1024 /* static shared memory counts towards the 48 KB default */ && (int)smem > cur) {
    CUDA_TRY(cudaFuncSetAttribute(action_kernel<TILE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    cur = (int)smem;
  }
  action_kernel<TILE><<<grid, TILE, smem, stream>>>(ap);
  CUDA_TRY(cudaGetLastError());
  return GFB_OK;
}

constexpr size_t kTableCapacityBytes = GFB_MAX_OBS_COLS * sizeof(DevObsCol) + (GFB_MAX_OBS_COLS / 4) * 17 * 4 + 64;

int upload_table(gfb_handle* h, PlanSlot& slot, const std::vector<int32_t>& table, cudaStream_t stream) {
  const size_t bytes = table.size() * sizeof(int32_t);
  if (bytes > kTableCapacityBytes) return fail(h, GFB_ERR_INVALID, "descriptor table too large");
  if (!slot.table_dev) CUDA_TRY(cudaMalloc(&slot.table_dev, kTableCapacityBytes));
  if (slot.table_host.size() != table.size() || (bytes && memcmp(slot.table_host.data(), table.data(), bytes) != 0)) {
    slot.table_host = table;
    if (bytes)
      CUDA_TRY(cudaMemcpyAsync(slot.table_dev, slot.table_host.data(), bytes, cudaMemcpyHostToDevice, stream));
  }
  return GFB_OK;
}

}  // namespace

// =============================================================================================
// C ABI
// =============================================================================================
extern "C" {

int gfb_abi_version(void) { return GFB_ABI_VERSION; }

int64_t gfb_abi_sizeof(int32_t which) {
  switch (which) {
    case 0: return (int64_t)sizeof(gfb_program);
    case 1: return (int64_t)sizeof(gfb_buffers);
    case 2: return (int64_t)sizeof(gfb_report);
    case 3: return (int64_t)sizeof(gfb_program_head);
    case 4: return (int64_t)GFB_B_COUNT;
    case 5: return (int64_t)sizeof(gfb_spawn);
    default: return -1;
  }
}

const char* gfb_last_error(const gfb_handle* h) { return h ? h->err.c_str() : "null handle"; }

int gfb_create(int32_t num_envs, int32_t device, gfb_handle** out) {
  if (!out || num_envs <= 0) return GFB_ERR_INVALID;
  *out = nullptr;
  if (device < 0) {  // host-only handle: term-table packing and specialisation descriptions
    gfb_handle* hh = new gfb_handle();
    hh->host_only = true;
    hh->device = -1;
    hh->num_envs = num_envs;
    const char* env_t = getenv("GFB_TILE");
    hh->force_tile = env_t ? atoi(env_t) : 0;
    const char* env_o = getenv("GFB_NO_OVERLAY");
    hh->disable_overlay = env_o && env_o[0] == '1';
    *out = hh;
    return GFB_OK;
  }
  int count = 0;
  if (cudaGetDeviceCount(&count) != cudaSuccess || count <= 0 || device >= count) return GFB_ERR_NO_DEVICE;
  gfb_handle* h = new gfb_handle();
  h->device = device;
  h->num_envs = num_envs;
  *out = h;  // returned even on failure so that gfb_last_error() works; caller destroys it
  CUDA_TRY(cudaSetDevice(device));
  const int nt = (num_envs + 31) / 32;
  h->scratch_tiles = nt;
  CUDA_TRY(cudaMalloc(&h->scratch.tile_bits, (size_t)(nt + 8) * sizeof(uint32_t)));  // (+ the tail slab's padding)
  CUDA_TRY(cudaMemset(h->scratch.tile_bits, 0, (size_t)(nt + 8) * sizeof(uint32_t)));
  CUDA_TRY(cudaMalloc(&h->scratch.term_count, GFB_MAX_TERMINATION_TERMS * sizeof(int32_t)));
  CUDA_TRY(cudaMalloc(&h->scratch.rew_acc, GFB_MAX_REWARD_TERMS * XS_WORDS * sizeof(unsigned long long)));
  CUDA_TRY(cudaMalloc(&h->scratch.rew_flags, GFB_MAX_REWARD_TERMS * sizeof(uint32_t)));
  CUDA_TRY(cudaMalloc(&h->scratch.counters, CTR_COUNT * sizeof(uint32_t)));
  CUDA_TRY(cudaMalloc(&h->scratch.status, sizeof(uint32_t)));
  CUDA_TRY(cudaMemset(h->scratch.term_count, 0, GFB_MAX_TERMINATION_TERMS * sizeof(int32_t)));
  CUDA_TRY(cudaMemset(h->scratch.rew_acc, 0, GFB_MAX_REWARD_TERMS * XS_WORDS * sizeof(unsigned long long)));
  CUDA_TRY(cudaMemset(h->scratch.rew_flags, 0, GFB_MAX_REWARD_TERMS * sizeof(uint32_t)));
  CUDA_TRY(cudaMemset(h->scratch.counters, 0, CTR_COUNT * sizeof(uint32_t)));
  CUDA_TRY(cudaMemset(h->scratch.status, 0, sizeof(uint32_t)));
  CUDA_TRY(cudaHostAlloc(&h->report_host, sizeof(gfb_report), cudaHostAllocMapped));
  memset(h->report_host, 0, sizeof(gfb_report));
  CUDA_TRY(cudaHostGetDevicePointer(reinterpret_cast<void**>(&h->scratch.report_host), h->report_host, 0));
  const char* env = getenv("GFB_DISABLE_TMA");
  h->disable_tma = env && env[0] == '1';
  env = getenv("GFB_NO_OVERLAY");
  h->disable_overlay = env && env[0] == '1';
  env = getenv("GFB_TILE");
  h->force_tile = env ? atoi(env) : 0;
  env = getenv("GFB_DEBUG");
  h->debug = env ? (uint32_t)atoi(env) : 0u;
  cudaDeviceGetAttribute(&h->num_sms, cudaDevAttrMultiProcessorCount, device);
  return GFB_OK;
}

void gfb_destroy(gfb_handle* h) {
  if (!h) return;
  for (auto& sp : h->specs)
    if (sp.dl) dlclose(sp.dl);
  if (h->host_only) {
    delete h;
    return;
  }
  cudaSetDevice(h->device);
  cudaFree(h->scratch.tile_bits);
  cudaFree(h->scratch.term_count);
  cudaFree(h->scratch.rew_acc);
  cudaFree(h->scratch.rew_flags);
  cudaFree(h->scratch.counters);
  cudaFree(h->scratch.status);
  if (h->report_host) cudaFreeHost(h->report_host);
  gfb_peer_disconnect(h);
  if (h->inbox_own) cudaFree(h->inbox_own);
  for (auto& s : h->slots)
    if (s.table_dev) cudaFree(s.table_dev);
  if (h->observe_slot.table_dev) cudaFree(h->observe_slot.table_dev);
  for (auto e : h->ev_aux) cudaEventDestroy(e);
  for (auto e : h->ev_post) cudaEventDestroy(e);
  for (auto e : h->ev_action) cudaEventDestroy(e);
  delete h;
}

int gfb_set_program(gfb_handle* h, const gfb_program* program) {
  if (!h || !program) return GFB_ERR_INVALID;
  const gfb_program_head& P = program->head;
  if (h->has_prog) {
    // the usual per-step call: nothing but the step index moved -> no validation, plans stay cached
    h->prog.head.step_index = P.step_index;
    if (memcmp(&h->prog, program, sizeof(gfb_program)) == 0) return GFB_OK;
  }
  if (P.num_envs != h->num_envs) return fail(h, GFB_ERR_INVALID, "program.num_envs differs from the handle's");
  if (P.num_dofs < 0 || P.num_dofs > GFB_MAX_DOFS) return fail(h, GFB_ERR_INVALID, "num_dofs out of range");
  if (P.n_reward < 0 || P.n_reward > GFB_MAX_REWARD_TERMS) return fail(h, GFB_ERR_INVALID, "n_reward out of range");
  if (P.n_termination < 0 || P.n_termination > GFB_MAX_TERMINATION_TERMS)
    return fail(h, GFB_ERR_INVALID, "n_termination out of range");
  if (P.n_command < 0 || P.n_command > GFB_MAX_COMMANDS) return fail(h, GFB_ERR_INVALID, "n_command out of range");
  if (P.n_contact < 0 || P.n_contact > GFB_MAX_CONTACT_MANAGERS) return fail(h, GFB_ERR_INVALID, "n_contact out of range");
  if (P.n_obs_groups < 0 || P.n_obs_groups > GFB_MAX_OBS_GROUPS) return fail(h, GFB_ERR_INVALID, "n_obs_groups out of range");
  for (int k = 0; k < P.n_command; ++k) {
    if (P.command[k].n_dims < 0 || P.command[k].n_dims > GFB_MAX_COMMAND_DIMS ||
        (P.command[k].n_dims == 0 && P.command[k].enabled))
      return fail(h, GFB_ERR_INVALID, "command n_dims out of range");
    if (P.command[k].enabled && P.command[k].resample_steps <= 0)
      return fail(h, GFB_ERR_INVALID, "command resample_steps must be positive");
  }
  for (int m = 0; m < P.n_contact; ++m) {
    if (P.contact[m].n_links <= 0 || P.contact[m].n_links > GFB_MAX_CONTACT_LINKS)
      return fail(h, GFB_ERR_INVALID, "contact n_links out of range");
    if (P.contact[m].n_with < 0 || P.contact[m].n_with > GFB_MAX_WITH_LINKS)
      return fail(h, GFB_ERR_INVALID, "contact n_with out of range");
    for (int t = 0; t < P.contact[m].n_links; ++t)
      if (P.contact[m].link_ids[t] < 0 || P.contact[m].link_ids[t] >= P.n_links_total)
        return fail(h, GFB_ERR_INVALID, "contact link id outside [0, n_links_total)");
  }
  for (int g = 0; g < P.n_obs_groups; ++g)
    if (P.obs_group[g].n_cols <= 0 || P.obs_group[g].history < 1 ||
        P.obs_group[g].col_begin + P.obs_group[g].n_cols > GFB_MAX_OBS_COLS)
      return fail(h, GFB_ERR_INVALID, "observation group out of range");
  for (int r = 0; r < P.n_reward; ++r) {
    const gfb_reward_term& t = P.reward[r];
    const bool contact_op = t.op == GFB_R_HAS_CONTACT || t.op == GFB_R_CONTACT_FORCE ||
                            t.op == GFB_R_FEET_AIR_TIME || t.op == GFB_R_FEET_SLIDE;
    if (contact_op && (t.mgr < 0 || t.mgr >= P.n_contact)) return fail(h, GFB_ERR_INVALID, "reward: bad contact manager");
    if (t.op == GFB_R_FEET_AIR_TIME && !P.contact[t.mgr].track_air_time)
      return fail(h, GFB_ERR_INVALID, "feet_air_time needs a contact manager with track_air_time");
    const bool cmd_op = t.op == GFB_R_STAND_STILL ||
                        ((t.op == GFB_R_TRACK_LIN_VEL || t.op == GFB_R_TRACK_ANG_VEL) && !(t.flags & GFB_RF_FIXED_COMMAND)) ||
                        (t.op == GFB_R_BASE_HEIGHT && (t.flags & GFB_RF_TARGET_FROM_COMMAND));
    if (cmd_op && (t.mgr < 0 || t.mgr >= P.n_command)) return fail(h, GFB_ERR_INVALID, "reward: bad command manager");
    if (t.op == GFB_R_FEET_AIR_TIME && t.i0 >= P.n_command) return fail(h, GFB_ERR_INVALID, "feet_air_time: bad command manager");

  }
  for (int t = 0; t < P.n_termination; ++t) {
    const gfb_termination_term& tt = P.termination[t];
    const bool contact_op = tt.op == GFB_T_HAS_CONTACT || tt.op == GFB_T_CONTACT_FORCE || tt.op == GFB_T_CONTACT_FORCE_GRACE;
    if (contact_op && (tt.mgr < 0 || tt.mgr >= P.n_contact)) return fail(h, GFB_ERR_INVALID, "termination: bad contact manager");

  }
  h->prog = *program;
  h->has_prog = true;
  h->prog_epoch += 1;
  return GFB_OK;
}

static int action_step_impl(gfb_handle* h, const gfb_buffers* b, const float* raw_env, const float* raw_mgr,
                            void* stream_, int ring) {
  if (!h || !b || !raw_env) return GFB_ERR_INVALID;
  if (h->host_only) return fail(h, GFB_ERR_NO_DEVICE, "host-only handle cannot launch kernels");
  if (!h->has_prog) return fail(h, GFB_ERR_INVALID, "gfb_set_program() first");
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  const gfb_program_head& P = h->prog.head;
  if (!raw_mgr) raw_mgr = raw_env;
  ActionParams ap{};
  ap.num_envs = P.num_envs;
  ap.num_dofs = P.num_dofs;
  ap.action_mode = P.action_mode;
  memcpy(ap.action_scale, P.action_scale, sizeof(ap.action_scale));
  memcpy(ap.action_offset, P.action_offset, sizeof(ap.action_offset));
  memcpy(ap.action_clip_lo, P.action_clip_lo, sizeof(ap.action_clip_lo));
  memcpy(ap.action_clip_hi, P.action_clip_hi, sizeof(ap.action_clip_hi));
  ap.raw_env = raw_env;
  ap.raw_mgr = raw_mgr;
  ap.env_actions = static_cast<float*>(b->buf[GFB_B_ENV_ACTIONS]);
  ap.env_last_actions = static_cast<float*>(b->buf[GFB_B_ENV_LAST_ACTIONS]);
  ap.targets = static_cast<float*>(b->buf[GFB_B_TARGETS]);
  ap.action_rate = static_cast<float*>(b->buf[GFB_B_ACTION_RATE]);
  ap.episode_length = static_cast<int32_t*>(b->buf[GFB_B_EPISODE_LENGTH]);
  ap.status = h->scratch.status;
  ap.check_finite = P.action_mode == 2 ? 0 : 1;  // position_within_limits.py:113-131 overrides the checks away
  ap.ring = ring;
  if (!ap.env_actions || !ap.env_last_actions) return fail(h, GFB_ERR_INVALID, "env action buffers missing");
  if (P.action_mode != 0 && !ap.targets) return fail(h, GFB_ERR_INVALID, "GFB_B_TARGETS missing");
  int tile = choose_tile(h);
  if (const char* at = getenv("GFB_ACTION_TILE")) {  // experiments: slab size of the action kernel alone
    const int t = atoi(at);
    if (t == 32 || t == 64 || t == 128 || t == 256) tile = t;
  }
  const int D = P.num_dofs;
  ap.tma_ok = !h->disable_tma && ((tile * D) % 4 == 0) && aligned16(raw_env) && aligned16(raw_mgr) &&
              aligned16(ap.env_actions) && aligned16(ap.env_last_actions) && (!ap.targets || aligned16(ap.targets));
  // raw, previous, targets (+ the delayed raw slab only with a delay FIFO): fewer bytes per block = more
  // blocks -- and more bytes in flight -- per SM
  const size_t smem = (size_t)tile * D * 4 * (raw_mgr != raw_env ? 4 : 3);
  const int grid = (P.num_envs + tile - 1) / tile;
  cudaEvent_t e0 = nullptr, e1 = nullptr;
  if (h->profiling && h->n_action + 2 <= (int)h->ev_action.size()) {
    e0 = h->ev_action[h->n_action++];
    e1 = h->ev_action[h->n_action++];
    cudaEventRecord(e0, stream);
  }
  int rc;
  if (tile == 32) rc = launch_action<32>(h, ap, smem, stream, grid);
  else if (tile == 64) rc = launch_action<64>(h, ap, smem, stream, grid);
  else if (tile == 128) rc = launch_action<128>(h, ap, smem, stream, grid);
  else rc = launch_action<256>(h, ap, smem, stream, grid);
  if (rc != GFB_OK) return rc;
  if (e1) cudaEventRecord(e1, stream);
  h->launches += 1;
  return GFB_OK;
}

int gfb_action_step(gfb_handle* h, const gfb_buffers* b, const float* raw_env, const float* raw_mgr, void* stream) {
  return action_step_impl(h, b, raw_env, raw_mgr, stream, 0);
}

int gfb_action_step_ring(gfb_handle* h, const gfb_buffers* b, const float* raw_env, const float* raw_mgr,
                         void* stream) {
  if (b && b->buf[GFB_B_ENV_ACTIONS] == b->buf[GFB_B_ENV_LAST_ACTIONS])
    return h ? fail(h, GFB_ERR_INVALID, "gfb_action_step_ring: the two action buffers must differ") : GFB_ERR_INVALID;
  return action_step_impl(h, b, raw_env, raw_mgr, stream, 1);
}

int gfb_post_physics(gfb_handle* h, const gfb_buffers* b, uint32_t phases, void* stream_) {
  if (!h || !b) return GFB_ERR_INVALID;
  if (h->host_only) return fail(h, GFB_ERR_NO_DEVICE, "host-only handle cannot launch kernels");
  if (!h->has_prog) return fail(h, GFB_ERR_INVALID, "gfb_set_program() first");
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  const gfb_program_head& P = h->prog.head;

  // required buffers for the requested phases
  auto need = [&](int id, const char* name) -> bool {
    if (b->buf[id]) return true;
    h->err = std::string("buffer ") + name + " is NULL";
    return false;
  };
  if (!need(GFB_B_EPISODE_LENGTH, "EPISODE_LENGTH")) return GFB_ERR_INVALID;
  if (P.base_max_episode_length > 0 && !need(GFB_B_MAX_EPISODE_LENGTH, "MAX_EPISODE_LENGTH")) return GFB_ERR_INVALID;
  if (phases & GFB_PHASE_TERMINATION)
    if (!need(GFB_B_TERMINATED, "TERMINATED") || !need(GFB_B_TRUNCATED, "TRUNCATED")) return GFB_ERR_INVALID;
  if (phases & GFB_PHASE_REWARD)
    if (!need(GFB_B_REWARD, "REWARD")) return GFB_ERR_INVALID;
  if ((phases & (GFB_PHASE_REWARD | GFB_PHASE_RESET)) && P.n_reward > 0)
    if (!need(GFB_B_EP_SUMS, "EP_SUMS") || !need(GFB_B_EP_SECONDS, "EP_SECONDS")) return GFB_ERR_INVALID;
  if (phases & GFB_PHASE_RESET)
    if (!need(GFB_B_RESET_IDX, "RESET_IDX")) return GFB_ERR_INVALID;
  if (phases & GFB_PHASE_CONTACT)
    for (int m = 0; m < P.n_contact; ++m) {
      if (!need(GFB_B_CONTACTS0 + m, "CONTACTS") || !need(GFB_B_CONTACT_POS0 + m, "CONTACT_POS")) return GFB_ERR_INVALID;
      if (P.contact[m].track_air_time && !need(GFB_B_AIR0 + m, "AIR")) return GFB_ERR_INVALID;
    }
  if (phases & GFB_PHASE_OBSERVE)
    for (int g = 0; g < P.n_obs_groups; ++g) {
      if (!need(GFB_B_OBS_OUT0 + g, "OBS_OUT")) return GFB_ERR_INVALID;
      if (P.obs_group[g].history > 1 && !need(GFB_B_OBS_PREV0 + g, "OBS_PREV")) return GFB_ERR_INVALID;
    }
  if (!(phases & GFB_PHASE_ENTITY) && (phases & (GFB_PHASE_REWARD | GFB_PHASE_TERMINATION | GFB_PHASE_OBSERVE)))
    if (!need(GFB_B_INV_BASE_QUAT, "INV_BASE_QUAT")) return GFB_ERR_INVALID;
  for (int r = 0; r < P.n_reward; ++r) {
    if (!(phases & GFB_PHASE_REWARD) || P.reward[r].weight == 0.0f) continue;
    const gfb_reward_term& t = P.reward[r];
    if (t.op == GFB_R_ACTION_RATE && !need(GFB_B_ACTION_RATE, "ACTION_RATE")) return GFB_ERR_INVALID;
    if (t.op == GFB_R_FEET_SLIDE && !need(GFB_B_LINKS_VEL, "LINKS_VEL")) return GFB_ERR_INVALID;
    if (t.op == GFB_R_BODY_ACC_EXP && !need(GFB_B_BODY_ACC_PREV, "BODY_ACC_PREV")) return GFB_ERR_INVALID;
    if (t.op == GFB_R_EXTERNAL && !need(GFB_B_EXT_VALUES, "EXT_VALUES")) return GFB_ERR_INVALID;
    if ((t.flags & GFB_RF_FIXED_COMMAND) && (t.op == GFB_R_TRACK_LIN_VEL || t.op == GFB_R_TRACK_ANG_VEL) &&
        !need(GFB_B_FIXED_COMMAND, "FIXED_COMMAND"))
      return GFB_ERR_INVALID;
    if (t.op == GFB_R_BASE_HEIGHT && (t.flags & GFB_RF_TARGET_FROM_TENSOR) && !need(GFB_B_TARGET_HEIGHT, "TARGET_HEIGHT"))
      return GFB_ERR_INVALID;
    if (t.op == GFB_R_BASE_HEIGHT && (t.flags & GFB_RF_TERRAIN_HEIGHT) && !need(GFB_B_HEIGHT_FIELD, "HEIGHT_FIELD"))
      return GFB_ERR_INVALID;
  }

  KParams kp{};
  const BufferKey key = buffer_key(*b);
  LaunchCache* lc = nullptr;
  for (auto& c : h->post_cache)
    if (c.valid && c.prog_epoch == h->prog_epoch && c.spec_gen == h->spec_gen && c.phases == phases && c.key == key) {
      lc = &c;
      break;
    }
  if (!lc) {
    LaunchCache& c = h->post_cache[h->post_cache_next];
    h->post_cache_next = (h->post_cache_next + 1) % kLaunchCaches;
    c.valid = false;
    int rc0 = plan_for_launch(h, *b, phases, c.plan, c.table, c.tile, c.n_stages);
    if (rc0 != GFB_OK) return rc0;
    c.tma_ok = tma_eligible(h, *b, c.plan, phases) ? 1 : 0;
    // a specialised kernel whose compile-time structure equals this launch's, if one is attached
    c.spec_index = -1;
    if (!h->specs.empty() && c.tma_ok) {
      gfb_program_head canon = P;
      canonicalize(canon);
      for (size_t i = 0; i < h->specs.size(); ++i) {
        const AttachedSpec& sp = h->specs[i];
        if (sp.tile == c.tile && sp.phases == phases && memcmp(&sp.plan, &c.plan, sizeof(Plan)) == 0 &&
            memcmp(&sp.canon, &canon, sizeof(canon)) == 0) {
          c.spec_index = (int)i;
          break;
        }
      }
    }
    // user-defined terms lowered to device code exist only in the specialised kernel generated for them
    if (c.spec_index < 0 && uses_user_terms(P, phases))
      return fail(h, GFB_ERR_UNSUPPORTED,
                  "the program has GFB_R_USER / GFB_T_USER terms or GFB_O_USER columns and no specialised kernel "
                  "generated for them is attached (the generic kernel does not evaluate them)");
    c.prog_epoch = h->prog_epoch;
    c.spec_gen = h->spec_gen;
    c.phases = phases;
    c.key = key;
    c.valid = true;
    lc = &c;
  }
  kp.plan = lc->plan;
  const std::vector<int32_t>& table = lc->table;
  const int tile = lc->tile;
  const size_t smem = (size_t)kp.plan.smem_words * 4;

  PlanSlot* slot = nullptr;
  for (auto& s : h->slots)
    if (s.used && s.phases == phases && s.tile == tile) slot = &s;
  if (!slot)
    for (auto& s : h->slots)
      if (!s.used) {
        slot = &s;
        break;
      }
  if (!slot) slot = &h->slots[0];
  slot->used = true;
  slot->phases = phases;
  slot->tile = tile;
  int rc = upload_table(h, *slot, table, stream);
  if (rc != GFB_OK) return rc;

  const int n_tiles = (P.num_envs + tile - 1) / tile;
  const AttachedSpec* spec = lc->spec_index >= 0 ? &h->specs[lc->spec_index] : nullptr;
  if (spec && spec->state_slots)  // the kernel reads and writes these rows in place
    for (int i = 0; i < 8; ++i)
      if (((spec->state_slots >> i) & 1u) && !b->buf[GFB_B_USER_STATE0 + i])
        return fail(h, GFB_ERR_INVALID,
                    "buffer USER_STATE" + std::to_string(i) + " is NULL (the attached specialised kernel keeps the "
                    "state of a lowered class-style term there)");
  // persistent grid: every block of the launch is resident from the start (the in-kernel ordered
  // compaction relies on it: a slab only waits for slabs that are already running)
  if (lc->resident_blocks == 0) {
    int per_sm = 0;
    if (spec && spec->blocks_per_sm) per_sm = spec->blocks_per_sm((unsigned)smem);
    else if (tile == 32) per_sm = blocks_per_sm<32>(h, smem);
    else if (tile == 64) per_sm = blocks_per_sm<64>(h, smem);
    else if (tile == 128) per_sm = blocks_per_sm<128>(h, smem);
    else per_sm = blocks_per_sm<256>(h, smem);
    if (per_sm <= 0) return fail(h, GFB_ERR_CUDA, "post kernel: no block fits on an SM with this slab plan");
    lc->resident_blocks = per_sm * std::max(h->num_sms, 1);
  }
  // Persistent loop: launches with 64-env slabs or more; debug bit 8 forces it (tests), bit 4 disables it.
  // (The intermittent "unspecified launch failure" of looped launches with short slab iterations was a
  //  corrupted mbarrier init value -- see the uniform-datapath note at the top of post_kernel.)
  const bool looped = (tile >= 64 || (h->debug & 8u)) && !(h->debug & 4u);
  const int grid = looped ? std::min(n_tiles, lc->resident_blocks) : n_tiles;

  const bool reports = (phases & GFB_PHASE_RESET) != 0;
  if (reports && !b->buf[GFB_B_RESET_IDX]) return fail(h, GFB_ERR_INVALID, "buffer RESET_IDX is NULL");
  h->epoch += 1;
  if (reports) h->report_seq += 1;
  kp.P = P;
  kp.b = *b;
  kp.s = h->scratch;
  kp.s.n_tiles = n_tiles;
  kp.s.epoch = h->epoch;
  kp.s.report_seq = h->report_seq;
  kp.cols = reinterpret_cast<const DevObsCol*>(slot->table_dev);
  kp.phases = phases;
  kp.tma_ok = lc->tma_ok;
  kp.debug = h->debug;
  kp.peer.world = 0;
  if (h->peer_world > 1 && reports) {
    if (!b->buf[GFB_B_LOG_ACC]) return fail(h, GFB_ERR_INVALID, "sharded logging needs GFB_B_LOG_ACC");
    for (int r = 0; r < h->peer_world; ++r) kp.peer.inbox[r] = h->inbox[r];
    kp.peer.rank = h->peer_rank;
    kp.peer.world = h->peer_world;
    kp.peer.seq = ++h->peer_seq;
    kp.peer.global_num_envs = h->global_num_envs;
  }

  cudaEvent_t e0 = nullptr, e1 = nullptr;
  if (h->profiling && h->n_post + 2 <= (int)h->ev_post.size()) {
    h->ev_post_obs_only[h->n_post / 2] = phases == GFB_PHASE_OBSERVE ? 1 : 0;
    e0 = h->ev_post[h->n_post++];
    e1 = h->ev_post[h->n_post++];
    cudaEventRecord(e0, stream);
  }
  if (spec) {
    if (spec->launch(&kp, grid, (unsigned)smem, stream) != 0)
      return fail(h, GFB_ERR_CUDA, std::string("specialised kernel launch: ") + cudaGetErrorString(cudaGetLastError()));
    h->n_spec_launches += 1;
    rc = GFB_OK;
  } else {
    if (tile == 32) rc = launch_post<32>(h, kp, smem, stream, grid);
    else if (tile == 64) rc = launch_post<64>(h, kp, smem, stream, grid);
    else if (tile == 128) rc = launch_post<128>(h, kp, smem, stream, grid);
    else rc = launch_post<256>(h, kp, smem, stream, grid);
    h->n_generic_launches += 1;
  }
  if (rc != GFB_OK) return rc;
  if (e1) cudaEventRecord(e1, stream);
  h->launches += 1;
  if (reports) {
    // the ascending index list from the slabs' reset masks: behind the post kernel, which has told the
    // host the counts by then -- this runs while the host wakes up (see compact_kernel)
    const int n_words = n_tiles * (tile / 32);
    const CompactGeometry g = compact_geometry(n_words);
    cudaEvent_t cmp_end = aux_begin(h, 0, stream);
    compact_kernel<<<g.n_blocks, CMP_THREADS, 0, stream>>>(h->scratch.tile_bits, n_words, g.words_per_block,
                                                         static_cast<int64_t*>(b->buf[GFB_B_RESET_IDX]));
    CUDA_TRY(cudaGetLastError());
    if (cmp_end) cudaEventRecord(cmp_end, stream);
    h->launches += 1;
  }
  return GFB_OK;
}

int gfb_read_report(gfb_handle* h, gfb_report* out, void* stream_) {
  if (!h || !out) return GFB_ERR_INVALID;
  if (h->host_only) return fail(h, GFB_ERR_NO_DEVICE, "host-only handle has no report");
  if (h->report_seq == 0) return fail(h, GFB_ERR_INVALID, "no launch with GFB_PHASE_RESET has been issued yet");
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  // The kernel stores the report into this (mapped, pinned) block and then its sequence number.
  // Spinning on that word costs ~1 us after the store; cudaStreamSynchronize would add the driver's
  // wake-up latency AND wait for the end of the kernel, which comes later than the report.
  volatile uint64_t* seq = &h->report_host->seq;
  const uint64_t want = h->report_seq;
  for (uint64_t spins = 1; *seq != want; ++spins) {
#if defined(__x86_64__) || defined(__i386__)
    __builtin_ia32_pause();
#endif
    if ((spins & 0x3fff) == 0) {  // every ~16 k spins: has the stream died or drained without a report?
      const cudaError_t q = cudaStreamQuery(stream);
      if (q == cudaSuccess) {
        if (*seq == want) break;
        return fail(h, GFB_ERR_CUDA, "the post-physics launch finished without delivering its report");
      }
      if (q != cudaErrorNotReady) return fail(h, GFB_ERR_CUDA, std::string("waiting for the report: ") + cudaGetErrorString(q));
    }
  }
  __atomic_thread_fence(__ATOMIC_ACQUIRE);
  memcpy(out, h->report_host, sizeof(gfb_report));
  return GFB_OK;
}

int gfb_read_report_local(gfb_handle* h, int32_t* n_reset, void* stream_) {
  if (!h || !n_reset) return GFB_ERR_INVALID;
  if (h->host_only) return fail(h, GFB_ERR_NO_DEVICE, "host-only handle has no report");
  if (h->report_seq == 0) return fail(h, GFB_ERR_INVALID, "no launch with GFB_PHASE_RESET has been issued yet");
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  volatile uint64_t* seq = &h->report_host->local_seq;
  const uint64_t want = h->report_seq;
  for (uint64_t spins = 1; *seq != want; ++spins) {
#if defined(__x86_64__) || defined(__i386__)
    __builtin_ia32_pause();
#endif
    if ((spins & 0x3fff) == 0) {  // has the stream died or drained without a report?
      const cudaError_t q = cudaStreamQuery(stream);
      if (q == cudaSuccess) {
        if (*seq == want) break;
        return fail(h, GFB_ERR_CUDA, "the post-physics launch finished without delivering its report");
      }
      if (q != cudaErrorNotReady) return fail(h, GFB_ERR_CUDA, std::string("waiting for the report: ") + cudaGetErrorString(q));
    }
  }
  __atomic_thread_fence(__ATOMIC_ACQUIRE);
  *n_reset = h->report_host->n_reset;
  return GFB_OK;
}

int gfb_post_physics_report(gfb_handle* h, const gfb_buffers* b, uint32_t phases, gfb_report* out, void* stream) {
  if (!(phases & GFB_PHASE_RESET)) return fail(h, GFB_ERR_INVALID, "gfb_post_physics_report needs GFB_PHASE_RESET");
  const int rc = gfb_post_physics(h, b, phases, stream);
  if (rc != GFB_OK) return rc;
  return gfb_read_report(h, out, stream);
}

int gfb_peer_export(gfb_handle* h, void* ipc_handle_out) {
  if (!h || !ipc_handle_out) return GFB_ERR_INVALID;
  if (h->host_only) return fail(h, GFB_ERR_NO_DEVICE, "host-only handle has no device memory to share");
  static_assert(sizeof(cudaIpcMemHandle_t) == GFB_IPC_HANDLE_BYTES, "IPC handle size");
  CUDA_TRY(cudaSetDevice(h->device));
  if (!h->inbox_own) CUDA_TRY(cudaMalloc(&h->inbox_own, sizeof(PeerInbox)));
  // (re)connecting restarts the sequence numbers: no stale flag may survive.  Peers write here only
  // after their gfb_peer_connect, i.e. after the handle exchange that follows this call.
  CUDA_TRY(cudaMemset(h->inbox_own, 0, sizeof(PeerInbox)));
  CUDA_TRY(cudaDeviceSynchronize());
  cudaIpcMemHandle_t ipc;
  CUDA_TRY(cudaIpcGetMemHandle(&ipc, h->inbox_own));
  memcpy(ipc_handle_out, &ipc, sizeof(ipc));
  return GFB_OK;
}

int gfb_peer_connect(gfb_handle* h, int32_t rank, int32_t world, const void* ipc_handles, int64_t global_num_envs) {
  if (!h || !ipc_handles) return GFB_ERR_INVALID;
  if (h->host_only) return fail(h, GFB_ERR_NO_DEVICE, "host-only handle cannot connect to peers");
  if (world < 1 || world > GFB_MAX_PEERS || rank < 0 || rank >= world)
    return fail(h, GFB_ERR_INVALID, "gfb_peer_connect: rank / world out of range");
  if (!h->inbox_own) return fail(h, GFB_ERR_INVALID, "gfb_peer_connect: call gfb_peer_export first");
  if (global_num_envs < h->num_envs) return fail(h, GFB_ERR_INVALID, "gfb_peer_connect: global_num_envs too small");
  gfb_peer_disconnect(h);
  CUDA_TRY(cudaSetDevice(h->device));
  const cudaIpcMemHandle_t* handles = static_cast<const cudaIpcMemHandle_t*>(ipc_handles);
  for (int r = 0; r < world; ++r) {
    if (r == rank) {
      h->inbox[r] = h->inbox_own;
      continue;
    }
    void* p = nullptr;
    cudaError_t e = cudaIpcOpenMemHandle(&p, handles[r], cudaIpcMemLazyEnablePeerAccess);
    if (e != cudaSuccess) {
      for (int q = 0; q < r; ++q)
        if (q != rank && h->inbox[q]) cudaIpcCloseMemHandle(h->inbox[q]);
      for (auto& q : h->inbox) q = nullptr;
      return fail(h, GFB_ERR_CUDA, std::string("cudaIpcOpenMemHandle (peer inbox): ") + cudaGetErrorString(e));
    }
    h->inbox[r] = static_cast<PeerInbox*>(p);
  }
  h->peer_rank = rank;
  h->peer_world = world;
  h->peer_seq = 0;
  h->global_num_envs = global_num_envs;
  return GFB_OK;
}

int gfb_peer_disconnect(gfb_handle* h) {
  if (!h) return GFB_ERR_INVALID;
  if (h->host_only) return GFB_OK;
  for (int r = 0; r < h->peer_world; ++r)
    if (r != h->peer_rank && h->inbox[r]) cudaIpcCloseMemHandle(h->inbox[r]);
  for (auto& q : h->inbox) q = nullptr;
  h->peer_world = 0;
  h->peer_rank = 0;
  return GFB_OK;
}

int gfb_observe(gfb_handle* h, const gfb_buffers* b, const int64_t* idx, int32_t n, void* stream_) {
  if (!h || !b) return GFB_ERR_INVALID;
  if (h->host_only) return fail(h, GFB_ERR_NO_DEVICE, "host-only handle cannot launch kernels");
  if (!h->has_prog) return fail(h, GFB_ERR_INVALID, "gfb_set_program() first");
  if (n <= 0) return GFB_OK;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  const gfb_program_head& P = h->prog.head;
  if (!b->buf[GFB_B_INV_BASE_QUAT]) return fail(h, GFB_ERR_INVALID, "INV_BASE_QUAT missing");
  ObserveParams op{};
  // observe-only plan: nothing is staged; the kernel reads staged-kind columns from their global buffer
  LaunchCache& oc = h->observe_cache;
  const BufferKey key = buffer_key(*b);
  int rc = GFB_OK;
  if (!(oc.valid && oc.prog_epoch == h->prog_epoch && oc.key == key)) {
    oc.valid = false;
    rc = build_plan(h, *b, GFB_PHASE_OBSERVE, kObserveTile, 1, oc.plan, oc.table, true);
    if (rc != GFB_OK) return rc;
    oc.prog_epoch = h->prog_epoch;
    oc.key = key;
    oc.valid = true;
  }
  op.plan = oc.plan;
  const std::vector<int32_t>& table = oc.table;
  if ((op.plan.needs & NEED_LIN) && !b->buf[GFB_B_VEL]) return fail(h, GFB_ERR_INVALID, "VEL missing");
  if ((op.plan.needs & NEED_ANG) && !b->buf[GFB_B_ANG]) return fail(h, GFB_ERR_INVALID, "ANG missing");
  // lowered user-defined observation terms: only the library generated for them (same structure, so the
  // same user_id) computes them -- into GFB_B_OBS_EXT1, which the plan's GFB_O_USER columns read
  const AttachedSpec* user_spec = nullptr;
  if (has_user_observations(P)) {
    gfb_program_head canon = P;
    canonicalize(canon);
    for (const AttachedSpec& sp : h->specs)
      if (sp.user_observe && memcmp(&sp.canon, &canon, sizeof(canon)) == 0) {
        user_spec = &sp;
        break;
      }
    if (!user_spec)
      return fail(h, GFB_ERR_UNSUPPORTED,
                  "gfb_observe: the program has GFB_O_USER columns and no specialised kernel generated for them is "
                  "attached (the generic kernel does not evaluate them)");
    for (int i = 0; i < 8; ++i)  // its class-style observation terms read and write these rows in place
      if (((user_spec->state_slots >> i) & 1u) && !b->buf[GFB_B_USER_STATE0 + i])
        return fail(h, GFB_ERR_INVALID,
                    "buffer USER_STATE" + std::to_string(i) + " is NULL (the attached specialised kernel keeps the "
                    "state of a lowered class-style term there)");
  }
  rc = upload_table(h, h->observe_slot, table, stream);
  if (rc != GFB_OK) return rc;
  op.P.n_contact = P.n_contact;
  op.P.n_obs_groups = P.n_obs_groups;
  op.P.rng_mode = P.rng_mode;
  op.P.rng_seed = P.rng_seed;
  op.P.step_index = P.step_index;
  for (int m = 0; m < P.n_contact; ++m) op.P.contact_links[m] = P.contact[m].n_links;
  memcpy(op.P.obs_group, P.obs_group, sizeof(op.P.obs_group));
  op.P.n_items = 0;
  for (int g = 0; g < P.n_obs_groups; ++g)
    for (int c = 0; c * 32 < P.obs_group[g].n_cols; ++c) {
      if (op.P.n_items >= OBS_MAX_ITEMS) return fail(h, GFB_ERR_UNSUPPORTED, "gfb_observe: too many observation columns");
      op.P.item_group[op.P.n_items] = (int8_t)g;
      op.P.item_chunk[op.P.n_items] = (int8_t)c;
      op.P.n_items += 1;
    }
  op.b = *b;
  op.cols = reinterpret_cast<const DevObsCol*>(h->observe_slot.table_dev);
  op.idx = idx;
  op.n = n;
  if (user_spec) {
    cudaEvent_t user_end = aux_begin(h, 3, stream);
    if (user_spec->user_observe(b, P.num_envs, idx, n, P.base_max_episode_length > 0 ? 1 : 0, stream) != 0)
      return fail(h, GFB_ERR_CUDA, std::string("user observation kernel: ") + cudaGetErrorString(cudaGetLastError()));
    if (user_end) cudaEventRecord(user_end, stream);
    h->n_user_observe_launches += 1;
    h->launches += 1;
  }
  const int grid = (n + OBS_WARPS * OBS_ROWS - 1) / (OBS_WARPS * OBS_ROWS);
  cudaEvent_t obs_end = aux_begin(h, 1, stream);
  observe_kernel<<<grid, OBS_WARPS * 32, 0, stream>>>(op);
  CUDA_TRY(cudaGetLastError());
  if (obs_end) cudaEventRecord(obs_end, stream);
  h->launches += 1;
  return GFB_OK;
}

int gfb_contact_forces(gfb_handle* h, const float* force, const float* position, const int32_t* link_a,
                       const int32_t* link_b, const float* links_quat, const int32_t* target_link_ids,
                       const int32_t* with_link_ids, float* out_forces, float* out_positions,
                       float* position_counts, int32_t n_envs, int32_t n_slots, int32_t n_links_total,
                       int32_t n_targets, int32_t n_with, int32_t has_with_filter, void* stream_) {
  if (!h || !force || !position || !link_a || !link_b || !links_quat || !target_link_ids || !out_forces ||
      !out_positions || !position_counts)
    return fail(h, GFB_ERR_INVALID, "gfb_contact_forces: null argument");
  if (n_envs <= 0 || n_targets <= 0) return GFB_OK;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  const int threads = 128;
  contact_kernel<<<(n_envs + threads - 1) / threads, threads, 0, stream>>>(
      force, position, link_a, link_b, reinterpret_cast<const float4*>(links_quat), target_link_ids, with_link_ids,
      out_forces, out_positions, position_counts, n_envs, n_slots, n_links_total, n_targets, n_with, has_with_filter);
  CUDA_TRY(cudaGetLastError());
  h->launches += 1;
  return GFB_OK;
}

int gfb_rotate(gfb_handle* h, const float* vec, const float* quat, float* out, int32_t n, int32_t conjugate,
               void* stream_) {
  if (!h || !quat || !out) return fail(h, GFB_ERR_INVALID, "gfb_rotate: null argument");
  if (n <= 0) return GFB_OK;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  rotate_kernel<<<(n + 255) / 256, 256, 0, stream>>>(vec, reinterpret_cast<const float4*>(quat), out, n, conjugate);
  CUDA_TRY(cudaGetLastError());
  h->launches += 1;
  return GFB_OK;
}

int gfb_spawn_pose(gfb_handle* h, const gfb_spawn* cfg, const int64_t* idx, int32_t n, int32_t n_rows,
                   const float* height_field, const float* u_x, const float* u_y, const float* u_rot_x,
                   const float* u_rot_y, const float* u_rot_z, float* position_buffer, float* rot_buffer,
                   float* quat_buffer, float* pos_out, float* quat_out, void* stream_) {
  if (!h || !cfg) return GFB_ERR_INVALID;
  if (h->host_only) return fail(h, GFB_ERR_NO_DEVICE, "host-only handle cannot launch kernels");
  if (n < 0 || n_rows < 0) return fail(h, GFB_ERR_INVALID, "gfb_spawn_pose: negative size");
  if (n == 0) return GFB_OK;
  if (!position_buffer) return fail(h, GFB_ERR_INVALID, "gfb_spawn_pose: position_buffer is NULL");
  if (!idx && n > n_rows) return fail(h, GFB_ERR_INVALID, "gfb_spawn_pose: n exceeds the buffer rows");
  if (height_field && (cfg->height_field_rows < 1 || cfg->height_field_cols < 1))
    return fail(h, GFB_ERR_INVALID, "gfb_spawn_pose: height field dimensions missing");
  if (cfg->with_rotation) {
    if (!rot_buffer || !quat_buffer) return fail(h, GFB_ERR_INVALID, "gfb_spawn_pose: rotation buffers missing");
    if (!aligned16(quat_buffer) || (quat_out && !aligned16(quat_out)))
      return fail(h, GFB_ERR_INVALID, "gfb_spawn_pose: quaternion buffers must be 16-byte aligned");
    for (int a = 0; a < 3; ++a)
      if (cfg->rot_mode[a] != GFB_SPAWN_ROT_KEEP && cfg->rot_mode[a] != GFB_SPAWN_ROT_DRAW)
        return fail(h, GFB_ERR_INVALID, "gfb_spawn_pose: bad rot_mode");
  }
  SpawnParams sp{};
  sp.cfg = *cfg;
  sp.idx = idx;
  sp.n = n;
  sp.height_field = height_field;
  sp.u_x = u_x;
  sp.u_y = u_y;
  sp.u_rot[0] = u_rot_x;
  sp.u_rot[1] = u_rot_y;
  sp.u_rot[2] = u_rot_z;
  sp.position_buffer = position_buffer;
  sp.rot_buffer = rot_buffer;
  sp.quat_buffer = quat_buffer;
  sp.pos_out = pos_out;
  sp.quat_out = quat_out;
  cudaEvent_t spawn_end = aux_begin(h, 2, static_cast<cudaStream_t>(stream_));
  spawn_kernel<<<(n + 127) / 128, 128, 0, static_cast<cudaStream_t>(stream_)>>>(sp);
  CUDA_TRY(cudaGetLastError());
  if (spawn_end) cudaEventRecord(spawn_end, static_cast<cudaStream_t>(stream_));
  h->launches += 1;
  return GFB_OK;
}

int gfb_reset_rows(gfb_handle* h, const int64_t* idx, int32_t n, int32_t width, int32_t mode, const float* base,
                   float a, float b, const float* draws, uint64_t seed, uint64_t counter, float* out, float* scatter,
                   void* stream_) {
  if (!h) return GFB_ERR_INVALID;
  if (h->host_only) return fail(h, GFB_ERR_NO_DEVICE, "host-only handle cannot launch kernels");
  if (n < 0 || width <= 0) return fail(h, GFB_ERR_INVALID, "gfb_reset_rows: bad shape");
  if (n == 0) return GFB_OK;
  if (!out) return fail(h, GFB_ERR_INVALID, "gfb_reset_rows: out is NULL");
  if (mode != GFB_ROWS_NOISE && mode != GFB_ROWS_UNIFORM) return fail(h, GFB_ERR_INVALID, "gfb_reset_rows: bad mode");
  if (mode == GFB_ROWS_NOISE && !base) return fail(h, GFB_ERR_INVALID, "gfb_reset_rows: base is NULL");
  ResetRowsParams p{};
  p.idx = idx; p.n = n; p.width = width; p.mode = mode; p.base = base; p.a = a; p.b = b; p.draws = draws;
  p.seed = seed; p.counter = counter; p.out = out; p.scatter = scatter;
  const long long total = (long long)n * width;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  reset_rows_kernel<<<(unsigned)((total + 255) / 256), 256, 0, stream>>>(p);
  CUDA_TRY(cudaGetLastError());
  h->launches += 1;
  return GFB_OK;
}

int gfb_spec_describe(gfb_handle* h, const gfb_buffers* b, uint32_t phases, void* canonical_head,
                      int32_t* plan_out, int32_t plan_cap, int32_t* plan_words, int32_t* tile_out) {
  if (!h || !b || !canonical_head || !plan_out || !plan_words || !tile_out) return GFB_ERR_INVALID;
  if (!h->has_prog) return fail(h, GFB_ERR_INVALID, "gfb_set_program() first");
  Plan plan;
  std::vector<int32_t> table;
  int tile = 0, n_stages = 1;
  int rc = plan_for_launch(h, *b, phases, plan, table, tile, n_stages);
  if (rc != GFB_OK) return rc;
  const int words = (int)(sizeof(Plan) / 4);
  *plan_words = words;
  if (plan_cap < words) return fail(h, GFB_ERR_INVALID, "plan_out too small");
  memcpy(plan_out, &plan, sizeof(Plan));
  gfb_program_head canon = h->prog.head;
  canonicalize(canon);
  memcpy(canonical_head, &canon, sizeof(canon));
  *tile_out = tile;
  return GFB_OK;
}

int gfb_spec_attach(gfb_handle* h, const char* path) {
  if (!h) return GFB_ERR_INVALID;
  if (!path) {
    for (auto& sp : h->specs)
      if (sp.dl) dlclose(sp.dl);
    h->specs.clear();
    h->spec_gen += 1;
    return GFB_OK;
  }
  void* dl = dlopen(path, RTLD_NOW | RTLD_LOCAL);
  if (!dl) return fail(h, GFB_ERR_INVALID, std::string("dlopen: ") + dlerror());
  using InfoFn = int (*)(int*, unsigned*, const void**, const void**, int*, int*);
  using LaunchFn = int (*)(const KParams*, int, unsigned, void*);
  InfoFn info = reinterpret_cast<InfoFn>(dlsym(dl, "gfb_spec_info"));
  LaunchFn launch = reinterpret_cast<LaunchFn>(dlsym(dl, "gfb_spec_launch"));
  if (!info || !launch) {
    dlclose(dl);
    return fail(h, GFB_ERR_INVALID, "not a gfb200 specialised kernel library");
  }
  AttachedSpec sp;
  const void *canon = nullptr, *plan = nullptr;
  int head_bytes = 0, plan_bytes = 0;
  info(&sp.tile, &sp.phases, &canon, &plan, &head_bytes, &plan_bytes);
  if (head_bytes != (int)sizeof(gfb_program_head) || plan_bytes != (int)sizeof(Plan)) {
    dlclose(dl);
    return fail(h, GFB_ERR_INVALID, "specialised kernel library was built against other struct layouts");
  }
  memcpy(&sp.canon, canon, sizeof(sp.canon));
  memcpy(&sp.plan, plan, sizeof(sp.plan));
  sp.dl = dl;
  sp.launch = launch;
  sp.blocks_per_sm = reinterpret_cast<int (*)(unsigned)>(dlsym(dl, "gfb_spec_blocks_per_sm"));
  sp.user_observe = reinterpret_cast<int (*)(const gfb_buffers*, int, const int64_t*, int, int, void*)>(
      dlsym(dl, "gfb_spec_user_observe"));
  if (auto slots = reinterpret_cast<unsigned (*)(void)>(dlsym(dl, "gfb_spec_state_slots"))) sp.state_slots = slots();
  h->specs.push_back(sp);
  h->spec_gen += 1;
  return GFB_OK;
}

int gfb_spec_stats(const gfb_handle* h, int64_t* specialised, int64_t* generic, int64_t* user_observe) {
  if (!h) return GFB_ERR_INVALID;
  if (specialised) *specialised = h->n_spec_launches;
  if (generic) *generic = h->n_generic_launches;
  if (user_observe) *user_observe = h->n_user_observe_launches;
  return GFB_OK;
}

int gfb_profile_enable(gfb_handle* h, int32_t enabled) {
  if (!h) return GFB_ERR_INVALID;
  if (enabled && h->ev_post.empty()) {
    h->ev_post.resize(kEventPairs * 2);
    h->ev_post_obs_only.assign(kEventPairs, 0);
    h->ev_action.resize(kEventPairs * 2);
    h->ev_aux.resize(kEventPairs * 4);
    h->ev_aux_kind.assign(kEventPairs * 2, 0);
    for (auto& e : h->ev_aux) CUDA_TRY(cudaEventCreate(&e));
    for (auto& e : h->ev_post) CUDA_TRY(cudaEventCreate(&e));
    for (auto& e : h->ev_action) CUDA_TRY(cudaEventCreate(&e));
  }
  h->profiling = enabled != 0;
  h->n_post = h->n_action = h->n_aux = 0;
  h->post_ms = h->action_ms = h->post_obs_ms = 0.f;
  h->post_count = h->action_count = h->post_obs_count = 0;
  for (int k = 0; k < 4; ++k) {
    h->aux_ms[k] = 0.f;
    h->aux_count[k] = 0;
  }
  return GFB_OK;
}

int gfb_profile_read(gfb_handle* h, float* post_ms_total, int32_t* post_launches, float* action_ms_total,
                     int32_t* action_launches) {
  if (!h) return GFB_ERR_INVALID;
  CUDA_TRY(cudaDeviceSynchronize());
  for (int i = 0; i + 1 < h->n_post; i += 2) {
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, h->ev_post[i], h->ev_post[i + 1]) == cudaSuccess) {
      if (h->ev_post_obs_only[i / 2]) {
        h->post_obs_ms += ms;
        h->post_obs_count += 1;
      } else {
        h->post_ms += ms;
        h->post_count += 1;
      }
    }
  }
  for (int i = 0; i + 1 < h->n_action; i += 2) {
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, h->ev_action[i], h->ev_action[i + 1]) == cudaSuccess) {
      h->action_ms += ms;
      h->action_count += 1;
    }
  }
  for (int i = 0; i + 1 < h->n_aux; i += 2) {
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, h->ev_aux[i], h->ev_aux[i + 1]) == cudaSuccess) {
      h->aux_ms[h->ev_aux_kind[i / 2]] += ms;
      h->aux_count[h->ev_aux_kind[i / 2]] += 1;
    }
  }
  h->n_post = h->n_action = h->n_aux = 0;
  if (post_ms_total) *post_ms_total = h->post_ms;
  if (post_launches) *post_launches = h->post_count;
  if (action_ms_total) *action_ms_total = h->action_ms;
  if (action_launches) *action_launches = h->action_count;
  return GFB_OK;
}

int gfb_profile_read_aux(gfb_handle* h, float* ms_total, int32_t* launches) {
  if (!h || !ms_total || !launches) return GFB_ERR_INVALID;
  int rc = gfb_profile_read(h, nullptr, nullptr, nullptr, nullptr);  // folds pending event pairs
  if (rc != GFB_OK) return rc;
  for (int k = 0; k < 4; ++k) {
    ms_total[k] = h->aux_ms[k];
    launches[k] = h->aux_count[k];
  }
  return GFB_OK;
}

int64_t gfb_launch_count(const gfb_handle* h) { return h ? h->launches : 0; }

}  // extern "C"
