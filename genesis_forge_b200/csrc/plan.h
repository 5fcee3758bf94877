// Host/device shared structures internal to libgfb200 (not part of the ABI).
#pragma once
#include <stdint.h>

#include "../../include/gfb200.h"

// typed view of an entry of the buffer table of the kernel parameter `K`
#define GFB_BUF(T_, id) (reinterpret_cast<T_*>(K.b.buf[id]))

namespace gfb {

// Observation column as the kernels consume it (built on the host from gfb_obs_col).
//   kind 0: constant zero
//   kind 1: slab-staged array: post kernel reads shared memory at `a + row*row_words + col`,
//           the observe kernel reads global buffer `gbuf`
//   kind 2: global buffer `gbuf` in both kernels
//   kind 3: per-env stash (derived values) at `stash + row*stash_stride + a`
//   vec  1: this column starts a 4-aligned run of 4 columns with the same contiguous source
struct DevObsCol {
  int32_t kind;
  int32_t a;
  int32_t row_words;
  int32_t col;
  float scale;
  float noise;
  int32_t gbuf;
  int32_t vec;
};

// needs mask: which body-frame vectors the term table uses
enum : uint32_t {
  NEED_LIN = 1u,
  NEED_ANG = 2u,
  NEED_GRAV = 4u,
  NEED_POS = 8u,
  NEED_DOF_POS = 16u,
  NEED_CONTACT_DATA = 32u,
};

// stash row layout (words, per env): [ang_b 3][lin_b 3][grav_b 3][per contact manager: norm[Lc], state 4*Lc]
struct Plan {
  int32_t tile;          // envs per thread block
  uint32_t needs;
  int32_t n_staged;
  // Two load groups.  Arrays [0, n_early) are loaded before the entity / contact phases.  Arrays
  // [n_early, n_staged) and (sums_late) the episode-sum rows are only read after the contact phase
  // and are loaded THEN, into the shared memory that held the contact slots -- the slab of a
  // contact-bearing table needs ~1/3 less shared memory, so more warps stay resident.
  // n_early == n_staged && !sums_late: everything is loaded up front (no contact slots staged).
  int32_t n_early;
  int32_t sums_late;
  // Arrays [0, n_prefetch) -- base quaternion, position, velocities -- are dead once the per-env
  // (owner) phase is over: the persistent kernel refills them with the NEXT slab's rows while the
  // current slab's observation rows are still being assembled.
  int32_t n_prefetch;
  int32_t staged_buf[GFB_MAX_STAGED];
  int32_t staged_words[GFB_MAX_STAGED];
  int32_t staged_off[GFB_MAX_STAGED];
  int32_t staged_store[GFB_MAX_STAGED];  // output buffer that receives a copy of the slab, or -1
  int32_t off_pos, off_quat, off_vel, off_ang, off_dof_pos;
  int32_t off_cmd[GFB_MAX_COMMANDS];
  int32_t off_cforce, off_cpos, off_cla, off_clb;
  int32_t stash_off, stash_stride;
  int32_t st_cnorm[GFB_MAX_CONTACT_MANAGERS];  // offsets inside a stash row
  int32_t st_air[GFB_MAX_CONTACT_MANAGERS];    // 4*Lc words: last_air, cur_air, last_contact, cur_contact
  int32_t sums_off;                            // (n_reward, tile) episode-sum slab
  int32_t cout_off[GFB_MAX_CONTACT_MANAGERS];  // (tile, 3*Lc) contact force output slab
  int32_t cposout_off[GFB_MAX_CONTACT_MANAGERS];
  int32_t cols_off;                            // descriptor table copy (DevObsCol | HeadCol | group SoA)
  int32_t n_cols_total;
  int32_t table_words;                         // total words of the descriptor table
  // 16-byte group path (observation groups whose frame width is a multiple of 4 and whose sources
  // are all in shared memory).  Inside the descriptor table:
  //   runs  (aligned contiguous run of one staged array):  int4 {off, stride, c4, scale}[n_runs],
  //                                                         float4 noise[n_runs]
  //   mixed (4 independent shared sources): int4 off[n_mixed], int4 stride[n_mixed],
  //                                         float4 scale[n_mixed], float4 noise[n_mixed], int c4[n_mixed]
  int32_t n_runs, run_off;
  int32_t n_mixed, mixed_off;
  int32_t grp_run_begin[GFB_MAX_OBS_GROUPS];   // -1 = per-element path for this observation group
  int32_t grp_run_count[GFB_MAX_OBS_GROUPS];
  int32_t grp_mixed_begin[GFB_MAX_OBS_GROUPS];
  int32_t grp_mixed_count[GFB_MAX_OBS_GROUPS];
  int32_t stage_words;                         // shared words of one ring stage
  int32_t n_stages;                            // 2 = prefetch ring, 1 = single buffer
  int32_t rew_acc_off;                         // exact episode-quotient sums (RESET launches, post_kernel.cuh)
  int32_t smem_words;                          // (last: spec.py reads it from the end of the plan)
};

// Logging exchange between the ranks of one NVLink domain (gfb_peer_connect): every rank owns an
// inbox with one slot per sender and step parity; senders store their partials
// straight into the peers' inboxes and publish them with a release store of the sequence number.
constexpr int PEER_VALS = GFB_MAX_REWARD_TERMS + GFB_MAX_TERMINATION_TERMS + 1;
struct PeerSlot {
  double vals[PEER_VALS];
  unsigned long long seq;
  unsigned long long _pad[64 - PEER_VALS - 1];
};
static_assert(sizeof(PeerSlot) == 512, "PeerSlot is padded to 512 bytes");
struct PeerInbox {
  PeerSlot slot[2][GFB_MAX_PEERS];  // [parity of the exchange number][sender]
};
struct PeerParams {
  PeerInbox* inbox[GFB_MAX_PEERS];  // [r] = rank r's inbox (own one for r == rank)
  int32_t rank, world;              // world <= 1: single rank, no exchange
  unsigned long long seq;           // sequence number of this exchange (same on every rank)
  int64_t global_num_envs;
};

// Scratch owned by the handle.  All counters are left at zero by the launch that used them.
enum : int {
  CTR_TICKET = 0,      // next slab to hand out (slabs [0, gridDim.x) belong to the blocks by index)
  CTR_COMPACT_DONE = 1,  // blocks of compact_kernel that have written their indices
  CTR_BLOCKS_DONE = 2, // blocks that have left the kernel (late logging at gridDim.x)
  CTR_TOTAL_RESET = 3, // number of reset envs of this launch
  CTR_COUNT = 8
};
struct Scratch {
  uint32_t* tile_bits;             // (ceil(N / 32) words, in env order) reset masks, 32 envs per word
  int32_t* term_count;             // (GFB_MAX_TERMINATION_TERMS) fire counts since the last report
  unsigned long long* rew_acc;     // (GFB_MAX_REWARD_TERMS x XS_WORDS) exact sums (tail_math.cuh)
  uint32_t* rew_flags;             // (GFB_MAX_REWARD_TERMS) non-finite episode quotients seen
  uint32_t* counters;              // CTR_*
  uint32_t* status;                // sticky status bits
  gfb_report* report_host;         // device address of the host's mapped report
  int32_t n_tiles;
  uint32_t epoch;                  // launch number
  unsigned long long report_seq;   // value of gfb_report.seq that announces this launch's report
};

struct KParams {
  gfb_program_head P;
  gfb_buffers b;
  Plan plan;
  Scratch s;
  PeerParams peer;
  const DevObsCol* cols;
  uint32_t phases;
  int32_t tma_ok;
  uint32_t debug;  // GFB_DEBUG experiments (0 in production): 1 no fences in the scan, 2 no scan, 4 one slab per block
};

}  // namespace gfb
