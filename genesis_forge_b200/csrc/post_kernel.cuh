// The fused post-physics kernel: one thread block per slab of TILE environments, one thread per
// environment for the per-env arithmetic, all threads together for slab loads/stores and for the
// observation assembly.
//
// Replaces, in one launch, managed_env.py:294-326 of the reference:
//   entity cache            entity_manager.py:189-195
//   contact net forces      contact_manager.py:384-432 + contact/kernel.py:35-90 (ordered sums)
//   air-time state machine  contact_manager.py:434-477
//   terminations            termination_manager.py:151-190, mdp/terminations.py
//   rewards + episode sums  reward_manager.py:166-195, mdp/rewards.py
//   command resample        command_manager.py:152-162, 290-303
//   in-library reset        genesis_env.py:233-252, contact_manager.py:316-329,
//                           reward_manager.py:197-222, command_manager.py:164-170
//   observations            observation_manager.py:218-256 (reset envs are re-observed afterwards by
//                           observe_kernel, because the reference observes after reset)
//
// Data movement: AoS rows ((N,3), (N,4), (N,D), (N,C,3) ...) of one slab are contiguous in HBM, so
// each staged array is ONE cp.async.bulk (TMA) transfer into shared memory, completion on one
// mbarrier; slab outputs go back with cp.async.bulk stores; (N,) arrays are plain coalesced
// accesses; observation rows are written with coalesced 16-byte stores straight from the gather.
//
// Persistent grid: as many blocks as are resident at once (or one per slab if fewer); a block takes
// slab blockIdx.x first and then draws further slabs from a ticket counter.  The logging reductions
// and the step report are part of this kernel (tail.cuh): its last block to finish writes the report
// into the host's mapped memory.
#pragma once
#include "device_utils.cuh"
#include "plan.h"
#include "tail.cuh"

// In a specialised build the term loops have compile-time trip counts and are fully unrolled.
#ifdef GFB_SPEC
#define GFB_UNROLL_TERMS _Pragma("unroll")
#else
#define GFB_UNROLL_TERMS
#endif

namespace gfb {

// fetch one observation value for slab row `row` (post kernel: staged arrays live in shared memory)
__device__ __forceinline__ float obs_fetch_post(const DevObsCol& d, const float* S, const gfb_buffers& b,
                                                const Plan& plan, int row, long long env) {
  switch (d.kind) {
    case 1:
      return S[d.a + row * d.row_words + d.col];
    case 2:
      return reinterpret_cast<const float*>(b.buf[d.gbuf])[env * d.row_words + d.col];
    case 3:
      return S[plan.stash_off + row * plan.stash_stride + d.a];
    default:
      return 0.0f;
  }
}

// v += u * noise for one 16-byte piece; u from the injected U(-1,1) buffer or Philox
__device__ __forceinline__ float4 add_noise(float4 v, const float4 nz, const float* noise, int row, int W0, int c4,
                                            const gfb_program_head& P, const Philox& rng, int e0, int col_begin,
                                            int rng_mode) {
  float4 u;
  if (rng_mode == 0) {
    u = noise ? reinterpret_cast<const float4*>(noise)[row * W0 + c4] : make_float4(0.f, 0.f, 0.f, 0.f);
  } else {
    const uint4 r4 = rng((uint32_t)(e0 + row), (uint32_t)P.step_index, (uint32_t)(P.step_index >> 32),
                         0x1000u + (uint32_t)(col_begin + (c4 << 2)));
    u = make_float4(sub(mul(u01(r4.x), 2.f), 1.f), sub(mul(u01(r4.y), 2.f), 1.f),
                    sub(mul(u01(r4.z), 2.f), 1.f), sub(mul(u01(r4.w), 2.f), 1.f));
  }
  if (nz.x != 0.f) v.x = add(v.x, mul(u.x, nz.x));
  if (nz.y != 0.f) v.y = add(v.y, mul(u.y, nz.y));
  if (nz.z != 0.f) v.z = add(v.z, mul(u.z, nz.z));
  if (nz.w != 0.f) v.w = add(v.w, mul(u.w, nz.w));
  return v;
}

// Issue the TMA loads of one slab: staged arrays [a_begin, a_end) of the plan (the early, the late or
// the prefetched group), `n_sum_rows` episode-sum rows, optionally the descriptor table.  All complete
// on `bar` (one arrival with the expected byte count).  Called by ALL lanes of warp 0, convergent: lane
// k describes transfer k (address arithmetic in parallel), the byte counts are summed across the warp
// for the expect-tx, and each lane's transfer is issued under a predicate -- no per-lane branch around
// an mbarrier / bulk-copy instruction (uniform-datapath rule, device_utils.cuh).
template <int TILE>
__device__ __forceinline__ void issue_slab_loads(const KParams& K, const Plan& plan, float* S, float* table_dst,
                                                 uint64_t* bar, int tile, int a_begin, int a_end, int n_sum_rows,
                                                 bool with_table, int lane, bool skip_cmd = false) {
  const int N = K.P.num_envs;
  const int e0 = tile * TILE;
  const uint32_t valid = (uint32_t)min(TILE, N - e0);
  const int n_arrays = a_end - a_begin;
  with_table = with_table && plan.table_words > 0;  // (phase sets without observation rows have no table)
  const int n_ops = n_arrays + n_sum_rows + (with_table ? 1 : 0);
  // (at most GFB_MAX_STAGED + GFB_MAX_REWARD_TERMS + 1 transfers: two sweeps of the warp)
  float* dst[2];
  const float* src[2];
  uint32_t bytes[2];
  uint32_t mine = 0;
#pragma unroll
  for (int sweep = 0; sweep < 2; ++sweep) {
    const int op = sweep * 32 + lane;
    dst[sweep] = S;
    src[sweep] = nullptr;
    bytes[sweep] = 0;
    if (op < n_arrays) {
      const int i = a_begin + op;
      const int buf = plan.staged_buf[i];
      // (skip_cmd: the command vectors keep their slot in the slab but are loaded and rewritten by their
      //  owner threads -- "split groups" in post_kernel)
      const bool skip = skip_cmd && buf >= GFB_B_COMMAND0 && buf < GFB_B_COMMAND0 + GFB_MAX_COMMANDS;
      dst[sweep] = S + plan.staged_off[i];
      src[sweep] = reinterpret_cast<const float*>(K.b.buf[buf]) + (size_t)e0 * plan.staged_words[i];
      bytes[sweep] = skip ? 0u : (uint32_t)plan.staged_words[i] * valid * 4u;
    } else if (op < n_arrays + n_sum_rows) {
      const int r = op - n_arrays;
      dst[sweep] = S + plan.sums_off + r * TILE;
      src[sweep] = GFB_BUF(const float, GFB_B_EP_SUMS) + (size_t)r * N + e0;
      bytes[sweep] = valid * 4u;
    } else if (op < n_ops) {
      dst[sweep] = table_dst;
      src[sweep] = reinterpret_cast<const float*>(K.cols);
      bytes[sweep] = (uint32_t)plan.table_words * 4u;
    }
    mine += bytes[sweep];
  }
  const uint32_t total = __reduce_add_sync(0xffffffffu, mine);
  mbar_expect_tx(lane == 0, bar, total);  // (also with total == 0: the phase then completes at once)
  __syncwarp();
#pragma unroll
  for (int sweep = 0; sweep < 2; ++sweep) {
    if (sweep * 32 < n_ops)  // (warp-uniform)
      bulk_load(bytes[sweep] != 0u, dst[sweep], src[sweep], bytes[sweep], bar);
  }
  __syncwarp();
}

// What a user-defined term lowered to device code (genesis_forge_b200/expr.py) reads: the slab rows and
// body-frame registers the plan already has (pos / quat / vel / ang, lin_b / ang_b / grav_b), otherwise its
// env's rows of the engine / environment arrays in global memory; the owner thread's registers (episode
// counters, this step's termination flags, the inverse base quaternion) and stash; its live params.
// The reset path of the observation terms (spec_kernel.cu) reads global memory only (S, st: null).
struct UserCtx {
  const gfb_buffers& b;
  size_t e;
  int ep_len, max_len;
  bool terminated, truncated;
  float iw;
  V3 iq;
  V3 lin_b, ang_b, grav_b;
  const float* S;
  int tid;
  const float* st;
  const Plan& plan;
  const float* p;
  int n_envs;  // (global-memory reads of the air-time planes)
  bool active;  // a real env: lanes that shadow env N-1 in a tail slab do not store state
};

// First stash word of the lowered user-defined observation values (gfb200.cu build_plan: st_user)
__device__ __forceinline__ int user_stash_base(const gfb_program_head& SP) {
  int s = 9;
  for (int m = 0; m < SP.n_contact; ++m) s += SP.contact[m].n_links * (SP.contact[m].track_air_time ? 5 : 1);
  return s;
}

#if defined(GFB_SPEC) && defined(GFB_SPEC_USER_TERMS)
// NaN propagating; on a tie (+0 / -0) the second operand.  amax / amin pass (element, accumulator), so a
// row's first element is kept on a tie, as torch-CPU does.
__device__ __forceinline__ float gfb_user_min(float a, float b) { return (a < b || a != a) ? a : b; }
__device__ __forceinline__ float gfb_user_max(float a, float b) { return (a > b || a != a) ? a : b; }
// torch.clamp: x is kept on a tie; a NaN bound propagates, except a NaN Python-scalar bound given alone
// (a Python float or a live param), which torch-CPU ignores
__device__ __forceinline__ float gfb_user_clamp_lo(float x, float lo) { return (x < lo || lo != lo) ? lo : x; }
__device__ __forceinline__ float gfb_user_clamp_hi(float x, float hi) { return (x > hi || hi != hi) ? hi : x; }
__device__ __forceinline__ float gfb_user_clamp_lo_scalar(float x, float lo) { return x < lo ? lo : x; }
__device__ __forceinline__ float gfb_user_clamp_hi_scalar(float x, float hi) { return x > hi ? hi : x; }
// float -> int32 as torch-CPU (x86 cvttss2si): truncation; NaN, +-Inf and |x| >= 2^31 give INT_MIN
__device__ __forceinline__ int gfb_user_f2i(float x) {
  return (x > -2147483904.0f && x < 2147483648.0f) ? __float2int_rz(x) : (int)0x80000000;
}
__device__ __forceinline__ int gfb_user_mod(int a, int b) {  // torch's remainder: the sign of the divisor
  const int r = a % b;
  return (r != 0 && ((r < 0) != (b < 0))) ? r + b : r;
}
GFB_SPEC_USER_TERMS
#endif

// Blocks per SM promised to the register allocator: the generic build assumes 768 threads per SM; a
// specialised build knows its slab's shared memory and promises only what that admits (spec.py)
#ifdef GFB_SPEC
#define GFB_MIN_BLOCKS(TILE_) (gfb_spec::MIN_BLOCKS)
#else
#define GFB_MIN_BLOCKS(TILE_) (768 / (TILE_))
#endif

template <int TILE>
__global__ void __launch_bounds__(TILE, GFB_MIN_BLOCKS(TILE)) post_kernel(const __grid_constant__ KParams K) {
  extern __shared__ __align__(128) float Sbase[];
  __shared__ __align__(8) uint64_t bars[3];  // [0] slab loads, [1] late load group, [2] prefetched arrays
  __shared__ int32_t s_term_count[GFB_MAX_TERMINATION_TERMS];
  __shared__ uint32_t s_rew_flags[GFB_MAX_REWARD_TERMS];
  __shared__ uint32_t s_reset_bits[TILE / 32];
  __shared__ uint32_t s_status;
  __shared__ int s_arrived;    // warps of this slab that are past the termination phase
  __shared__ int s_next_tile;  // the ticket drawn for the block's next slab

  // P: live values (weights, thresholds, ranges, dt, seeds) -- always the kernel parameters.
  // SP / plan / ph: the STRUCTURE of the term table and of the slab.  In the generic build they are
  // the kernel parameters too (an interpreter); in a specialised build (GFB_SPEC) they are
  // compile-time constants, so the term loops unroll, every switch folds to its one case and all
  // shared-memory offsets become immediates.
  const gfb_program_head& P = K.P;
#ifdef GFB_SPEC
  const gfb_program_head& SP = gfb_spec::kP;
  const Plan& plan = gfb_spec::kPlan;
  constexpr uint32_t ph = gfb_spec::PHASES;
  constexpr bool use_tma = true;  // the host only selects a specialised kernel when TMA is usable
#else
  const gfb_program_head& SP = K.P;
  const Plan& plan = K.plan;
  const uint32_t ph = K.phases;
  const bool use_tma = K.tma_ok != 0;
#endif
  constexpr int NW = TILE / 32;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int N = P.num_envs;
  const int D = SP.num_dofs;
  const bool stage_sums = (ph & (GFB_PHASE_REWARD | GFB_PHASE_RESET)) != 0 && SP.n_reward > 0;
  const int n_sum_rows = stage_sums ? SP.n_reward : 0;
  const int n_tiles = K.s.n_tiles;
  // two load groups (plan.h): the late one follows the contact phase into the contact slots' memory
  const bool two_groups = plan.n_early < plan.n_staged || plan.sums_late != 0;
  const int n_sum_rows_early = plan.sums_late ? 0 : n_sum_rows;
  // Split groups (no contact slots staged): what the per-env phase reads -- quat / pos / vel / ang and the
  // episode-sum rows -- is the PREFETCHED group (requested in the middle of the previous slab, bars[2]);
  // what only the observation rows read -- joint state, targets (bars[0], requested when the previous
  // slab was finished) -- is awaited just before the rows are assembled, so its latency hides behind the
  // per-env phase.  The command vectors (read by both) are loaded by their owner threads into registers
  // at the top of the slab and written to their slots before the rewards; the rewards read their own
  // joint positions from global memory.
  const bool split_x = !two_groups && plan.n_prefetch > 0;
  const int n_sum_rows_pf = split_x ? n_sum_rows : 0;
  const int n_sum_rows_main = split_x ? 0 : n_sum_rows_early;
  float* const S = Sbase;
  float* const Tbl = Sbase + plan.cols_off;  // descriptor table, loaded once per block
  const Philox rng(P.rng_seed);
  // reset_reward_log: the reset phase logs and clears the episode sums (reward manager enabled)
  const bool reward_log = SP.n_reward > 0 && !(SP.manager_flags & GFB_MF_REWARD_DISABLED);
  // exact sums of the episode quotients (tail_math.cuh), in the plan's shared memory (RESET launches): per
  // slab two 32-bit counters of 16-bit pieces per word, per block one 64-bit word (word i: thread i)
  const int n_acc_words = (ph & GFB_PHASE_RESET) && reward_log ? SP.n_reward * XS_WORDS : 0;
  int* const s_rew_acc = reinterpret_cast<int*>(Sbase + plan.rew_acc_off);
  unsigned long long* const s_rew_blk = reinterpret_cast<unsigned long long*>(s_rew_acc + 2 * n_acc_words);

  if (tid == 0) s_arrived = 0;
  for (int i = tid; i < n_acc_words; i += TILE) s_rew_blk[i] = 0ull;
  // barrier setup in straight-line code (thread 0 selected by predicate: uniform-datapath rule)
  mbar_init(tid == 0, &bars[0], 1);
  mbar_init(tid == 0, &bars[1], 1);
  mbar_init(tid == 0, &bars[2], 1);
  if (warp == 0) fence_mbar_init();  // (warp-uniform branch)
  __syncthreads();
  if (use_tma) {
    if (warp == 0 && (int)blockIdx.x < n_tiles) {
      if (plan.n_prefetch > 0)
        issue_slab_loads<TILE>(K, plan, Sbase, Tbl, &bars[2], blockIdx.x, 0, plan.n_prefetch, n_sum_rows_pf, false, lane);
      issue_slab_loads<TILE>(K, plan, Sbase, Tbl, &bars[0], blockIdx.x, plan.n_prefetch, plan.n_early, n_sum_rows_main,
                             true, lane, split_x);
    }
  } else {
    const int32_t* src = reinterpret_cast<const int32_t*>(K.cols);
    int32_t* dst = reinterpret_cast<int32_t*>(Tbl);
    for (int w = tid; w < plan.table_words; w += TILE) dst[w] = src[w];
  }

  // Slabs after the first come from a ticket counter.  A returning atomic takes microseconds while the
  // memory system is saturated and nothing a slab does may wait for a global round trip (tail.cuh), so
  // two tickets are kept in flight: the one drawn during the PREVIOUS slab names the next slab (it is
  // needed in the middle of this one, for the prefetch), the one drawn now the slab after that.
  uint32_t ticket = 0;  // (thread 0) drawn a slab ago
  if (tid == 0) ticket = atomicAdd(K.s.counters + CTR_TICKET, 1u);

  int it = 0;
  for (int tile = blockIdx.x; tile < n_tiles; ++it) {
  const int e0 = tile * TILE;
  const int valid = min(TILE, N - e0);
  const bool active = tid < valid;
  const int e = active ? e0 + tid : N - 1;  // inactive lanes shadow the last env and never write

  if (tid < GFB_MAX_TERMINATION_TERMS) s_term_count[tid] = 0;
  if (tid == 0) s_status = 0;
  for (int i = tid; i < 2 * n_acc_words; i += TILE) s_rew_acc[i] = 0;
  if (tid < GFB_MAX_REWARD_TERMS) s_rew_flags[tid] = 0u;

  // ------------------------------------------------------------------------------------------
  // slab loads: every staged array and the episode-sum rows are single cp.async.bulk transfers;
  // the lanes of warp 0 issue them in parallel, all complete on the stage's mbarrier
  // ------------------------------------------------------------------------------------------
  if (!use_tma) {
    for (int i = 0; i < plan.n_early; ++i) {
      const int words = plan.staged_words[i] * valid;
      const float* src = reinterpret_cast<const float*>(K.b.buf[plan.staged_buf[i]]) +
                         (size_t)e0 * plan.staged_words[i];
      float* dst = S + plan.staged_off[i];
      for (int w = tid; w < words; w += TILE) dst[w] = src[w];
    }
    if (stage_sums && !plan.sums_late) {
      const float* sums = GFB_BUF(const float, GFB_B_EP_SUMS);
      for (int r = 0; r < SP.n_reward; ++r)
        if (active) S[plan.sums_off + r * TILE + tid] = sums[(size_t)r * N + e];
    }
  }

  // per-env scalars straight into registers while the slab is in flight
  int ep_len = GFB_BUF(const int32_t, GFB_B_EPISODE_LENGTH)[e];
  int max_len = P.base_max_episode_length > 0 ? GFB_BUF(const int32_t, GFB_B_MAX_EPISODE_LENGTH)[e] : 0;
  float ep_secs = 0.0f, action_rate = 0.0f;
  if (ph & (GFB_PHASE_REWARD | GFB_PHASE_RESET)) {
    if (K.b.buf[GFB_B_EP_SECONDS]) ep_secs = GFB_BUF(const float, GFB_B_EP_SECONDS)[e];
  }
  if ((ph & GFB_PHASE_REWARD) && K.b.buf[GFB_B_ACTION_RATE])
    action_rate = GFB_BUF(const float, GFB_B_ACTION_RATE)[e];

#ifdef GFB_SPEC
  // specialised build: the tracked links are compile-time constants, so every link quaternion and
  // every air-time word of this env is requested here, while the slab is still in flight
  // (independent loads, their latency hidden behind the slab wait), instead of one dependent global
  // load per target inside the contact loops
  float4 tq_all[gfb_spec::N_TARGETS];
  float air_all[gfb_spec::N_TARGETS][4];
  if ((ph & GFB_PHASE_CONTACT) && SP.n_contact > 0) {
    const float4* lq = GFB_BUF(const float4, GFB_B_LINKS_QUAT) + (size_t)e * SP.n_links_total;
    int k = 0;
    GFB_UNROLL_TERMS
    for (int m = 0; m < SP.n_contact; ++m) {
      const int Lc = SP.contact[m].n_links;
      GFB_UNROLL_TERMS
      for (int t = 0; t < Lc; ++t, ++k) {
        tq_all[k] = lq[SP.contact[m].link_ids[t]];
        if (SP.contact[m].track_air_time) {
          const float* air = GFB_BUF(const float, GFB_B_AIR0 + m);
          const size_t base = (size_t)e * Lc + t, plane = (size_t)N * Lc;
          air_all[k][0] = air[base]; air_all[k][1] = air[plane + base];
          air_all[k][2] = air[2 * plane + base]; air_all[k][3] = air[3 * plane + base];
        }
      }
    }
  }
#endif

#ifdef GFB_SPEC
  float cmd_r[GFB_MAX_COMMANDS][GFB_MAX_COMMAND_DIMS];  // split groups: own command vectors, requested here
  if (split_x && (ph & (GFB_PHASE_REWARD | GFB_PHASE_COMMAND | GFB_PHASE_RESET | GFB_PHASE_OBSERVE))) {
    GFB_UNROLL_TERMS
    for (int k = 0; k < SP.n_command; ++k) {
      const int nd = SP.command[k].n_dims;
      if (nd == 0 || plan.off_cmd[k] < 0) continue;
      const float* cg = GFB_BUF(const float, GFB_B_COMMAND0 + k) + (size_t)e * nd;
      GFB_UNROLL_TERMS
      for (int i = 0; i < nd; ++i) cmd_r[k][i] = cg[i];
    }
  }
#endif

  // one warp polls the slab's mbarrier, the block barrier releases the rest
  if (use_tma && warp == 0) {
    if (plan.n_prefetch > 0) mbar_wait(&bars[2], (uint32_t)(it & 1));
    if (!split_x) mbar_wait(&bars[0], (uint32_t)(it & 1));
  }
  __syncthreads();

  // slab copies that need no arithmetic (entity cache: base_pos / base_quat are copies of pos / quat)
  if (ph & GFB_PHASE_ENTITY) {
    if (use_tma && !(K.debug & 16u)) {
      if (warp == 0) {  // lane i copies staged array i (predicated issue, every lane commits)
        const int i = min(lane, GFB_MAX_STAGED - 1);
        const bool mine = lane < plan.n_staged && plan.staged_store[i] >= 0 && K.b.buf[max(plan.staged_store[i], 0)] != nullptr;
        float* dst = mine ? reinterpret_cast<float*>(K.b.buf[plan.staged_store[i]]) + (size_t)e0 * plan.staged_words[i] : nullptr;
        bulk_store(mine, dst, S + plan.staged_off[i], (uint32_t)plan.staged_words[i] * (uint32_t)valid * 4u);
        bulk_commit();
        __syncwarp();
      }
    } else {
      for (int i = 0; i < plan.n_staged; ++i)
        if (plan.staged_store[i] >= 0 && K.b.buf[plan.staged_store[i]]) {
          float* dst = reinterpret_cast<float*>(K.b.buf[plan.staged_store[i]]) + (size_t)e0 * plan.staged_words[i];
          const float* src = S + plan.staged_off[i];
          const int words = plan.staged_words[i] * valid;
          for (int w = tid; w < words; w += TILE) dst[w] = src[w];
        }
    }
  }

  float* st = S + plan.stash_off + tid * plan.stash_stride;
  uint32_t status = 0;

  // ------------------------------------------------------------------------------------------
  // entity: inverse base quaternion and body-frame vectors
  // ------------------------------------------------------------------------------------------
  float iw = 1.0f;
  V3 iq = {0.f, 0.f, 0.f};
  if (ph & GFB_PHASE_ENTITY) {
    const float4 q = *reinterpret_cast<const float4*>(S + plan.off_quat + tid * 4);
    iw = q.x;  // q * (1,-1,-1,-1)
    iq.x = -q.y;
    iq.y = -q.z;
    iq.z = -q.w;
    if (active && K.b.buf[GFB_B_INV_BASE_QUAT])
      GFB_BUF(float4, GFB_B_INV_BASE_QUAT)[e] = make_float4(iw, iq.x, iq.y, iq.z);
  } else if (K.b.buf[GFB_B_INV_BASE_QUAT]) {
    const float4 q = GFB_BUF(const float4, GFB_B_INV_BASE_QUAT)[e];
    iw = q.x;
    iq.x = q.y;
    iq.y = q.z;
    iq.z = q.w;
  }
  V3 lin_b = {0.f, 0.f, 0.f}, ang_b = {0.f, 0.f, 0.f}, grav_b = {0.f, 0.f, 0.f};
  if (plan.needs & NEED_LIN) {
    const float* v = S + plan.off_vel + tid * 3;
    lin_b = rotate(V3{v[0], v[1], v[2]}, iw, iq);
    st[3] = lin_b.x; st[4] = lin_b.y; st[5] = lin_b.z;
  }
  if (plan.needs & NEED_ANG) {
    const float* v = S + plan.off_ang + tid * 3;
    ang_b = rotate(V3{v[0], v[1], v[2]}, iw, iq);
    st[0] = ang_b.x; st[1] = ang_b.y; st[2] = ang_b.z;
  }
  if (plan.needs & NEED_GRAV) {
    grav_b = rotate(V3{0.0f, 0.0f, -1.0f}, iw, iq);
    st[6] = grav_b.x; st[7] = grav_b.y; st[8] = grav_b.z;
  }

  // ------------------------------------------------------------------------------------------
  // contacts: ordered net force / mean position per tracked link, then air time
  // ------------------------------------------------------------------------------------------
  if ((ph & GFB_PHASE_CONTACT) && SP.n_contact > 0) {
    const int C = SP.n_contact_slots, L = SP.n_links_total;
    const int32_t* la = reinterpret_cast<const int32_t*>(S + plan.off_cla) + tid * C;
    const int32_t* lb = reinterpret_cast<const int32_t*>(S + plan.off_clb) + tid * C;
    const float* cf = S + plan.off_cforce + tid * C * 3;
    const float* cp = S + plan.off_cpos + tid * C * 3;
    // contact_manager.py:401-403: any NaN/Inf force is zeroed (and reported)
    bool bad = false;
    for (int k = 0; k < C * 3; ++k) bad |= !finite_f(cf[k]);
    if (bad && active) status |= GFB_STATUS_BAD_CONTACT;
    const float4* lq = GFB_BUF(const float4, GFB_B_LINKS_QUAT) + (size_t)e * L;
#ifdef GFB_SPEC
    int k_target = 0;
#endif

    GFB_UNROLL_TERMS
    for (int m = 0; m < SP.n_contact; ++m) {
      const gfb_contact_manager& cm = P.contact[m];
      const gfb_contact_manager& cs_ = SP.contact[m];
      const int Lc = cs_.n_links;
      if (cs_.disabled) {  // contact_manager.py:331-336: a disabled manager keeps its last results
        const float* cg = GFB_BUF(const float, GFB_B_CONTACTS0 + m) + (size_t)e * Lc * 3;
        for (int t = 0; t < Lc; ++t) {
          st[plan.st_cnorm[m] + t] = norm3(cg[t * 3], cg[t * 3 + 1], cg[t * 3 + 2]);
          if (cs_.track_air_time) {
            const float* air = GFB_BUF(const float, GFB_B_AIR0 + m);
            const size_t base = (size_t)e * Lc + t, plane = (size_t)N * Lc;
            float* sa = st + plan.st_air[m] + t * 4;
            sa[0] = air[base]; sa[1] = air[plane + base]; sa[2] = air[2 * plane + base]; sa[3] = air[3 * plane + base];
          }
        }
#ifdef GFB_SPEC
        k_target += Lc;
#endif
        continue;
      }
      // results go straight from registers to the (N, Lc, 3) outputs: staging them for a TMA store
      // would cost 6*Lc words of shared memory per env, i.e. resident warps
      float* fout = GFB_BUF(float, GFB_B_CONTACTS0 + m) + (size_t)e * Lc * 3;
      float* pout = GFB_BUF(float, GFB_B_CONTACT_POS0 + m) + (size_t)e * Lc * 3;
      GFB_UNROLL_TERMS
      for (int t = 0; t < Lc; ++t) {
        const int target = cs_.link_ids[t];
#ifdef GFB_SPEC
        const int kt = k_target++;
        const float4 tq = tq_all[kt];
#else
        const float4 tq = lq[target];
#endif
        float fx = 0.f, fy = 0.f, fz = 0.f, px = 0.f, py = 0.f, pz = 0.f, cnt = 0.f;
        // Which contact slots involve this link: a cheap compare pass builds a per-lane bit mask
        // (one word of hits, one of "the target is link_b"), then only the hits are
        // visited, in ascending slot order (= the oracle's summation order).  A warp iterates
        // max-over-lanes(#hits) times -- typically 1-2 -- instead of paying the rotate body for every
        // one of the C slots under divergence.
        for (int c0 = 0; c0 < C; c0 += 32) {  // 32 slots per mask word
          const int cn = min(32, C - c0);
          uint32_t hits = 0, hit_is_b = 0;
          for (int j = 0; j < cn; ++j) {
            const int a = la[c0 + j], b2 = lb[c0 + j];
            const bool is_a = a == target, is_b = b2 == target;
            bool hit = is_a | is_b;
            if (cs_.has_with_filter) {
              bool keep = false;
              for (int w = 0; w < cs_.n_with; ++w) {
                const int wl = cs_.with_ids[w];
                keep |= (is_a && b2 == wl) || (is_b && a == wl);
              }
              hit = hit && keep;
            }
            hits |= (hit ? 1u : 0u) << j;
            hit_is_b |= ((hit && is_b) ? 1u : 0u) << j;
          }
          while (hits) {
            const int j = __ffs(hits) - 1;
            const int c = c0 + j;
            const bool is_b = (hit_is_b >> j) & 1u;
            hits &= hits - 1;
            float x = cf[c * 3 + 0], y = cf[c * 3 + 1], z = cf[c * 3 + 2];
            if (bad) {
              x = finite_f(x) ? x : 0.f;
              y = finite_f(y) ? y : 0.f;
              z = finite_f(z) ? z : 0.f;
            }
            V3 f = is_b ? V3{x, y, z} : V3{-x, -y, -z};  // kernel.py:75-78
            f = inv_rotate_ti(f, tq.x, V3{tq.y, tq.z, tq.w});
            fx = add(fx, f.x); fy = add(fy, f.y); fz = add(fz, f.z);
            px = add(px, cp[c * 3 + 0]); py = add(py, cp[c * 3 + 1]); pz = add(pz, cp[c * 3 + 2]);
            cnt = add(cnt, 1.0f);
          }
        }
        if (cnt > 0.f) {  // kernel.py:85-90
          px = fdiv(px, cnt); py = fdiv(py, cnt); pz = fdiv(pz, cnt);
        }
        if (active) {
          fout[t * 3 + 0] = fx; fout[t * 3 + 1] = fy; fout[t * 3 + 2] = fz;
          pout[t * 3 + 0] = px; pout[t * 3 + 1] = py; pout[t * 3 + 2] = pz;
        }
        const float nrm = norm3(fx, fy, fz);
        st[plan.st_cnorm[m] + t] = nrm;

        if (cs_.track_air_time) {  // contact_manager.py:434-477
#ifdef GFB_SPEC
          float last_air = air_all[kt][0], cur_air = air_all[kt][1];
          float last_con = air_all[kt][2], cur_con = air_all[kt][3];
#else
          const float* air = GFB_BUF(const float, GFB_B_AIR0 + m);
          const size_t base = (size_t)e * Lc + t, plane = (size_t)N * Lc;
          float last_air = air[base], cur_air = air[plane + base];
          float last_con = air[2 * plane + base], cur_con = air[3 * plane + base];
#endif
          const float dt = cm.scene_dt;
          const bool is_contact = nrm > cm.air_time_threshold;
          const bool new_contact = (cur_air > 0.f) && is_contact;
          const bool new_detach = (cur_con > 0.f) && !is_contact;
          last_air = new_contact ? add(cur_air, dt) : last_air;
          const float cur_air2 = !is_contact ? add(cur_air, dt) : 0.f;
          last_con = new_detach ? add(cur_con, dt) : last_con;
          const float cur_con2 = is_contact ? add(cur_con, dt) : 0.f;
          float* sa = st + plan.st_air[m] + t * 4;
          sa[0] = last_air; sa[1] = cur_air2; sa[2] = last_con; sa[3] = cur_con2;
        }
      }
    }
  } else if (SP.n_contact > 0 && (ph & (GFB_PHASE_REWARD | GFB_PHASE_TERMINATION | GFB_PHASE_OBSERVE))) {
    // split execution: contact results of an earlier launch come back from global memory
    for (int m = 0; m < SP.n_contact; ++m) {
      const gfb_contact_manager& cm = P.contact[m];
      const gfb_contact_manager& cs_ = SP.contact[m];
      const float* cg = GFB_BUF(const float, GFB_B_CONTACTS0 + m) + (size_t)e * cs_.n_links * 3;
      for (int t = 0; t < cs_.n_links; ++t) {
        st[plan.st_cnorm[m] + t] = norm3(cg[t * 3], cg[t * 3 + 1], cg[t * 3 + 2]);
        if (cs_.track_air_time) {
          const float* air = GFB_BUF(const float, GFB_B_AIR0 + m);
          const size_t base = (size_t)e * cs_.n_links + t, plane = (size_t)N * cs_.n_links;
          float* sa = st + plan.st_air[m] + t * 4;
          sa[0] = air[base]; sa[1] = air[plane + base]; sa[2] = air[2 * plane + base]; sa[3] = air[3 * plane + base];
        }
      }
    }
  }

  {
    const uint32_t warp_status = __reduce_or_sync(0xffffffffu, status);
    if (lane == 0 && warp_status) atomicOr(&s_status, warp_status);
  }

  // ------------------------------------------------------------------------------------------
  // late load group: the arrays that only rewards / resample / reset / observations read (joint
  // state, targets, commands, episode-sum rows) now replace the contact slots in shared memory;
  // the terminations below run while they are in flight
  // ------------------------------------------------------------------------------------------
  if (two_groups) {
    __syncthreads();  // every thread is done with the contact slots
    if (use_tma) {
      if (warp == 0) {
        fence_async_smem();  // generic-proxy reads above, async-proxy writes below
        issue_slab_loads<TILE>(K, plan, S, Tbl, &bars[1], tile, plan.n_early, plan.n_staged,
                               plan.sums_late ? n_sum_rows : 0, false, lane);
      }
    } else {
      for (int i = plan.n_early; i < plan.n_staged; ++i) {
        const int words = plan.staged_words[i] * valid;
        const float* src = reinterpret_cast<const float*>(K.b.buf[plan.staged_buf[i]]) +
                           (size_t)e0 * plan.staged_words[i];
        float* dst = S + plan.staged_off[i];
        for (int w = tid; w < words; w += TILE) dst[w] = src[w];
      }
      if (stage_sums && plan.sums_late) {
        const float* sums = GFB_BUF(const float, GFB_B_EP_SUMS);
        for (int r = 0; r < SP.n_reward; ++r)
          if (active) S[plan.sums_off + r * TILE + tid] = sums[(size_t)r * N + e];
      }
    }
  }

  // ------------------------------------------------------------------------------------------
  // terminations
  // ------------------------------------------------------------------------------------------
  bool terminated = false, truncated = false;
  if (ph & GFB_PHASE_TERMINATION) {
    GFB_UNROLL_TERMS
    for (int t = 0; t < SP.n_termination; ++t) {
      const gfb_termination_term& tt = P.termination[t];
      const gfb_termination_term& ts = SP.termination[t];
      bool v = false;
      switch (ts.op) {
        case GFB_T_TIMEOUT:
          v = P.base_max_episode_length > 0 && ep_len > max_len;
          break;
        case GFB_T_BAD_ORIENTATION: {
          // asin(clamp(NaN, max=0.99)) > limit is False in the reference; fminf would drop the NaN
          const float tilt = norm2(grav_b.x, grav_b.y);
          v = !(ep_len <= ts.i0) && (tilt == tilt) && (fminf(tilt, 0.99f) >= tt.p[0]);
        } break;
        case GFB_T_BASE_HEIGHT_MIN:
          v = S[plan.off_pos + tid * 3 + 2] < tt.p[0];
          break;
        case GFB_T_OUT_OF_BOUNDS: {
          const float x = S[plan.off_pos + tid * 3], y = S[plan.off_pos + tid * 3 + 1];
          v = (x < tt.p[0]) | (x > tt.p[1]) | (y < tt.p[2]) | (y > tt.p[3]);
        } break;
        case GFB_T_HAS_CONTACT: {
          int n = 0;
          for (int l = 0; l < SP.contact[ts.mgr].n_links; ++l) n += st[plan.st_cnorm[ts.mgr] + l] > tt.p[0];
          v = n >= ts.i0;
        } break;
        case GFB_T_CONTACT_FORCE:
        case GFB_T_CONTACT_FORCE_GRACE: {
          bool any = false;
          for (int l = 0; l < SP.contact[ts.mgr].n_links; ++l) any |= st[plan.st_cnorm[ts.mgr] + l] > tt.p[0];
          v = any && (ts.op == GFB_T_CONTACT_FORCE || !(ep_len <= ts.i0));
        } break;
        case GFB_T_EXTERNAL:  // user-defined term evaluated on the host before this launch
          v = GFB_BUF(const float, GFB_B_EXT_VALUES)[(size_t)ts.i0 * N + e] != 0.0f;
          break;
#if defined(GFB_SPEC) && defined(GFB_SPEC_USER_TERMS)
        case GFB_T_USER:  // user-defined term lowered to device code (generated header)
          v = user_termination(t, UserCtx{K.b, (size_t)e, ep_len, max_len, false, false, iw, iq, lin_b, ang_b, grav_b, S, tid,
                                          st, plan, tt.p, N, active});
          break;
#endif
        default:
          break;
      }
      v = v && active;
      if (ts.time_out) truncated |= v; else terminated |= v;
      const uint32_t votes = __ballot_sync(0xffffffffu, v);
      if (lane == 0 && votes) atomicAdd(&s_term_count[t], __popc(votes));
    }
  } else if (ph & (GFB_PHASE_REWARD | GFB_PHASE_RESET)) {
    if (K.b.buf[GFB_B_TERMINATED]) terminated = GFB_BUF(const uint8_t, GFB_B_TERMINATED)[e] != 0;
    if (K.b.buf[GFB_B_TRUNCATED]) truncated = GFB_BUF(const uint8_t, GFB_B_TRUNCATED)[e] != 0;
  }

  bool reset = false;
  if (ph & GFB_PHASE_RESET) {
    if (ph & GFB_PHASE_FORCED_RESET) {
      const uint8_t* mask = GFB_BUF(const uint8_t, GFB_B_FORCE_RESET);
      reset = mask ? (mask[e] != 0) : true;
    } else {
      reset = terminated | truncated;  // managed_env.py:308-310
    }
    reset = reset && active;
  }

  // ------------------------------------------------------------------------------------------
  // the slab's terminations are final: fire counts, ordered reset indices, step report (tail.cuh).
  // The LAST warp of the slab to get here does this for the whole slab; the others carry on.
  // ------------------------------------------------------------------------------------------
  const uint32_t reset_votes = __ballot_sync(0xffffffffu, reset);
  int last = 0;  // this warp is the slab's last one past the terminations
  if (ph & (GFB_PHASE_TERMINATION | GFB_PHASE_RESET)) {
    if (lane == 0) {
      s_reset_bits[warp] = reset_votes;
      __threadfence_block();
      last = atomicAdd(&s_arrived, 1) == NW - 1;
    }
    last = __shfl_sync(0xffffffffu, last, 0);
    if (last) {
      __threadfence_block();
      if (lane == 0) s_arrived = 0;
      if ((ph & GFB_PHASE_TERMINATION) && lane < SP.n_termination) {
        const int fired = atomicAdd(&s_term_count[lane], 0);
        if (fired) atomicAdd(K.s.term_count + lane, fired);
      }
      if (lane == 0) {
        const uint32_t slab_status = atomicOr(&s_status, 0u);
        if (slab_status) atomicOr(K.s.status, slab_status);
      }
      if (ph & GFB_PHASE_RESET) {
        // Nothing here waits for memory: the number of reset envs is a sum (fire-and-forget integer
        // atomic), and the slab's reset mask goes to the scratch array from which compact_kernel,
        // enqueued right behind this kernel, expands the ascending index list (aux_kernels.cuh).
        const uint32_t bits = lane < NW ? atomicOr(&s_reset_bits[lane], 0u) : 0u;
        if (lane < NW) K.s.tile_bits[(size_t)tile * NW + lane] = bits;
        int slab_resets = __popc(bits);
#pragma unroll
        for (int o = NW / 2; o > 0; o >>= 1) slab_resets += __shfl_xor_sync(0xffffffffu, slab_resets, o);
        if (lane == 0 && slab_resets) atomicAdd(K.s.counters + CTR_TOTAL_RESET, (uint32_t)slab_resets);
      }
    }
  }

  if (two_groups) {  // the late group has landed
    if (use_tma && warp == 0) mbar_wait(&bars[1], (uint32_t)(it & 1));
    __syncthreads();
  }

  // split groups: the owner threads' command vectors -> their slots (the transfer group skips them)
  if (split_x && (ph & (GFB_PHASE_REWARD | GFB_PHASE_COMMAND | GFB_PHASE_RESET | GFB_PHASE_OBSERVE))) {
    GFB_UNROLL_TERMS
    for (int k = 0; k < SP.n_command; ++k) {
      const int nd = SP.command[k].n_dims;
      if (nd == 0 || plan.off_cmd[k] < 0) continue;
      float* cs = S + plan.off_cmd[k] + tid * nd;
#ifdef GFB_SPEC
      GFB_UNROLL_TERMS
      for (int i = 0; i < nd; ++i) cs[i] = cmd_r[k][i];
#else
      const float* cg = GFB_BUF(const float, GFB_B_COMMAND0 + k) + (size_t)e * nd;
      for (int i = 0; i < nd; ++i) cs[i] = cg[i];
#endif
    }
  }

  // ------------------------------------------------------------------------------------------
  // rewards
  // ------------------------------------------------------------------------------------------
  float reward = 0.0f;
  if (ph & GFB_PHASE_REWARD) {
    ep_secs = add(ep_secs, P.env_dt);  // reward_manager.py:178
    float dof_dev = 0.0f;
    bool have_dof_dev = false;
    GFB_UNROLL_TERMS
    for (int r = 0; r < SP.n_reward; ++r) {
      const gfb_reward_term& rt = P.reward[r];
      const gfb_reward_term& rs = SP.reward[r];
      if (rt.weight == 0.0f || rs.op == GFB_R_NONE) continue;  // reward_manager.py:181-182
      float v = 0.0f;
      switch (rs.op) {
        case GFB_R_IS_ALIVE:
          v = terminated ? 0.0f : 1.0f;
          break;
        case GFB_R_TERMINATED:
          v = terminated ? 1.0f : 0.0f;
          break;
        case GFB_R_BASE_HEIGHT: {
          float z = S[plan.off_pos + tid * 3 + 2];
          float off = 0.0f;
          if (rs.flags & GFB_RF_TERRAIN_FLAT) off = rt.p[1];
          if (rs.flags & GFB_RF_TERRAIN_HEIGHT) {
            const float x = S[plan.off_pos + tid * 3], y = S[plan.off_pos + tid * 3 + 1];
            off = terrain_height(x, y, P.terrain_bounds, P.height_field_rows, P.height_field_cols,
                                 GFB_BUF(const float, GFB_B_HEIGHT_FIELD));
          }
          float target = rt.p[0];
          if (rs.flags & GFB_RF_TARGET_FROM_COMMAND) target = S[plan.off_cmd[rs.mgr] + tid * SP.command[rs.mgr].n_dims];
          if (rs.flags & GFB_RF_TARGET_FROM_TENSOR) target = GFB_BUF(const float, GFB_B_TARGET_HEIGHT)[e];
          v = sq(sub(sub(z, off), target));
        } break;
        case GFB_R_DOF_SIMILAR:
        case GFB_R_STAND_STILL: {
          if (!have_dof_dev) {
            // (split groups: own row from global memory -- an L2 hit, the slab transfer of the same rows
            //  is in flight or done; the staged copy is only awaited for the observation rows)
            const float* q = split_x ? GFB_BUF(const float, GFB_B_DOF_POS) + (size_t)e * D
                                     : S + plan.off_dof_pos + tid * D;
            if ((D & 3) == 0) {
              for (int d4 = 0; d4 < D; d4 += 4) {
                const float4 qv = *reinterpret_cast<const float4*>(q + d4);
                dof_dev = add(dof_dev, fabsf(sub(qv.x, P.default_dof_pos[d4])));
                dof_dev = add(dof_dev, fabsf(sub(qv.y, P.default_dof_pos[d4 + 1])));
                dof_dev = add(dof_dev, fabsf(sub(qv.z, P.default_dof_pos[d4 + 2])));
                dof_dev = add(dof_dev, fabsf(sub(qv.w, P.default_dof_pos[d4 + 3])));
              }
            } else {
              for (int d = 0; d < D; ++d) dof_dev = add(dof_dev, fabsf(sub(q[d], P.default_dof_pos[d])));
            }
            have_dof_dev = true;
          }
          v = dof_dev;
          if (rs.op == GFB_R_STAND_STILL) {
            const float* c = S + plan.off_cmd[rs.mgr] + tid * SP.command[rs.mgr].n_dims;
            v = mul(dof_dev, norm2(c[0], c[1]) < rt.p[0] ? 1.0f : 0.0f);
          }
        } break;
        case GFB_R_LIN_VEL_Z:
          v = sq(lin_b.z);
          break;
        case GFB_R_ANG_VEL_XY:
          v = add(sq(ang_b.x), sq(ang_b.y));
          break;
        case GFB_R_FLAT_ORIENTATION:
          v = add(sq(grav_b.x), sq(grav_b.y));
          break;
        case GFB_R_ACTION_RATE:
          v = action_rate;
          break;
        case GFB_R_BODY_ACC_EXP: {
          // rewards.py:196-249: 1 - exp(-s * (|d lin_b / dt| + |d ang_b / dt|)); previous body-frame
          // velocities are term state that is NOT cleared on reset; the first evaluation sees zeros
          float* prev = GFB_BUF(float, GFB_B_BODY_ACC_PREV) + (size_t)e * 6;
          float ax = 0.f, ay = 0.f, az = 0.f, bx = 0.f, by = 0.f, bz = 0.f;
          if (rt.p[1] != 0.0f) {
            ax = fdiv(sub(lin_b.x, prev[0]), P.env_dt); ay = fdiv(sub(lin_b.y, prev[1]), P.env_dt);
            az = fdiv(sub(lin_b.z, prev[2]), P.env_dt);
            bx = fdiv(sub(ang_b.x, prev[3]), P.env_dt); by = fdiv(sub(ang_b.y, prev[4]), P.env_dt);
            bz = fdiv(sub(ang_b.z, prev[5]), P.env_dt);
          }
          if (active) {
            prev[0] = lin_b.x; prev[1] = lin_b.y; prev[2] = lin_b.z;
            prev[3] = ang_b.x; prev[4] = ang_b.y; prev[5] = ang_b.z;
          }
          const float motion = add(norm3(ax, ay, az), norm3(bx, by, bz));
          v = sub(1.0f, expf(mul(-rt.p[0], motion)));
        } break;
        case GFB_R_TRACK_LIN_VEL:
        case GFB_R_TRACK_ANG_VEL: {
          float c0, c1, c2;
          if (rs.flags & GFB_RF_FIXED_COMMAND) {
            const float* c = GFB_BUF(const float, GFB_B_FIXED_COMMAND) + (size_t)e * 3;
            c0 = c[0]; c1 = c[1]; c2 = c[2];
          } else {
            const float* c = S + plan.off_cmd[rs.mgr] + tid * SP.command[rs.mgr].n_dims;
            c0 = c[0]; c1 = c[1]; c2 = c[2];
          }
          float err;
          if (rs.op == GFB_R_TRACK_LIN_VEL)
            err = add(sq(sub(c0, lin_b.x)), sq(sub(c1, lin_b.y)));
          else
            err = sq(sub(c2, ang_b.z));
          v = expf(fdiv(-err, rt.p[0]));
        } break;
        case GFB_R_HAS_CONTACT: {
          int n = 0;
          for (int l = 0; l < SP.contact[rs.mgr].n_links; ++l) n += st[plan.st_cnorm[rs.mgr] + l] > rt.p[0];
          v = n >= rs.i0 ? 1.0f : 0.0f;
        } break;
        case GFB_R_CONTACT_FORCE: {
          for (int l = 0; l < SP.contact[rs.mgr].n_links; ++l)
            v = add(v, fmaxf(sub(st[plan.st_cnorm[rs.mgr] + l], rt.p[0]), 0.0f));
        } break;
        case GFB_R_FEET_AIR_TIME: {
          for (int l = 0; l < SP.contact[rs.mgr].n_links; ++l) {
            const float* sa = st + plan.st_air[rs.mgr] + l * 4;
            const bool made = (sa[3] > 0.0f) && (sa[3] < rt.p[2]);  // contact_manager.py:198-224
            float a = mul(sub(sa[0], rt.p[0]), made ? 1.0f : 0.0f);
            if (rs.flags & GFB_RF_HAS_MAX) a = fminf(a, rt.p[1]);
            v = add(v, a);
          }
          if (rs.i0 >= 0) {
            const float* c = S + plan.off_cmd[rs.i0] + tid * SP.command[rs.i0].n_dims;
            v = mul(v, norm2(c[0], c[1]) > 0.1f ? 1.0f : 0.0f);
          }
        } break;
        case GFB_R_FEET_SLIDE: {
          const int Lc = SP.contact[rs.mgr].n_links;
          const float* lv = GFB_BUF(const float, GFB_B_LINKS_VEL) + (size_t)e * Lc * 3;
          for (int l = 0; l < Lc; ++l) {
            const float speed = norm3(lv[l * 3], lv[l * 3 + 1], lv[l * 3 + 2]);
            v = add(v, mul(speed, st[plan.st_cnorm[rs.mgr] + l] > 1.0f ? 1.0f : 0.0f));
          }
        } break;
        case GFB_R_EXTERNAL:  // user-defined term evaluated on the host before this launch
          v = GFB_BUF(const float, GFB_B_EXT_VALUES)[(size_t)rs.ext_col * N + e];
          break;
#if defined(GFB_SPEC) && defined(GFB_SPEC_USER_TERMS)
        case GFB_R_USER:  // user-defined term lowered to device code (generated header)
          v = user_reward(r, UserCtx{K.b, (size_t)e, ep_len, max_len, terminated, truncated, iw, iq, lin_b, ang_b, grav_b,
                                     S, tid, st, plan, rt.p, N, active});
          break;
#endif
        default:
          break;
      }
      v = mul(v, rt.weight);
      reward = add(reward, v);                 // reward_manager.py:188-189
      float* sum = S + plan.sums_off + r * TILE + tid;
      *sum = add(*sum, v);                      // reward_manager.py:192-193
    }
  }

  // ------------------------------------------------------------------------------------------
  // command resample on the resample boundary (command_manager.py:152-162)
  // ------------------------------------------------------------------------------------------
  if (ph & GFB_PHASE_COMMAND) {
    for (int k = 0; k < SP.n_command; ++k) {
      const gfb_command_manager& cm = P.command[k];
      const gfb_command_manager& ks = SP.command[k];
      if (!ks.enabled) continue;
      if (active && (ep_len % cm.resample_steps) == 0) {
        float* cs = S + plan.off_cmd[k] + tid * ks.n_dims;
        float* cg = GFB_BUF(float, GFB_B_COMMAND0 + k) + (size_t)e * ks.n_dims;
        const float* inj = GFB_BUF(const float, GFB_B_INJ_CMD_STEP0 + k);
        for (int i = 0; i < ks.n_dims; ++i) {
          float val;
          if (SP.rng_mode == 0) {
            val = inj ? inj[(size_t)e * ks.n_dims + i] : cs[i];
          } else {
            const uint4 x = rng((uint32_t)e, (uint32_t)P.step_index, (uint32_t)(P.step_index >> 32), 0x100u + k * 16 + i);
            val = add(mul(u01(x.x), sub(cm.hi[i], cm.lo[i])), cm.lo[i]);
          }
          cs[i] = val;
          cg[i] = val;
        }
      }
    }
  }

  // ------------------------------------------------------------------------------------------
  // in-library part of reset() for the envs that terminated / truncated
  // ------------------------------------------------------------------------------------------
  if (ph & GFB_PHASE_RESET) {
    if (reset) {
      // genesis_env.py:233-252
      if (K.b.buf[GFB_B_ENV_ACTIONS]) {
        float* a = GFB_BUF(float, GFB_B_ENV_ACTIONS) + (size_t)e * D;
        float* la = GFB_BUF(float, GFB_B_ENV_LAST_ACTIONS) + (size_t)e * D;
        for (int d = 0; d < D; ++d) { a[d] = 0.0f; la[d] = 0.0f; }
      }
      ep_len = 0;
      if (P.max_len_random_span > 0.0f && P.base_max_episode_length > 0) {
        float u;
        if (SP.rng_mode == 0) {
          const float* inj = GFB_BUF(const float, GFB_B_INJ_MAX_LEN);
          u = inj ? inj[e] : 0.0f;
        } else {
          const uint4 x = rng((uint32_t)e, (uint32_t)P.step_index, (uint32_t)(P.step_index >> 32), 0x200u);
          u = sub(mul(u01(x.x), 2.0f), 1.0f);
        }
        max_len = (int)rintf(add((float)P.base_max_episode_length, mul(u, P.max_len_random_span)));
        GFB_BUF(int32_t, GFB_B_MAX_EPISODE_LENGTH)[e] = max_len;
      }
      GFB_BUF(int32_t, GFB_B_EPISODE_LENGTH)[e] = 0;
      // command_manager.py:164-170
      for (int k = 0; k < SP.n_command; ++k) {
        const gfb_command_manager& cm = P.command[k];
        const gfb_command_manager& ks = SP.command[k];
        if (!ks.enabled) continue;
        float* cs = S + plan.off_cmd[k] + tid * ks.n_dims;
        float* cg = GFB_BUF(float, GFB_B_COMMAND0 + k) + (size_t)e * ks.n_dims;
        const float* inj = GFB_BUF(const float, GFB_B_INJ_CMD_RESET0 + k);
        for (int i = 0; i < ks.n_dims; ++i) {
          float val;
          if (SP.rng_mode == 0) {
            val = inj ? inj[(size_t)e * ks.n_dims + i] : cs[i];
          } else {
            const uint4 x = rng((uint32_t)e, (uint32_t)P.step_index, (uint32_t)(P.step_index >> 32), 0x300u + k * 16 + i);
            val = add(mul(u01(x.x), sub(cm.hi[i], cm.lo[i])), cm.lo[i]);
          }
          cs[i] = val;
          cg[i] = val;
        }
      }
      // contact_manager.py:316-329
      for (int m = 0; m < SP.n_contact; ++m)
        if (SP.contact[m].track_air_time)
          for (int k = 0; k < SP.contact[m].n_links * 4; ++k) st[plan.st_air[m] + k] = 0.0f;
    }
    // reward_manager.py:197-222: per-term episode mean over the reset envs, then clear.  Resets are
    // sparse: every reset env adds its quotient to the slab's exact sums (tail_math.cuh): two words, as
    // four native 32-bit shared atomics without a return value (a 64-bit one is a compare-and-swap loop,
    // whose latency the reset lane's slab waits for at the next barrier).
    if (reset) {
      if (reward_log) {
        GFB_UNROLL_TERMS
        for (int r = 0; r < SP.n_reward; ++r) {
          float* sum = S + plan.sums_off + r * TILE + tid;
          if (P.reward[r].weight != 0.0f) {
            uint32_t fl = 0;
            long long lo, hi;
            const int k = xs_split(fdiv(*sum, ep_secs), lo, hi, fl);
            int* acc = s_rew_acc + (r * XS_WORDS + k) * 2;
            int p0, p1, p2, p3;
            xs_pieces(lo, p0, p1);
            xs_pieces(hi, p2, p3);
            if (p0) atomicAdd(acc, p0);
            if (p1) atomicAdd(acc + 1, p1);
            if (p2) atomicAdd(acc + 2, p2);
            if (p3) atomicAdd(acc + 3, p3);
            if (fl) atomicOr(&s_rew_flags[r], fl);
          }
          *sum = 0.0f;
        }
      }
      ep_secs = 1e-10f;
    }
  }

#if defined(GFB_SPEC) && defined(GFB_SPEC_USER_OBS)
  // lowered user-defined observation terms: from what a stock column of this launch sees (the post-resample
  // command, the body-frame registers, the staged rows) into the stash words the GFB_O_USER columns read.
  // Class-style terms among them (GFB_SPEC_USER_OBS_STATE) store their state once per evaluation: a reset env
  // of this launch is evaluated again by the reset path (gfb_observe), which stores it, so it does not store here.
  if (ph & GFB_PHASE_OBSERVE)
    user_observations(UserCtx{K.b, (size_t)e, ep_len, max_len, terminated, truncated, iw, iq, lin_b, ang_b, grav_b, S,
                              tid, st, plan, nullptr, N,
#ifdef GFB_SPEC_USER_OBS_STATE
                              active && !reset},
#else
                              active},
#endif
                      st + user_stash_base(SP));
#endif

  // ------------------------------------------------------------------------------------------
  // per-env outputs
  // ------------------------------------------------------------------------------------------
  if (active) {
    if (ph & GFB_PHASE_TERMINATION) {
      GFB_BUF(uint8_t, GFB_B_TERMINATED)[e] = terminated;
      GFB_BUF(uint8_t, GFB_B_TRUNCATED)[e] = truncated;
      if (K.b.buf[GFB_B_DONES]) GFB_BUF(uint8_t, GFB_B_DONES)[e] = terminated | truncated;
    }
    if (ph & GFB_PHASE_REWARD) GFB_BUF(float, GFB_B_REWARD)[e] = reward;
    if ((ph & (GFB_PHASE_REWARD | GFB_PHASE_RESET)) && K.b.buf[GFB_B_EP_SECONDS])
      GFB_BUF(float, GFB_B_EP_SECONDS)[e] = ep_secs;
    if (ph & (GFB_PHASE_CONTACT | GFB_PHASE_RESET)) {
      for (int m = 0; m < SP.n_contact; ++m) {
        const gfb_contact_manager& cm = P.contact[m];
        const gfb_contact_manager& cs_ = SP.contact[m];
        if (!cs_.track_air_time) continue;
        if (!(ph & GFB_PHASE_CONTACT) && !reset) continue;
        float* air = GFB_BUF(float, GFB_B_AIR0 + m);
        const size_t plane = (size_t)N * cs_.n_links;
        for (int t = 0; t < cs_.n_links; ++t) {
          const float* sa = st + plan.st_air[m] + t * 4;
          const size_t base = (size_t)e * cs_.n_links + t;
          air[base] = sa[0]; air[plane + base] = sa[1]; air[2 * plane + base] = sa[2]; air[3 * plane + base] = sa[3];
        }
      }
    }
  }
  if (use_tma) {
    fence_async_smem();
    // split groups: the arrays only the observation rows read have had the whole per-env phase to land
    if (split_x && warp == 0) mbar_wait(&bars[0], (uint32_t)(it & 1));
  }
  __syncthreads();
  // split groups: the episode sums leave first -- their rows are refilled by the prefetch below
  if (use_tma && split_x && warp == 0 && n_sum_rows > 0) {
    const bool mine = lane < n_sum_rows;
    const int i = mine ? lane : 0;
    bulk_store(mine, GFB_BUF(float, GFB_B_EP_SUMS) + (size_t)i * N + e0, S + plan.sums_off + i * TILE,
               (uint32_t)valid * 4u);
    bulk_commit();
    __syncwarp();
  }
  // the per-env phase is over: quat / pos / vel / ang of this slab are dead -- warp 0 refills them with
  // the next slab's rows, which land while the observation rows below are assembled
  int next_tile = 0;
  if (warp == 0) {
    next_tile = (int)gridDim.x + (int)__shfl_sync(0xffffffffu, ticket, 0);
    if (lane == 0) {
      s_next_tile = next_tile;
      ticket = atomicAdd(K.s.counters + CTR_TICKET, 1u);  // (names the slab after the next one)
    }
    if (use_tma && next_tile < n_tiles && plan.n_prefetch > 0) {
      bulk_wait_all_read();  // the entity-cache (and episode-sum) stores have read their slabs
      issue_slab_loads<TILE>(K, plan, Sbase, Tbl, &bars[2], next_tile, 0, plan.n_prefetch, n_sum_rows_pf, false, lane);
    }
  }

  // ------------------------------------------------------------------------------------------
  // slab outputs: episode sums
  // ------------------------------------------------------------------------------------------
  if (use_tma) {
    if (!split_x && warp == 0 && n_sum_rows > 0) {  // lane i stores row i (GFB_MAX_REWARD_TERMS <= 32)
      const bool mine = lane < n_sum_rows;
      const int i = mine ? lane : 0;
      bulk_store(mine, GFB_BUF(float, GFB_B_EP_SUMS) + (size_t)i * N + e0, S + plan.sums_off + i * TILE,
                 (uint32_t)valid * 4u);
      bulk_commit();
      __syncwarp();
    }
  } else {
    if (stage_sums && active) {
      float* sums = GFB_BUF(float, GFB_B_EP_SUMS);
      for (int r = 0; r < SP.n_reward; ++r) sums[(size_t)r * N + e] = S[plan.sums_off + r * TILE + tid];
    }
  }

  // ------------------------------------------------------------------------------------------
  // the slab's logging partials -> the block's sums (plain adds: thread i owns word i), flags -> the launch's
  // (rare; integer atomics: order-independent).  The block adds its sums to the launch's when it leaves: one
  // atomic per word and block instead of per slab, which would queue up behind each other in L2.
  // ------------------------------------------------------------------------------------------
  if ((ph & GFB_PHASE_RESET) && reward_log) {
    for (int i = tid; i < n_acc_words; i += TILE)
      s_rew_blk[i] += (unsigned long long)xs_join(s_rew_acc[2 * i], s_rew_acc[2 * i + 1]);
    if (tid < SP.n_reward && s_rew_flags[tid]) atomicOr(K.s.rew_flags + tid, s_rew_flags[tid]);
  }
  if (!(ph & (GFB_PHASE_TERMINATION | GFB_PHASE_RESET)) && tid == 0 && s_status) atomicOr(K.s.status, s_status);

  // ------------------------------------------------------------------------------------------
  // observations: every thread assembles 16-byte pieces of the slab's rows
  // (observation_manager.py:232-256: value * scale (+ U(-1,1) * noise), concatenated; history
  //  frames 1..H-1 are the previous step's frames 0..H-2, observation_manager.py:223-226)
  // ------------------------------------------------------------------------------------------
  if (ph & GFB_PHASE_OBSERVE) {
    const DevObsCol* cols_all = reinterpret_cast<const DevObsCol*>(Tbl);
    for (int g = 0; g < SP.n_obs_groups; ++g) {
      const gfb_obs_group& og = SP.obs_group[g];
      const int O = og.n_cols, OH = og.n_cols * og.history;
      const DevObsCol* cols = cols_all + og.col_begin;
      float* out = GFB_BUF(float, GFB_B_OBS_OUT0 + g) + (size_t)e0 * OH;
      const float* prev = GFB_BUF(const float, GFB_B_OBS_PREV0 + g);
      if (prev) prev += (size_t)e0 * OH;
      const float* noise = GFB_BUF(const float, GFB_B_OBS_NOISE0 + g);
      if (noise) noise += (size_t)e0 * O;
      const int W = OH >> 2, W0 = O >> 2;
      if (plan.grp_run_begin[g] >= 0) {
        // 16-byte path, three warp-uniform passes over the slab's rows.  Within a pass a thread
        // owns ONE piece position k of the row (its descriptor is read once, outside the loop) and
        // walks down the rows; consecutive threads hold consecutive pieces of TILE/n whole rows, so
        // a warp's stores land in a few contiguous segments of neighbouring rows.
        float4* out4 = reinterpret_cast<float4*>(out);
        // pass 1: contiguous runs of a staged array (one 16-byte shared load per piece)
        {
          const int n = plan.grp_run_count[g];
          const int rpp = n > 0 ? TILE / n : 0;  // rows per sweep
          if (n > 0 && n <= TILE && tid < rpp * n) {
            const int r0 = tid / n, k = tid - r0 * n;
            const int4 d = (reinterpret_cast<const int4*>(Tbl + plan.run_off) + plan.grp_run_begin[g])[k];
            const float4 nz =
                (reinterpret_cast<const float4*>(Tbl + plan.run_off + 4 * plan.n_runs) + plan.grp_run_begin[g])[k];
            const float sc = __int_as_float(d.w);
            const bool noisy = nz.x != 0.f || nz.y != 0.f || nz.z != 0.f || nz.w != 0.f;
            const float* src = S + d.x + r0 * d.y;
            float4* dst = out4 + r0 * W + d.z;
            const int sstep = rpp * d.y, dstep = rpp * W;
#pragma unroll 4
            for (int row = r0; row < valid; row += rpp) {
              float4 v = *reinterpret_cast<const float4*>(src);
              v.x = mul(v.x, sc); v.y = mul(v.y, sc); v.z = mul(v.z, sc); v.w = mul(v.w, sc);
              if (noisy) v = add_noise(v, nz, noise, row, W0, d.z, P, rng, e0, og.col_begin, SP.rng_mode);
              *dst = v;
              src += sstep;
              dst += dstep;
            }
          }
        }
        // pass 2: mixed groups (four independent shared sources: derived vectors, commands, ...)
        {
          const int n = plan.grp_mixed_count[g];
          const int rpp = n > 0 ? TILE / n : 0;
          if (n > 0 && n <= TILE && tid < rpp * n) {
            const int r0 = tid / n, k = tid - r0 * n;
            const int NM = plan.n_mixed, mb = plan.grp_mixed_begin[g];
            const int32_t* tab = reinterpret_cast<const int32_t*>(Tbl + plan.mixed_off);
            const int4 off = (reinterpret_cast<const int4*>(tab) + mb)[k];
            const int4 str = (reinterpret_cast<const int4*>(tab + 4 * NM) + mb)[k];
            const float4 sc = (reinterpret_cast<const float4*>(tab + 8 * NM) + mb)[k];
            const float4 nz = (reinterpret_cast<const float4*>(tab + 12 * NM) + mb)[k];
            const int c4 = (tab + 16 * NM + mb)[k];
            const bool noisy = nz.x != 0.f || nz.y != 0.f || nz.z != 0.f || nz.w != 0.f;
            const float *s0 = S + off.x + r0 * str.x, *s1 = S + off.y + r0 * str.y;
            const float *s2 = S + off.z + r0 * str.z, *s3 = S + off.w + r0 * str.w;
            float4* dst = out4 + r0 * W + c4;
            const int dstep = rpp * W;
#pragma unroll 2
            for (int row = r0; row < valid; row += rpp) {
              float4 v;
              v.x = mul(*s0, sc.x); v.y = mul(*s1, sc.y); v.z = mul(*s2, sc.z); v.w = mul(*s3, sc.w);
              if (noisy) v = add_noise(v, nz, noise, row, W0, c4, P, rng, e0, og.col_begin, SP.rng_mode);
              *dst = v;
              s0 += rpp * str.x; s1 += rpp * str.y; s2 += rpp * str.z; s3 += rpp * str.w;
              dst += dstep;
            }
          }
        }
        // pass 3: history frames 1..H-1 are the previous step's frames 0..H-2
        if (W > W0) {
          const int n = W - W0;
          const float4* prev4 = reinterpret_cast<const float4*>(prev);
          const int total = valid * n;
          int row = tid / n, k = tid - row * n;
          const int drow = TILE / n, dk = TILE - drow * n;
          for (int f = tid; f < total; f += TILE) {
            out4[row * W + W0 + k] = prev4[row * W + k];
            row += drow;
            k += dk;
            if (k >= n) { k -= n; ++row; }
          }
        }
      } else {
        const int total = valid * OH;
        for (int f = tid; f < total; f += TILE) {
          const int row = f / OH, col = f - row * OH;
          float v;
          if (col < O) {
            const DevObsCol d = cols[col];
            v = mul(obs_fetch_post(d, S, K.b, plan, row, e0 + row), d.scale);
            if (d.noise != 0.f) {
              float u;
              if (SP.rng_mode == 0) {
                u = noise ? noise[(size_t)row * O + col] : 0.f;
              } else {
                const uint4 x = rng((uint32_t)(e0 + row), (uint32_t)P.step_index, (uint32_t)(P.step_index >> 32),
                                    0x1000u + (uint32_t)(og.col_begin + (col & ~3)));
                const int j = col & 3;
                const uint32_t xj = j == 0 ? x.x : (j == 1 ? x.y : (j == 2 ? x.z : x.w));
                u = sub(mul(u01(xj), 2.f), 1.f);
              }
              v = add(v, mul(u, d.noise));
            }
          } else {
            v = prev[(size_t)row * OH + (col - O)];
          }
          out[(size_t)row * OH + col] = v;
        }
      }
    }
  }

  // everyone is done with the slab's shared memory before the rest of it is refilled
  __syncthreads();
  next_tile = s_next_tile;
  if (use_tma && next_tile < n_tiles && warp == 0) {
    bulk_wait_all_read();
    fence_async_smem();  // the slab's generic-proxy reads above, the async-proxy refill below
    issue_slab_loads<TILE>(K, plan, Sbase, Tbl, &bars[0], next_tile, plan.n_prefetch, plan.n_early, n_sum_rows_main,
                           false, lane, split_x);
  }

  tile = next_tile;
  }  // slab loop

  if (use_tma && warp == 0) bulk_wait_all();
  if ((ph & GFB_PHASE_RESET) && reward_log)  // only the nonzero words (no return value: RED, fire and forget)
    for (int i = tid; i < n_acc_words; i += TILE)
      if (s_rew_blk[i]) atomicAdd(K.s.rew_acc + i, s_rew_blk[i]);

  // ------------------------------------------------------------------------------------------
  // the last block to leave turns the reward sums into logged means and re-arms the counters
  // ------------------------------------------------------------------------------------------
  __shared__ int s_last_block;
  __syncthreads();
  if (tid == 0) {
    __threadfence();
    s_last_block = atomicAdd(K.s.counters + CTR_BLOCKS_DONE, 1u) == gridDim.x - 1u;
  }
  __syncthreads();
  if (s_last_block && warp == 0) {
    __threadfence();
    if (ph & GFB_PHASE_RESET) finalize_step(K, lane);  // logging values, the report, the word the host spins on
    __syncwarp();
    if (lane == 0) {
      K.s.counters[CTR_TICKET] = 0u;
      K.s.counters[CTR_BLOCKS_DONE] = 0u;
      K.s.counters[CTR_TOTAL_RESET] = 0u;
    }
  }
}

}  // namespace gfb
