// Pre-physics action kernel, the sparse re-observation kernel, the reset-side writers (spawn pose,
// reset rows) and the stand-alone contact scatter / rotation entry points.
#pragma once
#include "device_utils.cuh"
#include "plan.h"
#include "tail_math.cuh"

namespace gfb {

// ---------------------------------------------------------------------------------------------
// action_kernel: GenesisEnv.step bookkeeping + action manager (pre-physics)
//   genesis_env.py:196       episode_length += 1
//   genesis_env.py:202-203   last_actions <- actions ; actions <- raw   (ring mode: the caller has
//                            exchanged the two buffers, only actions <- raw is left to do)
//   position_action_manager.py:402-414   NaN/Inf flags; t = a*scale + offset; clamp(lo, hi)
//   position_within_limits.py:125-126    clamp(a,-1,1) * scale + offset
//   rewards.py:267-271       action_rate = sum((last_actions - actions)^2)   (consumed post-physics)
// One slab of TILE envs per block: the raw and previous action slabs are contiguous -> TMA in;
// last_actions / actions are pure copies -> TMA out of the very same shared-memory slabs.
// ---------------------------------------------------------------------------------------------
struct ActionParams {
  // the action part of the term table only (a launch copies its parameter block: 4 KB -> 0.6 KB)
  int32_t num_envs, num_dofs, action_mode, _pad;
  float action_scale[GFB_MAX_DOFS], action_offset[GFB_MAX_DOFS];
  float action_clip_lo[GFB_MAX_DOFS], action_clip_hi[GFB_MAX_DOFS];
  const float* raw_env;
  const float* raw_mgr;  // == raw_env unless a delay FIFO is active
  float* env_actions;
  float* env_last_actions;
  float* targets;
  float* action_rate;
  int32_t* episode_length;
  uint32_t* status;
  int32_t tma_ok;
  int32_t check_finite;
  int32_t ring;  // gfb_action_step_ring: env_last_actions already holds the previous actions (read only)
};

template <int TILE>
__global__ void __launch_bounds__(TILE) action_kernel(const __grid_constant__ ActionParams A) {
  extern __shared__ __align__(128) float S[];
  __shared__ __align__(8) uint64_t bar;
  const ActionParams& P = A;
  const int tid = threadIdx.x;
  const int N = P.num_envs, D = P.num_dofs;
  const int e0 = blockIdx.x * TILE;
  const int valid = min(TILE, N - e0);
  const bool active = tid < valid;
  const int e = e0 + tid;
  const bool use_tma = A.tma_ok && valid == TILE;
  const bool two_raw = A.raw_mgr != A.raw_env;

  float* s_raw = S;                   // (TILE, D) raw env actions
  float* s_prev = S + TILE * D;       // (TILE, D) previous env.actions
  float* s_tgt = S + 2 * TILE * D;    // (TILE, D) targets out
  float* s_rawm = S + 3 * TILE * D;   // (TILE, D) delayed raw (only with a FIFO)
  const uint32_t slab_bytes = (uint32_t)TILE * D * 4u;
  const size_t goff = (size_t)e0 * D;

  // (thread 0 is selected by predicate inside the wrappers, never by a branch: uniform-datapath rule,
  //  device_utils.cuh)
  mbar_init(tid == 0, &bar, 1);
  fence_mbar_init();
  __syncthreads();
  if (use_tma) {
    if (tid < 32) {
      mbar_expect_tx(tid == 0, &bar, slab_bytes * (two_raw ? 3u : 2u));
      bulk_load(tid == 0, s_raw, A.raw_env + goff, slab_bytes, &bar);
      bulk_load(tid == 0, s_prev, (A.ring ? A.env_last_actions : A.env_actions) + goff, slab_bytes, &bar);
      bulk_load(tid == 0 && two_raw, s_rawm, A.raw_mgr + goff, slab_bytes, &bar);
      __syncwarp();
    }
  } else {
    const int words = valid * D;
    for (int w = tid; w < words; w += TILE) {
      s_raw[w] = A.raw_env[goff + w];
      s_prev[w] = (A.ring ? A.env_last_actions : A.env_actions)[goff + w];
      if (two_raw) s_rawm[w] = A.raw_mgr[goff + w];
    }
  }
  int ep_len = 0;
  if (active && A.episode_length) ep_len = A.episode_length[e];  // in flight while the slabs arrive
  if (use_tma && tid < 32) mbar_wait(&bar, 0);  // one warp polls, the block barrier releases the rest
  __syncthreads();
  if (active && A.episode_length) A.episode_length[e] = ep_len + 1;  // genesis_env.py:195

  // pure copies first: last_actions <- previous actions, actions <- raw
  if (use_tma) {
    if (tid < 32) {
      bulk_store(tid == 0 && !A.ring, A.env_last_actions + goff, s_prev, slab_bytes);
      bulk_store(tid == 0, A.env_actions + goff, s_raw, slab_bytes);
      bulk_commit();
      __syncwarp();
    }
  } else {
    const int words = valid * D;
    for (int w = tid; w < words; w += TILE) {
      if (!A.ring) A.env_last_actions[goff + w] = s_prev[w];
      A.env_actions[goff + w] = s_raw[w];
    }
  }

  if (active) {
    const float* a = s_raw + tid * D;
    const float* p = s_prev + tid * D;
    const float* am = (two_raw ? s_rawm : s_raw) + tid * D;
    float* t = s_tgt + tid * D;
    float rate = 0.0f;
    uint32_t status = 0;
    auto one = [&](float x, float prev, float y, int d) -> float {
      rate = add(rate, sq(sub(prev, x)));
      if (A.check_finite) {
        if (y != y) status |= GFB_STATUS_NAN_ACTION;
        if (fabsf(y) == __int_as_float(0x7f800000)) status |= GFB_STATUS_INF_ACTION;
      }
      if (P.action_mode == 2) {
        // torch.clamp_ propagates NaN
        y = (y != y) ? y : fminf(fmaxf(y, -1.0f), 1.0f);
        y = add(mul(y, P.action_scale[d]), P.action_offset[d]);
      } else {
        y = add(mul(y, P.action_scale[d]), P.action_offset[d]);
        y = (y != y) ? y : fminf(fmaxf(y, P.action_clip_lo[d]), P.action_clip_hi[d]);
      }
      return y;
    };
    if ((D & 3) == 0) {
      // rows of D floats at a 4D-byte stride: 128-bit shared accesses are conflict-free and a
      // quarter of the instructions of the scalar walk (same element order: d ascending)
      for (int d = 0; d < D; d += 4) {
        const float4 x = *reinterpret_cast<const float4*>(a + d);
        const float4 pv = *reinterpret_cast<const float4*>(p + d);
        const float4 m = two_raw ? *reinterpret_cast<const float4*>(am + d) : x;
        float4 y;
        y.x = one(x.x, pv.x, m.x, d);
        y.y = one(x.y, pv.y, m.y, d + 1);
        y.z = one(x.z, pv.z, m.z, d + 2);
        y.w = one(x.w, pv.w, m.w, d + 3);
        *reinterpret_cast<float4*>(t + d) = y;
      }
    } else {
      for (int d = 0; d < D; ++d) t[d] = one(a[d], p[d], am[d], d);
    }
    if (A.action_rate) A.action_rate[e] = rate;
    if (status) atomicOr(A.status, status);
  }

  if (A.targets && P.action_mode != 0) {
    if (use_tma) {
      fence_async_smem();
      __syncthreads();
      if (tid < 32) {
        bulk_store(tid == 0, A.targets + goff, s_tgt, slab_bytes);
        bulk_commit();
        __syncwarp();
      }
    } else {
      __syncthreads();
      const int words = valid * D;
      for (int w = tid; w < words; w += TILE) A.targets[goff + w] = s_tgt[w];
    }
  }
  if (use_tma && tid < 32) bulk_wait_all();
}

// ---------------------------------------------------------------------------------------------
// compact_kernel: the ascending int64 list of reset env ids, identical to
// (terminated | truncated).nonzero() (managed_env.py:308-310), from the reset masks the post-physics
// kernel left in scratch memory (one 32-env word per warp of a slab, in env order).
// It is enqueued right behind the post kernel, whose last block has by then told the host how many
// envs reset: it runs while the host wakes up and walks through its reset fan-out, and whatever
// reads the list (engine setters, the re-observation) is enqueued behind it.
// Every block derives the number of reset envs before its own range by summing the population counts
// of all earlier words (the mask array is 128 KB at 1M envs: L2 hits), then scans its range.  The
// launch geometry (tail_math.cuh compact_geometry) starts every block inside the array.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(CMP_THREADS) compact_kernel(const uint32_t* __restrict__ words, int n_words,
                                                               int words_per_block, int64_t* __restrict__ out) {
  __shared__ int s_warp[CMP_THREADS / 32];
  __shared__ int s_base;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int w0 = blockIdx.x * words_per_block;
  if (w0 >= n_words) return;  // (block-uniform)
  const int w1 = min(w0 + words_per_block, n_words);
  // reset envs in all words before this block's range (w0 is a multiple of 256: 16-byte loads)
  int before = 0;
  const uint4* words4 = reinterpret_cast<const uint4*>(words);
#pragma unroll 4
  for (int w = tid; w < (w0 >> 2); w += CMP_THREADS) {
    const uint4 v = words4[w];
    before += __popc(v.x) + __popc(v.y) + __popc(v.z) + __popc(v.w);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) before += __shfl_xor_sync(0xffffffffu, before, o);
  if (lane == 0) s_warp[warp] = before;
  __syncthreads();
  if (tid == 0) {
    int total = 0;
    for (int k = 0; k < CMP_THREADS / 32; ++k) total += s_warp[k];
    s_base = total;
  }
  __syncthreads();
  int base = s_base;
  for (int v0 = w0; v0 < w1; v0 += CMP_THREADS) {
    const int w = v0 + tid;
    uint32_t bits = w < w1 ? words[w] : 0u;
    const int mine = __popc(bits);
    int incl = mine;  // inclusive scan over the sweep: within the warp, then over the warps
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int up = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += up;
    }
    __syncthreads();  // (s_warp is free again)
    if (lane == 31) s_warp[warp] = incl;
    __syncthreads();
    int warps_before = 0, sweep_total = 0;
    for (int k = 0; k < CMP_THREADS / 32; ++k) {
      const int c = s_warp[k];
      warps_before += k < warp ? c : 0;
      sweep_total += c;
    }
    int64_t* dst = out + base + warps_before + incl - mine;
    while (bits) {
      const int bit = __ffs(bits) - 1;
      bits &= bits - 1;
      *dst++ = (int64_t)w * 32 + bit;
    }
    base += sweep_total;
  }
}

// ---------------------------------------------------------------------------------------------
// observe_kernel: frame 0 of every observation group for a LIST of envs (or all envs), from the
// current engine state and the CACHED inverse base quaternion.  The reference observes after
// reset (managed_env.py:322-326) with post-reset engine getters but the pre-reset cached
// quaternion (entity_manager.py:134-146 vs :189-195; EntityManager.reset does not refresh it).
//
// A warp takes OBS_ROWS env rows, no shared memory, no block barrier: the lanes walk the rows' columns
// (consecutive columns of one source array are consecutive addresses, so loads and stores coalesce),
// each lane reads its column descriptor once for all rows; the env ids, cached quaternions and base
// velocities are warp-uniform broadcast loads.  The reset envs are scattered over the batch, so every
// access is a DRAM miss: the kernel is pure latency, a warp issues in order, and what matters is
// that all loads of a dependency level are issued before the first of them is used -- level 0: env
// ids + column descriptors; level 1: quaternions, velocities and the source values of two columns
// for all rows (unconditional loads from always-valid addresses, so no branch separates them).
// ---------------------------------------------------------------------------------------------
constexpr int OBS_MAX_ITEMS = 16;  // (group, 32-column chunk) pairs: 256 columns in at most 4 groups
struct ObserveHead {  // the observation part of the term table (instead of the whole 4 KB head)
  int32_t n_contact, n_obs_groups, rng_mode, n_items;
  uint64_t rng_seed, step_index;
  int32_t contact_links[GFB_MAX_CONTACT_MANAGERS];
  gfb_obs_group obs_group[GFB_MAX_OBS_GROUPS];
  int8_t item_group[OBS_MAX_ITEMS], item_chunk[OBS_MAX_ITEMS];
};

struct ObserveParams {
  ObserveHead P;
  gfb_buffers b;
  Plan plan;
  const DevObsCol* cols;
  const int64_t* idx;
  int32_t n;
};

constexpr int OBS_WARPS = 4;  // warps per block
constexpr int OBS_ROWS = 4;   // env rows per warp: their loads are issued together (memory-level parallelism)

// One (group, column) work item of a lane: its descriptor and the raw values of the warp's rows.
struct ObsItem {
  int4 d0, d1;  // DevObsCol: {kind, a, row_words, col}, {scale, noise, gbuf, vec}
  int g, col;
  bool on;
};
__device__ __forceinline__ ObsItem obs_item(const ObserveParams& K, int item, int lane) {
  ObsItem it;
  it.g = item < K.P.n_items ? K.P.item_group[item] : 0;
  const gfb_obs_group& og = K.P.obs_group[it.g];
  it.col = (item < K.P.n_items ? K.P.item_chunk[item] : 0) * 32 + lane;
  it.on = item < K.P.n_items && it.col < og.n_cols;
  const int4* dp = reinterpret_cast<const int4*>(K.cols + og.col_begin + (it.on ? it.col : 0));
  it.d0 = __ldg(dp);       // (issued unconditionally from a valid address: no branch ahead of the loads,
  it.d1 = __ldg(dp + 1);   //  so that the scheduler can put every load of a level in flight together)
  return it;
}

__global__ void __launch_bounds__(OBS_WARPS * 32, 7) observe_kernel(const __grid_constant__ ObserveParams K) {
  const ObserveHead& P = K.P;
  const Plan& plan = K.plan;
  const int lane = threadIdx.x & 31;
  const int i0 = (blockIdx.x * OBS_WARPS + (threadIdx.x >> 5)) * OBS_ROWS;
  if (i0 >= K.n) return;
  // level 0 (independent loads): the rows' env ids and the descriptors of this lane's first two columns
  long long e[OBS_ROWS];
#pragma unroll
  for (int r = 0; r < OBS_ROWS; ++r) {
    const int i = min(i0 + r, K.n - 1);  // (rows past the end repeat the last one and are not stored)
    e[r] = K.idx ? (long long)K.idx[i] : (long long)i;
  }
  ObsItem cur[2] = {obs_item(K, 0, lane), obs_item(K, 1, lane)};

  // level 1: cached inverse quaternion and base velocities of every row (warp-uniform broadcast loads).
  // Lane k < 9 keeps component k of [ang_b 3][lin_b 3][grav_b 3] (the stash layout of the post kernel,
  // plan.h) of every row; a column that wants one fetches it with a shuffle.
  float body[OBS_ROWS];
  {
    float4 q[OBS_ROWS];
    float va[OBS_ROWS][3], vl[OBS_ROWS][3];
#pragma unroll
    for (int r = 0; r < OBS_ROWS; ++r) {
      q[r] = GFB_BUF(const float4, GFB_B_INV_BASE_QUAT)[e[r]];
#pragma unroll
      for (int k = 0; k < 3; ++k) {
        va[r][k] = (plan.needs & NEED_ANG) ? GFB_BUF(const float, GFB_B_ANG)[e[r] * 3 + k] : 0.0f;
        vl[r][k] = (plan.needs & NEED_LIN) ? GFB_BUF(const float, GFB_B_VEL)[e[r] * 3 + k] : 0.0f;
      }
    }
#pragma unroll
    for (int r = 0; r < OBS_ROWS; ++r) {
      const V3 iq = {q[r].y, q[r].z, q[r].w};
      const V3 a = rotate(V3{va[r][0], va[r][1], va[r][2]}, q[r].x, iq);
      const V3 l = rotate(V3{vl[r][0], vl[r][1], vl[r][2]}, q[r].x, iq);
      const V3 g = rotate(V3{0.f, 0.f, -1.f}, q[r].x, iq);
      const float comp[9] = {a.x, a.y, a.z, l.x, l.y, l.z, g.x, g.y, g.z};
      float mine = 0.0f;
#pragma unroll
      for (int k = 0; k < 9; ++k) mine = lane == k ? comp[k] : mine;
      body[r] = mine;
    }
  }
  const Philox rng(P.rng_seed);
  const float* dummy = reinterpret_cast<const float*>(K.b.buf[GFB_B_INV_BASE_QUAT]);
  for (int item = 0; item < P.n_items; item += 2) {
    // level 1 (cont.): the source values of two columns x OBS_ROWS rows, all issued before any is used
    float raw[2][OBS_ROWS];
#pragma unroll
    for (int j = 0; j < 2; ++j) {
      const int kind = cur[j].d0.x;
      const bool global = cur[j].on && (kind == 1 || kind == 2);
      const float* src = global ? reinterpret_cast<const float*>(K.b.buf[cur[j].d1.z]) + cur[j].d0.w : dummy;
      const long long stride = global ? cur[j].d0.z : 0;
#pragma unroll
      for (int r = 0; r < OBS_ROWS; ++r) raw[j][r] = src[e[r] * stride];
    }
    // the next two descriptors are requested before this pair is finished
    ObsItem nxt[2] = {obs_item(K, item + 2, lane), obs_item(K, item + 3, lane)};
#pragma unroll
    for (int j = 0; j < 2; ++j) {
      const int kind = cur[j].d0.x, a = cur[j].d0.y, col = cur[j].col;
      const float scale = __int_as_float(cur[j].d1.x), nz = __int_as_float(cur[j].d1.y);
      const gfb_obs_group& og = P.obs_group[cur[j].g];
      const int O = og.n_cols, OH = og.n_cols * og.history;
      float* out = GFB_BUF(float, GFB_B_OBS_OUT0 + cur[j].g);
      const float* noise = GFB_BUF(const float, GFB_B_OBS_NOISE0 + cur[j].g);
      float v[OBS_ROWS];
#pragma unroll
      for (int r = 0; r < OBS_ROWS; ++r) v[r] = (kind == 1 || kind == 2) ? raw[j][r] : 0.0f;
      // (the shuffle is executed by every lane of the warp: no lane may skip it)
      const bool derived = cur[j].on && kind == 3 && a < 9;
#pragma unroll
      for (int r = 0; r < OBS_ROWS; ++r) {
        const float b = __shfl_sync(0xffffffffu, body[r], derived ? a : 0);
        if (derived) v[r] = b;
      }
      if (cur[j].on && kind == 3) {
        if (a >= 9) {  // |net contact force| of one tracked link (mdp/observations.py:181-193)
          for (int m = 0; m < P.n_contact; ++m) {
            const int t = a - plan.st_cnorm[m];
            if (t < 0 || t >= P.contact_links[m]) continue;
            const float* cg = GFB_BUF(const float, GFB_B_CONTACTS0 + m);
            if (!cg) continue;
#pragma unroll
            for (int r = 0; r < OBS_ROWS; ++r) {
              const float* c = cg + (e[r] * P.contact_links[m] + t) * 3;
              v[r] = norm3(c[0], c[1], c[2]);
            }
          }
        }
      }
      if (!cur[j].on) continue;  // (behind the shuffles: this lane has no column in this chunk)
#pragma unroll
      for (int r = 0; r < OBS_ROWS; ++r) {
        float x = mul(v[r], scale);
        if (nz != 0.f) {
          float u;
          if (P.rng_mode == 0) {
            u = noise ? noise[e[r] * O + col] : 0.f;
          } else {
            const uint4 w = rng((uint32_t)e[r], (uint32_t)P.step_index, (uint32_t)(P.step_index >> 32),
                                0x1000u + (uint32_t)(og.col_begin + (col & ~3)));
            const int jj = col & 3;
            const uint32_t wj = jj == 0 ? w.x : (jj == 1 ? w.y : (jj == 2 ? w.z : w.w));
            u = sub(mul(u01(wj), 2.f), 1.f);
          }
          x = add(x, mul(u, nz));
        }
        if (i0 + r < K.n) out[e[r] * OH + col] = x;
      }
    }
    cur[0] = nxt[0];
    cur[1] = nxt[1];
  }
}

// ---------------------------------------------------------------------------------------------
// contact_kernel: the reference's Taichi kernel (contact/kernel.py:5-90) on its own, with its
// argument list.  One thread per env, targets outer / contact slots inner, ordered sums.
// ---------------------------------------------------------------------------------------------
__global__ void contact_kernel(const float* __restrict__ force, const float* __restrict__ position,
                               const int32_t* __restrict__ link_a, const int32_t* __restrict__ link_b,
                               const float4* __restrict__ links_quat, const int32_t* __restrict__ targets,
                               const int32_t* __restrict__ withs, float* __restrict__ out_f,
                               float* __restrict__ out_p, float* __restrict__ counts, int n_envs, int C, int L,
                               int Lc, int Lw, int has_filter) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n_envs) return;
  const int32_t* la = link_a + (size_t)e * C;
  const int32_t* lb = link_b + (size_t)e * C;
  const float* cf = force + (size_t)e * C * 3;
  const float* cp = position + (size_t)e * C * 3;
  for (int t = 0; t < Lc; ++t) {
    const int target = targets[t];
    const float4 tq = links_quat[(size_t)e * L + target];
    float fx = 0.f, fy = 0.f, fz = 0.f, px = 0.f, py = 0.f, pz = 0.f, cnt = 0.f;
    for (int c = 0; c < C; ++c) {
      const int a = la[c], b = lb[c];
      const bool is_a = a == target, is_b = b == target;
      bool hit = is_a | is_b;
      if (hit && has_filter) {
        bool keep = false;
        for (int w = 0; w < Lw; ++w) keep |= (is_a && b == withs[w]) || (is_b && a == withs[w]);
        hit = keep;
      }
      if (hit) {
        const float x = cf[c * 3], y = cf[c * 3 + 1], z = cf[c * 3 + 2];
        V3 f = is_b ? V3{x, y, z} : V3{-x, -y, -z};
        f = inv_rotate_ti(f, tq.x, V3{tq.y, tq.z, tq.w});
        fx = add(fx, f.x); fy = add(fy, f.y); fz = add(fz, f.z);
        px = add(px, cp[c * 3]); py = add(py, cp[c * 3 + 1]); pz = add(pz, cp[c * 3 + 2]);
        cnt = add(cnt, 1.0f);
      }
    }
    if (cnt > 0.f) {
      px = fdiv(px, cnt); py = fdiv(py, cnt); pz = fdiv(pz, cnt);
    }
    float* of = out_f + ((size_t)e * Lc + t) * 3;
    float* op = out_p + ((size_t)e * Lc + t) * 3;
    of[0] = fx; of[1] = fy; of[2] = fz;
    op[0] = px; op[1] = py; op[2] = pz;
    counts[(size_t)e * Lc + t] = cnt;
  }
}

// ---------------------------------------------------------------------------------------------
// rotate_kernel: transform_by_quat(vec, q or conj(q)) for stand-alone getter calls
// ---------------------------------------------------------------------------------------------
__global__ void rotate_kernel(const float* __restrict__ vec, const float4* __restrict__ quat,
                              float* __restrict__ out, int n, int conjugate) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float4 q = quat[i];
  const V3 qv = conjugate ? V3{-q.y, -q.z, -q.w} : V3{q.y, q.z, q.w};
  const V3 v = vec ? V3{vec[i * 3], vec[i * 3 + 1], vec[i * 3 + 2]} : V3{0.f, 0.f, -1.f};
  const V3 r = rotate(v, q.x, qv);
  out[i * 3] = r.x;
  out[i * 3 + 1] = r.y;
  out[i * 3 + 2] = r.z;
}

// ---------------------------------------------------------------------------------------------
// reset_rows_kernel: the value rows a reset hands to the engine setters (SURVEY.md 8(f) rank 1), one
// launch instead of a chain of indexed torch ops per setter:
//   mode GFB_ROWS_NOISE    out[i, j] = base[j] + u * a, u ~ U(-1, 1)        (PositionActionManager
//                          ._add_random_noise, position_action_manager.py:516-525: gains -- one row --
//                          and the default joint positions of the reset envs, :432-464)
//   mode GFB_ROWS_UNIFORM  out[i, j] = U(a, b)                               (randomize_link_mass_shift,
//                          mdp/reset.py:229-284)
// Draws are injected (`draws`, (n, width): the reference's own numbers in the parity harness) or
// Philox4x32-10 keyed by (seed, env id, counter, column).  `scatter` (rows, width), if given, receives
// row idx[i] as well (the manager's persistent per-env buffer).
// ---------------------------------------------------------------------------------------------
struct ResetRowsParams {
  const int64_t* idx;
  int32_t n, width, mode, _pad;
  const float* base;
  float a, b;
  const float* draws;
  uint64_t seed, counter;
  float* out;
  float* scatter;
};

__global__ void __launch_bounds__(256) reset_rows_kernel(const ResetRowsParams p) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long long)p.n * p.width) return;
  const int row = (int)(i / p.width), col = (int)(i - (long long)row * p.width);
  const long long e = p.idx ? (long long)p.idx[row] : (long long)row;
  float u;  // U(-1, 1) for NOISE, the final value (injected) or U(0, 1) for UNIFORM
  if (p.draws) {
    u = p.draws[i];
  } else {
    const Philox rng(p.seed);
    const uint4 r = rng((uint32_t)e, (uint32_t)((uint64_t)e >> 32) ^ 0x52455354u, (uint32_t)p.counter,
                        (uint32_t)(p.counter >> 32) ^ (uint32_t)(col >> 2));  // stream tag 'REST'
    const int j = col & 3;
    const float u01v = u01(j == 0 ? r.x : (j == 1 ? r.y : (j == 2 ? r.z : r.w)));
    u = p.mode == GFB_ROWS_NOISE ? sub(mul(u01v, 2.0f), 1.0f) : u01v;
  }
  float v;
  if (p.mode == GFB_ROWS_NOISE) v = add(p.base[col], mul(u, p.a));
  else v = p.draws ? u : add(mul(u, sub(p.b, p.a)), p.a);
  p.out[i] = v;
  if (p.scatter) p.scatter[e * p.width + col] = v;
}

// ---------------------------------------------------------------------------------------------
// spawn_kernel: spawn pose of the reset envs in one launch (gfb_spawn_pose, include/gfb200.h).
// One thread per reset env; every scattered row belongs to exactly one thread.
// ---------------------------------------------------------------------------------------------
struct SpawnParams {
  gfb_spawn cfg;
  const int64_t* idx;
  int32_t n;
  const float* height_field;
  const float* u_x;
  const float* u_y;
  const float* u_rot[3];
  float* position_buffer;
  float* rot_buffer;
  float* quat_buffer;
  float* pos_out;
  float* quat_out;
};

__global__ void __launch_bounds__(128) spawn_kernel(const SpawnParams p) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= p.n) return;
  const gfb_spawn& c = p.cfg;
  const int64_t e = p.idx ? p.idx[i] : (int64_t)i;
  const Philox rng(c.rng_seed);
  const uint32_t e_lo = (uint32_t)e, e_hi = (uint32_t)((uint64_t)e >> 32);
  const uint32_t k_lo = (uint32_t)c.rng_counter, k_hi = (uint32_t)(c.rng_counter >> 32);

  float ux, uy;
  if (p.u_x && p.u_y) {
    ux = p.u_x[i];
    uy = p.u_y[i];
  } else {
    const uint4 r = rng(e_lo, e_hi ^ 0x53504157u, k_lo, k_hi);  // stream tag 'SPAW'
    ux = p.u_x ? p.u_x[i] : u01(r.x);
    uy = p.u_y ? p.u_y[i] : u01(r.y);
  }
  const float x = add(mul(ux, c.x_span), c.x_lo);
  const float y = add(mul(uy, c.y_span), c.y_lo);
  const float ground = p.height_field
                           ? terrain_height(x, y, c.terrain_bounds, c.height_field_rows, c.height_field_cols, p.height_field)
                           : c.flat_height;
  const float z = add(ground, c.height_offset);
  float* row = p.position_buffer + e * 3;
  row[0] = x;
  row[1] = y;
  row[2] = z;
  if (p.pos_out) {
    p.pos_out[(size_t)i * 3] = x;
    p.pos_out[(size_t)i * 3 + 1] = y;
    p.pos_out[(size_t)i * 3 + 2] = z;
  }
  if (!c.with_rotation) return;

  float ang[3];
  uint4 r{};
  bool drawn = false;
#pragma unroll
  for (int a = 0; a < 3; ++a) {
    float* cell = p.rot_buffer + e * 3 + a;
    if (c.rot_mode[a] == GFB_SPAWN_ROT_DRAW) {
      float v;
      if (p.u_rot[a]) {
        v = p.u_rot[a][i];
      } else {
        if (!drawn) {
          r = rng(e_lo, e_hi ^ 0x53505254u, k_lo, k_hi);  // stream tag 'SPRT'
          drawn = true;
        }
        const uint32_t bits = a == 0 ? r.x : (a == 1 ? r.y : r.z);
        v = add(mul(u01(bits), sub(c.rot_hi[a], c.rot_lo[a])), c.rot_lo[a]);
      }
      *cell = v;
      ang[a] = v;
    } else {
      ang[a] = *cell;
    }
  }
  // xyz_to_quat (genesis.utils.geom; mdp/reset.py:63,194): extrinsic x-y-z, w first
  const float hx = mul(ang[0], 0.5f), hy = mul(ang[1], 0.5f), hz = mul(ang[2], 0.5f);
  const float cx = cosf(hx), cy = cosf(hy), cz = cosf(hz);
  const float sx = sinf(hx), sy = sinf(hy), sz = sinf(hz);
  const float qw = sub(mul(mul(cx, cy), cz), mul(mul(sx, sy), sz));
  const float qx = add(mul(mul(sx, cy), cz), mul(mul(cx, sy), sz));
  const float qy = sub(mul(mul(cx, sy), cz), mul(mul(sx, cy), sz));
  const float qz = add(mul(mul(cx, cy), sz), mul(mul(sx, sy), cz));
  const float4 q = make_float4(qw, qx, qy, qz);
  reinterpret_cast<float4*>(p.quat_buffer)[e] = q;
  if (p.quat_out) reinterpret_cast<float4*>(p.quat_out)[i] = q;
}

}  // namespace gfb
