// Logging reductions and the step report as device functions of the post-physics kernel (they used
// to be most of a second, "finalize" kernel):
//
//   * termination fire counts and the number of reset envs are integer atomics, fire and forget.
//   * the episode means of the reward terms over the reset envs (reward_manager.py:205-216) are
//     accumulated as exact integer sums of the fp32 quotients (tail_math.cuh: XS_WORDS words per term;
//     integer atomics commute, so the logged values are run-to-run deterministic) and turned into means
//     by the last block to leave the kernel.  Contract of a logged mean, S the exact sum of the n
//     quotients: NaN if a quotient is NaN or both infinities occur, else an infinite quotient; +-Inf if
//     S rounded to fp32 overflows (as an fp32 sum of the same values does); else S / n within 1 fp32 ulp,
//     +0 for a zero sum.  Sharded over ranks, each rank's S travels as a double and the doubles are
//     summed in rank order: deterministic, but within W * 2^-53 * sum|q| rather than exact.
//   * that block also writes the step report into the host's mapped memory and, last, its sequence
//     word, on which the host spins.
//   * envs sharded over ranks: both reductions are exchanged over NVLink peer memory (plan.h PeerInbox).
//
// The ORDERED list of reset env ids (GFB_B_RESET_IDX == (terminated | truncated).nonzero(),
// managed_env.py:308-310) is not needed by the host, only by work enqueued behind this launch: the
// slabs leave their reset masks in scratch memory and compact_kernel (aux_kernels.cuh), enqueued right
// behind the post kernel, expands them while the host is still waking up from the report.
//
// RULE learnt on the way here (1M envs, config 2; the kernel without any compaction takes 110 us):
// while the memory system is saturated a global round trip costs microseconds, so NOTHING a slab does
// may wait for one before its next block barrier -- no returning atomic whose result is used at once,
// no fence behind a batch of stores.  In-kernel variants of the ordered compaction that were built and
// measured: decoupled look-back per slab right after the terminations 251 us (the resident blocks run
// in lock-step waves, every slab of a wave polled the same cache lines); two-level (per chunk of 32
// slabs, last arriver scans the chunk, look-back over chunks) at that place 156-162 us; the same with
// the chunk work moved to the end of the slab iteration 128-137 us (a finisher that waits for earlier
// chunks stalls its whole slab at the next barrier, and the late slabs convoy).
#pragma once
#include "device_utils.cuh"
#include "plan.h"
#include "tail_math.cuh"

namespace gfb {

__device__ __forceinline__ void st_release_sys(unsigned long long* p, unsigned long long v) {
  asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long ld_acquire_sys(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ unsigned long long ld_relaxed_gpu(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_relaxed_gpu(unsigned long long* p, unsigned long long v) {
  asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ uint32_t ld_acquire_gpu_u32(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ unsigned long long global_timer_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}

// ---------------------------------------------------------------------------------------------
// exchange of the logging partials between the ranks (one warp).  Lane i owns two elements of the
// vector: a[i] (i < n_a: termination fire counts, then the number of reset envs) and b[i] (i < n_b:
// reward episode-quotient sums); they travel in one inbox slot.  On return a / b hold the sums over
// ranks in rank order (bit-identical on all ranks).  Returns false if a peer did not show up.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ bool peer_exchange(const PeerParams& pp, double& a, int n_a, double& b, int n_b, int lane) {
  const int parity = (int)(pp.seq & 1ull);
  const int me = pp.rank, W = pp.world;
  for (int p = 0; p < W; ++p) {
    PeerSlot& slot = pp.inbox[p]->slot[parity][me];
    if (lane < n_a) slot.vals[lane] = a;
    if (lane < n_b) slot.vals[n_a + lane] = b;
  }
  __threadfence_system();
  __syncwarp();
  if (lane < W) st_release_sys(&pp.inbox[lane]->slot[parity][me].seq, pp.seq);
  int late = 0;
  if (lane < W) {
    const unsigned long long* flag = &pp.inbox[me]->slot[parity][lane].seq;
    const unsigned long long t0 = global_timer_ns();
    while (ld_acquire_sys(flag) != pp.seq) {
      if (global_timer_ns() - t0 > 2000000000ull) {  // ~2 s: a peer never issued this exchange
        late = 1;
        break;
      }
      __nanosleep(200);
    }
  }
  if (__any_sync(0xffffffffu, late)) return false;
  __threadfence_system();
  double ga = 0.0, gb = 0.0;
  for (int r = 0; r < W; ++r) {
    const PeerSlot& slot = pp.inbox[me]->slot[parity][r];
    if (lane < n_a) ga += __ldcv(&slot.vals[lane]);
    if (lane < n_b) gb += __ldcv(&slot.vals[n_a + lane]);
  }
  a = ga;
  b = gb;
  return true;
}

// ---------------------------------------------------------------------------------------------
// End of the launch (one warp of the last block to leave the kernel): logging values and the report.
//   termination_manager.py:178-182  fired fraction per term
//   reward_manager.py:205-216       mean over the reset envs of (episode sum / episode seconds)
//   managed_env.py:308-310          number of reset envs (compact_kernel writes the indices)
// The GPU is idle while this runs, so every read is issued before the first one is used (one round
// trip), then the values are stored, and last -- behind a system-scope fence -- the report's sequence
// word, on which the host spins.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void finalize_step(const KParams& K, int lane) {
  const gfb_program_head& P = K.P;
  const Scratch& sc = K.s;
  const int n_t = P.n_termination, n_r = P.n_reward;
  __threadfence();
  // reads (and re-arming: every accumulator is left at zero for the next launch)
  const int n_reset = (int)ld_acquire_gpu_u32(sc.counters + CTR_TOTAL_RESET);  // every slab has added its share
  const int count = lane < n_t ? atomicExch(sc.term_count + lane, 0) : 0;
  uint32_t status = lane == 0 ? atomicExch(sc.status, 0u) : 0u;
  long long acc[XS_WORDS];  // lane = reward term
#pragma unroll
  for (int k = 0; k < XS_WORDS; ++k) acc[k] = lane < n_r ? (long long)atomicExch(sc.rew_acc + lane * XS_WORDS + k, 0ull) : 0ll;
  const uint32_t acc_flags = lane < n_r ? atomicExch(sc.rew_flags + lane, 0u) : 0u;

  double counts = lane < n_t ? (double)count : (lane == n_t ? (double)n_reset : 0.0);  // lane n_t: reset envs
  double sum = lane < n_r ? xs_to_double(acc, acc_flags) : 0.0;
  double* log_acc = GFB_BUF(double, GFB_B_LOG_ACC);
  float* log_out = GFB_BUF(float, GFB_B_LOG_OUT);
  if (log_acc) {  // local partials (what the NCCL fallback path all-reduces)
    if (lane < n_r) log_acc[lane] = sum;
    if (lane <= n_t) log_acc[n_r + lane] = counts;
  }
  // first stage of the report: the rank's own counts -- all the host needs to start its reset fan-out --
  // before the exchange below waits for the slowest peer
  gfb_report* rep = sc.report_host;
  if (lane < n_t) rep->termination_count[lane] = count;
  if (lane == 0) {
    rep->n_reset = n_reset;
    rep->status = status;
  }
  const bool staged = K.peer.world > 1 && log_acc;  // single rank: both stages are released together below
  if (staged) {
    __threadfence_system();
    __syncwarp();
    if (lane == 0) st_release_sys(reinterpret_cast<unsigned long long*>(&rep->local_seq), sc.report_seq);
  }

  long long denom = P.num_envs;
  if (K.peer.world > 1 && log_acc) {
    if (peer_exchange(K.peer, counts, n_t + 1, sum, n_r, lane)) denom = K.peer.global_num_envs;
    else if (lane == 0) status |= GFB_STATUS_PEER_TIMEOUT;
  }
  const double g_reset = __shfl_sync(0xffffffffu, counts, n_t);
  if (lane < n_t) {
    rep->global_termination_count[lane] = (long long)counts;
    if (log_out) log_out[n_r + lane] = fdiv((float)counts, (float)denom);
  }
  if (lane < n_r && log_out) {
    const bool logged = P.reward[lane].weight != 0.0f;  // reward_manager.py:208-209
    log_out[lane] = (g_reset > 0.0 && logged) ? xs_mean(sum, g_reset) : 0.0f;
  }
  if (lane == n_t) rep->global_n_reset = (long long)counts;
  if (lane == 0) rep->status = status;  // (again: the exchange may have added GFB_STATUS_PEER_TIMEOUT)
  __threadfence_system();
  __syncwarp();
  if (lane == 0) {
    if (!staged) st_release_sys(reinterpret_cast<unsigned long long*>(&rep->local_seq), sc.report_seq);
    st_release_sys(reinterpret_cast<unsigned long long*>(&rep->seq), sc.report_seq);
  }
}

}  // namespace gfb
