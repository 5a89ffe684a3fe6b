// Shared definitions of the gradient-aggregation kernels (csrc/fused_sync.cu: single-kernel K-of-N / interval path;
// csrc/fused_bucket.cu: bucketed, overlapped K == N path): the symmetric control block, the peer pointer tables and the
// system-scope memory / multimem helpers.
#pragma once

#include <stddef.h>
#include <string.h>

#include "common.cuh"
#include "host_utils.h"

namespace dm {

constexpr int SYNC_MAX_RANKS = 8;
constexpr int SYNC_RING = 64;          // commit-word ring (steps)
constexpr int SYNC_THREADS = 512;
constexpr int TIMING_RING = 1024;      // per-rank arrival-timestamp ring (steps)

// Control block, one per rank, in symmetric memory.  Words written remotely are spread over
// separate 128-byte lines.
struct SyncCtrl {
  // ---- written by peers -----------------------------------------------------------------
  volatile uint32_t arrive[SYNC_MAX_RANKS * 32];     // [p*32]: peer p arrived for epoch (value = epoch+1)
  volatile uint32_t done[SYNC_MAX_RANKS * 32];       // [p*32]: peer p's pushes for step s landed (value = s+1)
  volatile unsigned long long commit_local[SYNC_RING];  // ((step+1) << 32) | mask, broadcast by the committer
  // ---- authoritative on the chief only ------------------------------------------------------
  unsigned int bitmap[SYNC_RING];                    // arrival bitmap of step s at [s % RING]
  unsigned long long commit[SYNC_RING];              // ((step+1) << 32) | mask
  volatile uint32_t global_step;                     // number of committed steps
  volatile uint32_t last_in_mask[SYNC_MAX_RANKS];    // (last step in whose mask rank q was) + 1
  uint32_t pad0[32];
  // ---- local ----------------------------------------------------------------------------------
  uint32_t epoch;                // global step of my weights (device-resident so CUDA graphs replay)
  uint32_t cta_counter;          // grid-wide completion counter
  volatile uint32_t decided_tag; // epoch+1 once `decided_mask` is valid for this launch
  volatile uint32_t decided_mask;
  volatile uint32_t decided_late;   // 1: my gradient is not part of the mean
  volatile uint32_t decided_target; // epoch to move to after this launch
  uint32_t error;                // watchdog: 1 = arrival timeout, 2 = done timeout
  uint32_t accepted_steps, dropped_steps;
  uint32_t last_mask, last_count, last_late;
  uint32_t pad1[32];
  unsigned long long t_arrive[TIMING_RING];   // %globaltimer at arrival, per local step (cdf telemetry)
  unsigned long long t_start[TIMING_RING];    // %globaltimer stamped by the step's first kernel
  unsigned long long t_phase[8];              // last launch: kernel start, decided, reduced, pushed, landed, shadowed
  // ---- bucketed (overlapped) aggregation: the early bucket has its own handshake words ---------------------------
  volatile uint32_t arrive_e[SYNC_MAX_RANKS * 32];   // [p*32]: peer p's early-bucket gradients are complete (epoch+1)
  volatile uint32_t done_e[SYNC_MAX_RANKS * 32];     // [p*32]: peer p's early-bucket pushes have landed (epoch+1)
  uint32_t cta_counter_e;
  uint32_t cta_counter2;         // late bucket kernel: CTAs that have finished (the last one closes the step)
  uint32_t pad2[30];
  unsigned long long t_phase_e[8];            // early kernel: start, arrived, reduced (CTA 0), all pushed, all landed, applied (CTA 0)
  // ---- device-side interval mode (mode C, csrc/fused_interval.cu) ------------------------------------------------------------
  volatile unsigned long long iv_state;    // ((step+1) << 32) | gradients accumulated for that step -- read by the committer
  volatile uint32_t iv_busy;               // step+1 while an accumulate for that step is in flight (Dekker pair of commit_local)
  volatile uint32_t iv_last_total;         // written by the committer: divisor of the tick that produced my current weights
  unsigned long long iv_deadline;          // local %globaltimer deadline of the current tick
  unsigned long long iv_interval_ns;
  uint32_t iv_adopted;                     // this iteration adopted new weights: refresh the bf16 shadow
  uint32_t iv_go;                          // this iteration's gradient may be accumulated (its step is still open)
  uint32_t iv_commit_go;                   // step+1: I won the commit of that step -> the apply kernel reduces + pushes
  uint32_t iv_commit_mask;                 // contributors of the tick I am committing
  uint32_t iv_commit_total;                // its divisor (sum of the contributors' counts)
  uint32_t iv_ticks_committed;             // ticks this rank committed (statistics)
  uint32_t cta_counter_iv;
  // ---- host mirror of the status words: the kernel that closes a step writes (epoch, error, accepted, dropped, last_mask,
  // last_count, last_late, seq) into page-locked HOST memory (zero-copy store over PCIe) so the training loop learns a step's
  // outcome without a device read or a memcpy node in the step graph (a D2H memcpy node costs the graph ~10 us) ------------------
  uint32_t status_seq;                     // number of steps closed so far (ring index of the mirror slot = seq & 3)
  uint32_t* host_mirror;                   // 4 slots x 8 words in mapped pinned host memory, or null
  uint32_t decider_claim;                  // step+1 of the newest launch whose arrival/commit decision a CTA has claimed
  uint32_t bar_seq;                        // device barriers completed so far (dm_device_barrier)
  uint32_t pad3[14];
  volatile uint32_t bar[SYNC_MAX_RANKS * 32];   // [p*32]: peer p entered device barrier number (value)
};

struct SyncPeers {
  SyncCtrl* ctrl[SYNC_MAX_RANKS];
  float* params[SYNC_MAX_RANKS];
  const float* grads[SYNC_MAX_RANKS];
};

struct SyncArgs {
  int rank, nranks, k;
  int numel4;                 // arena length in float4
  float lr0, decay_rate;      // staircase exponential decay evaluated on device (reference K12)
  int decay_steps;
  float drop_keep;            // gradient drop-connect keep probability, <= 0: off (reference K14)
  uint32_t drop_seed;
  unsigned long long timeout_ns;
  __nv_bfloat16* shadow;      // local bf16 copy of the parameter arena (tensor-core operand source)
  // NVLS (NVSwitch multicast) views of the two arenas, null when the fabric has none.  A load from mc_grads returns the
  // SUM over all ranks computed inside the switch; a store to mc_params lands in every rank's arena.
  const float* mc_grads;
  float* mc_params;
};

// ---- system-scope memory helpers ----------------------------------------------------------------
DMNIST_DEVICE uint32_t ld_acquire_sys(const volatile uint32_t* p) {
  uint32_t v;
  asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
DMNIST_DEVICE unsigned long long ld_acquire_sys64(const volatile unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
// Polling loads: RELAXED (an acquire load costs a CCTL.IVALL -- it invalidates the SM's whole L1 -- on EVERY poll, which is
// poison for the tensor-core kernels the small aggregation CTAs are co-resident with); the one acquire fence a wait needs is
// issued by spin_until() when the wait is over.
DMNIST_DEVICE uint32_t ld_relaxed_sys(const volatile uint32_t* p) {
  uint32_t v;
  asm volatile("ld.relaxed.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
DMNIST_DEVICE unsigned long long ld_relaxed_sys64(const volatile unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.relaxed.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
DMNIST_DEVICE void fence_acq_rel_sys() { asm volatile("fence.acq_rel.sys;" ::: "memory"); }
DMNIST_DEVICE void st_release_sys(volatile uint32_t* p, uint32_t v) {
  asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
DMNIST_DEVICE void st_release_sys64(volatile unsigned long long* p, unsigned long long v) {
  asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
DMNIST_DEVICE float4 ld_peer_f4(const float* p) {   // peer data: read once, keep out of L1
  float4 v;
  asm volatile("ld.global.L1::no_allocate.v4.f32 {%0, %1, %2, %3}, [%4];"
               : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w)
               : "l"(p)
               : "memory");
  return v;
}
DMNIST_DEVICE void st_peer_f4(float* p, float4 v) {
  asm volatile("st.global.L1::no_allocate.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z),
               "f"(v.w)
               : "memory");
}

// In-switch reduction: one 16-byte load returns the element-wise fp32 sum of the same address on every rank.
DMNIST_DEVICE float4 multimem_ld_reduce_f4(const float* mc) {
  float4 v;
  asm volatile("multimem.ld_reduce.relaxed.sys.global.add.v4.f32 {%0, %1, %2, %3}, [%4];"
               : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w)
               : "l"(mc)
               : "memory");
  return v;
}
// Multicast store: the switch replicates the 16 bytes into every rank's copy.
DMNIST_DEVICE void multimem_st_f4(float* mc, float4 v) {
  asm volatile("multimem.st.relaxed.sys.global.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(mc), "f"(v.x), "f"(v.y), "f"(v.z),
               "f"(v.w)
               : "memory");
}

// Host mirror of a step's outcome.  Called by ONE thread per step, as EARLY as the outcome is known (the values are passed
// in, the control-block words themselves are updated when the step closes): the stores travel to page-locked host memory over
// PCIe while the kernel does its work, and are complete when the kernel -- hence the step's completion event -- is.  No fence:
// the host only reads the slot after waiting for that event, and checks the seq word against the step it expects.
DMNIST_DEVICE void publish_status(SyncCtrl* me, uint32_t epoch_after, uint32_t accepted, uint32_t dropped, uint32_t mask,
                                  uint32_t count, uint32_t late) {
  const uint32_t seq = me->status_seq;
  uint32_t* m = me->host_mirror;
  if (m != nullptr) {
    m += 8 * (seq & 3u);
    *reinterpret_cast<uint4*>(m) = make_uint4(epoch_after, me->error, accepted, dropped);
    *reinterpret_cast<uint4*>(m + 4) = make_uint4(mask, count, late, seq + 1);
  }
  me->status_seq = seq + 1;
}

DMNIST_DEVICE float device_lr(const SyncArgs& a, uint32_t step) {
  const float p = (float)(step / (uint32_t)max(a.decay_steps, 1));
  return a.lr0 * __powf(a.decay_rate, p);
}

// ---- update rules: the one place that spells the optimizer formulas for every aggregation kernel -----------------------
// TF 1.x semantics (distributedmnist_b200/optim.py is the host twin):
//   SGD       w -= lr * g
//   MOMENTUM  a = momentum * a + g;  w -= lr * a                                       (ApplyMomentum, no Nesterov)
//   RMSPROP   ms += (g * g - ms) * (1 - decay);  mom = momentum * mom + lr * g / sqrt(ms + eps);  w -= mom   (ApplyRMSProp)
// with g = (sum over the contributors) / divisor.  The rule is a template parameter: the SGD instantiations compile to the
// same instructions as the kernels had before state existed (the divisor stays folded into the rate there).
enum : int { RULE_SGD = 0, RULE_MOMENTUM = 1, RULE_RMSPROP = 2 };

// Per-parameter state: fp32 arenas with the parameter arena's layout, one per slot and rank (symmetric memory).
struct OptArgs {
  float* s0[SYNC_MAX_RANKS];    // momentum: accumulator a;  RMSProp: ms
  float* s1[SYNC_MAX_RANKS];    // RMSProp: mom
  float* mc_s0;                 // NVLS multicast views of the state arenas (set exactly when the parameter arena's is)
  float* mc_s1;
  float momentum, decay, eps;
  float divisor;                // > 0: the mean's divisor instead of the contributor count (host-driven interval ticks)
};

template <int RULE>
struct Update {
  static constexpr int SLOTS = RULE == RULE_SGD ? 0 : (RULE == RULE_MOMENTUM ? 1 : 2);
  float scale;                  // SGD: lr / count;  stateful rules: 1 / count (the mean is formed before the state sees it)
  float lr, momentum, decay1, eps;

  DMNIST_DEVICE Update(const OptArgs& o, float lr_, float count) {
    if constexpr (RULE == RULE_SGD) {
      scale = lr_ / count;
      lr = momentum = decay1 = eps = 0.f;
    } else {
      scale = __frcp_rn(o.divisor > 0.f ? o.divisor : count);
      lr = lr_;
      momentum = o.momentum;
      decay1 = 1.f - o.decay;
      eps = o.eps;
    }
  }
  // One element: `sum` = gradient sum over the contributors, `a` / `b` = its state slots.  Returns the new weight.
  DMNIST_DEVICE float step(float w, float sum, float& a, float& b) const {
    if constexpr (RULE == RULE_SGD) {
      return w - scale * sum;
    } else if constexpr (RULE == RULE_MOMENTUM) {
      const float g = sum * scale;
      a = momentum * a + g;
      return w - lr * a;
    } else {
      const float g = sum * scale;
      a += (g * g - a) * decay1;
      b = momentum * b + __fdiv_rn(lr * g, __fsqrt_rn(a + eps));   // correctly rounded under --use_fast_math too
      return w - b;
    }
  }
  DMNIST_DEVICE float4 step4(float4 w, float4 s, float4& a, float4& b) const {
    w.x = step(w.x, s.x, a.x, b.x);
    w.y = step(w.y, s.y, a.y, b.y);
    w.z = step(w.z, s.z, a.z, b.z);
    w.w = step(w.w, s.w, a.w, b.w);
    return w;
  }
  // state of arena float4 `i` in replica `r`'s arenas
  DMNIST_DEVICE static void load(const OptArgs& o, int r, size_t i, float4& a, float4& b) {
    if constexpr (SLOTS > 0) a = reinterpret_cast<const float4*>(o.s0[r])[i];
    if constexpr (SLOTS > 1) b = reinterpret_cast<const float4*>(o.s1[r])[i];
  }
  DMNIST_DEVICE static void store(const OptArgs& o, int r, size_t i, float4 a, float4 b) {
    if constexpr (SLOTS > 0) reinterpret_cast<float4*>(o.s0[r])[i] = a;
    if constexpr (SLOTS > 1) reinterpret_cast<float4*>(o.s1[r])[i] = b;
  }
  // the owner of a shard replicates its new state into every replica's arenas, next to the weights: multicast (NVLS) or
  // peer stores.  Must be issued before the fence that precedes the owner's "pushed" flag.
  DMNIST_DEVICE static void push(const OptArgs& o, int nranks, size_t i, float4 a, float4 b, bool multicast) {
    if constexpr (SLOTS > 0) {
      if (multicast) multimem_st_f4(o.mc_s0 + 4 * i, a);
      else for (int q = 0; q < nranks; ++q) st_peer_f4(o.s0[q] + 4 * i, a);
    }
    if constexpr (SLOTS > 1) {
      if (multicast) multimem_st_f4(o.mc_s1 + 4 * i, b);
      else for (int q = 0; q < nranks; ++q) st_peer_f4(o.s1[q] + 4 * i, b);
    }
  }
};

// Every kernel of the step runs with the same L1/shared split, so CTAs of different kernels can share an SM.
template <class Kern>
inline cudaError_t set_max_shared_carveout(Kern kern) {
  return cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
}

// Pointer tables of the state arenas (index = rank, like SyncPeers), hyper-parameters, divisor override.
inline OptArgs make_opt_args(void* const* s0, void* const* s1, int rank, int nranks, void* mc_s0, void* mc_s1,
                             float momentum, float decay, float eps, float divisor) {
  OptArgs o;
  for (int i = 0; i < SYNC_MAX_RANKS; ++i) {
    const int j = i < nranks ? i : rank;
    o.s0[i] = s0 != nullptr ? reinterpret_cast<float*>(s0[j]) : nullptr;
    o.s1[i] = s1 != nullptr ? reinterpret_cast<float*>(s1[j]) : nullptr;
  }
  o.mc_s0 = reinterpret_cast<float*>(mc_s0);
  o.mc_s1 = reinterpret_cast<float*>(mc_s1);
  o.momentum = momentum; o.decay = decay; o.eps = eps; o.divisor = divisor;
  return o;
}

// Poll (RELAXED loads inside pred) until pred() or the watchdog fires, then ONE acquire load of the flag the wait was about
// (`acq`: LDG.STRONG.SYS + a single CCTL.IVALL; a fence.acq_rel.sys here would be a MEMBAR.ALL.SYS, which also waits for every
// outstanding store of the SM -- measured: +4 us per step at N = 2 -- and an acquire load on every poll invalidates the SM's
// L1 thousands of times under the co-resident tensor-core kernels).
template <class Pred>
DMNIST_DEVICE bool spin_until(Pred pred, unsigned long long timeout_ns, const volatile uint32_t* acq) {
  bool ok = true;
  if (!pred()) {
    const unsigned long long t0 = globaltimer_ns();
    unsigned spins = 0;
    while (!pred()) {
      if (++spins > 64) {          // busy-poll first (the common wait is a few microseconds), then back off
        __nanosleep(64);
        if ((spins & 255) == 0 && globaltimer_ns() - t0 > timeout_ns) { ok = false; break; }
      }
    }
  }
  (void)ld_acquire_sys(acq);
  return ok;
}

}  // namespace dm
