// Device-side interval aggregation (mode C of the reference: every `interval_ms` the parameter server applies the MEAN OF
// WHATEVER GRADIENTS HAVE ARRIVED and workers never block -- src/sync_replicas_optimizer_modified/
// sync_replicas_optimizer_modified.py:208-215 (chief timer), :373 (take_grad(1)), :59-62 (stale pushes dropped)).
//
// No timer thread and no host collective: every replica free-runs its own CUDA graph; per local iteration
//
//   iv_adopt     (1 warp)   a commit for my step has landed (commit word + the committer's "weights pushed" flag)?
//                           -> move to the new step, arm the next tick's deadline = now + interval (%globaltimer)
//   iv_shadow    (grid)     ... and refresh the bf16 shadow of the weights the committer pushed into my arena
//   <forward / backward of the model>
//   iv_gate      (1 warp)   Dekker gate against a concurrent commit: busy := step+1; fence.sc; commit word present?
//                           -> my gradient is stale (computed from weights that are being replaced): dropped
//   iv_accumulate(grid)     acc (+)= gradient          (symmetric accumulator, one per replica; nobody else writes it)
//   iv_close     (1 warp)   count++, busy := 0.  Tick deadline passed?  -> read every replica's (step, count) word, mask =
//                           replicas with count > 0 for this step, CAS the chief's commit word (exactly one winner, the
//                           arrival-bitmap/commit ring of the K-of-N path), broadcast it, wait until no contributor is
//                           mid-accumulate, re-read the counts: divisor = total number of accumulated gradients
//   iv_apply     (grid)     winner only: sum the contributors' accumulators over NVLink (peer loads), / total, update rule,
//                           push the new weights and optimizer state into EVERY replica's arenas (multimem.st / peer stores),
//                           release the "pushed" flags
//
// A replica that is mid-iteration at the deadline is simply not in the mask (its count is 0) or contributes what it had; it
// never waits for anybody and nobody waits for it.  Replicas hold bit-identical weights whenever no push is in flight.
#include "fused_sync.cuh"

namespace dm {

constexpr int IV_THREADS = 512;

DMNIST_DEVICE void fence_sc_sys() { asm volatile("fence.sc.sys;" ::: "memory"); }

struct IntervalArgs {
  float* acc[SYNC_MAX_RANKS];      // symmetric gradient accumulators (fp32, arena layout)
};

__global__ void iv_arm_kernel(SyncCtrl* me, unsigned long long interval_ns) {
  if (threadIdx.x == 0) {
    me->iv_interval_ns = interval_ns;
    me->iv_deadline = globaltimer_ns() + interval_ns;
    me->iv_state = ((unsigned long long)(me->epoch + 1) << 32);
    me->iv_busy = 0;
    me->iv_commit_go = 0;
  }
}

__global__ void iv_adopt_kernel(SyncCtrl* me) {
  pdl_wait();
  if (threadIdx.x != 0) return;
  uint32_t e = me->epoch, adopted = 0, mask = 0;
  for (int it = 0; it < SYNC_RING / 2; ++it) {
    const unsigned long long cw = ld_acquire_sys64(&me->commit_local[e % SYNC_RING]);
    if ((uint32_t)(cw >> 32) != e + 1) break;
    const uint32_t committer = ((uint32_t)cw >> 8) & 0xffu;
    if (ld_acquire_sys(&me->done[committer * 32]) < e + 1) break;     // its pushes are still landing in my arena
    mask = (uint32_t)cw & 0xffu;
    ++e; ++adopted;
  }
  if (adopted) {
    me->epoch = e;
    me->iv_deadline = globaltimer_ns() + me->iv_interval_ns;
    me->last_mask = mask;
    me->last_count = me->iv_last_total;
    __threadfence();
    st_release_sys64(&me->iv_state, (unsigned long long)(e + 1) << 32);   // new step, nothing accumulated yet
  }
  me->iv_adopted = adopted;
  me->t_start[e % TIMING_RING] = globaltimer_ns();
}

__global__ void __launch_bounds__(IV_THREADS) iv_shadow_kernel(const SyncCtrl* me, const float* __restrict__ params,
                                                               __nv_bfloat16* __restrict__ shadow, int numel4) {
  pdl_wait();
  if (!me->iv_adopted || shadow == nullptr) return;
  for (int i = blockIdx.x * IV_THREADS + threadIdx.x; i < numel4; i += gridDim.x * IV_THREADS) {
    const float4 v = __ldcv(reinterpret_cast<const float4*>(params) + i);   // pushed by a peer: not through L1
    uint2 o;
    o.x = pack_bf16x2(v.x, v.y);
    o.y = pack_bf16x2(v.z, v.w);
    *reinterpret_cast<uint2*>(shadow + 4 * (size_t)i) = o;
  }
}

__global__ void iv_gate_kernel(SyncCtrl* me) {
  pdl_wait();
  if (threadIdx.x != 0) return;
  const uint32_t e = me->epoch;
  me->iv_busy = e + 1;
  fence_sc_sys();                                   // Dekker: my busy flag is visible before I look at the commit word
  const unsigned long long cw = ld_acquire_sys64(&me->commit_local[e % SYNC_RING]);
  const uint32_t go = ((uint32_t)(cw >> 32) >= e + 1) ? 0u : 1u;
  if (!go) st_release_sys(&me->iv_busy, 0u);
  me->iv_go = go;
  me->t_arrive[e % TIMING_RING] = globaltimer_ns();
}

__global__ void __launch_bounds__(IV_THREADS) iv_accumulate_kernel(const SyncCtrl* me, float* __restrict__ acc,
                                                                   const float* __restrict__ grads, int numel4) {
  pdl_wait();
  if (!me->iv_go) return;
  const bool first = (uint32_t)me->iv_state == 0u;      // first gradient of this step overwrites: nothing to zero
  for (int i = blockIdx.x * IV_THREADS + threadIdx.x; i < numel4; i += gridDim.x * IV_THREADS) {
    float4 g = reinterpret_cast<const float4*>(grads)[i];
    if (!first) {
      const float4 a = reinterpret_cast<const float4*>(acc)[i];
      g.x += a.x; g.y += a.y; g.z += a.z; g.w += a.w;
    }
    reinterpret_cast<float4*>(acc)[i] = g;
  }
}

// One thread: close my accumulate; after the deadline try to commit the tick.
DMNIST_DEVICE void iv_close(const SyncPeers& P, const SyncArgs& a, SyncCtrl* me) {
  const uint32_t e = me->epoch;
  const uint32_t slot = e % SYNC_RING;
  me->iv_commit_go = 0;
  if (!me->iv_go) {                     // stale gradient (reference: push dropped, the worker proceeds)
    me->dropped_steps += 1;
    me->last_late = 1;
    return;
  }
  me->accepted_steps += 1;
  me->last_late = 0;
  const unsigned long long st = me->iv_state + 1ull;
  __threadfence();                      // the accumulator (previous kernel) is complete before the count says so
  st_release_sys64(&me->iv_state, st);
  st_release_sys(&me->iv_busy, 0u);
  if (globaltimer_ns() < me->iv_deadline) return;

  // ---- the tick is due: whoever gets here first commits it with the replicas that have something accumulated ----------------
  SyncCtrl* chief = P.ctrl[0];
  unsigned long long old = ld_acquire_sys64((volatile unsigned long long*)&chief->commit[slot]);
  if ((uint32_t)(old >> 32) >= e + 1) return;            // somebody else already did
  uint32_t mask = 0;
  for (int q = 0; q < a.nranks; ++q) {
    const unsigned long long sq = q == a.rank ? st : ld_acquire_sys64(&P.ctrl[q]->iv_state);
    if ((uint32_t)(sq >> 32) == e + 1 && (uint32_t)sq > 0u) mask |= 1u << q;
  }
  const unsigned long long mine = ((unsigned long long)(e + 1) << 32) | ((uint32_t)a.rank << 8) | mask;
  if (atomicCAS_system(&chief->commit[slot], old, mine) != old) return;   // exactly one winner
  for (int q = 0; q < a.nranks; ++q) st_release_sys64(&P.ctrl[q]->commit_local[slot], mine);
  fence_sc_sys();                                        // Dekker: the commit word is out before I look at the busy flags
  uint32_t total = 0;
  for (int q = 0; q < a.nranks; ++q) {
    if (!((mask >> q) & 1u)) continue;
    if (q != a.rank) {
      const bool ok = spin_until([&] { return ld_relaxed_sys(&P.ctrl[q]->iv_busy) != e + 1; }, a.timeout_ns, &P.ctrl[q]->iv_busy);
      if (!ok) me->error = 1;
    }
    const unsigned long long sq = q == a.rank ? st : ld_acquire_sys64(&P.ctrl[q]->iv_state);
    total += (uint32_t)sq;                               // final count: an accumulate that was in flight is included
  }
  me->iv_commit_mask = mask;
  me->iv_commit_total = total;
  me->iv_ticks_committed += 1;
  me->iv_commit_go = e + 1;
}

__global__ void iv_close_kernel(SyncPeers P, SyncArgs a) {
  SyncCtrl* me = P.ctrl[a.rank];
  pdl_wait();
  if (threadIdx.x != 0) return;
  iv_close(P, a, me);
  // the iteration's outcome (step, accepted / dropped) for the host loop
  publish_status(me, me->epoch, me->accepted_steps, me->dropped_steps, me->last_mask, me->last_count, me->last_late);
}

template <int RULE>
__global__ void __launch_bounds__(IV_THREADS, 1) iv_apply_kernel(SyncPeers P, SyncArgs a, IntervalArgs r, OptArgs o) {
  using U = Update<RULE>;
  SyncCtrl* me = P.ctrl[a.rank];
  __shared__ uint32_t s_last;
  pdl_wait();
  const uint32_t e = me->epoch;
  if (me->iv_commit_go != e + 1) return;
  const uint32_t mask = me->iv_commit_mask, total = me->iv_commit_total;
  const U up(o, device_lr(a, e), (float)max(total, 1u));
  int contrib[SYNC_MAX_RANKS];
  int nc = 0;
  for (int q = 0; q < a.nranks; ++q)
    if ((mask >> q) & 1u) contrib[nc++] = q;
  const float* wsrc = P.params[a.rank];
  for (int i = blockIdx.x * IV_THREADS + threadIdx.x; i < a.numel4; i += gridDim.x * IV_THREADS) {
    float4 g[SYNC_MAX_RANKS];
#pragma unroll
    for (int c = 0; c < SYNC_MAX_RANKS; ++c)
      g[c] = c < nc ? ld_peer_f4(r.acc[contrib[c]] + 4 * (size_t)i) : make_float4(0.f, 0.f, 0.f, 0.f);
    const float4 w0 = *reinterpret_cast<const float4*>(wsrc + 4 * (size_t)i);
    float4 sa, sb;
    U::load(o, a.rank, (size_t)i, sa, sb);
    float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int c = 0; c < SYNC_MAX_RANKS; ++c)
      if (c < nc) { s.x += g[c].x; s.y += g[c].y; s.z += g[c].z; s.w += g[c].w; }
    const float4 nw = up.step4(w0, s, sa, sb);
    if (a.mc_params != nullptr) {
      multimem_st_f4(a.mc_params + 4 * (size_t)i, nw);
      *reinterpret_cast<float4*>(P.params[a.rank] + 4 * (size_t)i) = nw;     // my own copy also through the local path
      U::push(o, a.nranks, (size_t)i, sa, sb, true);
      U::store(o, a.rank, (size_t)i, sa, sb);
    } else {
      for (int q = 0; q < a.nranks; ++q) st_peer_f4(P.params[q] + 4 * (size_t)i, nw);
      U::push(o, a.nranks, (size_t)i, sa, sb, false);
    }
  }
  // ---- all pushes (weights and state) are out -> publish the step ---------------------------------------------------------------------------------
  __syncthreads();
  if (threadIdx.x == 0) {
    fence_sc_sys();
    s_last = (atomicAdd(&me->cta_counter_iv, 1u) == gridDim.x - 1) ? 1u : 0u;
  }
  __syncthreads();
  if (s_last && threadIdx.x == 0) {
    me->cta_counter_iv = 0;
    atomicMax_system((unsigned int*)&P.ctrl[0]->global_step, e + 1);
    for (int q = 0; q < a.nranks; ++q) P.ctrl[q]->iv_last_total = total;
    fence_sc_sys();
    for (int q = 0; q < a.nranks; ++q) st_release_sys(&P.ctrl[q]->done[a.rank * 32], e + 1);
  }
}

}  // namespace dm

extern "C" {

// Arm the interval clock on this replica: the first tick is due `interval_ms` from now (reference: start_interval_updates).
int dm_interval_arm(void* ctrl, double interval_ms, void* stream_) {
  dm::iv_arm_kernel<<<1, 32, 0, reinterpret_cast<cudaStream_t>(stream_)>>>(reinterpret_cast<dm::SyncCtrl*>(ctrl),
                                                                         (unsigned long long)(interval_ms * 1e6));
  return (int)cudaGetLastError();
}

// First two kernels of an interval-mode iteration: adopt freshly pushed weights (+ bf16 shadow refresh).
int dm_interval_begin(void* ctrl, const void* params, void* shadow_bf16, long long numel, void* stream_) {
  using namespace dm;
  if (numel & 3) return -1;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream_);
  cudaError_t e = launch_kernel(iv_adopt_kernel, dim3(1), dim3(32), 0, st, reinterpret_cast<SyncCtrl*>(ctrl));
  if (e != cudaSuccess) return (int)e;
  return (int)launch_kernel(iv_shadow_kernel, dim3(148), dim3(IV_THREADS), 0, st, reinterpret_cast<const SyncCtrl*>(ctrl),
                            reinterpret_cast<const float*>(params), reinterpret_cast<__nv_bfloat16*>(shadow_bf16),
                            (int)(numel / 4));
}

// Last four kernels of an interval-mode iteration: gate, accumulate, close (+ commit attempt), apply (winner only).
int dm_interval_end(void* const* ctrl, void* const* params, void* const* grads, void* const* acc, int rank, int nranks,
                    long long numel, float lr0, float decay_rate, int decay_steps, double timeout_ms, int ctas, void* stream_,
                    void* mc_params, int rule, void* const* s0, void* const* s1, void* mc_s0, void* mc_s1, float momentum,
                    float decay, float eps) {
  using namespace dm;
  if (nranks < 1 || nranks > SYNC_MAX_RANKS || (numel & 3)) return -1;
  if (rule < RULE_SGD || rule > RULE_RMSPROP || (rule != RULE_SGD && s0 == nullptr) || (rule == RULE_RMSPROP && s1 == nullptr)) return -4;
  if (rule != RULE_SGD && nranks > 1 && mc_params != nullptr && (mc_s0 == nullptr || (rule == RULE_RMSPROP && mc_s1 == nullptr))) return -4;
  SyncPeers P;
  IntervalArgs r;
  for (int i = 0; i < SYNC_MAX_RANKS; ++i) {
    const int j = i < nranks ? i : rank;
    P.ctrl[i] = reinterpret_cast<SyncCtrl*>(ctrl[j]);
    P.params[i] = reinterpret_cast<float*>(params[j]);
    P.grads[i] = reinterpret_cast<const float*>(grads[j]);
    r.acc[i] = reinterpret_cast<float*>(acc[j]);
  }
  SyncArgs a;
  a.rank = rank; a.nranks = nranks; a.k = 1; a.numel4 = (int)(numel / 4);
  a.lr0 = lr0; a.decay_rate = decay_rate; a.decay_steps = decay_steps;
  a.drop_keep = 0.f; a.drop_seed = 0;
  a.timeout_ns = (unsigned long long)(timeout_ms * 1e6);
  a.shadow = nullptr; a.mc_grads = nullptr;
  a.mc_params = nranks > 1 ? reinterpret_cast<float*>(mc_params) : nullptr;
  const OptArgs o = make_opt_args(s0, s1, rank, nranks, nranks > 1 ? mc_s0 : nullptr, nranks > 1 ? mc_s1 : nullptr,
                                  momentum, decay, eps, 0.f);
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream_);
  if (ctas < 1 || ctas > 148) ctas = 148;
  SyncCtrl* me = P.ctrl[rank];
  cudaError_t e = launch_kernel(iv_gate_kernel, dim3(1), dim3(32), 0, st, me);
  if (e != cudaSuccess) return (int)e;
  e = launch_kernel(iv_accumulate_kernel, dim3(ctas), dim3(IV_THREADS), 0, st, (const SyncCtrl*)me, r.acc[rank],
                    P.grads[rank], a.numel4);
  if (e != cudaSuccess) return (int)e;
  e = launch_kernel(iv_close_kernel, dim3(1), dim3(32), 0, st, P, a);
  if (e != cudaSuccess) return (int)e;
  if (rule == RULE_MOMENTUM) return (int)launch_kernel(iv_apply_kernel<RULE_MOMENTUM>, dim3(ctas), dim3(IV_THREADS), 0, st, P, a, r, o);
  if (rule == RULE_RMSPROP) return (int)launch_kernel(iv_apply_kernel<RULE_RMSPROP>, dim3(ctas), dim3(IV_THREADS), 0, st, P, a, r, o);
  return (int)launch_kernel(iv_apply_kernel<RULE_SGD>, dim3(ctas), dim3(IV_THREADS), 0, st, P, a, r, o);
}

}  // extern "C"
