// The gradient-aggregation hot path as ONE kernel:  arrival -> commit mask -> reduce over
// NVLink peer memory -> x 1/count -> SGD -> replicate weights -> bf16 shadow.
//
// Replaces, per training step, the reference's parameter-server round trip (SURVEY §2.5
// X1-X8; src/sync_replicas_optimizer_modified/sync_replicas_optimizer_modified.py:330-398):
//   X1 apply_grad (worker->PS reduce with staleness filter)  -> arrival bit + peer loads
//   X2 take_grad(K|N|1) (mean over accepted gradients)       -> commit mask, sum, x 1/popcount
//   X3 apply_gradients + global_step++ on the PS             -> SGD in the same loop, epoch word
//   X4 weight pulls by every worker                          -> owner pushes its shard to all peers
//   X5/X6 token enqueue / dequeue barrier                    -> done flags
// No NCCL call and no separate scale / optimizer kernel runs on this path.
//
// Every rank launches this kernel on its own GPU.  All buffers live in symmetric memory
// (same layout on every rank, peers mapped through CUDA IPC / VMM), so a kernel addresses a
// peer's gradient arena, parameter arena and control block directly.
//
// Two arrival policies:
//   FULL  (K == N):  all-to-all arrival flags, one NVLink hop.
//   KOFN  (K <  N):  arrival bitmap + commit word owned by the chief (rank 0): a rank ORs its
//                    bit into the chief's bitmap; whoever first observes popcount >= K publishes
//                    the frozen bitmap with a CAS and broadcasts it to every rank's control
//                    block.  Ranks in the mask form the reduce team: team member i of c owns
//                    shard i of c, sums the *masked* contributors, divides by c and pushes the
//                    new weights to ALL N ranks.  A rank that is not in the mask ("late") or
//                    arrives for an already committed step ("stale", reference …modified.py:59-62)
//                    has its gradient discarded, waits until the pushes have landed, fast-forwards
//                    to the newest global step and continues: replicas never diverge and nobody
//                    waits for a straggler.
#include "fused_sync.cuh"

namespace dm {

// ---------------------------------------------------------------------------------------------------
// Arrival + commit decision (executed by CTA 0, warp 0).  Publishes decided_* in the local ctrl.
// ---------------------------------------------------------------------------------------------------
template <bool KOFN>
DMNIST_DEVICE void decide(const SyncPeers& P, const SyncArgs& a, SyncCtrl* me, uint32_t epoch) {
  const int lane = threadIdx.x;
  const uint32_t full_mask = (a.nranks >= 32) ? 0xffffffffu : ((1u << a.nranks) - 1u);
  uint32_t mask = full_mask, late = 0, target = epoch + 1;
  if (lane == 0) { const unsigned long long now = globaltimer_ns(); me->t_arrive[epoch % TIMING_RING] = now; me->t_phase[0] = now; }
  // The gradient arena was written by earlier kernels of this stream: it is complete in my L2, which is
  // where peers read it over NVLink; the release on the flag store below orders it for them.
  if (!KOFN) {
    if (lane < a.nranks) st_release_sys(&P.ctrl[lane]->arrive[a.rank * 32], epoch + 1);
    bool ok = true;
    if (lane < a.nranks)
      ok = spin_until([&] { return ld_relaxed_sys(&me->arrive[lane * 32]) >= epoch + 1; }, a.timeout_ns, &me->arrive[lane * 32]);
    if (!__all_sync(0xffffffffu, ok) && lane == 0) me->error = 1;
  } else {
    SyncCtrl* chief = P.ctrl[0];
    const int slot = epoch % SYNC_RING;
    if (lane == 0) {
      const unsigned long long want_tag = (unsigned long long)(epoch + 1);
      // Commit words are broadcast into every rank's control block, so "is my step already
      // committed?" is a local read (no NVLink round trip on the common path).
      unsigned long long cw = ld_acquire_sys64(&me->commit_local[slot]);
      if ((cw >> 32) < want_tag) {
        // Not committed as far as I can see: OR my bit into the chief's bitmap.  Bitmap slots carry
        // no tag: the committer of step s clears the slot of step s + RING/2, so a bit that lands
        // after its step committed (the race below) is wiped half a lap before the slot is reused.
        const unsigned int now = (atomicOr_system(&chief->bitmap[slot], 1u << a.rank) | (1u << a.rank)) & full_mask;
        if (__popc(now) >= a.k) {
          unsigned long long old = ld_acquire_sys64((volatile unsigned long long*)&chief->commit[slot]);
          if ((old >> 32) < want_tag) {
            const unsigned long long mine = (want_tag << 32) | (unsigned long long)now;
            // exactly one winner publishes the frozen bitmap as the step's commit mask
            if (atomicCAS_system(&chief->commit[slot], old, mine) == old) {
              for (int q = 0; q < a.nranks; ++q)
                if ((now >> q) & 1u) chief->last_in_mask[q] = epoch + 1;
              __threadfence_system();
              atomicMax_system((unsigned int*)&chief->global_step, epoch + 1);
              for (int q = 0; q < a.nranks; ++q) st_release_sys64(&P.ctrl[q]->commit_local[slot], mine);
              atomicExch_system(&chief->bitmap[(slot + SYNC_RING / 2) % SYNC_RING], 0u);
            }
          }
        }
        // wait for the commit word of my step to reach my control block
        const bool ok = spin_until(
            [&] { cw = ld_relaxed_sys64(&me->commit_local[slot]); return (cw >> 32) >= want_tag; }, a.timeout_ns,
            reinterpret_cast<const volatile uint32_t*>(&me->commit_local[slot]));
        if (!ok) me->error = 1;
      }
      if ((cw >> 32) == want_tag) {
        mask = (uint32_t)cw;
        late = ((mask >> a.rank) & 1u) ? 0u : 1u;
      } else {
        mask = 0;   // committed at least one ring lap ago: stale beyond the ring
        late = 1;
      }
      if (late) {
        // stale / late (reference: push dropped, worker proceeds with the newest step): fast-forward
        const uint32_t g = ld_acquire_sys(&chief->global_step);
        target = g > epoch + 1 ? g : epoch + 1;
      }
    }
    mask = __shfl_sync(0xffffffffu, mask, 0);
    late = __shfl_sync(0xffffffffu, late, 0);
    target = __shfl_sync(0xffffffffu, target, 0);
  }
  if (lane == 0) {
    me->decided_mask = mask;
    me->decided_late = late;
    me->decided_target = target;
    __threadfence();
    st_release_sys(&me->decided_tag, epoch + 1);
  }
}

template <bool KOFN, int RULE>
__global__ void __launch_bounds__(SYNC_THREADS, 1) fused_sync_sgd_kernel(SyncPeers P, SyncArgs a, OptArgs o) {
  using U = Update<RULE>;
  SyncCtrl* me = P.ctrl[a.rank];
  __shared__ uint32_t s_mask, s_late, s_target, s_last;
  pdl_wait();      // the gradient arena is complete only when the backward kernels have finished
  const uint32_t epoch = me->epoch;   // stable for the whole launch (only the last CTA writes it, at exit)

  const bool solo = a.nranks == 1;     // single replica: no arrival / commit / done protocol at all
  if (solo) {
    if (threadIdx.x == 0) {
      s_mask = 1u; s_late = 0u; s_target = epoch + 1;
      if (blockIdx.x == 0) {
        const unsigned long long now = globaltimer_ns();
        me->t_arrive[epoch % TIMING_RING] = now;
        me->t_phase[0] = now;
        me->t_phase[1] = now;
      }
    }
  } else {
    // The arrival / commit decision is taken by whichever CTA gets here first (its warp 0), not by a fixed block index:
    // CUDA does not promise that block 0 is resident before the polling CTAs fill the machine (side-stream kernels or an
    // evaluator sharing the GPU may hold SMs), and every other CTA only spins on a LOCAL word.
    if (threadIdx.x < 32) {
      uint32_t won = 0;
      if (threadIdx.x == 0) won = atomicMax(&me->decider_claim, epoch + 1) < epoch + 1 ? 1u : 0u;
      won = __shfl_sync(0xffffffffu, won, 0);
      if (won) decide<KOFN>(P, a, me, epoch);
    }
    if (threadIdx.x == 0) {
      spin_until([&] { return ld_relaxed_sys(&me->decided_tag) == epoch + 1; }, a.timeout_ns * 2, &me->decided_tag);
      s_mask = me->decided_mask;
      s_late = me->decided_late;
      s_target = me->decided_target;
      if (blockIdx.x == 0) me->t_phase[1] = globaltimer_ns();
    }
  }
  __syncthreads();
  const uint32_t mask = s_mask, late = s_late;
  const int count = __popc(mask);
  if (blockIdx.x == 0 && threadIdx.x == 0)     // the step's outcome is decided: tell the host now, the PCIe trip overlaps the reduction
    publish_status(me, s_target, me->accepted_steps + (late ? 0u : 1u), me->dropped_steps + (late ? 1u : 0u), mask, (uint32_t)count, late);
  int own_begin = 0, own_end = 0;   // float4 range whose shadow this rank writes in the update loop

  if (!late && count > 0) {
    // ---- reduce my shard over the contributors, SGD, push to every rank -------------------------
    const int my_idx = __popc(mask & ((1u << a.rank) - 1u));
    const int shard = (a.numel4 + count - 1) / count;
    const int begin = my_idx * shard;
    const int end = min(begin + shard, a.numel4);
    own_begin = begin;
    own_end = end;
    const U up(o, device_lr(a, epoch), (float)count);
    const uint32_t drop_thresh = a.drop_keep > 0.f ? (uint32_t)(a.drop_keep * 16777216.f) : 0u;
    int contrib[SYNC_MAX_RANKS];
    int nc = 0;
    for (int q = 0; q < a.nranks; ++q)
      if ((mask >> q) & 1u) contrib[nc++] = q;
    const float* wsrc = P.params[a.rank];
    const uint32_t full_mask = (1u << a.nranks) - 1u;
    if (a.mc_grads != nullptr && a.mc_params != nullptr && !solo && mask == full_mask && drop_thresh == 0u) {
      // ---- NVLS path (every replica contributes): the reduction happens inside the NVSwitch and the update is
      // multicast back, so each GPU's links carry |shard| once in and once out instead of (N-1) x |shard| each way.
      constexpr int V = 4;
      const int stride = gridDim.x * SYNC_THREADS;
      for (int i0 = begin + blockIdx.x * SYNC_THREADS + threadIdx.x; i0 < end; i0 += V * stride) {
        float4 g[V], w[V], sa[V], sb[V];
#pragma unroll
        for (int u = 0; u < V; ++u) {
          const int i = i0 + u * stride;
          if (i < end) {
            g[u] = multimem_ld_reduce_f4(a.mc_grads + 4 * (size_t)i);
            w[u] = *reinterpret_cast<const float4*>(wsrc + 4 * (size_t)i);
            U::load(o, a.rank, (size_t)i, sa[u], sb[u]);
          }
        }
#pragma unroll
        for (int u = 0; u < V; ++u) {
          const int i = i0 + u * stride;
          if (i >= end) continue;
          const float4 nw = up.step4(w[u], g[u], sa[u], sb[u]);
          multimem_st_f4(a.mc_params + 4 * (size_t)i, nw);
          U::push(o, a.nranks, (size_t)i, sa[u], sb[u], true);
          if (a.shadow != nullptr) {
            uint2 o;
            o.x = pack_bf16x2(nw.x, nw.y);
            o.y = pack_bf16x2(nw.z, nw.w);
            *reinterpret_cast<uint2*>(a.shadow + 4 * (size_t)i) = o;
          }
        }
      }
    } else {
    // Latency is the enemy here (a remote load is ~2 us): every thread issues the loads of ALL contributors
    // for U elements before it touches any of them, so one NVLink round trip covers the whole reduction of
    // its elements (at N = 8 a shard is so small that most threads make exactly one trip).
    constexpr int UN = 2;
    const int stride = gridDim.x * SYNC_THREADS;
    for (int i0 = begin + blockIdx.x * SYNC_THREADS + threadIdx.x; i0 < end; i0 += UN * stride) {
      float4 g[UN][SYNC_MAX_RANKS], w[UN], sa[UN], sb[UN];
#pragma unroll
      for (int u = 0; u < UN; ++u) {
        const int i = i0 + u * stride;
#pragma unroll
        for (int c = 0; c < SYNC_MAX_RANKS; ++c)
          g[u][c] = (c < nc && i < end) ? ld_peer_f4(P.grads[contrib[c]] + 4 * (size_t)i) : make_float4(0.f, 0.f, 0.f, 0.f);
        if (i < end) {
          w[u] = *reinterpret_cast<const float4*>(wsrc + 4 * (size_t)i);
          U::load(o, a.rank, (size_t)i, sa[u], sb[u]);
        }
      }
#pragma unroll
      for (int u = 0; u < UN; ++u) {
        const int i = i0 + u * stride;
        if (i >= end) continue;
        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int c = 0; c < SYNC_MAX_RANKS; ++c) {
          if (c < nc) {
            float4 v = g[u][c];
            if (drop_thresh) {   // drop-connect: contributor's Bernoulli mask, no 1/p rescale (reference :414-416)
              const uint32_t sm = a.drop_seed + epoch * 0x9E3779B9u + (uint32_t)contrib[c] * 0x85EBCA77u;
              v.x = dropout_keep(sm, 4u * i + 0, drop_thresh) ? v.x : 0.f;
              v.y = dropout_keep(sm, 4u * i + 1, drop_thresh) ? v.y : 0.f;
              v.z = dropout_keep(sm, 4u * i + 2, drop_thresh) ? v.z : 0.f;
              v.w = dropout_keep(sm, 4u * i + 3, drop_thresh) ? v.w : 0.f;
            }
            acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
          }
        }
        const float4 nw = up.step4(w[u], acc, sa[u], sb[u]);
        for (int q = 0; q < a.nranks; ++q) st_peer_f4(P.params[q] + 4 * (size_t)i, nw);
        U::push(o, a.nranks, (size_t)i, sa[u], sb[u], false);
        if (a.shadow != nullptr) {   // my shard's bf16 shadow straight from registers
          uint2 o;
          o.x = pack_bf16x2(nw.x, nw.y);
          o.y = pack_bf16x2(nw.z, nw.w);
          *reinterpret_cast<uint2*>(a.shadow + 4 * (size_t)i) = o;
        }
      }
    }
    }   // P2P path
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) me->t_phase[2] = globaltimer_ns();

  // ---- grid-wide: all my pushes are out -> tell every rank ------------------------------------------
  __syncthreads();
  if (threadIdx.x == 0) {
    if (!solo) __threadfence_system();
    s_last = (atomicAdd(&me->cta_counter, 1u) == gridDim.x - 1) ? 1u : 0u;
  }
  __syncthreads();
  if (!solo && s_last && !late && threadIdx.x < a.nranks) st_release_sys(&P.ctrl[threadIdx.x]->done[a.rank * 32], epoch + 1);
  if (s_last && threadIdx.x == 0) me->t_phase[3] = globaltimer_ns();

  // ---- wait until every team member's shard has landed in MY arena ---------------------------------
  if (!solo && threadIdx.x < a.nranks) {
    const int q = threadIdx.x;
    uint32_t need = ((mask >> q) & 1u) ? epoch + 1 : 0u;
    if (KOFN && late) need = ld_acquire_sys(&P.ctrl[0]->last_in_mask[q]);   // fast-forward: everything committed so far
    const bool ok = spin_until([&] { return ld_relaxed_sys(&me->done[q * 32]) >= need; }, a.timeout_ns, &me->done[q * 32]);
    if (!ok) me->error = 2;
  }
  __syncthreads();
  if (blockIdx.x == 0 && threadIdx.x == 0) me->t_phase[4] = globaltimer_ns();

  // ---- local bf16 shadow of the fresh weights (operand source for the tcgen05 kernels) --------------
  if (a.shadow != nullptr) {
    const float* w = P.params[a.rank];
    for (int i = blockIdx.x * SYNC_THREADS + threadIdx.x; i < a.numel4; i += gridDim.x * SYNC_THREADS) {
      if (i >= own_begin && i < own_end) continue;                       // done in the update loop
      const float4 v = __ldcv(reinterpret_cast<const float4*>(w) + i);   // bypass L1: peers just wrote it
      uint2 o;
      o.x = pack_bf16x2(v.x, v.y);
      o.y = pack_bf16x2(v.z, v.w);
      *reinterpret_cast<uint2*>(a.shadow + 4 * (size_t)i) = o;
    }
  }

  // ---- bookkeeping by the last CTA ---------------------------------------------------------------------
  if (s_last && threadIdx.x == 0) {
    me->last_mask = mask;
    me->last_count = count;
    me->last_late = late;
    if (late) me->dropped_steps += 1; else me->accepted_steps += 1;
    me->cta_counter = 0;
    me->t_phase[5] = globaltimer_ns();
    me->epoch = s_target;
  }
}

// =====================================================================================================================
// Bucketed aggregation (K == N, more than one replica): the step's gradients become available in two waves --
//   early bucket  fc1/fc2 parameters, 96.9 % of the bytes, complete ~45 % into the backward pass,
//   late bucket   conv1/conv2 parameters, 3 % of the bytes, complete at the very end --
// so the bulk of the NVLink traffic is moved under the remaining backward kernels:
//
//   sync_early (a few CTAs, side branch of the step graph, runs NEXT TO conv2 dgrad/wgrad + conv1 wgrad)
//       arrive_e all-to-all -> two-shot: reduce my shard of the bucket (NVLS multimem.ld_reduce or P2P loads) -> SGD ->
//       push to every rank (multimem.st / P2P stores) -> done_e flags.  Does NOT wait for the peers' pushes.
//   sync_late (whole GPU, end of the step)
//       arrive all-to-all -> ONE-shot for the small bucket: every rank sums all N contributions itself in rank order
//       (bit-identical everywhere, no push phase, one NVLink round trip) -> SGD locally -> done flags (peers may now
//       overwrite nothing I still read) -> wait done_e (the early pushes have landed here) -> bf16 shadow -> epoch + 1.
// The exposed communication per step is one flag hop + one round trip on 208 KB instead of the whole 6.6 MB exchange.
// =====================================================================================================================
struct BucketArgs {
  int begin4, end4;               // early kernel: the early bucket; late kernel: the whole arena (float4 units)
  int early_begin4, early_end4;   // late kernel: the early bucket (skipped by the one-shot, refreshed in the shadow)
};

// NR = number of replicas (compile time: the peer loop keeps 16 independent 16-byte loads in flight per thread).
// CTAs are SMALL (128 threads = one warp per scheduler, <= 96 registers, no shared memory) and there is one per SM: they fit
// next to the tensor-core CTAs of conv2 dgrad/wgrad and conv1 wgrad, whose six warps leave the schedulers mostly idle,
// so the exchange borrows issue slots instead of whole SMs.  (A first version used 20 full-size CTAs on reserved SMs:
// an SM sustains only ~10 GB/s of peer traffic -- its outstanding-request budget over a ~3 us round trip -- so 20 of
// them needed 33 us for the 2 x 3.2 MB, longer than the backward pass they were hiding under; see
// profiles/bench_r1_call26_2gpu_bucketed.txt.)
constexpr int EARLY_THREADS = 128;   // one warp per scheduler, 3 K registers each: fits next to conv2_dgrad / conv1_wgrad CTAs
template <int NR>
__global__ void __launch_bounds__(EARLY_THREADS) fused_sync_early_kernel(SyncPeers P, SyncArgs a, BucketArgs r) {
  SyncCtrl* me = P.ctrl[a.rank];
  __shared__ uint32_t s_last;
  pdl_wait();
  const uint32_t epoch = me->epoch;
  if (blockIdx.x == 0 && threadIdx.x == 0) me->t_phase_e[0] = globaltimer_ns();
  // arrival: CTA 0 tells every peer, every CTA watches the local flags (local polls are free)
  if (threadIdx.x < a.nranks) {
    if (blockIdx.x == 0) st_release_sys(&P.ctrl[threadIdx.x]->arrive_e[a.rank * 32], epoch + 1);
    const bool ok = spin_until([&] { return ld_relaxed_sys(&me->arrive_e[threadIdx.x * 32]) >= epoch + 1; }, a.timeout_ns, &me->arrive_e[threadIdx.x * 32]);
    if (!ok) me->error = 1;
  }
  __syncthreads();
  if (blockIdx.x == 0 && threadIdx.x == 0) me->t_phase_e[1] = globaltimer_ns();

  const int n4 = r.end4 - r.begin4;
  const int shard = (n4 + a.nranks - 1) / a.nranks;
  const int begin = r.begin4 + a.rank * shard;
  const int end = min(begin + shard, r.end4);
  const float scale = device_lr(a, epoch) / (float)a.nranks;
  const float* wsrc = P.params[a.rank];
  const int stride = gridDim.x * EARLY_THREADS;
  if (a.mc_grads != nullptr && a.mc_params != nullptr) {
    constexpr int V = 8;
    for (int i0 = begin + blockIdx.x * EARLY_THREADS + threadIdx.x; i0 < end; i0 += V * stride) {
      float4 g[V], w[V];
#pragma unroll
      for (int u = 0; u < V; ++u) {
        const int i = i0 + u * stride;
        if (i < end) {
          g[u] = multimem_ld_reduce_f4(a.mc_grads + 4 * (size_t)i);
          w[u] = *reinterpret_cast<const float4*>(wsrc + 4 * (size_t)i);
        }
      }
#pragma unroll
      for (int u = 0; u < V; ++u) {
        const int i = i0 + u * stride;
        if (i >= end) continue;
        float4 nw = w[u];
        nw.x -= scale * g[u].x; nw.y -= scale * g[u].y; nw.z -= scale * g[u].z; nw.w -= scale * g[u].w;
        multimem_st_f4(a.mc_params + 4 * (size_t)i, nw);
        if (a.shadow != nullptr) {
          uint2 o;
          o.x = pack_bf16x2(nw.x, nw.y);
          o.y = pack_bf16x2(nw.z, nw.w);
          *reinterpret_cast<uint2*>(a.shadow + 4 * (size_t)i) = o;
        }
      }
    }
  } else {
    constexpr int U = 16 / NR;
    for (int i0 = begin + blockIdx.x * EARLY_THREADS + threadIdx.x; i0 < end; i0 += U * stride) {
      float4 g[U][NR], w[U];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int i = i0 + u * stride;
#pragma unroll
        for (int c = 0; c < NR; ++c)
          g[u][c] = i < end ? ld_peer_f4(P.grads[c] + 4 * (size_t)i) : make_float4(0.f, 0.f, 0.f, 0.f);
        if (i < end) w[u] = *reinterpret_cast<const float4*>(wsrc + 4 * (size_t)i);
      }
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int i = i0 + u * stride;
        if (i >= end) continue;
        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int c = 0; c < NR; ++c) { acc.x += g[u][c].x; acc.y += g[u][c].y; acc.z += g[u][c].z; acc.w += g[u][c].w; }
        float4 nw = w[u];
        nw.x -= scale * acc.x; nw.y -= scale * acc.y; nw.z -= scale * acc.z; nw.w -= scale * acc.w;
#pragma unroll
        for (int q = 0; q < NR; ++q) st_peer_f4(P.params[q] + 4 * (size_t)i, nw);
        if (a.shadow != nullptr) {
          uint2 o;
          o.x = pack_bf16x2(nw.x, nw.y);
          o.y = pack_bf16x2(nw.z, nw.w);
          *reinterpret_cast<uint2*>(a.shadow + 4 * (size_t)i) = o;
        }
      }
    }
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) me->t_phase_e[2] = globaltimer_ns();
  // all my pushes are out -> tell every rank (they wait for it in their late kernel)
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence_system();
    s_last = (atomicAdd(&me->cta_counter_e, 1u) == gridDim.x - 1) ? 1u : 0u;
  }
  __syncthreads();
  if (s_last) {
    if (threadIdx.x < a.nranks) st_release_sys(&P.ctrl[threadIdx.x]->done_e[a.rank * 32], epoch + 1);
    if (threadIdx.x == 0) { me->cta_counter_e = 0; me->t_phase_e[3] = globaltimer_ns(); }
  }
}

__global__ void __launch_bounds__(SYNC_THREADS, 1) fused_sync_late_kernel(SyncPeers P, SyncArgs a, BucketArgs r) {
  SyncCtrl* me = P.ctrl[a.rank];
  __shared__ uint32_t s_last;
  pdl_wait();
  const uint32_t epoch = me->epoch;
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    const unsigned long long now = globaltimer_ns();
    me->t_arrive[epoch % TIMING_RING] = now;
    me->t_phase[0] = now;
    publish_status(me, epoch + 1, me->accepted_steps + 1, me->dropped_steps, (1u << a.nranks) - 1u, (uint32_t)a.nranks, 0u);
  }
  if (threadIdx.x < a.nranks) {
    if (blockIdx.x == 0) st_release_sys(&P.ctrl[threadIdx.x]->arrive[a.rank * 32], epoch + 1);
    const bool ok = spin_until([&] { return ld_relaxed_sys(&me->arrive[threadIdx.x * 32]) >= epoch + 1; }, a.timeout_ns, &me->arrive[threadIdx.x * 32]);
    if (!ok) me->error = 1;
  }
  __syncthreads();
  if (blockIdx.x == 0 && threadIdx.x == 0) me->t_phase[1] = globaltimer_ns();

  // ---- one-shot on the late bucket: every rank sums all contributions in rank order and updates its own copy -------------
  const float scale = device_lr(a, epoch) / (float)a.nranks;
  float* wdst = P.params[a.rank];
  const int stride = gridDim.x * SYNC_THREADS;
  // late bucket = [begin4, end4) minus the early range: walk a compacted index
  const int early_n = r.early_end4 - r.early_begin4;
  const int n_late = (r.end4 - r.begin4) - early_n;
  for (int j = blockIdx.x * SYNC_THREADS + threadIdx.x; j < n_late; j += stride) {
    const int i = (r.begin4 + j < r.early_begin4) ? r.begin4 + j : r.begin4 + j + early_n;
    float4 g[SYNC_MAX_RANKS];
#pragma unroll
    for (int c = 0; c < SYNC_MAX_RANKS; ++c)
      g[c] = c < a.nranks ? ld_peer_f4(P.grads[c] + 4 * (size_t)i) : make_float4(0.f, 0.f, 0.f, 0.f);
    float4 nw = *reinterpret_cast<const float4*>(wdst + 4 * (size_t)i);
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int c = 0; c < SYNC_MAX_RANKS; ++c)
      if (c < a.nranks) { acc.x += g[c].x; acc.y += g[c].y; acc.z += g[c].z; acc.w += g[c].w; }
    nw.x -= scale * acc.x; nw.y -= scale * acc.y; nw.z -= scale * acc.z; nw.w -= scale * acc.w;
    *reinterpret_cast<float4*>(wdst + 4 * (size_t)i) = nw;
    if (a.shadow != nullptr) {
      uint2 o;
      o.x = pack_bf16x2(nw.x, nw.y);
      o.y = pack_bf16x2(nw.z, nw.w);
      *reinterpret_cast<uint2*>(a.shadow + 4 * (size_t)i) = o;
    }
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) me->t_phase[2] = globaltimer_ns();

  // ---- my reads of the peers' gradient arenas are complete -> release them (their next step overwrites those arenas) ---------
  __syncthreads();
  if (threadIdx.x == 0) s_last = (atomicAdd(&me->cta_counter, 1u) == gridDim.x - 1) ? 1u : 0u;
  __syncthreads();
  if (s_last && threadIdx.x < a.nranks) st_release_sys(&P.ctrl[threadIdx.x]->done[a.rank * 32], epoch + 1);
  if (s_last && threadIdx.x == 0) me->t_phase[3] = globaltimer_ns();

  // ---- the early bucket's pushes (sent while the backward pass was still running) have landed in my arena? -------------------
  if (threadIdx.x < a.nranks) {
    const bool ok = spin_until([&] { return ld_relaxed_sys(&me->done_e[threadIdx.x * 32]) >= epoch + 1; }, a.timeout_ns, &me->done_e[threadIdx.x * 32]);
    if (!ok) me->error = 2;
  }
  __syncthreads();
  if (blockIdx.x == 0 && threadIdx.x == 0) me->t_phase[4] = globaltimer_ns();
  if (a.shadow != nullptr) {
    // bf16 shadow of the early bucket, except my own shard (written from registers by the early kernel)
    const int n4 = r.early_end4 - r.early_begin4;
    const int shard = (n4 + a.nranks - 1) / a.nranks;
    const int own_begin = r.early_begin4 + a.rank * shard, own_end = min(own_begin + shard, r.early_end4);
    for (int i = r.early_begin4 + blockIdx.x * SYNC_THREADS + threadIdx.x; i < r.early_end4; i += stride) {
      if (i >= own_begin && i < own_end) continue;
      const float4 v = __ldcv(reinterpret_cast<const float4*>(wdst) + i);
      uint2 o;
      o.x = pack_bf16x2(v.x, v.y);
      o.y = pack_bf16x2(v.z, v.w);
      *reinterpret_cast<uint2*>(a.shadow + 4 * (size_t)i) = o;
    }
  }
  // ---- last CTA: nobody may still be reading MY gradient arena when the next step starts overwriting it ------------------------
  if (s_last) {
    if (threadIdx.x < a.nranks) {
      const bool ok = spin_until([&] { return ld_relaxed_sys(&me->done[threadIdx.x * 32]) >= epoch + 1; }, a.timeout_ns, &me->done[threadIdx.x * 32]);
      if (!ok) me->error = 2;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
      const uint32_t full = (1u << a.nranks) - 1u;
      me->last_mask = full;
      me->last_count = a.nranks;
      me->last_late = 0;
      me->accepted_steps += 1;
      me->cta_counter = 0;
      me->t_phase[5] = globaltimer_ns();
      me->epoch = epoch + 1;
    }
  }
}

// fp32 -> bf16 shadow refresh (after init / checkpoint restore, outside the hot loop).
__global__ void f32_to_bf16_kernel(const float* __restrict__ src, __nv_bfloat16* __restrict__ dst, int n4) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += gridDim.x * blockDim.x) {
    const float4 v = reinterpret_cast<const float4*>(src)[i];
    uint2 o;
    o.x = pack_bf16x2(v.x, v.y);
    o.y = pack_bf16x2(v.z, v.w);
    reinterpret_cast<uint2*>(dst)[i] = o;
  }
}

// Device-side straggler injection: with probability `prob` (hash of the step) spin for `usec`.
__global__ void straggler_delay_kernel(const SyncCtrl* ctrl, float prob, unsigned int usec, uint32_t seed) {
  const uint32_t step = ctrl->epoch;
  if (dropout_keep(seed, step, (uint32_t)(prob * 16777216.f))) {
    const unsigned long long t0 = globaltimer_ns();
    while (globaltimer_ns() - t0 < (unsigned long long)usec * 1000ull) __nanosleep(1000);
  }
}

// Device-side barrier over NVLink flags: returns on every replica within a flag hop (~2 us) of the LAST replica entering it.
// Used to align the replicas' streams (e.g. right before a timed region: a host-side barrier leaves tens of microseconds of
// start skew between the processes).
__global__ void device_barrier_kernel(SyncPeers P, int rank, int nranks, unsigned long long timeout_ns) {
  SyncCtrl* me = P.ctrl[rank];
  const uint32_t seq = me->bar_seq + 1;
  if (threadIdx.x < nranks) {
    st_release_sys(&P.ctrl[threadIdx.x]->bar[rank * 32], seq);
    if (!spin_until([&] { return ld_relaxed_sys(&me->bar[threadIdx.x * 32]) >= seq; }, timeout_ns, &me->bar[threadIdx.x * 32])) me->error = 1;
  }
  __syncthreads();
  if (threadIdx.x == 0) me->bar_seq = seq;
}

// Stamp the start of a step's compute (%globaltimer) for the cdf-mode telemetry.
__global__ void stamp_start_kernel(SyncCtrl* ctrl) { ctrl->t_start[ctrl->epoch % TIMING_RING] = globaltimer_ns(); }
// Stamp "my gradient is complete": launched on the compute chain after the last backward kernel and BEFORE the chain joins the
// exchange branch, so a replica's compute time never contains the wait for a slower replica's gradients
// (reference: finished - dequeued, src/timeout_manager.py:55-61).  The aggregation kernels keep an existing stamp of this step.
__global__ void stamp_arrive_kernel(SyncCtrl* ctrl) {
  pdl_wait();
  ctrl->t_arrive[ctrl->epoch % TIMING_RING] = globaltimer_ns();
}

}  // namespace dm

extern "C" {

int dm_sync_ctrl_bytes() { return (int)sizeof(dm::SyncCtrl); }

// Offsets of host-readable fields (the Python side reads the control block through a view).
int dm_sync_ctrl_offset(const char* field) {
  using dm::SyncCtrl;
#define DM_OFF(name) if (strcmp(field, #name) == 0) return (int)offsetof(SyncCtrl, name)
  DM_OFF(epoch); DM_OFF(error); DM_OFF(accepted_steps); DM_OFF(dropped_steps); DM_OFF(last_mask);
  DM_OFF(last_count); DM_OFF(last_late); DM_OFF(global_step); DM_OFF(t_arrive); DM_OFF(t_start);
  DM_OFF(cta_counter); DM_OFF(t_phase); DM_OFF(t_phase_e); DM_OFF(arrive); DM_OFF(done); DM_OFF(arrive_e); DM_OFF(done_e);
  DM_OFF(commit_local); DM_OFF(bitmap); DM_OFF(commit); DM_OFF(last_in_mask); DM_OFF(decided_tag); DM_OFF(decided_mask);
  DM_OFF(decided_late); DM_OFF(decided_target); DM_OFF(cta_counter_e); DM_OFF(cta_counter2);
  DM_OFF(status_seq); DM_OFF(host_mirror); DM_OFF(decider_claim); DM_OFF(iv_state); DM_OFF(iv_busy); DM_OFF(iv_deadline); DM_OFF(iv_ticks_committed);
#undef DM_OFF
  return -1;
}

// peers: arrays of `nranks` device pointers (index = rank; own entries are the local buffers).
int dm_fused_sync_sgd(void* const* ctrl, void* const* params, void* const* grads, int rank, int nranks, int k,
                      long long numel, float lr0, float decay_rate, int decay_steps, float drop_keep,
                      unsigned int drop_seed, double timeout_ms, void* shadow_bf16, int ctas, void* stream_,
                      const void* mc_grads, void* mc_params, int rule, void* const* s0, void* const* s1, void* mc_s0,
                      void* mc_s1, float momentum, float decay, float eps, float divisor) {
  using namespace dm;
  if (nranks < 1 || nranks > SYNC_MAX_RANKS || (numel & 3) || k < 1 || k > nranks) return -1;
  if (rule < RULE_SGD || rule > RULE_RMSPROP || (rule != RULE_SGD && s0 == nullptr) || (rule == RULE_RMSPROP && s1 == nullptr)) return -4;
  if (rule != RULE_SGD && mc_params != nullptr && (mc_s0 == nullptr || (rule == RULE_RMSPROP && mc_s1 == nullptr))) return -4;
  SyncPeers P;
  for (int i = 0; i < SYNC_MAX_RANKS; ++i) {
    const int j = i < nranks ? i : rank;
    P.ctrl[i] = reinterpret_cast<SyncCtrl*>(ctrl[j]);
    P.params[i] = reinterpret_cast<float*>(params[j]);
    P.grads[i] = reinterpret_cast<const float*>(grads[j]);
  }
  SyncArgs a;
  a.rank = rank; a.nranks = nranks; a.k = k; a.numel4 = (int)(numel / 4);
  a.lr0 = lr0; a.decay_rate = decay_rate; a.decay_steps = decay_steps;
  a.drop_keep = drop_keep; a.drop_seed = drop_seed;
  a.timeout_ns = (unsigned long long)(timeout_ms * 1e6);
  a.shadow = reinterpret_cast<__nv_bfloat16*>(shadow_bf16);
  a.mc_grads = reinterpret_cast<const float*>(mc_grads);
  a.mc_params = reinterpret_cast<float*>(mc_params);
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  const OptArgs o = make_opt_args(s0, s1, rank, nranks, mc_s0, mc_s1, momentum, decay, eps, divisor);
  if (ctas < 1) ctas = 64;
  static bool configured = false;
  if (!configured) {     // every kernel of the step runs with the same L1/shared split, so CTAs of different kernels can share an SM
    DM_CUDA_OK(set_max_shared_carveout(fused_sync_sgd_kernel<true, RULE_SGD>));
    DM_CUDA_OK(set_max_shared_carveout(fused_sync_sgd_kernel<false, RULE_SGD>));
    DM_CUDA_OK(set_max_shared_carveout(fused_sync_sgd_kernel<true, RULE_MOMENTUM>));
    DM_CUDA_OK(set_max_shared_carveout(fused_sync_sgd_kernel<false, RULE_MOMENTUM>));
    DM_CUDA_OK(set_max_shared_carveout(fused_sync_sgd_kernel<true, RULE_RMSPROP>));
    DM_CUDA_OK(set_max_shared_carveout(fused_sync_sgd_kernel<false, RULE_RMSPROP>));
    configured = true;
  }
  const dim3 g(ctas), b(SYNC_THREADS);
  switch (rule * 2 + (k < nranks ? 1 : 0)) {
    case 2 * RULE_SGD + 1: return (int)launch_kernel(fused_sync_sgd_kernel<true, RULE_SGD>, g, b, 0, stream, P, a, o);
    case 2 * RULE_MOMENTUM: return (int)launch_kernel(fused_sync_sgd_kernel<false, RULE_MOMENTUM>, g, b, 0, stream, P, a, o);
    case 2 * RULE_MOMENTUM + 1: return (int)launch_kernel(fused_sync_sgd_kernel<true, RULE_MOMENTUM>, g, b, 0, stream, P, a, o);
    case 2 * RULE_RMSPROP: return (int)launch_kernel(fused_sync_sgd_kernel<false, RULE_RMSPROP>, g, b, 0, stream, P, a, o);
    case 2 * RULE_RMSPROP + 1: return (int)launch_kernel(fused_sync_sgd_kernel<true, RULE_RMSPROP>, g, b, 0, stream, P, a, o);
    default: return (int)launch_kernel(fused_sync_sgd_kernel<false, RULE_SGD>, g, b, 0, stream, P, a, o);
  }
}

// Bucketed aggregation, K == N.  phase 1 = early bucket [begin, end) floats, phase 2 = late bucket [begin, end) with the
// early bucket [early_begin, early_end) named for the shadow refresh.  All offsets are multiples of 4 floats.
int dm_fused_sync_bucket(void* const* ctrl, void* const* params, void* const* grads, int rank, int nranks, int phase,
                         long long begin, long long end, long long early_begin, long long early_end, float lr0,
                         float decay_rate, int decay_steps, double timeout_ms, void* shadow_bf16, int ctas, void* stream_,
                         const void* mc_grads, void* mc_params) {
  using namespace dm;
  if (nranks < 2 || nranks > SYNC_MAX_RANKS || ((begin | end | early_begin | early_end) & 3) || phase < 1 || phase > 2) return -1;
  SyncPeers P;
  for (int i = 0; i < SYNC_MAX_RANKS; ++i) {
    const int j = i < nranks ? i : rank;
    P.ctrl[i] = reinterpret_cast<SyncCtrl*>(ctrl[j]);
    P.params[i] = reinterpret_cast<float*>(params[j]);
    P.grads[i] = reinterpret_cast<const float*>(grads[j]);
  }
  SyncArgs a;
  a.rank = rank; a.nranks = nranks; a.k = nranks; a.numel4 = 0;
  a.lr0 = lr0; a.decay_rate = decay_rate; a.decay_steps = decay_steps;
  a.drop_keep = 0.f; a.drop_seed = 0;
  a.timeout_ns = (unsigned long long)(timeout_ms * 1e6);
  a.shadow = reinterpret_cast<__nv_bfloat16*>(shadow_bf16);
  a.mc_grads = reinterpret_cast<const float*>(mc_grads);
  a.mc_params = reinterpret_cast<float*>(mc_params);
  BucketArgs r;
  r.begin4 = (int)(begin / 4); r.end4 = (int)(end / 4);
  r.early_begin4 = (int)(early_begin / 4); r.early_end4 = (int)(early_end / 4);
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  if (ctas < 1) ctas = 148;
  if (phase == 1) {
    // The early kernel must be CO-RESIDENT with the tensor-core kernels of the backward pass.  CTAs of kernels that run
    // with different L1/shared splits cannot share an SM (observed: the early kernel only got SMs as conv2_dgrad CTAs
    // exited, profiles/bench_r1_call27_2gpu.txt), so EVERY kernel of the step asks for the same split (max shared).
    static bool configured = false;
    if (!configured) {
      DM_CUDA_OK(cudaFuncSetAttribute(fused_sync_early_kernel<2>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
      DM_CUDA_OK(cudaFuncSetAttribute(fused_sync_early_kernel<4>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
      DM_CUDA_OK(cudaFuncSetAttribute(fused_sync_early_kernel<8>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
      DM_CUDA_OK(cudaFuncSetAttribute(fused_sync_late_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
      configured = true;
    }
    if (nranks == 2) return (int)launch_kernel(fused_sync_early_kernel<2>, dim3(ctas), dim3(EARLY_THREADS), 0, stream, P, a, r);
    if (nranks == 4) return (int)launch_kernel(fused_sync_early_kernel<4>, dim3(ctas), dim3(EARLY_THREADS), 0, stream, P, a, r);
    if (nranks == 8) return (int)launch_kernel(fused_sync_early_kernel<8>, dim3(ctas), dim3(EARLY_THREADS), 0, stream, P, a, r);
    return -5;     // bucketed path is instantiated for 2, 4 and 8 replicas; the caller falls back to the single kernel
  }
  return (int)launch_kernel(fused_sync_late_kernel, dim3(ctas), dim3(SYNC_THREADS), 0, stream, P, a, r);
}

// Point the control block's host mirror at `host_ptr` (page-locked, device-accessible host memory: 4 slots x 8 words) or null.
int dm_sync_set_host_mirror(void* ctrl, void* host_ptr) {
  using dm::SyncCtrl;
  DM_CUDA_OK(cudaMemcpy(reinterpret_cast<char*>(ctrl) + offsetof(SyncCtrl, host_mirror), &host_ptr, sizeof(void*),
                        cudaMemcpyHostToDevice));
  return 0;
}

int dm_f32_to_bf16(const void* src, void* dst, long long numel, void* stream_) {
  if (numel & 3) return -1;
  dm::f32_to_bf16_kernel<<<148, 512, 0, reinterpret_cast<cudaStream_t>(stream_)>>>(
      reinterpret_cast<const float*>(src), reinterpret_cast<__nv_bfloat16*>(dst), (int)(numel / 4));
  return (int)cudaGetLastError();
}

int dm_straggler_delay(const void* ctrl, float prob, unsigned int usec, unsigned int seed, void* stream_) {
  dm::straggler_delay_kernel<<<1, 1, 0, reinterpret_cast<cudaStream_t>(stream_)>>>(
      reinterpret_cast<const dm::SyncCtrl*>(ctrl), prob, usec, seed);
  return (int)cudaGetLastError();
}

int dm_device_barrier(void* const* ctrl, int rank, int nranks, double timeout_ms, void* stream_) {
  using namespace dm;
  if (nranks < 1 || nranks > SYNC_MAX_RANKS) return -1;
  SyncPeers P;
  for (int i = 0; i < SYNC_MAX_RANKS; ++i) {
    P.ctrl[i] = reinterpret_cast<SyncCtrl*>(ctrl[i < nranks ? i : rank]);
    P.params[i] = nullptr;
    P.grads[i] = nullptr;
  }
  device_barrier_kernel<<<1, 32, 0, reinterpret_cast<cudaStream_t>(stream_)>>>(P, rank, nranks, (unsigned long long)(timeout_ms * 1e6));
  return (int)cudaGetLastError();
}

int dm_stamp_arrive(void* ctrl, void* stream_) {
  return (int)dm::launch_kernel(dm::stamp_arrive_kernel, dim3(1), dim3(1), 0, reinterpret_cast<cudaStream_t>(stream_),
                                reinterpret_cast<dm::SyncCtrl*>(ctrl));
}

int dm_stamp_start(void* ctrl, void* stream_) {
  dm::stamp_start_kernel<<<1, 1, 0, reinterpret_cast<cudaStream_t>(stream_)>>>(reinterpret_cast<dm::SyncCtrl*>(ctrl));
  return (int)cudaGetLastError();
}

}  // extern "C"
