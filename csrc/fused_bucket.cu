// Bucketed, overlapped gradient aggregation for the headline configuration (every replica contributes, K == N, on 1/2/4/8
// replicas): the reference's per-step parameter-server round trip (SURVEY §2.5 X1-X6;
// src/sync_replicas_optimizer_modified/sync_replicas_optimizer_modified.py:330-398) as TWO kernels per step, neither of
// which calls NCCL or leaves an elementwise kernel behind:
//
//   bucket_early_kernel   side branch of the step graph, co-resident with conv2 dgrad/wgrad + conv1 wgrad.
//       The fc1 weight gradient (96.5 % of the model's bytes) travels as **bf16**: fc1_wgrad's epilogue stores bf16 into a
//       symmetric buffer g16; rank r reduces shard r of everybody's g16 *in place* -- `multimem.ld_reduce.add.acc::f32.bf16x2`
//       (fp32 accumulation inside the NVSwitch) + `multimem.st`, or peer loads/stores where the fabric has no multicast --
//       so each GPU moves |g16| (1 + 1/N) bytes per direction instead of 2x that in fp32.  After the all-to-all "my shard is
//       out" flags every rank applies SGD to ITS OWN fp32 master copy of fc1 from the now identical bf16 sum (master weights
//       never cross NVLink) and rewrites the bf16 shadow the tensor-core kernels read.  All of it runs under the backward pass.
//   bucket_late_ll_kernel end of the step; the only exposed communication (default for a late bucket <= 1 MB: LeNet, 236 KB).
//       The small bucket (conv1/conv2/fc2 parameters + all biases) is PUSHED as LL lines {bf16x2, tag, bf16x2, tag} with
//       tag = step + 1: every rank multicasts its lines into slot [rank] of every replica's inbox (`multimem.st`; peer stores
//       without NVLS) and polls its own inbox until all N - 1 slots carry this step's tag -- data and "it is there" arrive in
//       the same 16-byte store, so ONE NVLink store latency is exposed: no flags, no fences, no grid barrier.  Rank-ordered
//       sum (bit-identical everywhere), SGD locally.  The inbox is double-buffered on the parity of the global step, so no
//       rank ever waits for a peer to finish *reading* (why that is safe: parallel/protocol.py::BucketV2Model, explored
//       schedule by schedule in tests/test_protocol.py).
//   bucket_late_kernel    the same push with plain fp32 data + one release flag per peer: for late buckets of megabytes (the
//       MLPs), which are bandwidth-bound -- LL lines would double their bytes.
//
// Replicas stay bit-identical: every rank applies the same bf16 sums / the same rank-ordered fp32 sums to identical weights.
#include "fused_sync.cuh"

namespace dm {

struct BucketV2 {
  int fc1_b4, fc1_e4;                    // fc1 weights inside the fp32 arena (float4 units)
  int numel4;                            // arena length (float4 units)
  __nv_bfloat16* g16[SYNC_MAX_RANKS];    // bf16 fc1 gradient of every rank (symmetric; reduced in place)
  float* inbox[SYNC_MAX_RANKS];          // late-bucket inbox of every rank: [2 parities][nranks][n_late] floats
  __nv_bfloat16* mc_g16;                 // NVLS multicast views (null: peer loads / stores)
  float* mc_inbox;
};

// 16 bytes = 8 bf16: in-switch sum over all ranks, accumulated in fp32, returned rounded to bf16.
DMNIST_DEVICE uint4 multimem_ld_reduce_bf16x8(const __nv_bfloat16* mc) {
  uint4 v;
  asm volatile("multimem.ld_reduce.relaxed.sys.global.add.acc::f32.v4.bf16x2 {%0, %1, %2, %3}, [%4];"
               : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w)
               : "l"(mc)
               : "memory");
  return v;
}
DMNIST_DEVICE void multimem_st_b128(void* mc, uint4 v) {
  asm volatile("multimem.st.relaxed.sys.global.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(mc), "r"(v.x), "r"(v.y), "r"(v.z),
               "r"(v.w)
               : "memory");
}
DMNIST_DEVICE uint4 ld_peer_b128(const void* p) {
  uint4 v;
  asm volatile("ld.global.L1::no_allocate.v4.u32 {%0, %1, %2, %3}, [%4];"
               : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w)
               : "l"(p)
               : "memory");
  return v;
}
DMNIST_DEVICE void st_peer_b128(void* p, uint4 v) {
  asm volatile("st.global.L1::no_allocate.v4.u32 [%0], {%1, %2, %3, %4};" ::"l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w)
               : "memory");
}
DMNIST_DEVICE float bf16_lo(uint32_t w) { return __uint_as_float(w << 16); }
DMNIST_DEVICE float bf16_hi(uint32_t w) { return __uint_as_float(w & 0xffff0000u); }

// ---------------------------------------------------------------------------------------------------------------------
// early bucket
// ---------------------------------------------------------------------------------------------------------------------
// CTAs are small (128 threads, no shared memory, <= 96 registers) and there is one per SM: they sit next to the
// tensor-core CTAs of the backward pass and borrow their idle issue slots (profiles/coresidency_probe_r1.txt).
constexpr int EARLY2_THREADS = 128;

// parts: bit 0 = exchange (arrival flags, in-place reduce of my shard, "shard out" flags), bit 1 = apply (wait for every
// shard, SGD on the local fp32 master copy, bf16 shadow).  The LeNet step launches both at once; the MLP step launches the
// exchange right after the big weight-gradient GEMM -- it touches neither weights nor shadow, so it may run next to the
// data-gradient GEMM that still reads that layer's shadow -- and the apply after it.
template <int NR, int RULE>
__global__ void __launch_bounds__(EARLY2_THREADS) bucket_early_kernel(SyncPeers P, SyncArgs a, BucketV2 r, int parts, OptArgs o) {
  using U = Update<RULE>;
  SyncCtrl* me = P.ctrl[a.rank];
  __shared__ uint32_t s_last;
  pdl_wait();
  const uint32_t epoch = me->epoch;
  const int n8 = (r.fc1_e4 - r.fc1_b4) >> 1;       // 16-byte chunks of 8 bf16
  const int stride = gridDim.x * EARLY2_THREADS;
  const int tid = blockIdx.x * EARLY2_THREADS + threadIdx.x;
  __nv_bfloat16* mine = r.g16[a.rank];
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    const unsigned long long now = globaltimer_ns();
    me->t_phase_e[0] = now;
    if (NR == 1) { me->t_phase_e[1] = now; me->t_phase_e[2] = now; me->t_phase_e[3] = now; me->t_phase_e[4] = now; }
  }

  if (NR > 1 && (parts & 1)) {
    // ---- every rank's fc1_wgrad is complete (all-to-all flags: CTA 0 tells the peers, everybody watches the local words) ----
    if (threadIdx.x < NR) {
      if (blockIdx.x == 0) st_release_sys(&P.ctrl[threadIdx.x]->arrive_e[a.rank * 32], epoch + 1);
      const bool ok = spin_until([&] { return ld_relaxed_sys(&me->arrive_e[threadIdx.x * 32]) >= epoch + 1; }, a.timeout_ns, &me->arrive_e[threadIdx.x * 32]);
      if (!ok) me->error = 1;
    }
    __syncthreads();
    if (blockIdx.x == 0 && threadIdx.x == 0) me->t_phase_e[1] = globaltimer_ns();

    // ---- reduce shard `rank` of all N gradients in place, on every replica ----------------------------------------------------
    const int shard = (n8 + NR - 1) / NR;
    const int begin = a.rank * shard, end = min(begin + shard, n8);
    if (r.mc_g16 != nullptr) {
      constexpr int V = 4;
      for (int c0 = begin + tid; c0 < end; c0 += V * stride) {
        uint4 g[V];
#pragma unroll
        for (int u = 0; u < V; ++u) {
          const int c = c0 + u * stride;
          if (c < end) g[u] = multimem_ld_reduce_bf16x8(r.mc_g16 + 8 * (size_t)c);
        }
#pragma unroll
        for (int u = 0; u < V; ++u) {
          const int c = c0 + u * stride;
          if (c >= end) continue;
          multimem_st_b128(r.mc_g16 + 8 * (size_t)c, g[u]);
          // my own copy also through the local path (same bits): the apply loop below must not depend on the multicast
          // store's trip through the switch having come back
          *reinterpret_cast<uint4*>(mine + 8 * (size_t)c) = g[u];
        }
      }
    } else {
      constexpr int U = NR >= 8 ? 2 : (NR == 4 ? 4 : 8);     // 16 independent 16-byte peer loads in flight per thread
      for (int c0 = begin + tid; c0 < end; c0 += U * stride) {
        uint4 g[U][NR];
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const int c = c0 + u * stride;
#pragma unroll
          for (int q = 0; q < NR; ++q) g[u][q] = c < end ? ld_peer_b128(r.g16[q] + 8 * (size_t)c) : make_uint4(0, 0, 0, 0);
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const int c = c0 + u * stride;
          if (c >= end) continue;
          float s[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
#pragma unroll
          for (int q = 0; q < NR; ++q) {       // rank order, fp32
            s[0] += bf16_lo(g[u][q].x); s[1] += bf16_hi(g[u][q].x); s[2] += bf16_lo(g[u][q].y); s[3] += bf16_hi(g[u][q].y);
            s[4] += bf16_lo(g[u][q].z); s[5] += bf16_hi(g[u][q].z); s[6] += bf16_lo(g[u][q].w); s[7] += bf16_hi(g[u][q].w);
          }
          const uint4 o = make_uint4(pack_bf16x2(s[0], s[1]), pack_bf16x2(s[2], s[3]), pack_bf16x2(s[4], s[5]),
                                     pack_bf16x2(s[6], s[7]));
#pragma unroll
          for (int q = 0; q < NR; ++q) st_peer_b128(r.g16[q] + 8 * (size_t)c, o);
        }
      }
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) me->t_phase_e[2] = globaltimer_ns();

    // ---- all my stores are out -> tell every rank; then wait until every shard has landed here --------------------------------
    __syncthreads();
    if (threadIdx.x == 0) {
      __threadfence_system();
      s_last = (atomicAdd(&me->cta_counter_e, 1u) == gridDim.x - 1) ? 1u : 0u;
    }
    __syncthreads();
    if (s_last) {
      if (threadIdx.x < NR) st_release_sys(&P.ctrl[threadIdx.x]->done_e[a.rank * 32], epoch + 1);
      if (threadIdx.x == 0) { me->cta_counter_e = 0; me->t_phase_e[3] = globaltimer_ns(); }
    }
  }
  if (!(parts & 2)) return;
  if (NR > 1) {
    if (threadIdx.x < NR) {
      const bool ok = spin_until([&] { return ld_relaxed_sys(&me->done_e[threadIdx.x * 32]) >= epoch + 1; }, a.timeout_ns, &me->done_e[threadIdx.x * 32]);
      if (!ok) me->error = 2;
    }
    __syncthreads();
    if (blockIdx.x == 0 && threadIdx.x == 0) me->t_phase_e[4] = globaltimer_ns();
  }

  // ---- update my fp32 master copy of fc1 (and its local state) from the (identical everywhere) bf16 gradient sum; fresh bf16
  // shadow ---------------------------------------------------------------------------------------------------------------
  const U up(o, device_lr(a, epoch), (float)NR);
  float* w = P.params[a.rank] + 4 * (size_t)r.fc1_b4;
  __nv_bfloat16* sh = a.shadow != nullptr ? a.shadow + 4 * (size_t)r.fc1_b4 : nullptr;
  const size_t st4 = (size_t)r.fc1_b4;                                // fc1 inside the state arenas (float4 units)
  constexpr int A = RULE == RULE_RMSPROP ? 1 : 2;                     // RMSProp's four state vectors: stay within 96 registers
  for (int c0 = tid; c0 < n8; c0 += A * stride) {
    uint4 g[A];
    float4 w0[A], w1[A], sa0[A], sa1[A], sb0[A], sb1[A];
#pragma unroll
    for (int u = 0; u < A; ++u) {
      const int c = c0 + u * stride;
      if (c < n8) {
        g[u] = __ldcv(reinterpret_cast<const uint4*>(mine) + c);      // peers / the switch just wrote it: not through L1
        w0[u] = *reinterpret_cast<const float4*>(w + 8 * (size_t)c);
        w1[u] = *reinterpret_cast<const float4*>(w + 8 * (size_t)c + 4);
        U::load(o, a.rank, st4 + 2 * (size_t)c, sa0[u], sb0[u]);
        U::load(o, a.rank, st4 + 2 * (size_t)c + 1, sa1[u], sb1[u]);
      }
    }
#pragma unroll
    for (int u = 0; u < A; ++u) {
      const int c = c0 + u * stride;
      if (c >= n8) continue;
      const float4 a0 = up.step4(w0[u], make_float4(bf16_lo(g[u].x), bf16_hi(g[u].x), bf16_lo(g[u].y), bf16_hi(g[u].y)), sa0[u], sb0[u]);
      const float4 a1 = up.step4(w1[u], make_float4(bf16_lo(g[u].z), bf16_hi(g[u].z), bf16_lo(g[u].w), bf16_hi(g[u].w)), sa1[u], sb1[u]);
      *reinterpret_cast<float4*>(w + 8 * (size_t)c) = a0;
      *reinterpret_cast<float4*>(w + 8 * (size_t)c + 4) = a1;
      U::store(o, a.rank, st4 + 2 * (size_t)c, sa0[u], sb0[u]);
      U::store(o, a.rank, st4 + 2 * (size_t)c + 1, sa1[u], sb1[u]);
      if (sh != nullptr)
        *reinterpret_cast<uint4*>(sh + 8 * (size_t)c) =
            make_uint4(pack_bf16x2(a0.x, a0.y), pack_bf16x2(a0.z, a0.w), pack_bf16x2(a1.x, a1.y), pack_bf16x2(a1.z, a1.w));
    }
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) me->t_phase_e[5] = globaltimer_ns();
}

// ---------------------------------------------------------------------------------------------------------------------
// late bucket
// ---------------------------------------------------------------------------------------------------------------------
constexpr int LATE2_THREADS = 512;

template <int RULE>
__global__ void __launch_bounds__(LATE2_THREADS, 1) bucket_late_kernel(SyncPeers P, SyncArgs a, BucketV2 r, OptArgs o) {
  using U = Update<RULE>;
  SyncCtrl* me = P.ctrl[a.rank];
  __shared__ uint32_t s_last;
  pdl_wait();
  const uint32_t epoch = me->epoch;
  const int NR = a.nranks;
  const int early_n4 = r.fc1_e4 - r.fc1_b4;
  const int n_late4 = r.numel4 - early_n4;
  const int stride = gridDim.x * LATE2_THREADS;
  const int tid = blockIdx.x * LATE2_THREADS + threadIdx.x;
  const float* g_local = P.grads[a.rank];
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    const unsigned long long now = globaltimer_ns();
    if (me->t_arrive[epoch % TIMING_RING] < me->t_start[epoch % TIMING_RING] || me->t_start[epoch % TIMING_RING] == 0)
      me->t_arrive[epoch % TIMING_RING] = now;   // "gradient complete" stamp (unless the compute chain stamped it already)
    me->t_phase[0] = now;
    if (NR == 1) me->t_phase[1] = now;
  }
  const size_t half = (size_t)(epoch & 1u) * (size_t)NR * (size_t)n_late4;   // inbox half of this step (float4 units)

  if (NR > 1) {
    // ---- push my late-bucket gradients into slot [rank] of every replica's inbox -------------------------------------------
    const size_t slot = half + (size_t)a.rank * (size_t)n_late4;
    for (int j = tid; j < n_late4; j += stride) {
      const int i = (j < r.fc1_b4) ? j : j + early_n4;
      const float4 v = *reinterpret_cast<const float4*>(g_local + 4 * (size_t)i);
      if (r.mc_inbox != nullptr) {
        multimem_st_f4(r.mc_inbox + 4 * (slot + j), v);
      } else {
        for (int q = 0; q < NR; ++q)
          if (q != a.rank) st_peer_f4(r.inbox[q] + 4 * (slot + j), v);
      }
    }
    __syncthreads();
    if (threadIdx.x == 0) {
      __threadfence_system();
      s_last = (atomicAdd(&me->cta_counter, 1u) == gridDim.x - 1) ? 1u : 0u;
    }
    __syncthreads();
    if (s_last) {
      if (threadIdx.x < NR) st_release_sys(&P.ctrl[threadIdx.x]->arrive[a.rank * 32], epoch + 1);
      if (threadIdx.x == 0) { me->cta_counter = 0; me->t_phase[1] = globaltimer_ns(); }
    }
    // ---- every replica's push has landed in MY inbox? ------------------------------------------------------------------------
    if (threadIdx.x < NR) {
      const bool ok = spin_until([&] { return ld_relaxed_sys(&me->arrive[threadIdx.x * 32]) >= epoch + 1; }, a.timeout_ns, &me->arrive[threadIdx.x * 32]);
      if (!ok) me->error = 1;
    }
    __syncthreads();
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    me->t_phase[2] = globaltimer_ns();
    // K == N: the outcome is known; published AFTER this CTA's fence.sys (which would otherwise wait for the PCIe store)
    publish_status(me, epoch + 1, me->accepted_steps + 1, me->dropped_steps, (NR >= 32) ? 0xffffffffu : ((1u << NR) - 1u), (uint32_t)NR, 0u);
  }

  // ---- sum the N contributions in rank order, update my copy (and my state), bf16 shadow ----------------------------------
  const U up(o, device_lr(a, epoch), (float)NR);
  float* wdst = P.params[a.rank];
  const float* inbox = r.inbox[a.rank];
  for (int j = tid; j < n_late4; j += stride) {
    const int i = (j < r.fc1_b4) ? j : j + early_n4;
    float4 g[SYNC_MAX_RANKS];
    const float4 own = *reinterpret_cast<const float4*>(g_local + 4 * (size_t)i);
#pragma unroll
    for (int c = 0; c < SYNC_MAX_RANKS; ++c) {
      if (c < NR)
        g[c] = (c == a.rank) ? own : __ldcv(reinterpret_cast<const float4*>(inbox) + half + (size_t)c * (size_t)n_late4 + j);
    }
    const float4 w0 = *reinterpret_cast<const float4*>(wdst + 4 * (size_t)i);
    float4 sa, sb;
    U::load(o, a.rank, (size_t)i, sa, sb);
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int c = 0; c < SYNC_MAX_RANKS; ++c)
      if (c < NR) { acc.x += g[c].x; acc.y += g[c].y; acc.z += g[c].z; acc.w += g[c].w; }
    const float4 nw = up.step4(w0, acc, sa, sb);
    *reinterpret_cast<float4*>(wdst + 4 * (size_t)i) = nw;
    U::store(o, a.rank, (size_t)i, sa, sb);
    if (a.shadow != nullptr) {
      uint2 o;
      o.x = pack_bf16x2(nw.x, nw.y);
      o.y = pack_bf16x2(nw.z, nw.w);
      *reinterpret_cast<uint2*>(a.shadow + 4 * (size_t)i) = o;
    }
  }
  // ---- the last CTA to finish closes the step -------------------------------------------------------------------------------
  __syncthreads();
  if (threadIdx.x == 0) {
    if (atomicAdd(&me->cta_counter2, 1u) == gridDim.x - 1) {
      const uint32_t full = (NR >= 32) ? 0xffffffffu : ((1u << NR) - 1u);
      me->last_mask = full;
      me->last_count = NR;
      me->last_late = 0;
      me->accepted_steps += 1;
      me->cta_counter2 = 0;
      const unsigned long long now = globaltimer_ns();
      me->t_phase[3] = now; me->t_phase[4] = now; me->t_phase[5] = now;
      me->epoch = epoch + 1;
    }
  }
}

// ---------------------------------------------------------------------------------------------------------------------
// late bucket, LL protocol (default): every 16-byte line carries its own validity tags -- {d0, tag, d1, tag}, tag = step + 1 --
// so data and "it has arrived" travel in ONE store: no flag word, no fence.sys round trip before the flag, no grid-wide
// barrier.  A thread multicasts its lines (multimem.st; peer stores without NVLS) and then polls the matching lines of the
// other replicas in its own inbox until all four tags of a float4 are current.  Exposed communication = one NVLink store
// latency (~1.5 us) instead of store + ack + flag (~7 us measured at N = 2).  The inbox is double-buffered on the step's parity
// (a replica can be at most one step ahead of a reader) and costs 2x the bytes of the small bucket -- 475 KB per replica.
// ---------------------------------------------------------------------------------------------------------------------
DMNIST_DEVICE uint4 ld_volatile_b128(const void* p) {
  uint4 v;
  asm volatile("ld.volatile.global.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p) : "memory");
  return v;
}

// BF16 = true (default): a line carries FOUR gradients as bf16 -- {bf16x2, tag, bf16x2, tag} -- i.e. one line per float4, half the
// bytes: at N = 8 every GPU ingests 7 slots, and 7 x 475 KB of fp32 lines were ~4 us of pure NVLink ingress on the critical path.
// Every replica sums the SAME bf16-rounded contributions (its own included) in fp32, so the replicas stay bit-identical.
template <bool BF16, int RULE>
__global__ void __launch_bounds__(LATE2_THREADS) bucket_late_ll_kernel(SyncPeers P, SyncArgs a, BucketV2 r, OptArgs o) {
  using U = Update<RULE>;
  SyncCtrl* me = P.ctrl[a.rank];
  pdl_wait();
  const uint32_t epoch = me->epoch;
  const uint32_t tag = epoch + 1;
  const int NR = a.nranks;
  const int early_n4 = r.fc1_e4 - r.fc1_b4;
  const int n_late4 = r.numel4 - early_n4;
  const int stride = gridDim.x * LATE2_THREADS;
  const int tid = blockIdx.x * LATE2_THREADS + threadIdx.x;
  const float* g_local = P.grads[a.rank];
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    const unsigned long long now = globaltimer_ns();
    if (me->t_arrive[epoch % TIMING_RING] < me->t_start[epoch % TIMING_RING] || me->t_start[epoch % TIMING_RING] == 0)
      me->t_arrive[epoch % TIMING_RING] = now;   // "gradient complete" stamp (unless the compute chain stamped it already)
    me->t_phase[0] = now;
  }
  // line index space of an inbox: [2 parities][NR slots][2 * n_late4 lines of 16 bytes]
  constexpr int LPE = BF16 ? 1 : 2;                  // lines per float4
  const size_t lines_per_slot = LPE * (size_t)n_late4;
  const size_t half = (size_t)(epoch & 1u) * (size_t)NR * lines_per_slot;

  if (NR > 1) {
    const size_t slot = half + (size_t)a.rank * lines_per_slot;
    for (int j = tid; j < n_late4; j += stride) {
      const int i = (j < r.fc1_b4) ? j : j + early_n4;
      const float4 v = *reinterpret_cast<const float4*>(g_local + 4 * (size_t)i);
      const uint4 l0 = BF16 ? make_uint4(pack_bf16x2(v.x, v.y), tag, pack_bf16x2(v.z, v.w), tag)
                            : make_uint4(__float_as_uint(v.x), tag, __float_as_uint(v.y), tag);
      const uint4 l1 = make_uint4(__float_as_uint(v.z), tag, __float_as_uint(v.w), tag);
      const size_t li = slot + LPE * (size_t)j;
      if (r.mc_inbox != nullptr) {
        multimem_st_b128(reinterpret_cast<uint4*>(r.mc_inbox) + li, l0);
        if (!BF16) multimem_st_b128(reinterpret_cast<uint4*>(r.mc_inbox) + li + 1, l1);
      } else {
        for (int q = 0; q < NR; ++q) {
          if (q == a.rank) continue;
          st_peer_b128(reinterpret_cast<uint4*>(r.inbox[q]) + li, l0);
          if (!BF16) st_peer_b128(reinterpret_cast<uint4*>(r.inbox[q]) + li + 1, l1);
        }
      }
    }
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    me->t_phase[1] = globaltimer_ns();
    // every line of mine is on its way; nothing below fences, so this PCIe store rides along with the exchange
    publish_status(me, epoch + 1, me->accepted_steps + 1, me->dropped_steps, (NR >= 32) ? 0xffffffffu : ((1u << NR) - 1u), (uint32_t)NR, 0u);
  }

  // ---- receive: poll my inbox until the other replicas' lines of this step are there; rank-ordered sum; update; shadow ----
  const U up(o, device_lr(a, epoch), (float)NR);
  float* wdst = P.params[a.rank];
  const uint4* inbox = reinterpret_cast<const uint4*>(r.inbox[a.rank]);
  for (int j = tid; j < n_late4; j += stride) {
    const int i = (j < r.fc1_b4) ? j : j + early_n4;
    float4 own = *reinterpret_cast<const float4*>(g_local + 4 * (size_t)i);
    if (BF16) {                                     // my own contribution exactly as the others see it
      const uint32_t p0 = pack_bf16x2(own.x, own.y), p1 = pack_bf16x2(own.z, own.w);
      own = make_float4(bf16_lo(p0), bf16_hi(p0), bf16_lo(p1), bf16_hi(p1));
    }
    float4 g[SYNC_MAX_RANKS];
    // all N-1 slots are polled TOGETHER: the loads of every replica's lines are in flight at once (a line that has just
    // landed from NVLink costs a full memory latency; polling the slots one after the other serialised 7 of those at N = 8)
    const uint4* src = inbox + half + LPE * (size_t)j;
    uint32_t pending = ((NR >= 32) ? 0xffffffffu : ((1u << NR) - 1u)) & ~(1u << a.rank);
#pragma unroll
    for (int c = 0; c < SYNC_MAX_RANKS; ++c)
      if (c == a.rank) g[c] = own;                  // (compile-time indices: g[] stays in registers)
    unsigned long long t0 = 0;
    unsigned spins = 0;
    while (pending) {
      uint4 l0[SYNC_MAX_RANKS], l1[SYNC_MAX_RANKS];
#pragma unroll
      for (int c = 0; c < SYNC_MAX_RANKS; ++c) {
        if ((pending >> c) & 1u) {
          l0[c] = ld_volatile_b128(src + (size_t)c * lines_per_slot);
          if (!BF16) l1[c] = ld_volatile_b128(src + (size_t)c * lines_per_slot + 1);
        }
      }
#pragma unroll
      for (int c = 0; c < SYNC_MAX_RANKS; ++c) {
        if (((pending >> c) & 1u) && l0[c].y == tag && l0[c].w == tag && (BF16 || (l1[c].y == tag && l1[c].w == tag))) {
          g[c] = BF16 ? make_float4(bf16_lo(l0[c].x), bf16_hi(l0[c].x), bf16_lo(l0[c].z), bf16_hi(l0[c].z))
                      : make_float4(__uint_as_float(l0[c].x), __uint_as_float(l0[c].z), __uint_as_float(l1[c].x), __uint_as_float(l1[c].z));
          pending &= ~(1u << c);
        }
      }
      if (pending && ++spins > 64) {            // busy-poll first, then back off; watchdog instead of a hang
        if (t0 == 0) t0 = globaltimer_ns();
        __nanosleep(64);
        if ((spins & 255) == 0 && globaltimer_ns() - t0 > a.timeout_ns) { me->error = 1; break; }
      }
    }
    if (pending) {
#pragma unroll
      for (int c = 0; c < SYNC_MAX_RANKS; ++c)
        if ((pending >> c) & 1u) g[c] = make_float4(0.f, 0.f, 0.f, 0.f);
    }
    const float4 w0 = *reinterpret_cast<const float4*>(wdst + 4 * (size_t)i);
    float4 sa, sb;
    U::load(o, a.rank, (size_t)i, sa, sb);
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int c = 0; c < SYNC_MAX_RANKS; ++c)
      if (c < NR) { acc.x += g[c].x; acc.y += g[c].y; acc.z += g[c].z; acc.w += g[c].w; }
    const float4 nw = up.step4(w0, acc, sa, sb);
    *reinterpret_cast<float4*>(wdst + 4 * (size_t)i) = nw;
    U::store(o, a.rank, (size_t)i, sa, sb);
    if (a.shadow != nullptr) {
      uint2 o;
      o.x = pack_bf16x2(nw.x, nw.y);
      o.y = pack_bf16x2(nw.z, nw.w);
      *reinterpret_cast<uint2*>(a.shadow + 4 * (size_t)i) = o;
    }
  }
  // ---- the last CTA to finish closes the step -------------------------------------------------------------------------------
  __syncthreads();
  if (threadIdx.x == 0) {
    if (atomicAdd(&me->cta_counter2, 1u) == gridDim.x - 1) {
      const uint32_t full = (NR >= 32) ? 0xffffffffu : ((1u << NR) - 1u);
      me->last_mask = full;
      me->last_count = NR;
      me->last_late = 0;
      me->accepted_steps += 1;
      me->cta_counter2 = 0;
      const unsigned long long now = globaltimer_ns();
      me->t_phase[2] = now; me->t_phase[3] = now; me->t_phase[4] = now; me->t_phase[5] = now;
      me->epoch = epoch + 1;
    }
  }
}

template <int RULE>
cudaError_t configure_bucket_kernels() {
  cudaError_t e = cudaSuccess;
  for (cudaError_t x : {set_max_shared_carveout(bucket_early_kernel<1, RULE>), set_max_shared_carveout(bucket_early_kernel<2, RULE>),
                        set_max_shared_carveout(bucket_early_kernel<4, RULE>), set_max_shared_carveout(bucket_early_kernel<8, RULE>),
                        set_max_shared_carveout(bucket_late_kernel<RULE>), set_max_shared_carveout(bucket_late_ll_kernel<true, RULE>),
                        set_max_shared_carveout(bucket_late_ll_kernel<false, RULE>)})
    if (e == cudaSuccess) e = x;
  return e;
}

template <int RULE>
int launch_bucket(const SyncPeers& P, const SyncArgs& a, const BucketV2& r, const OptArgs& o, int phase, int ctas,
                  cudaStream_t stream, int late_ll, int late_bf16) {
  const int nranks = a.nranks;
  if (phase != 2) {
    if (ctas < 1) ctas = 148;
    const dim3 g(ctas), b(EARLY2_THREADS);
    const int parts = phase == 1 ? 3 : (phase == 3 ? 1 : 2);
    if (nranks == 1) return (int)launch_kernel(bucket_early_kernel<1, RULE>, g, b, 0, stream, P, a, r, parts, o);
    if (nranks == 2) return (int)launch_kernel(bucket_early_kernel<2, RULE>, g, b, 0, stream, P, a, r, parts, o);
    if (nranks == 4) return (int)launch_kernel(bucket_early_kernel<4, RULE>, g, b, 0, stream, P, a, r, parts, o);
    if (nranks == 8) return (int)launch_kernel(bucket_early_kernel<8, RULE>, g, b, 0, stream, P, a, r, parts, o);
    return -5;    // instantiated for 1, 2, 4 and 8 replicas; the caller falls back to the single kernel
  }
  if (nranks > 1 && r.inbox[0] == nullptr) return -3;
  const int n_late4 = r.numel4 - (r.fc1_e4 - r.fc1_b4);
  int grid = (n_late4 + LATE2_THREADS - 1) / LATE2_THREADS;      // one float4 per thread: a single round of loads
  if (grid < 1) grid = 1;
  // LL lines double the bytes and poll per element: the right protocol for a latency-bound SMALL bucket (LeNet: 236 KB); a
  // large late bucket (the MLPs: megabytes) is bandwidth-bound and goes as plain data + release flags
  if (late_ll && (long long)n_late4 * 16 <= (1ll << 20)) {        // no in-kernel barrier: any grid size is safe
    if (grid > 296) grid = 296;
    if (late_bf16) return (int)launch_kernel(bucket_late_ll_kernel<true, RULE>, dim3(grid), dim3(LATE2_THREADS), 0, stream, P, a, r, o);
    return (int)launch_kernel(bucket_late_ll_kernel<false, RULE>, dim3(grid), dim3(LATE2_THREADS), 0, stream, P, a, r, o);
  }
  if (ctas >= 1 && grid > ctas) grid = ctas;
  if (grid > 148) grid = 148;                                     // all CTAs must be co-resident (in-kernel barrier)
  return (int)launch_kernel(bucket_late_kernel<RULE>, dim3(grid), dim3(LATE2_THREADS), 0, stream, P, a, r, o);
}

}  // namespace dm

extern "C" {

// phase 1 = early bucket (the big weight matrix, bf16 wire, side branch): exchange + apply; 3 = exchange only; 4 = apply only;
// phase 2 = late bucket + end of the step.
//   ctrl/params/grads: tables of `nranks` peer pointers (index = rank);  g16 / inbox: same, for the bf16 fc1 gradient buffer
//   and the late-bucket inbox (2 parities x nranks slots x (numel - fc1 numel) x 8 bytes: LL lines);  mc_*: NVLS multicast views
//   or null;  late_ll: 1 = LL protocol for the late bucket (default), 0 = data + release flags;  late_bf16: LL lines carry
//   bf16 (default) or fp32 gradients.
//   fc1_begin/fc1_end/numel in floats, all multiples of 8 / 8 / 4.
int dm_bucket_sync(void* const* ctrl, void* const* params, void* const* grads, void* const* g16, void* const* inbox, int rank,
                   int nranks, int phase, long long fc1_begin, long long fc1_end, long long numel, float lr0,
                   float decay_rate, int decay_steps, double timeout_ms, void* shadow_bf16, int ctas, void* stream_,
                   void* mc_g16, void* mc_inbox, int late_ll, int late_bf16, int rule, void* const* s0, void* const* s1,
                   float momentum, float decay, float eps) {
  using namespace dm;
  if (nranks < 1 || nranks > SYNC_MAX_RANKS || phase < 1 || phase > 4) return -1;
  if (rule < RULE_SGD || rule > RULE_RMSPROP || (rule != RULE_SGD && s0 == nullptr) || (rule == RULE_RMSPROP && s1 == nullptr)) return -4;
  // every rank updates its own state from the identical sums: no state crosses NVLink, no multicast views
  const OptArgs o = make_opt_args(s0, s1, rank, nranks, nullptr, nullptr, momentum, decay, eps, 0.f);
  if ((fc1_begin & 7) || (fc1_end & 7) || (numel & 3) || fc1_begin < 0 || fc1_end < fc1_begin || fc1_end > numel) return -2;
  SyncPeers P;
  BucketV2 r;
  for (int i = 0; i < SYNC_MAX_RANKS; ++i) {
    const int j = i < nranks ? i : rank;
    P.ctrl[i] = reinterpret_cast<SyncCtrl*>(ctrl[j]);
    P.params[i] = reinterpret_cast<float*>(params[j]);
    P.grads[i] = reinterpret_cast<const float*>(grads[j]);
    r.g16[i] = reinterpret_cast<__nv_bfloat16*>(g16[j]);
    r.inbox[i] = inbox != nullptr ? reinterpret_cast<float*>(inbox[j]) : nullptr;
  }
  SyncArgs a;
  a.rank = rank; a.nranks = nranks; a.k = nranks; a.numel4 = (int)(numel / 4);
  a.lr0 = lr0; a.decay_rate = decay_rate; a.decay_steps = decay_steps;
  a.drop_keep = 0.f; a.drop_seed = 0;
  a.timeout_ns = (unsigned long long)(timeout_ms * 1e6);
  a.shadow = reinterpret_cast<__nv_bfloat16*>(shadow_bf16);
  a.mc_grads = nullptr; a.mc_params = nullptr;
  r.fc1_b4 = (int)(fc1_begin / 4); r.fc1_e4 = (int)(fc1_end / 4); r.numel4 = (int)(numel / 4);
  r.mc_g16 = nranks > 1 ? reinterpret_cast<__nv_bfloat16*>(mc_g16) : nullptr;
  r.mc_inbox = nranks > 1 ? reinterpret_cast<float*>(mc_inbox) : nullptr;
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  static bool configured = false;
  if (!configured) {   // same L1/shared split as every other kernel of the step, or the CTAs cannot share an SM with them
    DM_CUDA_OK(configure_bucket_kernels<RULE_SGD>());
    DM_CUDA_OK(configure_bucket_kernels<RULE_MOMENTUM>());
    DM_CUDA_OK(configure_bucket_kernels<RULE_RMSPROP>());
    configured = true;
  }
  if (rule == RULE_MOMENTUM) return launch_bucket<RULE_MOMENTUM>(P, a, r, o, phase, ctas, stream, late_ll, late_bf16);
  if (rule == RULE_RMSPROP) return launch_bucket<RULE_RMSPROP>(P, a, r, o, phase, ctas, stream, late_ll, late_bf16);
  return launch_bucket<RULE_SGD>(P, a, r, o, phase, ctas, stream, late_ll, late_bf16);
}

}  // extern "C"
