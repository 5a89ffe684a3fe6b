"""FusedBackend: gradient aggregation by the single sm_100a kernel of ``csrc/fused_sync.cu``.

The product path for SURVEY §2.5 X1-X8: the parameter arena, the gradient arena and a
control block live in symmetric memory; one kernel per step publishes arrival, obtains
the commit mask (all-to-all flags for K == N, chief-owned bitmap + CAS for K < N), sums
the contributors' gradients straight out of peer HBM over NVLink, divides by
``popcount(mask)``, applies the update rule (SGD, momentum or RMSProp, ``optim.py``) on
its shard and pushes the new weights -- and the rule's state -- into every rank's arenas,
then refreshes the local bf16 shadow used by the tensor-core kernels.
No NCCL collective and no separate elementwise kernel is launched.

Two ways to drive it:

* ``sync_step`` -- eager, host-visible result (tests, the reference-style training loop);
* ``enqueue`` -- stream-ordered launch with the LR schedule evaluated on the device from
  the device-resident step counter, so the whole training step replays as a CUDA graph
  with no per-step host input.
"""
from __future__ import annotations

import ctypes
import os
from typing import Dict, List, Optional

import torch

from ..ops.lib import check, load, require_blackwell, stream_ptr
from ..optim import rule_or_sgd
from .backends import Backend, StepInfo
from .context import ReplicaContext
from .symm_mem import SymmetricBuffer, allocate_symmetric


class FusedBackend(Backend):
    name = "fused"
    _STATUS = ("epoch", "error", "accepted_steps", "dropped_steps", "last_mask", "last_count", "last_late")

    def __init__(self, ctx: ReplicaContext, ctas: int = 0, timeout_ms: float = 30000.0, use_nvls: Optional[bool] = None,
                 debug_sync: bool = False):
        super().__init__(ctx)
        assert ctx.on_gpu, "FusedBackend needs a GPU"
        self.lib = load()
        require_blackwell(ctx.device)
        check(self.lib.dm_set_device(ctx.device.index or 0), "dm_set_device")
        # programmatic dependent launch between the kernels of a step (DMNIST_PDL=0 disables)
        self.lib.dm_set_pdl(0 if os.environ.get("DMNIST_PDL", "1") == "0" else 1)
        self.ctas = ctas or int(os.environ.get("DMNIST_SYNC_CTAS", "148"))
        # NVLS (in-switch reduction + multicast store) for the arenas when the fabric offers it; DMNIST_NVLS=0 -> P2P only
        #   DMNIST_NVLS unset: allocate multicast-capable arenas, use multimem from 4 replicas up (at 2 the peer path is
        #   faster: measured 106 vs 115 us/step, profiles/bench_r1_call23_2gpu.txt); =1 always; =0 never (CUDA-IPC arenas)
        #   (--use_nvls=false forces the P2P kernels and CUDA-IPC arenas, like DMNIST_NVLS=0)
        nv = os.environ.get("DMNIST_NVLS", "") if use_nvls is None else ("1" if use_nvls else "0")
        self.want_nvls = nv != "0"
        self.use_nvls = nv == "1" or (nv == "" and ctx.world_size >= 4)
        self.timeout_ms = timeout_ms
        self._buffers: List[SymmetricBuffer] = []
        self._by_ptr: Dict[int, SymmetricBuffer] = {}
        nbytes = int(self.lib.dm_sync_ctrl_bytes())
        self.ctrl = SymmetricBuffer(nbytes, ctx.rank, ctx.world_size, ctx.device)
        self._ctrl_bytes = self.ctrl.view(torch.uint8)
        self._off = {f: int(self.lib.dm_sync_ctrl_offset(f.encode())) for f in
                     ("epoch", "error", "accepted_steps", "dropped_steps", "last_mask", "last_count", "last_late",
                      "global_step", "t_arrive", "t_start", "cta_counter", "t_phase", "t_phase_e", "arrive", "done",
                      "arrive_e", "done_e", "commit_local", "bitmap", "commit", "last_in_mask", "decided_tag",
                      "decided_mask", "decided_late", "decided_target", "cta_counter_e", "cta_counter2", "status_seq",
                      "host_mirror", "iv_state", "iv_busy", "iv_deadline", "iv_ticks_committed", "decider_claim")}
        assert all(v >= 0 for v in self._off.values()), self._off
        # the host-readable status words (epoch .. last_late) sit next to each other: ONE device->host copy per query
        self._status_lo = min(self._off[f] for f in self._STATUS)
        self._status_hi = max(self._off[f] for f in self._STATUS) + 4
        self.debug_sync = debug_sync or os.environ.get("DMNIST_DEBUG_SYNC", "0") == "1"
        self.late_ll = os.environ.get("DMNIST_LATE_LL", "1") != "0"     # LL lines (data + tags in one store) for the late bucket
        self.late_bf16 = os.environ.get("DMNIST_LATE_BF16", "1") != "0"  # ... carrying bf16 gradients (half the bytes)
        # host mirror of the status words: the kernel that closes a step stores them into page-locked host memory itself
        self._mirror = torch.zeros(4 * 8, dtype=torch.int32).pin_memory()
        check(self.lib.dm_sync_set_host_mirror(ctypes.c_void_p(self.ctrl.local_ptr), ctypes.c_void_p(self._mirror.data_ptr())),
              "dm_sync_set_host_mirror")
        self._mirror_np = self._mirror.numpy().view("<u4")
        self.shadow: Optional[torch.Tensor] = None     # bf16 copy of the parameter arena
        self.drop_keep = 0.0
        self.drop_seed = 0

    # ---- memory ---------------------------------------------------------------------------
    def allocate(self, numel: int) -> torch.Tensor:
        buf = allocate_symmetric(numel * 4, self.ctx.rank, self.ctx.world_size, self.ctx.device, self.want_nvls)
        self._buffers.append(buf)
        t = buf.view(torch.float32, 0, numel)
        self._by_ptr[t.data_ptr()] = buf
        return t

    def allocate_buffer(self, nbytes: int):
        """Raw symmetric allocation (peer-mapped, NVLS-multicast-mapped when available): the bf16 gradient buffer and the
        late-bucket inbox of the bucketed aggregation.  Collective: every rank calls it in the same order."""
        buf = allocate_symmetric(int(nbytes), self.ctx.rank, self.ctx.world_size, self.ctx.device, self.want_nvls)
        self._buffers.append(buf)
        return buf

    def attach_shadow(self, params: torch.Tensor) -> torch.Tensor:
        """Create the local bf16 shadow arena of ``params`` and fill it."""
        self.shadow = torch.empty(params.numel(), dtype=torch.bfloat16, device=params.device)
        self.refresh_shadow(params)
        return self.shadow

    def refresh_shadow(self, params: torch.Tensor) -> None:
        if self.shadow is not None:
            check(self.lib.dm_f32_to_bf16(ctypes.c_void_p(params.data_ptr()), ctypes.c_void_p(self.shadow.data_ptr()),
                                          ctypes.c_longlong(params.numel()), stream_ptr()), "dm_f32_to_bf16")

    # ---- control-block access ---------------------------------------------------------------
    def _read_u32(self, field: str, index: int = 0) -> int:
        off = self._off[field] + 4 * index
        return int(self._ctrl_bytes[off:off + 4].view(torch.int32).item()) & 0xFFFFFFFF

    def _write_u32(self, field: str, value: int) -> None:
        off = self._off[field]
        self._ctrl_bytes[off:off + 4].view(torch.int32).fill_(value if value < 2 ** 31 else value - 2 ** 32)

    @property
    def device_epoch(self) -> int:
        return self._read_u32("epoch")

    def set_global_step(self, step: int) -> None:
        """Checkpoint restore: every rank starts from ``step`` (also the chief's commit counter)."""
        self._write_u32("epoch", step)
        self._write_u32("global_step", step)
        self._write_u32("decider_claim", step)
        torch.cuda.synchronize()
        self.barrier()

    def read_status(self) -> Dict[str, int]:
        """epoch / error / accepted / dropped / last_mask / last_count / last_late with ONE device->host copy (synchronises
        the current stream)."""
        raw = self._ctrl_bytes[self._status_lo:self._status_hi].cpu().numpy().view("<u4")
        return {f: int(raw[(self._off[f] - self._status_lo) // 4]) for f in self._STATUS}

    @property
    def status_seq(self) -> int:
        """Number of steps closed on the device so far (device read)."""
        return self._read_u32("status_seq")

    def mirror_info(self, seq: int, check: bool = False) -> StepInfo:
        """StepInfo of the ``seq``-th closed step (1-based) from the host mirror -- valid once that step's completion event
        has been waited for; no device read.  Falls back to a device read if the slot was already overwritten (the host
        fell more than three steps behind) or the mirror is not in use."""
        m = self._mirror_np[8 * ((seq - 1) & 3):8 * ((seq - 1) & 3) + 8]
        if int(m[7]) != seq:
            return self.last_step_info(check=check)
        st = dict(zip(self._STATUS, (int(x) for x in m[:7])))
        if check:
            self.check_error(st)
        late = st["last_late"]
        return StepInfo(global_step=st["epoch"], accepted=not late, mask=st["last_mask"], count=st["last_count"],
                        stale=bool(late))

    def check_error(self, status: Optional[Dict[str, int]] = None) -> None:
        e = (status or self.read_status())["error"]
        if e:
            if self.debug_sync:
                import sys
                self.debug_dump(sys.stderr)
            raise RuntimeError("fused sync watchdog fired on rank %d: %s timeout (DMNIST_DEBUG_SYNC=1 / --debug_sync dumps "
                               "the control block)" % (self.ctx.rank, {1: "arrival", 2: "push-complete"}.get(e, str(e))))

    def debug_dump(self, out=None) -> str:
        """The accumulator / token-queue state of the reference's debug Print ops (…modified.py:230-234,383-387), here: every
        handshake word of this rank's control block -- which peers have arrived / finished for which step, the chief's
        arrival bitmap and commit ring, the local decision.  Printed when a watchdog fires under ``--debug_sync``."""
        n = self.ctx.world_size
        raw = self._ctrl_bytes.cpu().numpy()
        u32 = lambda off: int(raw[off:off + 4].view("<u4")[0])           # noqa: E731
        u64 = lambda off: int(raw[off:off + 8].view("<u8")[0])           # noqa: E731
        lines = ["[sync-debug rank %d/%d] epoch=%d error=%d accepted=%d dropped=%d last(mask=%#x count=%d late=%d) global_step=%d"
                 % (self.ctx.rank, n, u32(self._off["epoch"]), u32(self._off["error"]), u32(self._off["accepted_steps"]),
                    u32(self._off["dropped_steps"]), u32(self._off["last_mask"]), u32(self._off["last_count"]),
                    u32(self._off["last_late"]), u32(self._off["global_step"]))]
        for f in ("arrive", "done", "arrive_e", "done_e"):
            lines.append("  %-9s per peer (value = step+1): %s" % (f, [u32(self._off[f] + 128 * q) for q in range(n)]))
        lines.append("  decided: tag=%d mask=%#x late=%d target=%d   cta counters: %d / %d / %d"
                     % (u32(self._off["decided_tag"]), u32(self._off["decided_mask"]), u32(self._off["decided_late"]),
                        u32(self._off["decided_target"]), u32(self._off["cta_counter"]), u32(self._off["cta_counter_e"]),
                        u32(self._off["cta_counter2"])))
        ep = u32(self._off["epoch"])
        slots = sorted({(ep + d) % 64 for d in (-2, -1, 0, 1)})
        lines.append("  commit_local[slot]=(step+1, mask): %s"
                     % {sl: (u64(self._off["commit_local"] + 8 * sl) >> 32, hex(u64(self._off["commit_local"] + 8 * sl) & 0xffffffff))
                        for sl in slots})
        if self.ctx.rank == 0:
            lines.append("  chief bitmap[slot]: %s   commit[slot]: %s   last_in_mask: %s"
                         % ({sl: hex(u32(self._off["bitmap"] + 4 * sl)) for sl in slots},
                            {sl: (u64(self._off["commit"] + 8 * sl) >> 32, hex(u64(self._off["commit"] + 8 * sl) & 0xffffffff)) for sl in slots},
                            [u32(self._off["last_in_mask"] + 4 * q) for q in range(n)]))
        txt = "\n".join(lines)
        if out is not None:
            print(txt, file=out, flush=True)
        return txt

    def read_phases(self):
        """%globaltimer stamps of the last launch: start, decided, reduced, pushed, landed, end (ns, relative)."""
        t = self._ctrl_bytes[self._off["t_phase"]:self._off["t_phase"] + 48].view(torch.int64).cpu().tolist()
        return [x - t[0] for x in t]

    def read_phases_early(self):
        """Early-bucket kernel of the last step: start, arrived, reduced (CTA 0), all pushes out, all shards landed,
        applied (CTA 0) (ns, relative)."""
        t = self._ctrl_bytes[self._off["t_phase_e"]:self._off["t_phase_e"] + 48].view(torch.int64).cpu().tolist()
        return [x - t[0] for x in t]

    def read_timing(self, first_step: int, last_step: int):
        """(start_ns, arrive_ns) %globaltimer stamps of local steps [first, last] (cdf telemetry)."""
        ring = 1024
        ta = self._ctrl_bytes[self._off["t_arrive"]:self._off["t_arrive"] + 8 * ring].view(torch.int64).cpu()
        ts = self._ctrl_bytes[self._off["t_start"]:self._off["t_start"] + 8 * ring].view(torch.int64).cpu()
        return [(int(ts[s % ring]), int(ta[s % ring])) for s in range(first_step, last_step + 1)]

    # ---- launches -------------------------------------------------------------------------------
    def _state_args(self, rule, slots, multicast: bool):
        """C arguments of the update rule: code, the two state-arena pointer tables, their multicast views (only when the
        weights travel by multicast too), momentum, decay, epsilon."""
        rule = rule_or_sgd(rule)
        if len(slots) != rule.num_slots:
            raise ValueError("update rule %s keeps %d state arenas, got %d" % (rule.name, rule.num_slots, len(slots)))
        bufs = [self._by_ptr[t.data_ptr()] for t in slots] + [None, None]
        tables = [b.ptr_table() if b is not None else None for b in bufs[:2]]
        mc = [ctypes.c_void_p(b.multicast_ptr if (multicast and b is not None) else 0) for b in bufs[:2]]
        return [int(rule.code)] + tables + mc + [ctypes.c_float(x) for x in rule.hyper]

    def enqueue(self, params: torch.Tensor, grads: torch.Tensor, k: int, lr0: float, decay_rate: float = 1.0,
                decay_steps: int = 1, stream: Optional[torch.cuda.Stream] = None, rule=None, slots=(),
                divisor: float = 0.0) -> None:
        """``rule`` / ``slots``: update rule and its state arenas (symmetric, from :meth:`allocate`); ``divisor`` > 0 replaces
        the contributor count as the mean's divisor (stateful rules only)."""
        pb, gb = self._by_ptr[params.data_ptr()], self._by_ptr[grads.data_ptr()]
        mcg, mcp = self._mc_ptrs(pb, gb, slots)
        rc = self.lib.dm_fused_sync_sgd(
            self.ctrl.ptr_table(), pb.ptr_table(), gb.ptr_table(), self.ctx.rank, self.ctx.world_size, int(k),
            ctypes.c_longlong(params.numel()), ctypes.c_float(lr0), ctypes.c_float(decay_rate), int(decay_steps),
            ctypes.c_float(self.drop_keep), ctypes.c_uint(self.drop_seed), ctypes.c_double(self.timeout_ms),
            ctypes.c_void_p(0 if self.shadow is None else self.shadow.data_ptr()), int(self.ctas), stream_ptr(stream),
            mcg, mcp, *self._state_args(rule, slots, bool(mcp.value)), ctypes.c_float(divisor))
        check(rc, "dm_fused_sync_sgd")

    def _mc_ptrs(self, pb, gb, slots=()):
        on = self.use_nvls and pb.multicast_ptr and gb.multicast_ptr \
            and all(self._by_ptr[t.data_ptr()].multicast_ptr for t in slots)
        return ctypes.c_void_p(gb.multicast_ptr if on else 0), ctypes.c_void_p(pb.multicast_ptr if on else 0)

    def enqueue_bucket(self, params: torch.Tensor, grads: torch.Tensor, phase: int, begin: int, end: int,
                       early_begin: int, early_end: int, lr0: float, decay_rate: float = 1.0, decay_steps: int = 1,
                       ctas: int = 0, stream: Optional[torch.cuda.Stream] = None) -> None:
        """Bucketed aggregation (K == N, world_size > 1): ``phase`` 1 = early bucket ``[begin, end)`` (floats) on a few
        CTAs next to the remaining backward kernels, 2 = late bucket + completion of the step (csrc/fused_sync.cu)."""
        pb, gb = self._by_ptr[params.data_ptr()], self._by_ptr[grads.data_ptr()]
        rc = self.lib.dm_fused_sync_bucket(
            self.ctrl.ptr_table(), pb.ptr_table(), gb.ptr_table(), self.ctx.rank, self.ctx.world_size, int(phase),
            ctypes.c_longlong(begin), ctypes.c_longlong(end), ctypes.c_longlong(early_begin), ctypes.c_longlong(early_end),
            ctypes.c_float(lr0), ctypes.c_float(decay_rate), int(decay_steps), ctypes.c_double(self.timeout_ms),
            ctypes.c_void_p(0 if self.shadow is None else self.shadow.data_ptr()), int(ctas), stream_ptr(stream),
            *self._mc_ptrs(pb, gb))
        check(rc, "dm_fused_sync_bucket")

    def enqueue_bucket_v2(self, params: torch.Tensor, grads: torch.Tensor, g16, inbox, phase: int, fc1_begin: int,
                          fc1_end: int, lr0: float, decay_rate: float = 1.0, decay_steps: int = 1, ctas: int = 0,
                          stream: Optional[torch.cuda.Stream] = None, rule=None, slots=()) -> None:
        """Bucketed aggregation, bf16 wire (csrc/fused_bucket.cu).  ``phase`` 1: reduce the bf16 fc1 gradient buffer ``g16``
        in place over NVLink (NVLS or P2P) and apply the update rule to the local fp32 fc1 weights and state -- a side
        branch of the step graph; ``phase`` 2: push the small bucket into every replica's ``inbox``, sum in rank order,
        update, close the step.  Every rank updates its own state from the identical sums: state never crosses NVLink."""
        pb, gb = self._by_ptr[params.data_ptr()], self._by_ptr[grads.data_ptr()]
        on = self.use_nvls and self.ctx.world_size > 1
        mc_g16 = g16.multicast_ptr if on else 0
        mc_inbox = inbox.multicast_ptr if (on and inbox is not None) else 0
        rc = self.lib.dm_bucket_sync(
            self.ctrl.ptr_table(), pb.ptr_table(), gb.ptr_table(), g16.ptr_table(),
            inbox.ptr_table() if inbox is not None else None, self.ctx.rank, self.ctx.world_size, int(phase),
            ctypes.c_longlong(fc1_begin), ctypes.c_longlong(fc1_end), ctypes.c_longlong(params.numel()),
            ctypes.c_float(lr0), ctypes.c_float(decay_rate), int(decay_steps), ctypes.c_double(self.timeout_ms),
            ctypes.c_void_p(0 if self.shadow is None else self.shadow.data_ptr()), int(ctas), stream_ptr(stream),
            ctypes.c_void_p(mc_g16), ctypes.c_void_p(mc_inbox), int(self.late_ll), int(self.late_bf16),
            *[x for i, x in enumerate(self._state_args(rule, slots, False)) if i not in (3, 4)])
        check(rc, "dm_bucket_sync(phase %d)" % phase)

    # ---- device-side interval mode (mode C, csrc/fused_interval.cu) ----------------------------------------------------------
    def interval_arm(self, interval_ms: float) -> None:
        """Start the interval clock on this replica (reference ``start_interval_updates``): first tick due in ``interval_ms``."""
        self.barrier()                       # replicas start their clocks together (each uses its own %globaltimer afterwards)
        check(self.lib.dm_interval_arm(ctypes.c_void_p(self.ctrl.local_ptr), ctypes.c_double(interval_ms), stream_ptr()),
              "dm_interval_arm")
        torch.cuda.synchronize()
        self.barrier()

    def enqueue_interval_begin(self, params: torch.Tensor, stream: Optional[torch.cuda.Stream] = None) -> None:
        """Start of an interval-mode iteration: adopt weights a committer has pushed (step counter, bf16 shadow)."""
        check(self.lib.dm_interval_begin(ctypes.c_void_p(self.ctrl.local_ptr), ctypes.c_void_p(params.data_ptr()),
                                         ctypes.c_void_p(0 if self.shadow is None else self.shadow.data_ptr()),
                                         ctypes.c_longlong(params.numel()), stream_ptr(stream)), "dm_interval_begin")

    def enqueue_interval_end(self, params: torch.Tensor, grads: torch.Tensor, acc: torch.Tensor, lr0: float,
                             decay_rate: float = 1.0, decay_steps: int = 1,
                             stream: Optional[torch.cuda.Stream] = None, rule=None, slots=()) -> None:
        """End of an interval-mode iteration: accumulate the gradient locally; after the tick's deadline try to commit the
        tick (mean of whatever every replica has accumulated) -- never blocks on another replica's progress.  The committer
        pushes the new weights and the rule's state into every replica."""
        pb, gb, ab = self._by_ptr[params.data_ptr()], self._by_ptr[grads.data_ptr()], self._by_ptr[acc.data_ptr()]
        on = self.use_nvls and pb.multicast_ptr and all(self._by_ptr[t.data_ptr()].multicast_ptr for t in slots)
        mc = pb.multicast_ptr if on else 0
        check(self.lib.dm_interval_end(self.ctrl.ptr_table(), pb.ptr_table(), gb.ptr_table(), ab.ptr_table(), self.ctx.rank,
                                       self.ctx.world_size, ctypes.c_longlong(params.numel()), ctypes.c_float(lr0),
                                       ctypes.c_float(decay_rate), int(decay_steps), ctypes.c_double(self.timeout_ms),
                                       int(self.ctas), stream_ptr(stream), ctypes.c_void_p(mc),
                                       *self._state_args(rule, slots, bool(mc))), "dm_interval_end")

    @property
    def nvls_active(self) -> bool:
        return self.use_nvls and bool(self._buffers) and all(b.multicast_ptr for b in self._buffers[:2])

    def enqueue_straggler_delay(self, prob: float, usec: float, seed: int = 12345,
                                stream: Optional[torch.cuda.Stream] = None) -> None:
        check(self.lib.dm_straggler_delay(ctypes.c_void_p(self.ctrl.local_ptr), ctypes.c_float(prob),
                                          ctypes.c_uint(int(usec)), ctypes.c_uint(seed), stream_ptr(stream)),
              "dm_straggler_delay")

    def device_barrier(self, stream: Optional[torch.cuda.Stream] = None) -> None:
        """Stream-ordered barrier over NVLink flags (csrc/fused_sync.cu): every replica's stream passes it within a flag hop of
        the last replica reaching it -- aligns the replicas far tighter than a host-side barrier can."""
        if self.ctx.world_size > 1:
            check(self.lib.dm_device_barrier(self.ctrl.ptr_table(), self.ctx.rank, self.ctx.world_size,
                                             ctypes.c_double(self.timeout_ms), stream_ptr(stream)), "dm_device_barrier")

    def enqueue_stamp_arrive(self, stream: Optional[torch.cuda.Stream] = None) -> None:
        """cdf telemetry: "my gradient is complete" on the compute chain, before it joins the exchange branch."""
        check(self.lib.dm_stamp_arrive(ctypes.c_void_p(self.ctrl.local_ptr), stream_ptr(stream)), "dm_stamp_arrive")

    def enqueue_stamp_start(self, stream: Optional[torch.cuda.Stream] = None) -> None:
        check(self.lib.dm_stamp_start(ctypes.c_void_p(self.ctrl.local_ptr), stream_ptr(stream)), "dm_stamp_start")

    def drop_connect_(self, grads: torch.Tensor, keep_prob: float, step: int) -> None:
        # Applied inside the fused kernel's load stage (per contributor); just arm it.
        self.drop_keep = float(keep_prob)
        self.drop_seed = 0x2545F491

    def last_step_info(self, check: bool = False) -> StepInfo:
        st = self.read_status()
        if check:
            self.check_error(st)
        late = st["last_late"]
        return StepInfo(global_step=st["epoch"], accepted=not late, mask=st["last_mask"], count=st["last_count"],
                        stale=bool(late))

    def sync_step(self, params, grads, lr, local_step, k, delay_s: float = 0.0, rule=None, slots=()) -> StepInfo:
        if delay_s > 0:
            self.enqueue_straggler_delay(1.0, delay_s * 1e6)
        self.enqueue(params, grads, k, lr0=float(lr), rule=rule, slots=slots)
        return self.last_step_info(check=True)   # one device -> host read (synchronises)

    def interval_tick(self, params, acc, count, lr, tick, rule=None, slots=()) -> StepInfo:
        """Mode C tick: every rank joins; ranks with an empty accumulator contribute zeros and the
        divisor is the total number of accumulated gradients (mean of whatever arrived)."""
        counts = self.all_gather_object(int(count))
        total = sum(counts)
        mask = sum(1 << i for i, c in enumerate(counts) if c > 0)
        if total == 0:
            return StepInfo(self.device_epoch, False, 0, 0, applied=False)
        if rule_or_sgd(rule).num_slots == 0:
            # lr/total instead of lr/popcount: fold the ratio into lr0 (kernel divides by N contributors)
            self.enqueue(params, acc, self.ctx.world_size, lr0=float(lr) * self.ctx.world_size / total)
        else:
            # with state the mean has to be formed before the rule sees it: pass the divisor itself
            self.enqueue(params, acc, self.ctx.world_size, lr0=float(lr), rule=rule, slots=slots, divisor=float(total))
        info = self.last_step_info()
        self.check_error()
        return StepInfo(info.global_step, count > 0, mask, total)

    def close(self) -> None:
        torch.cuda.synchronize()
        self.barrier()
        for b in self._buffers + [self.ctrl]:
            b.close()
