"""sm_100a compute engine: the reference convnet's training step as 11 hand-written kernels
replayed from one CUDA graph.

Step = (reference src/distributed_train.py:332 ``sess.run(apply_gradients_op)``)::

    memset(small grads, loss)                              2 memset nodes
    conv1_fwd        conv+bias+ReLU+pool (SIMT, K=25)       csrc/lenet_simt.cu
    conv2_fwd        tcgen05 implicit GEMM + bias/ReLU/pool csrc/conv2_tc.cu
    fc1_fwd          tcgen05 GEMM, split-K into fp32        csrc/gemm_tc.cu
    fc2_fwd_bwd      bias+ReLU+dropout, fc2, softmax-CE,
                     accuracy, dlogits, d(fc1)              csrc/lenet_simt.cu
    fc2_wgrad        fc2 weight/bias + fc1 bias gradients   (side branch)
    fc1_wgrad        tcgen05 GEMM (MN-major x MN-major) -> gradient arena
    fc1_dgrad        tcgen05 GEMM -> bf16
    unpool2          maxpool2/ReLU2 backward + conv2 bias grad
    conv2_wgrad      tcgen05, K = pixels, fp32 atomics -> gradient arena
    conv2_dgrad      tcgen05
    conv1_wgrad      maxpool1/ReLU1 backward + conv1 weight/bias grad
    fused_sync_sgd   arrival -> mask -> NVLink reduce -> 1/count -> SGD -> push -> bf16 shadow

Weights live in TF layouts in one flat fp32 arena (symmetric memory); the tensor-core
kernels read the bf16 shadow arena the fused kernel refreshes.  Nothing on this path
calls cuDNN, cuBLAS or NCCL.
"""
from __future__ import annotations

import ctypes
import os
from typing import Optional, Tuple

import numpy as np
import torch

from .engine import ComputeEngine
from .models import get_model
from .models.lenet import dropout_seed_mix
from .ops import gemm as G
from .ops.lib import check, load, ptr, stream_ptr
from .optim import rule_or_sgd
from .parallel.backends import StepInfo
from .parallel.fused import FusedBackend


class _RunnerEvent:
    """Completion of a step launched through the native runner: ``synchronize()`` like a ``torch.cuda.Event``."""

    def __init__(self, lib, runner, slot: int):
        self.lib, self.runner, self.slot = lib, runner, slot

    def synchronize(self) -> None:
        rc = self.lib.dm_runner_wait(self.runner, self.slot)
        if rc != 0:
            raise RuntimeError("dm_runner_wait failed: CUDA error %d" % rc)

    def query(self) -> bool:
        return self.lib.dm_runner_query(self.runner, self.slot) == 1


class CudaLeNetEngine(ComputeEngine):
    def __init__(self, batch_size: int, backend: FusedBackend, seed: int = 66478, rank: int = 0,
                 keep_prob: float = 0.5, use_graph: bool = True):
        self.lib = load()
        self.backend = backend
        self.device = backend.ctx.device
        self.spec, _ = get_model("lenet")
        self.batch_size = B = batch_size
        self.seed, self.rank, self.keep_prob = seed, rank, keep_prob
        self.use_graph = use_graph
        dev = self.device
        self.params = backend.allocate(self.spec.arena_numel)
        self.params.copy_(self.spec.init_flat(seed).to(dev))
        self.grads = backend.allocate(self.spec.arena_numel)
        self.shadow = backend.attach_shadow(self.params)
        self.p = self.spec.views(self.params)
        self.g = self.spec.views(self.grads)
        self.pb = self.spec.views(self.shadow)
        bf, u8, f32 = torch.bfloat16, torch.uint8, torch.float32
        # two input slots so the H2D copy of step i+1 overlaps the compute of step i
        # (images and labels of a slot share one allocation so a packed host batch moves with ONE host->device copy)
        self._in_bytes = B * 784 * 4 + B * 8
        self.in_dev = [torch.zeros(self._in_bytes, dtype=u8, device=dev) for _ in range(2)]
        self.images = [t[:B * 784 * 4].view(f32).view(B, 28, 28) for t in self.in_dev]
        self.labels = [t[B * 784 * 4:].view(torch.int64) for t in self.in_dev]
        self.h_images = [torch.zeros(B, 28, 28, dtype=f32).pin_memory() for _ in range(2)]
        self.h_labels = [torch.zeros(B, dtype=torch.int64).pin_memory() for _ in range(2)]
        self.a1 = torch.zeros(B, 14, 14, 32, dtype=bf, device=dev)
        self.code1 = torch.zeros(B, 14, 14, 32, dtype=u8, device=dev)
        self.a2 = torch.zeros(B, 3136, dtype=bf, device=dev)
        self.code2 = torch.zeros(B, 3136, dtype=u8, device=dev)
        self.fc1_splits = 7                                         # 49 k-blocks of 64 -> 7 per CTA
        self.h_part = torch.zeros(self.fc1_splits, B, 512, dtype=f32, device=dev)   # fc1 split-K partial sums
        self.dh = torch.zeros(B, 512, dtype=bf, device=dev)
        self.h_act = torch.zeros(B, 512, dtype=f32, device=dev)      # post ReLU/dropout fc1 activations (fc2_wgrad operand)
        self.dlogits = torch.zeros(B, 12, dtype=f32, device=dev)     # d loss / d logits, 48-byte rows
        self.dxfc = torch.zeros(B, 3136, dtype=bf, device=dev)
        self.dy2 = torch.zeros(B, 14, 14, 64, dtype=bf, device=dev)
        self.dx1 = torch.zeros(B, 14, 14, 32, dtype=bf, device=dev)
        self.d_loss_acc = torch.zeros(2, dtype=f32, device=dev)
        self.h_loss_bufs = [torch.zeros(2, dtype=f32).pin_memory() for _ in range(2)]
        self.h_loss_acc = self.h_loss_bufs[0]
        self._loss_reads = 0
        self._slot = 0            # input slot the next step computes from
        self._loaded = 0
        self._h2d_bytes = B * 784 * 4 + B * 8
        self.copy_stream = torch.cuda.Stream(device=dev)
        # the data-gradient chain is the critical path: it is captured on a high-priority stream, the weight-gradient
        # side branches on low-priority ones, so the block scheduler serves the chain first whenever both have CTAs pending
        lo, hi = (0, -1)
        self._side = [torch.cuda.Stream(device=dev, priority=lo) for _ in range(4)]
        self._main_priority = hi if os.environ.get("DMNIST_PRIO", "1") != "0" else lo
        self._wgrad_late = os.environ.get("DMNIST_WGRAD_LATE", "1") != "0"
        self._branches = os.environ.get("DMNIST_BRANCHES", "1") != "0"
        self._fuse_unpool = os.environ.get("DMNIST_FUSE_UNPOOL", "1") != "0"
        self._conv1_tc = os.environ.get("DMNIST_CONV1_TC", "1") != "0"    # conv1 fwd / wgrad on tcgen05 (csrc/conv1_tc.cu)
        self._copy_done = [torch.cuda.Event() for _ in range(2)]
        self._slot_free = [torch.cuda.Event() for _ in range(2)]
        self._graphs = [None, None]
        self._opt_args: Optional[dict] = None
        self._straggler = None
        self._stamp = False
        p_fc1 = self.spec.param("fc1_weights")
        self._zero_ranges = [(0, p_fc1.offset), (p_fc1.offset + p_fc1.numel, self.spec.arena_numel)]
        self._seed_mix0 = dropout_seed_mix(seed, 0, rank)
        # early bucket = fc1_weights (96.5 % of the bytes, final as soon as fc1_wgrad is done); everything else is late
        self._bucket_split = p_fc1.offset
        self._bucket_early = (p_fc1.offset, p_fc1.offset + p_fc1.numel)
        self._bucketed = False
        self._bucket_v2 = False       # bf16-wire early bucket + pushed late bucket (csrc/fused_bucket.cu)
        self._g16 = self._g16_view = self._inbox = None
        self._epoch_ptr = ctypes.c_void_p(backend.ctrl.local_ptr + backend._off["epoch"])
        self.launches_per_step = 0

    # ---- inputs ------------------------------------------------------------------------------
    def _leave_native_runner(self) -> None:
        """The torch-dispatched path takes over again: its events know nothing about steps the native runner launched."""
        if getattr(self, "_runner", None) is not None:
            torch.cuda.synchronize()
            self.lib.dm_runner_destroy(self._runner)
            self._runner = None

    def load_batch(self, images, labels) -> None:
        """Pinned host staging -> device slot, on the copy stream (overlaps the previous step)."""
        self._leave_native_runner()
        s = self._loaded & 1
        if isinstance(images, torch.Tensor) and images.dtype == torch.float32 and labels.dtype == torch.int64 \
                and ((images.is_pinned() and labels.is_pinned()) or (images.is_cuda and labels.is_cuda)):
            # already page-locked (or device-resident): DMA straight from the caller's buffers (they must stay untouched
            # until the copy has run, i.e. until the step that consumes them has been enqueued twice)
            hi, hl = images.view(self.images[0].shape), labels
        else:
            hi, hl = self.h_images[s], self.h_labels[s]
            if isinstance(images, np.ndarray):
                hi.copy_(torch.from_numpy(images).view(hi.shape))
                hl.copy_(torch.from_numpy(labels))
            else:
                hi.copy_(images.reshape(hi.shape))
                hl.copy_(labels)
        with torch.cuda.stream(self.copy_stream):
            self.copy_stream.wait_event(self._slot_free[s])   # the step that last read this slot is done
            self.images[s].copy_(hi, non_blocking=True)
            self.labels[s].copy_(hl, non_blocking=True)
            self._copy_done[s].record(self.copy_stream)
        self._slot = s
        self._loaded += 1

    def pack_batch(self, images, labels, pin: bool = True) -> torch.Tensor:
        """One contiguous (page-locked) host buffer holding a batch in the device slot's layout: fp32 images
        ``[B,28,28]`` followed by int64 labels ``[B]``.  Input pipelines that fill such buffers hand each batch to
        :meth:`load_packed`, which is a single DMA."""
        B = self.batch_size
        buf = torch.empty(self._in_bytes, dtype=torch.uint8)
        if pin:
            buf = buf.pin_memory()
        img = torch.as_tensor(images, dtype=torch.float32).reshape(B * 784)
        buf[:B * 784 * 4].view(torch.float32).copy_(img)
        buf[B * 784 * 4:].view(torch.int64).copy_(torch.as_tensor(labels, dtype=torch.int64).reshape(B))
        return buf

    def load_packed(self, packed: torch.Tensor) -> None:
        """Packed batch (see :meth:`pack_batch`; pinned host or device memory) -> device slot with one copy on the copy
        stream.  The buffer must stay untouched until the step after the next one has been enqueued."""
        self._leave_native_runner()
        s = self._loaded & 1
        with torch.cuda.stream(self.copy_stream):
            self.copy_stream.wait_event(self._slot_free[s])
            self.in_dev[s].copy_(packed, non_blocking=True)
            self._copy_done[s].record(self.copy_stream)
        self._slot = s
        self._loaded += 1

    def h2d_bytes_per_step(self) -> int:
        return self._h2d_bytes

    # ---- native step executor (csrc/step_runner.cu) ----------------------------------------------------------------------
    def step_packed(self, packed: torch.Tensor):
        """One whole training step from a packed batch (see :meth:`pack_batch`; pinned host or device memory): input DMA,
        event chaining and the graph launch happen in ONE native call once both slot graphs exist (``DMNIST_NATIVE_RUNNER=0``
        keeps the torch-dispatched path).  Returns ``(waitable, loss buffer, seq)`` like :meth:`read_result_async`."""
        r = getattr(self, "_runner", None)
        if r is None and self.use_graph and self._opt_args is not None and os.environ.get("DMNIST_NATIVE_RUNNER", "1") != "0" \
                and all(g is not None and g[1] for g in self._graphs):
            r = self._make_runner()
        if r is None:
            self.load_packed(packed)
            self.train_step()
            return self.read_result_async()
        s = int(self.lib.dm_runner_step(r, ctypes.c_void_p(packed.data_ptr())))
        if s < 0:
            raise RuntimeError("dm_runner_step failed: CUDA error %d" % -s)
        self._keep_alive[s] = packed                     # the DMA reads it asynchronously
        self._slot = s
        self._loaded += 1
        self._steps_launched += 1
        return _RunnerEvent(self.lib, r, s), self.h_loss_bufs[s], self._seq0 + self._steps_launched

    def _make_runner(self):
        torch.cuda.synchronize()                         # hand-over point: nothing of the torch-dispatched path is in flight
        lib = self.lib
        lib.dm_runner_create.restype = ctypes.c_void_p
        cur = torch.cuda.current_stream()
        r = lib.dm_runner_create(ctypes.c_void_p(cur.cuda_stream), ctypes.c_void_p(self.copy_stream.cuda_stream),
                                 ctypes.c_void_p(self._graphs[0][0].raw_cuda_graph_exec()),
                                 ctypes.c_void_p(self._graphs[1][0].raw_cuda_graph_exec()),
                                 ctypes.c_void_p(self.in_dev[0].data_ptr()), ctypes.c_void_p(self.in_dev[1].data_ptr()),
                                 ctypes.c_ulonglong(self._in_bytes), int(self._loaded & 1))
        if not r:
            return None
        self._runner = ctypes.c_void_p(r)
        self._keep_alive = [None, None]
        return self._runner

    # ---- optimizer binding ------------------------------------------------------------------------
    def attach_optimizer(self, opt) -> None:
        """Bind the aggregation policy so the whole step (compute + fused sync) is one graph."""
        sched = opt.lr_schedule
        k = getattr(opt, "replicas_to_aggregate", opt.total_num_replicas)
        # update rule + its state arenas (symmetric, parameter-arena layout, NVLS-mapped when the fabric has multicast): the
        # optimizer owns them, every aggregation launch of the step reads and writes them
        rule = rule_or_sgd(getattr(opt, "update_rule", None))
        slots = opt.ensure_slots(self.spec.arena_numel) if rule.num_slots else []
        self.slots = slots
        self._opt_args = dict(k=int(k), lr0=float(sched.initial_learning_rate), decay_rate=float(sched.decay_rate),
                              decay_steps=int(sched.decay_steps), rule=rule, slots=slots)
        if getattr(opt, "drop_connect_probability", None) is not None:
            self.backend.drop_connect_(self.grads, opt.drop_connect_probability, 0)
        self._straggler = getattr(opt, "_straggler", None)
        self._stamp = getattr(opt, "mode", "") == "cdf"
        self._graphs = [None, None]
        self._runner = None                  # graphs are re-captured: the native runner is rebuilt on demand
        # mode C on the device (csrc/fused_interval.cu): every iteration adds its gradient to a symmetric accumulator; ticks
        # are committed by whichever replica first passes the %globaltimer deadline
        self._interval = getattr(opt, "mode", "") == "interval"
        if self._interval and getattr(self, "_acc", None) is None:
            self._acc = self.backend.allocate(self.spec.arena_numel)
        # Bucketed aggregation (csrc/fused_sync.cu): full participation on 2/4/8 replicas.  fc1's weight gradient (96.5 % of
        # the bytes) is exchanged by small co-resident CTAs NEXT TO conv2 dgrad/wgrad + conv1 wgrad; the rest goes one-shot.
        #   DMNIST_BUCKET=2 (default): csrc/fused_bucket.cu -- fc1's gradient leaves the GEMM epilogue as bf16, is reduced in
        #     place over NVLink (in-switch fp32 accumulation) and applied to the local fp32 master weights under the backward
        #     pass; the small bucket is pushed into every replica's inbox.  Also used on ONE replica (no exchange, the fc1
        #     update still leaves the critical path).   =1: round-1 fp32 two-shot / one-shot kernels.   =0: single kernel.
        n = self.backend.ctx.world_size
        mode = os.environ.get("DMNIST_BUCKET", "2")
        can = (hasattr(self, "_bucket_split") and int(k) == n and self._branches and self.backend.drop_keep <= 0.0
               and getattr(opt, "mode", "") != "interval")
        self._bucket_v2 = can and mode == "2" and n in (1, 2, 4, 8)
        # the round-1 bucket kernels apply SGD only: a stateful rule takes the single kernel there
        self._bucketed = can and ((mode == "1" and n in (2, 4, 8) and rule.num_slots == 0) or self._bucket_v2)
        if self._bucket_v2 and self._g16 is None:
            e0, e1 = self._bucket_early
            assert e0 % 8 == 0 and (e1 - e0) % 8 == 0, "fc1 weights must start on a 32-byte boundary of the arena"
            self._g16 = self.backend.allocate_buffer((e1 - e0) * 2)
            self._g16_view = self._g16.view(torch.bfloat16, 0, e1 - e0).view(*getattr(self, "_g16_shape", (3136, 512)))
            n_late = self.spec.arena_numel - (e1 - e0)
            self._inbox = self.backend.allocate_buffer(2 * n * n_late * 8) if n > 1 else None   # LL lines: 8 bytes per float
        # early-bucket grid: the CTAs share SMs with the tensor-core kernels of the backward pass and every one of them fences
        # at system scope once; measured at N = 4 (profiles/r2/bench_call12_4gpu.txt): 296 CTAs 90.8, 148 CTAs 85.8, 74 CTAs
        # 82.5 us/step -- half the SMs carry the exchange, the kernel still ends before the backward pass does
        self._early_ctas = int(os.environ.get("DMNIST_EARLY_CTAS", "0")) or (74 if n > 1 else 148)
        torch.cuda.synchronize()
        self._seq0 = self.backend.status_seq       # steps closed on this control block before the engine's first one
        self._steps_launched = 0
        self.lib.dm_set_max_ctas(int(os.environ.get("DMNIST_MAX_CTAS", "148")))

    def params_updated(self) -> None:
        """Parameters were written from the host (init / restore): refresh the bf16 shadow."""
        self.backend.refresh_shadow(self.params)

    # ---- kernel sequence ------------------------------------------------------------------------------
    def _launch_forward(self, images: torch.Tensor, labels: torch.Tensor, B: int, train: bool,
                        logits_out: Optional[torch.Tensor] = None) -> int:
        lib, sp, p, pb = self.lib, stream_ptr(), self.p, self.pb
        conv1_fwd = lib.dm_conv1_fwd_tc if self._conv1_tc else lib.dm_conv1_fwd
        check(conv1_fwd(ptr(images), ptr(p["conv1_weights"]), ptr(p["conv1_biases"]), ptr(self.a1),
                        ptr(self.code1), B, *self._zero_args(train), sp), "conv1_fwd")
        check(lib.dm_conv2_fwd(ptr(self.a1), ptr(pb["conv2_weights"]), ptr(p["conv2_biases"]), ptr(self.a2),
                               ptr(self.code2), B, sp), "conv2_fwd")
        # fc1: a2[B,3136] (K-major) * W1[3136,512] (MN-major), split-K: 7 partial tiles stored side by side
        # (no atomics, nothing to zero); fc2_fwd_bwd sums them while applying bias + ReLU + dropout
        stride = self.h_part.stride(0)
        G.gemm_bf16_raw(self.a2, pb["fc1_weights"], self.h_part, B, 512, 3136, 3136, 512, 512, False, True,
                        G.EPI_STORE_F32, splits=self.fc1_splits, bn=64, split_stride=stride)
        check(lib.dm_fc2_fwd_bwd(ptr(self.h_part), ctypes.c_longlong(stride), self.fc1_splits, ptr(p["fc1_biases"]),
                                 ptr(p["fc2_weights"]), ptr(p["fc2_biases"]), ptr(labels), ptr(self.dh), ptr(self.h_act),
                                 ptr(self.dlogits), ptr(self.d_loss_acc), ptr(logits_out), B, int(train),
                                 ctypes.c_uint(self._seed_mix0), self._epoch_ptr if train else ctypes.c_void_p(0),
                                 ctypes.c_float(self.keep_prob), sp), "fc2_fwd_bwd")
        return 4

    def _launch_backward(self, images: torch.Tensor, B: int, early_sync: bool = False) -> int:
        """Backward as a small DAG: the weight-gradient kernels have no consumer before the aggregation, so they run
        on low-priority side streams (captured as parallel graph branches) next to the data-gradient chain
        fc1_dgrad(+unpool) -> conv2_dgrad -> conv1_wgrad.  ``early_sync``: bucketed aggregation -- the early-bucket
        kernel joins the fc1_wgrad branch and the small fc gradients get a branch of their own."""
        lib, g, pb = self.lib, self.g, self.pb
        main = torch.cuda.current_stream()
        branch = self._branches
        if branch:
            fork1 = torch.cuda.Event()
            fork1.record(main)
            self._side[0].wait_event(fork1)
            # (loss, accuracy) are final after fc2_fwd_bwd: their copy into the slot's page-locked host buffer is a branch of
            # the step (a memcpy node of the graph) that runs under the backward pass -- reading the result costs the host
            # no extra call, only a wait on the step's completion event
            # (its own branch, joined only at the very end of the step: a memcpy node in front of the aggregation kernel
            # would cost that kernel its programmatic launch edge)
            self._side[3].wait_event(fork1)
            with torch.cuda.stream(self._side[3]):
                self.h_loss_bufs[self._slot].copy_(self.d_loss_acc, non_blocking=True)
                self._join_loss = torch.cuda.Event()
                self._join_loss.record(self._side[3])
        else:
            self.h_loss_bufs[self._slot].copy_(self.d_loss_acc, non_blocking=True)
        sp = stream_ptr()
        # fc1 dgrad: dxfc[B,3136] = dh[B,512] (K-major) * W1[3136,512] (rows = in, K = out contiguous)
        if self._fuse_unpool:
            # ... with maxpool2/ReLU2 backward and the conv2 bias gradient in the GEMM epilogue (no [B,3136] intermediate)
            check(lib.dm_fc1_dgrad_unpool(ptr(self.dh), ptr(pb["fc1_weights"]), ptr(self.code2), ptr(self.dy2),
                                          ptr(g["conv2_biases"]), B, sp), "fc1_dgrad_unpool")
        else:
            G.gemm_bf16_raw(self.dh, pb["fc1_weights"], self.dxfc, B, 3136, 512, 512, 512, 3136, False, False,
                            G.EPI_STORE_BF16, bn=64)
            check(lib.dm_unpool2(ptr(self.dxfc), ptr(self.code2), ptr(self.dy2), ptr(g["conv2_biases"]), B, sp), "unpool2")
        # (the side branch is issued AFTER the chain's kernel: both become ready together and the first one dispatched takes
        #  the SMs -- the data-gradient GEMM must be that one)
        with torch.cuda.stream(self._side[0] if branch else main):
            # fc1 wgrad: dW1[3136,512] = a2^T (A MN-major) * dh (B MN-major), K = batch; straight into the arena
            if early_sync and self._bucket_v2:
                # ... as bf16 into the symmetric wire buffer: half the epilogue stores, half the NVLink bytes
                G.gemm_bf16_raw(self.a2, self.dh, self._g16_view, 3136, 512, B, 3136, 512, 512, True, True,
                                G.EPI_STORE_BF16, bn=128)
            else:
                G.gemm_bf16_raw(self.a2, self.dh, g["fc1_weights"], 3136, 512, B, 3136, 512, 512, True, True,
                                G.EPI_STORE_F32, bn=128)
            if not early_sync:
                # fc2 weight/bias + fc1 bias gradients: only the aggregation kernel consumes them
                check(lib.dm_fc2_wgrad(ptr(self.h_act), ptr(self.dlogits), ptr(self.dh), ptr(g["fc2_weights"]),
                                       ptr(g["fc2_biases"]), ptr(g["fc1_biases"]), B, stream_ptr()), "fc2_wgrad")
            if branch and not early_sync:
                join1 = torch.cuda.Event()
                join1.record(self._side[0])
        if early_sync:
            # early bucket (fc1 weights): final once fc1_wgrad is done; the kernel also rewrites my shard of the fc1 bf16
            # shadow, which fc1_dgrad (launched above on the main stream) still reads -> ordered after it
            ev_du = torch.cuda.Event()
            ev_du.record(main)
            with torch.cuda.stream(self._side[0]):
                self._side[0].wait_event(ev_du)
                if self._straggler is not None and not getattr(self, "_delay_in_chain", False):
                    self.backend.enqueue_straggler_delay(self._straggler.prob, self._straggler.usec, stream=self._side[0])
                oa = self._opt_args
                e0, e1 = self._bucket_early
                if self._bucket_v2:
                    self.backend.enqueue_bucket_v2(self.params, self.grads, self._g16, self._inbox, 1, e0, e1, oa["lr0"],
                                                   oa["decay_rate"], oa["decay_steps"], ctas=self._early_ctas,
                                                   stream=self._side[0], rule=oa["rule"], slots=oa["slots"])
                else:
                    self.backend.enqueue_bucket(self.params, self.grads, 1, e0, e1, e0, e1, oa["lr0"], oa["decay_rate"],
                                                oa["decay_steps"], ctas=self._early_ctas, stream=self._side[0])
                join1 = torch.cuda.Event()
                join1.record(self._side[0])
            # the small fc gradients (fc2 weights/biases, fc1 biases) belong to the late bucket: their own branch
            self._side[2].wait_event(fork1)
            with torch.cuda.stream(self._side[2]):
                check(lib.dm_fc2_wgrad(ptr(self.h_act), ptr(self.dlogits), ptr(self.dh), ptr(g["fc2_weights"]),
                                       ptr(g["fc2_biases"]), ptr(g["fc1_biases"]), B, stream_ptr()), "fc2_wgrad")
                join3 = torch.cuda.Event()
                join3.record(self._side[2])
        late = branch and self._wgrad_late
        if late:
            # conv2 dgrad and wgrad each fill the machine (1 CTA/SM, ~200 KB smem): side by side they only slow the chain
            # down.  wgrad is forked AFTER dgrad instead and shares the SMs with conv1_wgrad (LDS/FMA-bound, 37 KB/CTA).
            check(lib.dm_conv2_dgrad(ptr(self.dy2), ptr(pb["conv2_weights"]), ptr(self.dx1), B, sp), "conv2_dgrad")
        if branch:
            fork2 = torch.cuda.Event()
            fork2.record(main)
            self._side[1].wait_event(fork2)
        with torch.cuda.stream(self._side[1] if branch else main):
            check(lib.dm_conv2_wgrad(ptr(self.a1), ptr(self.dy2), ptr(g["conv2_weights"]), B, stream_ptr()), "conv2_wgrad")
            if branch:
                join2 = torch.cuda.Event()
                join2.record(self._side[1])
        if not late:
            check(lib.dm_conv2_dgrad(ptr(self.dy2), ptr(pb["conv2_weights"]), ptr(self.dx1), B, sp), "conv2_dgrad")
        conv1_wgrad = lib.dm_conv1_wgrad_tc if self._conv1_tc else lib.dm_conv1_wgrad
        check(conv1_wgrad(ptr(images), ptr(self.dx1), ptr(self.code1), ptr(g["conv1_weights"]),
                          ptr(g["conv1_biases"]), B, sp), "conv1_wgrad")
        if branch:
            main.wait_event(join2)
            if self._stamp and early_sync:
                # every backward kernel of THIS replica is done (conv1_wgrad on the chain, conv2_wgrad joined): stamp it before
                # waiting for the exchange branch, which contains the all-to-all with the other replicas
                main.wait_event(join3)
                self.backend.enqueue_stamp_arrive()
            main.wait_event(join1)
            if early_sync:
                main.wait_event(join3)
        return 6 if self._fuse_unpool else 7

    def _zero_args(self, train: bool):
        """Regions conv1_fwd clears at the start of a training step (atomically accumulated gradients + loss)."""
        if not train:
            return (ctypes.c_void_p(0), 0, ctypes.c_void_p(0), 0, ptr(self.d_loss_acc), 2)
        base = self.grads.data_ptr()
        (a0, b0), (a1, b1) = self._zero_ranges
        return (ctypes.c_void_p(base + 4 * a0), b0 - a0, ctypes.c_void_p(base + 4 * a1), b1 - a1,
                ptr(self.d_loss_acc), 2)

    def _launch_zero(self) -> int:
        return 0    # folded into conv1_fwd

    def time_kernels(self, iters: int = 20) -> dict:
        """Average device time of every kernel of the step, measured in place with CUDA events between
        eager launches (caches warm, as in the replayed graph; includes the launch gap)."""
        names = ["memsets", "conv1_fwd", "conv2_fwd", "fc1_fwd", "fc2_fwd_bwd", "fc1_wgrad", "fc2_wgrad", "fc1_dgrad", "unpool2",
                 "conv2_wgrad", "conv2_dgrad", "conv1_wgrad", "fused_sync_sgd"]
        tot = {n: 0.0 for n in names}
        B, s = self.batch_size, self._slot
        img, lbl = self.images[s], self.labels[s]
        lib, sp, g, p, pb = self.lib, stream_ptr(), self.g, self.p, self.pb

        def seq():
            yield "memsets", lambda: self._launch_zero()
            fw = []
            # forward / backward are issued kernel by kernel so an event can sit between any two
            yield "conv1_fwd", lambda: check((lib.dm_conv1_fwd_tc if self._conv1_tc else lib.dm_conv1_fwd)(ptr(img), ptr(p["conv1_weights"]), ptr(p["conv1_biases"]),
                                                              ptr(self.a1), ptr(self.code1), B, *self._zero_args(True), sp),
                                             "conv1_fwd")
            yield "conv2_fwd", lambda: check(lib.dm_conv2_fwd(ptr(self.a1), ptr(pb["conv2_weights"]), ptr(p["conv2_biases"]),
                                                              ptr(self.a2), ptr(self.code2), B, sp), "conv2_fwd")
            stride = self.h_part.stride(0)
            yield "fc1_fwd", lambda: G.gemm_bf16_raw(self.a2, pb["fc1_weights"], self.h_part, B, 512, 3136, 3136, 512, 512,
                                                     False, True, G.EPI_STORE_F32, splits=self.fc1_splits, bn=64,
                                                     split_stride=stride)
            yield "fc2_fwd_bwd", lambda: check(lib.dm_fc2_fwd_bwd(
                ptr(self.h_part), ctypes.c_longlong(stride), self.fc1_splits, ptr(p["fc1_biases"]), ptr(p["fc2_weights"]),
                ptr(p["fc2_biases"]), ptr(lbl), ptr(self.dh), ptr(self.h_act), ptr(self.dlogits), ptr(self.d_loss_acc),
                ctypes.c_void_p(0), B, 1, ctypes.c_uint(self._seed_mix0), self._epoch_ptr, ctypes.c_float(self.keep_prob), sp),
                "fc2_fwd_bwd")
            yield "fc1_wgrad", lambda: G.gemm_bf16_raw(self.a2, self.dh, g["fc1_weights"], 3136, 512, B, 3136, 512, 512,
                                                       True, True, G.EPI_STORE_F32, bn=128)
            yield "fc2_wgrad", lambda: check(lib.dm_fc2_wgrad(ptr(self.h_act), ptr(self.dlogits), ptr(self.dh),
                                                              ptr(g["fc2_weights"]), ptr(g["fc2_biases"]),
                                                              ptr(g["fc1_biases"]), B, sp), "fc2_wgrad")
            if self._fuse_unpool:
                yield "fc1_dgrad", lambda: check(lib.dm_fc1_dgrad_unpool(ptr(self.dh), ptr(pb["fc1_weights"]), ptr(self.code2),
                                                                         ptr(self.dy2), ptr(g["conv2_biases"]), B, sp),
                                                 "fc1_dgrad_unpool")
            else:
                yield "fc1_dgrad", lambda: G.gemm_bf16_raw(self.dh, pb["fc1_weights"], self.dxfc, B, 3136, 512, 512, 512, 3136,
                                                           False, False, G.EPI_STORE_BF16, bn=64)
                yield "unpool2", lambda: check(lib.dm_unpool2(ptr(self.dxfc), ptr(self.code2), ptr(self.dy2),
                                                              ptr(g["conv2_biases"]), B, sp), "unpool2")
            yield "conv2_wgrad", lambda: check(lib.dm_conv2_wgrad(ptr(self.a1), ptr(self.dy2), ptr(g["conv2_weights"]), B, sp),
                                               "conv2_wgrad")
            yield "conv2_dgrad", lambda: check(lib.dm_conv2_dgrad(ptr(self.dy2), ptr(pb["conv2_weights"]), ptr(self.dx1), B, sp),
                                               "conv2_dgrad")
            yield "conv1_wgrad", lambda: check((lib.dm_conv1_wgrad_tc if self._conv1_tc else lib.dm_conv1_wgrad)(ptr(img), ptr(self.dx1), ptr(self.code1),
                                                                  ptr(g["conv1_weights"]), ptr(g["conv1_biases"]), B, sp),
                                               "conv1_wgrad")
            yield "fused_sync_sgd", lambda: self.backend.enqueue(self.params, self.grads, **self._opt_args)

        for it in range(iters + 3):
            evs = [torch.cuda.Event(enable_timing=True)]
            evs[0].record()
            order = []
            for name, fn in seq():
                fn()
                e = torch.cuda.Event(enable_timing=True)
                e.record()
                evs.append(e)
                order.append(name)
            torch.cuda.synchronize()
            if self.backend.ctx.world_size > 1:
                self.backend.barrier()
            if it >= 3:
                for i, name in enumerate(order):
                    tot[name] += evs[i].elapsed_time(evs[i + 1]) * 1e3 / iters
        return tot

    def _launch_step(self, slot: int, with_sync: bool) -> None:
        n = 0
        interval = with_sync and getattr(self, "_interval", False)
        bucketed = with_sync and self._bucketed and not interval
        self._delay_in_chain = False
        if self._stamp:
            self.backend.enqueue_stamp_start()
            n += 1
            if bucketed and self._straggler is not None:
                # cdf telemetry: the injected delay is part of THIS replica's compute (start stamp .. gradient-complete stamp)
                self.backend.enqueue_straggler_delay(self._straggler.prob, self._straggler.usec)
                self._delay_in_chain = True
                n += 1
        if interval:
            self.backend.enqueue_interval_begin(self.params)
            n += 2
        n += self._launch_zero()
        n += self._launch_forward(self.images[slot], self.labels[slot], self.batch_size, True)
        n += self._launch_backward(self.images[slot], self.batch_size, early_sync=bucketed)
        if bucketed:
            oa = self._opt_args
            e0, e1 = self._bucket_early
            if self._bucket_v2:
                self.backend.enqueue_bucket_v2(self.params, self.grads, self._g16, self._inbox, 2, e0, e1, oa["lr0"],
                                               oa["decay_rate"], oa["decay_steps"], rule=oa["rule"], slots=oa["slots"])
            else:
                self.backend.enqueue_bucket(self.params, self.grads, 2, 0, self.spec.arena_numel, e0, e1,
                                            oa["lr0"], oa["decay_rate"], oa["decay_steps"])
            n += 2 + (1 if self._straggler is not None else 0)
        elif with_sync:
            if self._straggler is not None:
                self.backend.enqueue_straggler_delay(self._straggler.prob, self._straggler.usec)
                n += 1
            if interval:
                oa = self._opt_args
                self.backend.enqueue_interval_end(self.params, self.grads, self._acc, oa["lr0"], oa["decay_rate"], oa["decay_steps"],
                                                  rule=oa["rule"], slots=oa["slots"])
                n += 4
            else:
                self.backend.enqueue(self.params, self.grads, **self._opt_args)
                n += 1
        if self._branches:
            torch.cuda.current_stream().wait_event(self._join_loss)      # the loss read-back branch rejoins at the end of the step
        self.launches_per_step = n

    def _run(self, with_sync: bool) -> None:
        s = self._slot
        cur = torch.cuda.current_stream()
        cur.wait_event(self._copy_done[s])
        if self.use_graph:
            key = s
            if self._graphs[key] is None or self._graphs[key][1] != with_sync:
                self._launch_step(s, False)           # warm-up (gradients only): sets func attributes outside capture
                torch.cuda.synchronize()
                gr = torch.cuda.CUDAGraph()
                # thread_local: other threads (NCCL watchdog, pin-memory) may call CUDA while we capture
                cap = torch.cuda.Stream(device=self.device, priority=getattr(self, "_main_priority", 0))
                with torch.cuda.graph(gr, stream=cap, capture_error_mode="thread_local"):
                    self._launch_step(s, with_sync)
                self._graphs[key] = (gr, with_sync)
            self._graphs[key][0].replay()
        else:
            self._launch_step(s, with_sync)
        if with_sync:
            self._steps_launched = getattr(self, "_steps_launched", 0) + 1
        self._slot_free[s].record(cur)

    # ---- public step API ----------------------------------------------------------------------------------
    def forward_backward(self, step: int) -> None:
        """Gradients only (the aggregation is launched separately by the optimizer)."""
        self._run(with_sync=False)

    def train_step(self) -> None:
        """Whole step incl. the fused allreduce+SGD kernel, as one CUDA graph replay."""
        assert self._opt_args is not None, "attach_optimizer() first"
        self._run(with_sync=True)

    def read_loss_async(self):
        """``(event, buffer)`` of the step enqueued last: the step copies (loss, accuracy) into a pinned host buffer
        (two alternate, one per input slot) as its final node; wait on the event, then read ``buffer[0]`` / ``buffer[1]``."""
        s = self._slot                      # the step just enqueued copied its result into this slot's buffer itself
        self.h_loss_acc = self.h_loss_bufs[s]
        return self._slot_free[s], self.h_loss_bufs[s]

    def read_result_async(self):
        """``(event, loss buffer, seq)`` of the step enqueued last: wait on the event, then ``loss[0]``/``loss[1]`` are (loss,
        accuracy) and ``backend.mirror_info(seq)`` is the step's StepInfo -- both were written into page-locked host memory
        by the step's own kernels, so the host never issues a device read."""
        s = self._slot
        return self._slot_free[s], self.h_loss_bufs[s], self._seq0 + self._steps_launched

    def loss_acc(self) -> Tuple[float, float]:
        ev, buf = self.read_loss_async()
        ev.synchronize()
        return float(buf[0]), float(buf[1])

    def step_info(self) -> StepInfo:
        return self.backend.last_step_info(check=True)     # one packed device->host read

    # ---- inference ------------------------------------------------------------------------------------------
    @torch.no_grad()
    def evaluate(self, images, labels) -> Tuple[float, float]:
        if isinstance(images, np.ndarray):
            images, labels = torch.from_numpy(np.ascontiguousarray(images)), torch.from_numpy(np.ascontiguousarray(labels))
        images = images.reshape(-1, 28, 28).to(self.device, torch.float32)
        labels = labels.to(self.device, torch.int64)
        n, B = images.shape[0], self.batch_size
        tot_loss = tot_hit = 0.0
        for s in range(0, n, B):
            m = min(B, n - s)
            self._launch_forward(images[s:s + m].contiguous(), labels[s:s + m].contiguous(), m, False)
            la = self.d_loss_acc.cpu()
            tot_loss += float(la[0]) * m      # kernel scales by 1/m
            tot_hit += float(la[1]) * m
        return tot_loss / n, tot_hit / n

    def forward_logits(self, images: torch.Tensor, labels: torch.Tensor, train: bool) -> torch.Tensor:
        """Debug/test helper: logits of one batch through the CUDA forward."""
        B = images.shape[0]
        out = torch.zeros(B, 10, dtype=torch.float32, device=self.device)
        self.d_loss_acc.zero_()
        self._launch_forward(images.reshape(B, 28, 28).contiguous(), labels, B, train, logits_out=out)
        return out


class CudaMlpEngine(ComputeEngine):
    """2-/3-layer MLP on the sm_100a kernels: hidden layers = tcgen05 GEMM with bias+ReLU fused in the
    epilogue, output layer + softmax-CE = SIMT (csrc/mlp_simt.cu), every weight gradient = tcgen05 GEMM
    with MN-major operands writing straight into the gradient arena."""

    def __init__(self, model: str, batch_size: int, backend: FusedBackend, hidden: int = 1024, seed: int = 66478,
                 rank: int = 0, use_graph: bool = True):
        assert hidden % 64 == 0, "--mlp_hidden must be a multiple of 64 on the GPU path"
        self.lib, self.backend, self.device = load(), backend, backend.ctx.device
        self.spec, _ = get_model(model, hidden)
        self.model, self.batch_size, self.hidden = model, batch_size, hidden
        self.n_layers = len(self.spec.params) // 2
        self.use_graph = use_graph
        # 128 x 256 GEMM tiles when the hidden width allows: half the L2->SM operand traffic per FLOP of 128 x 128
        self._bn = 256 if (hidden % 256 == 0 and os.environ.get("DMNIST_GEMM_BN256", "1") != "0") else 128
        B, dev, bf = batch_size, self.device, torch.bfloat16
        self.params = backend.allocate(self.spec.arena_numel)
        self.params.copy_(self.spec.init_flat(seed).to(dev))
        self.grads = backend.allocate(self.spec.arena_numel)
        self.shadow = backend.attach_shadow(self.params)
        self.p, self.g, self.pb = (self.spec.views(t) for t in (self.params, self.grads, self.shadow))
        self._in_bytes = B * 784 * 4 + B * 8
        self.in_dev = [torch.zeros(self._in_bytes, dtype=torch.uint8, device=dev) for _ in range(2)]
        self.images = [t[:B * 784 * 4].view(torch.float32).view(B, 784) for t in self.in_dev]
        self.labels = [t[B * 784 * 4:].view(torch.int64) for t in self.in_dev]
        self.h_images = [torch.zeros(B, 784, dtype=torch.float32).pin_memory() for _ in range(2)]
        self.h_labels = [torch.zeros(B, dtype=torch.int64).pin_memory() for _ in range(2)]
        self.x16 = torch.zeros(B, 784, dtype=bf, device=dev)
        self.h = [torch.zeros(B, hidden, dtype=bf, device=dev) for _ in range(self.n_layers - 1)]
        self.dh = [torch.zeros(B, hidden, dtype=bf, device=dev) for _ in range(self.n_layers - 1)]
        self.dl_pad = torch.zeros(B, 64, dtype=bf, device=dev)
        self.d_loss_acc = torch.zeros(2, dtype=torch.float32, device=dev)
        self.h_loss_bufs = [torch.zeros(2, dtype=torch.float32).pin_memory() for _ in range(2)]
        self._loss_reads = 0
        self._slot = self._loaded = 0
        self.copy_stream = torch.cuda.Stream(device=dev)
        self._copy_done = [torch.cuda.Event() for _ in range(2)]
        self._slot_free = [torch.cuda.Event() for _ in range(2)]
        self._graphs = [None, None]
        self._opt_args: Optional[dict] = None
        self._straggler = None
        self.launches_per_step = 0
        # bucketed aggregation (csrc/fused_bucket.cu): the largest weight matrix is the early bucket (bf16 wire, exchanged next
        # to the remaining backward GEMMs), everything else the pushed late bucket
        big = max((q for q in self.spec.params if q.name.endswith("weights")), key=lambda q: q.numel)
        self._early_name = big.name
        self._bucket_split = big.offset
        self._bucket_early = (big.offset, big.offset + big.numel)
        self._g16_shape = (784 if big.name == "fc1_weights" else hidden, hidden if big.name != "fc%d_weights" % self.n_layers else 10)
        self._branches = True
        self._bucketed = self._bucket_v2 = False
        self._g16 = self._g16_view = self._inbox = None
        self._side = [torch.cuda.Stream(device=dev)]
        # everything except the weight matrices (written whole by GEMM stores) is accumulated with atomics
        stored = sorted((q.offset, q.offset + q.numel) for q in self.spec.params if q.name.endswith("weights"))
        self._zero_ranges, pos = [], 0
        for (a0, a1) in stored:
            if a0 > pos:
                self._zero_ranges.append((pos, a0))
            pos = a1
        if pos < self.spec.arena_numel:
            self._zero_ranges.append((pos, self.spec.arena_numel))

    # shared plumbing with the convnet engine
    load_batch = CudaLeNetEngine.load_batch
    _leave_native_runner = CudaLeNetEngine._leave_native_runner
    step_packed = CudaLeNetEngine.step_packed
    _make_runner = CudaLeNetEngine._make_runner
    pack_batch = CudaLeNetEngine.pack_batch
    load_packed = CudaLeNetEngine.load_packed
    attach_optimizer = CudaLeNetEngine.attach_optimizer
    params_updated = CudaLeNetEngine.params_updated
    _run = CudaLeNetEngine._run
    forward_backward = CudaLeNetEngine.forward_backward
    train_step = CudaLeNetEngine.train_step
    read_loss_async = CudaLeNetEngine.read_loss_async
    read_result_async = CudaLeNetEngine.read_result_async
    loss_acc = CudaLeNetEngine.loss_acc
    step_info = CudaLeNetEngine.step_info
    _stamp = False

    def h2d_bytes_per_step(self) -> int:
        return self.batch_size * (784 * 4 + 8)

    def _forward(self, images: torch.Tensor, labels: torch.Tensor, B: int, train: bool,
                 logits_out: Optional[torch.Tensor] = None) -> int:
        lib, sp, p, pb, H = self.lib, stream_ptr(), self.p, self.pb, self.hidden
        n = 0
        check(lib.dm_f32_to_bf16(ptr(images), ptr(self.x16), ctypes.c_longlong(B * 784), sp), "f32_to_bf16")
        src, K = self.x16, 784
        for i in range(1, self.n_layers):
            # h_i = relu(src @ W_i + b_i): A K-major, B = W_i [in,out] MN-major, bias+ReLU in the epilogue
            G.gemm_bf16_raw(src, pb["fc%d_weights" % i], self.h[i - 1], B, H, K, K, H, H, False, True,
                            G.EPI_BIAS_RELU_BF16, bn=self._bn, bias=p["fc%d_biases" % i])
            src, K = self.h[i - 1], H
            n += 1
        L = self.n_layers
        check(lib.dm_dense10_xent(ptr(src), ptr(p["fc%d_weights" % L]), ptr(p["fc%d_biases" % L]), ptr(labels),
                                  ptr(self.dh[-1]), ptr(self.dl_pad), ptr(self.g["fc%d_biases" % L]),
                                  ptr(self.d_loss_acc), ptr(logits_out), B, H, int(train), sp), "dense10_xent")
        return n + 2

    def _backward(self, B: int, early_sync: bool = False) -> int:
        """``early_sync``: bucketed aggregation -- the big layer's weight gradient is stored as bf16 into the wire buffer and its
        exchange (phase 3) starts on a side stream at once, next to the data-gradient GEMM; the apply (phase 4) follows that
        GEMM, which is the last reader of the layer's bf16 shadow."""
        lib, sp, g, pb, H, L = self.lib, stream_ptr(), self.g, self.pb, self.hidden, self.n_layers
        n = 0
        main = torch.cuda.current_stream()
        oa, be = self._opt_args, self.backend
        self._join_early = None
        # output layer: dW_L[H,10] = h_last^T (MN-major) * dl (MN-major, 64-wide zero-padded rows, N = 10)
        G.gemm_bf16_raw(self.h[-1], self.dl_pad, g["fc%d_weights" % L], H, 10, B, H, 64, 10, True, True,
                        G.EPI_STORE_F32, bn=64)
        check(lib.dm_relu_bwd_colsum(ptr(self.dh[-1]), ctypes.c_void_p(0), ctypes.c_void_p(0),
                                     ptr(g["fc%d_biases" % (L - 1)]), B, H, sp), "colsum")
        n += 2
        for i in range(L - 1, 0, -1):
            src, K = (self.h[i - 2], H) if i > 1 else (self.x16, 784)
            early = early_sync and self._early_name == "fc%d_weights" % i
            # dW_i[in,H] = src^T (MN-major) * dh_i (MN-major), K = batch
            if early:
                G.gemm_bf16_raw(src, self.dh[i - 1], self._g16_view, K, H, B, K, H, H, True, True, G.EPI_STORE_BF16, bn=self._bn)
                e0, e1 = self._bucket_early
                ev = torch.cuda.Event()
                ev.record(main)
                side = self._side[0]
                side.wait_event(ev)
                be.enqueue_bucket_v2(self.params, self.grads, self._g16, self._inbox, 3 if i > 1 else 1, e0, e1, oa["lr0"],
                                     oa["decay_rate"], oa["decay_steps"], stream=side, rule=oa["rule"], slots=oa["slots"])
                n += 1
                if i == 1:
                    self._join_early = torch.cuda.Event()
                    self._join_early.record(side)
            else:
                G.gemm_bf16_raw(src, self.dh[i - 1], g["fc%d_weights" % i], K, H, B, K, H, H, True, True,
                                G.EPI_STORE_F32, bn=self._bn)
            n += 1
            if i > 1:
                # dh_{i-1} = (dh_i @ W_i^T) * relu'(h_{i-1});  W_i [in,out]: rows = in (N), K = out contiguous
                G.gemm_bf16_raw(self.dh[i - 1], pb["fc%d_weights" % i], self.dh[i - 2], B, H, H, H, H, H, False, False,
                                G.EPI_STORE_BF16, bn=self._bn)
                if early:
                    # the data-gradient GEMM above was the last reader of this layer's bf16 shadow: the apply may rewrite it
                    ev2 = torch.cuda.Event()
                    ev2.record(main)
                    side = self._side[0]
                    side.wait_event(ev2)
                    be.enqueue_bucket_v2(self.params, self.grads, self._g16, self._inbox, 4, e0, e1, oa["lr0"],
                                         oa["decay_rate"], oa["decay_steps"], stream=side, rule=oa["rule"], slots=oa["slots"])
                    n += 1
                    self._join_early = torch.cuda.Event()
                    self._join_early.record(side)
                check(lib.dm_relu_bwd_colsum(ptr(self.dh[i - 2]), ptr(self.h[i - 2]), ptr(self.dh[i - 2]),
                                             ptr(g["fc%d_biases" % (i - 1)]), B, H, sp), "relu_bwd_colsum")
                n += 2
        if self._join_early is not None:
            main.wait_event(self._join_early)
        return n

    def _launch_zero(self) -> int:
        sp, base = stream_ptr(), self.grads.data_ptr()
        for (a, b) in self._zero_ranges:
            check(self.lib.dm_memset_async(ctypes.c_void_p(base + 4 * a), 0, ctypes.c_ulonglong(4 * (b - a)), sp), "memset")
        check(self.lib.dm_memset_async(ptr(self.d_loss_acc), 0, ctypes.c_ulonglong(8), sp), "memset")
        return 0

    def _launch_step(self, slot: int, with_sync: bool) -> None:
        B = self.batch_size
        n = 0
        interval = with_sync and getattr(self, "_interval", False)
        if interval:
            self.backend.enqueue_interval_begin(self.params)
            n += 2
        bucketed = with_sync and self._bucket_v2 and not interval
        n += self._launch_zero()
        n += self._forward(self.images[slot], self.labels[slot], B, True)
        n += self._backward(B, early_sync=bucketed)
        if bucketed:
            if self._straggler is not None:
                self.backend.enqueue_straggler_delay(self._straggler.prob, self._straggler.usec)
                n += 1
            oa = self._opt_args
            e0, e1 = self._bucket_early
            self.backend.enqueue_bucket_v2(self.params, self.grads, self._g16, self._inbox, 2, e0, e1, oa["lr0"],
                                           oa["decay_rate"], oa["decay_steps"], rule=oa["rule"], slots=oa["slots"])
            n += 1
        elif with_sync:
            if self._straggler is not None:
                self.backend.enqueue_straggler_delay(self._straggler.prob, self._straggler.usec)
                n += 1
            if interval:
                oa = self._opt_args
                self.backend.enqueue_interval_end(self.params, self.grads, self._acc, oa["lr0"], oa["decay_rate"], oa["decay_steps"],
                                                  rule=oa["rule"], slots=oa["slots"])
                n += 4
            else:
                self.backend.enqueue(self.params, self.grads, **self._opt_args)
                n += 1
        self.h_loss_bufs[slot].copy_(self.d_loss_acc, non_blocking=True)     # result read-back is part of the step
        self.launches_per_step = n

    @torch.no_grad()
    def evaluate(self, images, labels) -> Tuple[float, float]:
        if isinstance(images, np.ndarray):
            images, labels = torch.from_numpy(np.ascontiguousarray(images)), torch.from_numpy(np.ascontiguousarray(labels))
        images = images.reshape(-1, 784).to(self.device, torch.float32)
        labels = labels.to(self.device, torch.int64)
        n, B = images.shape[0], self.batch_size
        tot_loss = tot_hit = 0.0
        for s in range(0, n, B):
            m = min(B, n - s)
            self.d_loss_acc.zero_()
            self._forward(images[s:s + m].contiguous(), labels[s:s + m].contiguous(), m, False)
            la = self.d_loss_acc.cpu()
            tot_loss += float(la[0]) * m
            tot_hit += float(la[1]) * m
        return tot_loss / n, tot_hit / n


def make_cuda_engine(flags, ctx, backend) -> ComputeEngine:
    if not isinstance(backend, FusedBackend):
        raise RuntimeError("the sm_100a engine needs the fused backend")
    if flags.model == "lenet":
        return CudaLeNetEngine(flags.batch_size, backend, seed=flags.seed, rank=ctx.rank,
                               keep_prob=flags.dropout_keep_prob, use_graph=flags.use_cuda_graph)
    return CudaMlpEngine(flags.model, flags.batch_size, backend, hidden=flags.mlp_hidden, seed=flags.seed,
                         rank=ctx.rank, use_graph=flags.use_cuda_graph)


def make_cuda_eval_engine(flags, device: torch.device) -> ComputeEngine:
    from .parallel.context import ReplicaContext
    ctx = ReplicaContext(0, 1, device.index or 0, device, "none")
    backend = FusedBackend(ctx)
    if flags.model == "lenet":
        return CudaLeNetEngine(1000, backend, seed=flags.seed, keep_prob=flags.dropout_keep_prob, use_graph=False)
    return CudaMlpEngine(flags.model, 1000, backend, hidden=flags.mlp_hidden, seed=flags.seed, use_graph=False)
