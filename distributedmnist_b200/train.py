"""Training driver: the per-replica hot loop.

reference: ``distributed_train.train(target, dataset, dataset_test, cluster_spec)``
(src/distributed_train.py:109-408).  Behaviour kept: K defaults to the number of
workers (:118-121); replica 0 is the chief (:130); staircase LR decay with the /K
rule (:143-156); mode selection from ``--interval_method`` /
``--worker_times_cdf_method`` (:176-188); optional drop-connect in the default mode
only (:194-203); chief restores the latest checkpoint at start (Supervisor,
:244-262) and saves every ``--save_interval_secs`` plus once at the end (:252,
405-408); start-up barrier (:277); the log-line formats (:296,325,341-342,367-371,
398-399); ``worker<id>_time_acc.npy`` every ``--save_results_period`` global steps
(:373-379); per-step chrome timelines (:354-358); loop exit when
``step > max_steps`` checked after the work (:360).

Dropped on purpose (SURVEY §5.9): the second forward pass per iteration that the
reference runs only to log loss/accuracy (:334), ``sess.kill()/reset_kill()``
(:391-396, not in stock TF), ``np.set_printoptions(threshold=np.nan)`` (:31).
"""
from __future__ import annotations

import os
import threading
import time
from datetime import datetime
from typing import Dict, Optional

import numpy as np
import torch

from .checkpoint import Saver
from .engine import make_engine
from .flags import FLAGS
from .optim import UpdateRule
from .parallel.aggregators import (SyncReplicasOptimizer, TimeoutReplicasOptimizer,
                                   parse_straggler_spec)
from .parallel.backends import make_backend
from .parallel.context import ReplicaContext
from .parallel.timeout_manager import launch_manager
from .schedule import LearningRateSchedule
from .utils.logging import get_logger
from .utils.summary import SummaryWriter
from .utils.timeline import Timeline, cupti_device_spans, timeline_path

log = get_logger()

LOG_FORMAT = ("Worker %d: %s: step %d, loss = %f, train_acc = %f, test_acc = %f"
              "(%.1f examples/sec; %.3f  sec/batch)")


class _AsyncCheckpointer:
    """Chief-side saver: snapshot on the training thread, file IO on a helper thread.  The optimizer's state arenas are
    snapshotted at the same drained point as the weights and saved under TF's slot names (``Variable_4/Momentum``)."""

    def __init__(self, train_dir: str, spec, interval_s: float, step_fn=None, opt=None):
        self.train_dir, self.spec, self.interval_s = train_dir, spec, interval_s
        self.step_fn = step_fn       # GPU path: drain the step in flight and read the device step counter (consistent snapshot)
        self.opt = opt               # update rule + state arenas (opt.slots)
        self.saver = Saver()
        self._next = time.time() + interval_s
        self._thread: Optional[threading.Thread] = None

    def maybe_save(self, params: torch.Tensor, global_step: int) -> None:
        if time.time() >= self._next:
            self._next = time.time() + self.interval_s
            self.save(params, global_step, blocking=False)

    def save(self, params: torch.Tensor, global_step: int, blocking: bool = True) -> None:
        if self.step_fn is not None:
            global_step = self.step_fn()         # the host loop runs one step ahead of what it has consumed
        state = self.spec.to_state_dict(params)  # consistent snapshot (device -> host copy)
        if self.opt is not None and self.opt.update_rule.num_slots:
            state.update(self.opt.update_rule.slots_to_state_dict(self.spec, self.opt.ensure_slots(params.numel())))
        if self._thread is not None:
            self._thread.join()
        self._thread = threading.Thread(target=self.saver.save, args=(self.train_dir, state, global_step))
        self._thread.start()
        if blocking:
            self._thread.join()

    def close(self) -> None:
        if self._thread is not None:
            self._thread.join()


class _BatchPacker:
    """Input pipeline of the GPU path: a helper thread draws batches from the DataSet and packs each into one page-locked
    buffer (fp32 images then int64 labels, the device slot's layout), a few batches ahead of the training loop, so a step's
    input is ONE host->device DMA and the hot loop never touches numpy.  Buffers rotate through a ring deep enough that a
    buffer is not rewritten before the copy that reads it has run (the engine double-buffers its device slots)."""

    def __init__(self, engine, dataset, batch_size: int, depth: int = 8, workers: int = 2):
        import queue
        self.engine, self.dataset, self.batch_size = engine, dataset, batch_size
        B = batch_size
        self._nimg = B * 784 * 4
        self.workers = max(1, workers)
        # every worker owns a private ring segment deep enough that a buffer is never rewritten while the DMA that reads it
        # may still be pending (the queue bounds how far ahead of the training loop the workers can run)
        self.rings = [[torch.empty(B * 784 * 4 + B * 8, dtype=torch.uint8).pin_memory() for _ in range(depth + 4)]
                      for _ in range(self.workers)]
        self.ready: "queue.Queue" = queue.Queue(maxsize=depth)
        self._draw = threading.Lock()          # batches are drawn from the DataSet one at a time; the gathers run in parallel
        self._stop = False
        # fast path: gather the batch's rows straight from the dataset arrays into the page-locked buffer with torch
        # (multi-threaded, releases the GIL -- the training loop's interpreter is not held up by the packer)
        self._src = None
        if hasattr(dataset, "next_batch_indices") and not getattr(dataset, "fake_data", False):
            imgs = np.ascontiguousarray(dataset.images, dtype=np.float32).reshape(dataset.num_examples, -1)
            if imgs.shape[1] == 784:
                self._src = (torch.from_numpy(imgs), torch.from_numpy(np.ascontiguousarray(dataset.labels)).to(torch.int64))
        self._threads = [threading.Thread(target=self._run, args=(w,), daemon=True) for w in range(self.workers)]
        for t in self._threads:
            t.start()

    def _run(self, w: int) -> None:
        i = 0
        ring = self.rings[w]
        while not self._stop:
            buf = ring[i % len(ring)]
            if self._src is not None:
                with self._draw:
                    idx = torch.from_numpy(self.dataset.next_batch_indices(self.batch_size).copy())
                torch.index_select(self._src[0], 0, idx, out=buf[:self._nimg].view(torch.float32).view(self.batch_size, 784))
                torch.index_select(self._src[1], 0, idx, out=buf[self._nimg:].view(torch.int64))
            else:
                with self._draw:
                    images, labels = self.dataset.next_batch(self.batch_size)
                buf[:self._nimg].view(torch.float32).copy_(torch.from_numpy(np.ascontiguousarray(images, dtype=np.float32)).reshape(-1))
                buf[self._nimg:].view(torch.int64).copy_(torch.from_numpy(np.ascontiguousarray(labels)).to(torch.int64).reshape(-1))
            while not self._stop:
                try:
                    self.ready.put(buf, timeout=0.1)
                    break
                except Exception:  # noqa: BLE001  (queue.Full)
                    continue
            i += 1

    def next(self) -> torch.Tensor:
        return self.ready.get()

    def close(self) -> None:
        self._stop = True
        try:
            while True:
                self.ready.get_nowait()
        except Exception:  # noqa: BLE001  (queue.Empty)
            pass
        for t in self._threads:
            t.join(timeout=2.0)


def train(ctx: ReplicaContext, dataset, dataset_test=None, flags=FLAGS) -> Dict:
    num_workers = ctx.world_size
    # reference distributed_train.py:118-121
    if flags.num_replicas_to_aggregate == -1:
        num_replicas_to_aggregate = num_workers
    else:
        num_replicas_to_aggregate = flags.num_replicas_to_aggregate
    assert num_workers > 0
    is_chief = ctx.is_chief

    backend = make_backend(ctx, flags.backend, flags)
    engine = make_engine(flags, ctx, backend)
    spec = engine.spec
    lr_schedule = LearningRateSchedule.from_flags(flags, dataset.num_examples, num_replicas_to_aggregate)
    straggler = parse_straggler_spec(flags.inject_straggler)
    rule = UpdateRule.from_flags(flags)

    if flags.interval_method or flags.worker_times_cdf_method:
        # reference :179-183 -- interval wins when both are set, as there.
        mode = "interval" if flags.interval_method else "cdf"
        opt = TimeoutReplicasOptimizer(backend, lr_schedule, total_num_replicas=num_workers, mode=mode,
                                       interval_ms=flags.interval_ms, straggler=straggler, seed=flags.seed,
                                       update_rule=rule)
    else:
        opt = SyncReplicasOptimizer(
            backend, lr_schedule, replicas_to_aggregate=num_replicas_to_aggregate,
            total_num_replicas=num_workers,
            drop_connect_probability=flags.drop_connect_probability if flags.drop_connect else None,
            straggler=straggler, seed=flags.seed, update_rule=rule)
    # GPU path: every mode runs as one CUDA graph per step -- K-of-N / full barrier through the fused aggregation kernels,
    # interval through the device-side deadline protocol (csrc/fused_interval.cu)
    fused_step = hasattr(engine, "attach_optimizer")
    if fused_step:
        engine.attach_optimizer(opt)   # GPU path: compute + fused allreduce/SGD replay as one CUDA graph
    slots = opt.ensure_slots(spec.arena_numel) if rule.num_slots else []   # optimizer state, initial values

    # Supervisor semantics: chief restores the newest checkpoint, everyone gets it.
    restored_step = 0
    if is_chief:
        os.makedirs(flags.train_dir, exist_ok=True)
        latest = Saver.latest(flags.train_dir)
        if latest is not None:
            state, restored_step = Saver.restore(latest)
            engine.params.copy_(spec.from_state_dict(state).to(engine.params.device))
            log.info("Restored model from %s at step=%d" % (latest, restored_step))
            if slots:
                if rule.has_slots(spec, state):
                    for t, flat in zip(slots, rule.slots_from_state_dict(spec, state)):
                        t.copy_(flat.to(t.device))
                    log.info("Restored %s optimizer slots (%s)" % (rule.name, ", ".join(rule.slot_names)))
                else:
                    log.info("Checkpoint has no %s optimizer slots (%s): they start from their initial values"
                             % (rule.name, ", ".join(rule.slot_names)))
    if num_workers > 1:
        restored_step = backend.all_gather_object(restored_step)[0]
        if restored_step > 0:
            backend.broadcast_(engine.params, 0)
            for t in slots:
                backend.broadcast_(t, 0)
    if restored_step > 0:
        opt.local_step = restored_step
        if hasattr(backend, "set_global_step"):
            backend.set_global_step(restored_step)
    if hasattr(engine, "params_updated"):
        engine.params_updated()
    log.info("%s Supervisor" % datetime.now())

    def _device_step() -> int:
        torch.cuda.synchronize()
        return int(backend.device_epoch)
    ckpt = _AsyncCheckpointer(flags.train_dir, spec, flags.save_interval_secs,
                              step_fn=_device_step if (fused_step and hasattr(backend, "device_epoch")) else None, opt=opt) \
        if is_chief else None
    summary = SummaryWriter(flags.train_dir) if (is_chief and flags.should_summarize) else None

    # Even if not using timeout, we want to wait until all machines are ready (reference :275-277).
    timeout_client, timeout_server = launch_manager(backend, flags)

    next_summary_time = time.time() + flags.save_summaries_secs
    begin_time = time.time()
    cur_iteration = -1
    if flags.interval_method:
        if fused_step and hasattr(backend, "interval_arm"):
            backend.interval_arm(float(flags.interval_ms))   # reference :287-288 (chief timer) -> %globaltimer deadline on the device
        else:
            opt.start_interval_updates()   # CPU plumbing path: shared absolute host-clock deadlines

    time_acc_list = []
    step = restored_step
    loss_value = train_acc_value = float("nan")
    results = {"steps": [], "losses": [], "accepted": 0, "dropped": 0}
    # cdf telemetry (reference timeout_manager.py:55-61): compute time = gradient done - token dequeued, the barrier wait
    # NOT included.  interval wins when both flags are set (as in the reference) and its replicas are not in lock step, so
    # the collective flush of the cdf tables must not run then.
    cdf = bool(flags.worker_times_cdf_method and not flags.interval_method)
    device_times = cdf and fused_step and hasattr(backend, "read_timing")   # %globaltimer stamps written by the step's kernels
    cdf_pushed = 0                 # first iteration whose device stamps have not been handed to the timeout client yet
    # GPU path: the host runs ONE step ahead of the device -- step i+1 is enqueued before step i's (loss, status words) are
    # read from the page-locked buffers the step's graph copied them to, so no iteration ever waits for a device sync, and
    # batches are packed into page-locked buffers by a helper thread (`_BatchPacker`).
    pipelined = bool(fused_step and getattr(flags, "pipeline_steps", True) and hasattr(engine, "read_result_async")
                     and not flags.timeline_logging)
    packer = _BatchPacker(engine, dataset, flags.batch_size) if pipelined else None
    every = max(flags.log_every, 1)
    pending = None                 # (iteration, start_time, result token) of the step in flight
    launched = 0
    exact = isinstance(opt, SyncReplicasOptimizer) and num_replicas_to_aggregate == num_workers or cdf
    stop = False

    def finish_iteration(it: int, start_time: float, info, loss_acc) -> None:
        nonlocal step, loss_value, train_acc_value, next_summary_time, stop
        step = info.global_step
        do_log = (it % every == 0)
        if loss_acc is not None:
            loss_value, train_acc_value = loss_acc
        if do_log:
            log.info("Global step attained: %d" % step)
            log.info("DONE RUNNING SESSION...")
        finish_time = time.time()
        if step > flags.max_steps:
            stop = True
            return
        test_acc_value = 0.0   # hard-wired in the reference too (:363)
        duration = finish_time - start_time
        examples_per_sec = flags.batch_size / float(max(duration, 1e-9))
        if do_log:
            log.info(LOG_FORMAT % (ctx.rank, datetime.now(), step, loss_value, train_acc_value,
                                   test_acc_value, examples_per_sec, duration))
        time_acc_list.append((finish_time, train_acc_value, test_acc_value, loss_value))
        results["steps"].append(step)
        results["losses"].append(loss_value)
        if step % flags.save_results_period == 0:
            np.save(os.path.join(flags.train_dir, "worker%d_time_acc.npy" % ctx.rank), np.array(time_acc_list))
        if is_chief:
            ckpt.maybe_save(engine.params, step)
            if summary is not None and next_summary_time < time.time():
                log.info("Running Summary operation on the chief.")
                summary.add_scalars({"loss": loss_value, "train_acc": train_acc_value,
                                     "learning_rate": lr_schedule(step)}, step)
                log.info("Finished running Summary operation.")
                next_summary_time += flags.save_summaries_secs

    def push_device_times(upto: int) -> None:
        """Hand the %globaltimer stamps of iterations [cdf_pushed, upto] to the timeout client: 'dequeued' = the step's first
        kernel started, 'finished' = the aggregation kernel was entered (gradient complete, barrier not yet waited for)."""
        nonlocal cdf_pushed
        if upto < cdf_pushed:
            return
        pairs = backend.read_timing(restored_step + cdf_pushed, restored_step + upto)
        for it, (ts, ta) in zip(range(cdf_pushed, upto + 1), pairs):
            timeout_client.broadcast_worker_dequeued_token(it, ts * 1e-9)
            timeout_client.broadcast_worker_finished_computing_gradients(it, ta * 1e-9)
        cdf_pushed = upto + 1

    last_consume = time.time()
    while not stop:
        cur_iteration += 1
        do_log = (cur_iteration % every == 0)
        if do_log:
            log.info("A new iteration...")

        if cdf and not device_times:
            t_deq = opt.wait_op()
            timeout_client.broadcast_worker_dequeued_token(cur_iteration, t_deq)

        if pipelined:
            if do_log:
                log.info("RUNNING SESSION... %f" % time.time())
            token = (cur_iteration, engine.step_packed(packer.next()))   # input DMA + step graph: one native call
            launched += 1
            prev, pending = pending, token
            if prev is not None:
                it, (ev, lbuf, seq) = prev
                ev.synchronize()
                info = opt._account(backend.mirror_info(seq, check=True))
                now = time.time()
                finish_iteration(it, last_consume, info, (float(lbuf[0]), float(lbuf[1])))
                last_consume = now
                if device_times and it > 10 and (it % 50 == 0 or it == 500):
                    push_device_times(it)
            # K == N: the global step after `launched` steps is known without reading anything -> stop launching exactly there
            if exact and restored_step + launched > flags.max_steps:
                break
            continue

        tl = Timeline(pid=ctx.rank) if flags.timeline_logging else None
        start_time = time.time()
        images, labels = dataset.next_batch(flags.batch_size)
        if tl:
            tl.add_span("next_batch", 0.0, (time.time() - start_time) * 1e6)
        if do_log:
            log.info("RUNNING SESSION... %f" % time.time())

        t0 = time.perf_counter()
        engine.load_batch(images, labels)
        t1 = time.perf_counter()
        t_fin = None
        dev_spans = None
        if fused_step:
            if tl and ctx.on_gpu:
                # reference: RunOptions(trace_level=FULL_TRACE) per step (src/distributed_train.py:317-319) -> here CUPTI around
                # the graph replay: every kernel / copy of the step with its stream, start and duration
                dev_spans = cupti_device_spans(engine.train_step)
            else:
                engine.train_step()
            t2 = time.perf_counter()
            info = opt._account(engine.step_info())   # device -> host read of the step's outcome (one packed copy)
        else:
            engine.forward_backward(opt.local_step)
            t2 = time.perf_counter()
            t_fin = time.time()                       # gradient complete; the barrier / reduction comes after this stamp
            info = opt.apply_gradients(engine.params, engine.grads) if not isinstance(opt, TimeoutReplicasOptimizer) \
                else opt.apply_gradients(engine.params, engine.grads, ctx.rank, cdf)
            if info.applied and hasattr(engine, "params_updated") and not hasattr(engine, "train_step"):
                engine.params_updated()
        la = engine.loss_acc() if (do_log or flags.timeline_logging) else None
        t3 = time.perf_counter()

        if cdf:
            if device_times:
                if cur_iteration > 10 and (cur_iteration % 50 == 0 or cur_iteration == 500):
                    push_device_times(cur_iteration)
            else:
                opt.finish_times.append(t_fin if t_fin is not None else time.time())
                timeout_client.broadcast_worker_finished_computing_gradients(cur_iteration, opt.finish_times[-1])

        if tl:
            base = (t0 - tl._t0) * 1e6
            tl.add_span("load_batch(H2D)", base, (t1 - t0) * 1e6)
            tl.add_span("forward_backward", base + (t1 - t0) * 1e6, (t2 - t1) * 1e6)
            tl.add_span("aggregate+apply", base + (t2 - t0) * 1e6, (t3 - t2) * 1e6)
            if dev_spans:
                tl.add_device_spans(dev_spans, base + (t1 - t0) * 1e6)
            with open(timeline_path(flags.train_dir, ctx.rank, info.global_step), "w") as f:
                f.write(tl.generate_chrome_trace_format())
        finish_iteration(cur_iteration, start_time, info, la)

    if pending is not None:          # drain the step still in flight
        it, (ev, lbuf, seq) = pending
        ev.synchronize()
        info = opt._account(backend.mirror_info(seq, check=True))
        finish_iteration(it, last_consume, info, (float(lbuf[0]), float(lbuf[1])))
        pending = None
    if packer is not None:
        packer.close()
    if device_times:
        push_device_times(cur_iteration)

    if is_chief:
        log.info("Elapsed Time: %f" % (time.time() - begin_time))
    if cdf:
        timeout_client.flush()
        if ctx.rank == 0 and device_times:
            timeout_server.report()

    # Save after the training ends (reference :405-408).
    if is_chief:
        ckpt.save(engine.params, step, blocking=True)
        ckpt.close()
    if summary is not None:
        summary.close()
    results.update(final_step=step, accepted=opt.accepted_steps, dropped=opt.dropped_steps,
                   params=engine.params, elapsed=time.time() - begin_time,
                   timeout_server=timeout_server, engine=engine, optimizer=opt)
    return results
