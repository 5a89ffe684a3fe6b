"""Gradient-aggregation policies: the three synchronisation modes of the reference.

====================  =====================================================  =========================
mode                  reference                                              here
====================  =====================================================  =========================
A  K-of-N (default)   stock ``tf.train.SyncReplicasOptimizer`` selected at   :class:`SyncReplicasOptimizer`
                      src/distributed_train.py:185-188
B  full barrier +     ``TimeoutReplicasOptimizer`` with ``take_grad(N)``,     :class:`TimeoutReplicasOptimizer`
   timing ("cdf")     per-worker token queues, ``_wait_op`` run first         (``mode="cdf"``)
                      (sync_replicas_optimizer_modified.py:198-206,278-279,
                      370-371; distributed_train.py:305-307,344-345)
C  interval           ``take_grad(1)`` from a chief-side timer every          :class:`TimeoutReplicasOptimizer`
                      ``--interval_ms`` (…modified.py:208-215,373)            (``mode="interval"``)
====================  =====================================================  =========================

Optional gradient drop-connect (Bernoulli(p) 0/1 mask on every gradient element
before aggregation, no 1/p rescale, mode A only -- distributed_train.py:194-196,
202-203,414-416) and straggler injection (new; the reference relied on naturally
slow EC2 ``t2`` instances) are applied here, before the backend moves any bytes.
"""
from __future__ import annotations

import random
import time
from dataclasses import dataclass
from typing import Callable, Dict, List, Optional

import torch

from ..optim import UpdateRule, rule_or_sgd
from .backends import Backend, StepInfo


@dataclass
class StragglerSpec:
    prob: float
    usec: float


def parse_straggler_spec(text: str) -> Dict[int, StragglerSpec]:
    """``"3:0.5:2000,5:1:500"`` -> {3: (p=.5, 2000us), 5: (p=1, 500us)}."""
    out: Dict[int, StragglerSpec] = {}
    for item in filter(None, (s.strip() for s in (text or "").split(","))):
        parts = item.split(":")
        if len(parts) != 3:
            raise ValueError("--inject_straggler wants rank:prob:usec, got %r" % item)
        out[int(parts[0])] = StragglerSpec(float(parts[1]), float(parts[2]))
    return out


class _AggregatorBase:
    def __init__(self, backend: Backend, lr_schedule: Callable[[int], float], total_num_replicas: int,
                 straggler: Optional[Dict[int, StragglerSpec]] = None, seed: int = 0,
                 update_rule: Optional[UpdateRule] = None):
        self.backend = backend
        self.update_rule = rule_or_sgd(update_rule)
        self.slots: List[torch.Tensor] = []     # optimizer state arenas (parameter-arena layout), see ensure_slots()
        self.lr_schedule = lr_schedule
        self.total_num_replicas = int(total_num_replicas)
        self.local_step = 0          # global step of the weights my next gradient is computed from (X7)
        self.last_info: Optional[StepInfo] = None
        self._straggler = (straggler or {}).get(backend.ctx.rank)
        self._rng = random.Random(seed * 7919 + backend.ctx.rank)
        self.accepted_steps = 0
        self.dropped_steps = 0

    @property
    def global_step(self) -> int:
        return self.local_step

    def ensure_slots(self, numel: int) -> List[torch.Tensor]:
        """The update rule's state arenas, allocated through the backend (symmetric memory on the fused backend) and set to
        their initial values on first use.  Every rank calls it in the same order (the allocation may be collective)."""
        if len(self.slots) != self.update_rule.num_slots:
            self.slots = self.update_rule.allocate_slots(self.backend.allocate, numel)
        return self.slots

    def _delay_s(self) -> float:
        s = self._straggler
        if s is not None and self._rng.random() < s.prob:
            return s.usec * 1e-6
        return 0.0

    def _rule_kw(self, params: torch.Tensor) -> dict:
        if self.update_rule.num_slots == 0:
            return {}          # SGD: the backends' call is exactly what it was before state existed
        return dict(rule=self.update_rule, slots=self.ensure_slots(params.numel()))

    def _account(self, info: StepInfo) -> StepInfo:
        self.last_info = info
        self.local_step = info.global_step
        if info.applied:
            if info.accepted:
                self.accepted_steps += 1
            else:
                self.dropped_steps += 1
        return info

    # API-shape parity with the reference's optimizer objects; the queue runner /
    # token machinery has no work left to do (SURVEY §2.5 X5, X6, X8).
    def get_chief_queue_runner(self):
        return None

    def get_init_tokens_op(self):
        return None


class SyncReplicasOptimizer(_AggregatorBase):
    """Mode A: synchronous SGD that commits on the first K of N gradients."""

    def __init__(self, backend: Backend, lr_schedule, replicas_to_aggregate: int, total_num_replicas: int,
                 drop_connect_probability: Optional[float] = None, straggler=None, seed: int = 0,
                 update_rule: Optional[UpdateRule] = None):
        super().__init__(backend, lr_schedule, total_num_replicas, straggler, seed, update_rule)
        if not 1 <= replicas_to_aggregate <= total_num_replicas:
            raise ValueError("replicas_to_aggregate=%d must be in [1, %d]" % (replicas_to_aggregate, total_num_replicas))
        self.replicas_to_aggregate = int(replicas_to_aggregate)
        self.drop_connect_probability = drop_connect_probability
        self._dc_gen: Optional[torch.Generator] = None

    def _drop_connect(self, grads: torch.Tensor) -> torch.Tensor:
        p = self.drop_connect_probability
        if p is None:
            return grads
        if hasattr(self.backend, "drop_connect_"):
            self.backend.drop_connect_(grads, p, self.local_step)   # device-side hash mask
            return grads
        if self._dc_gen is None:
            self._dc_gen = torch.Generator(device="cpu")
            self._dc_gen.manual_seed(1009 * (self.backend.ctx.rank + 1))
        keep = (torch.rand(grads.shape, generator=self._dc_gen) < p).to(grads.dtype).to(grads.device)
        return grads.mul_(keep)

    def apply_gradients(self, params: torch.Tensor, grads: torch.Tensor) -> StepInfo:
        grads = self._drop_connect(grads)
        lr = self.lr_schedule(self.local_step)
        info = self.backend.sync_step(params, grads, lr, self.local_step, self.replicas_to_aggregate,
                                      delay_s=self._delay_s(), **self._rule_kw(params))
        return self._account(info)


class TimeoutReplicasOptimizer(_AggregatorBase):
    """Modes B ("cdf": full barrier + per-iteration timing) and C ("interval")."""

    def __init__(self, backend: Backend, lr_schedule, total_num_replicas: int, mode: str = "cdf",
                 interval_ms: int = 1000, straggler=None, seed: int = 0,
                 clock: Callable[[], float] = time.monotonic, update_rule: Optional[UpdateRule] = None):
        super().__init__(backend, lr_schedule, total_num_replicas, straggler, seed, update_rule)
        assert mode in ("cdf", "interval")
        self.mode = mode
        self.interval_s = interval_ms / 1000.0
        self._clock = clock
        self._acc: Optional[torch.Tensor] = None
        self._acc_count = 0
        self._tick = 0
        self._t0: Optional[float] = None
        self.dequeue_times: List[float] = []      # mode B telemetry (host clock)
        self.finish_times: List[float] = []

    # ---- mode B ---------------------------------------------------------------
    def wait_op(self) -> float:
        """Acquire half of the barrier: the reference's per-worker token dequeue
        (``_wait_op``, …modified.py:278-279).  With a commit protocol the token *is*
        the previous step's commit, which ``apply_gradients`` already waited for, so
        this only stamps the time (the event ``worker_dequeued_token`` reports)."""
        t = time.time()
        self.dequeue_times.append(t)
        return t

    def mark_finished(self) -> float:
        t = time.time()
        self.finish_times.append(t)
        return t

    # ---- mode C ---------------------------------------------------------------
    def start_interval_updates(self, t0: Optional[float] = None) -> None:
        """Arm the interval clock (reference ``start_interval_updates``, …modified.py:208-215).

        Deadlines are absolute: tick k fires at ``t0 + (k+1)*interval``.  All replicas
        live on one box and share ``CLOCK_MONOTONIC``, so the chief's t0 (shared at
        start-up) gives every replica the same deadlines without a timer thread."""
        if t0 is None:
            t0 = self.backend.all_gather_object(self._clock())[0]
        self._t0 = t0

    def _deadline(self, tick: int) -> float:
        assert self._t0 is not None, "call start_interval_updates() first"
        return self._t0 + (tick + 1) * self.interval_s

    def apply_gradients(self, params: torch.Tensor, grads: torch.Tensor, worker_id: int = 0,
                        collect_cdfs: bool = False) -> StepInfo:
        if self.mode == "cdf":
            lr = self.lr_schedule(self.local_step)
            info = self.backend.sync_step(params, grads, lr, self.local_step, self.total_num_replicas,
                                          delay_s=self._delay_s(), **self._rule_kw(params))
            return self._account(info)
        # interval: push into the local accumulator, never block on other replicas
        # until a deadline has passed.
        d = self._delay_s()
        if d > 0:
            time.sleep(d)
        if self._acc is None:
            self._acc = self.backend.allocate(grads.numel())   # symmetric on the fused backend
        self._acc.add_(grads)
        self._acc_count += 1
        info = StepInfo(self.local_step, False, 0, 0, applied=False)
        if self._clock() >= self._deadline(self._tick):
            # ONE tick per call (every replica joins tick t exactly once, in its first call after deadline t), and after a
            # late tick the next deadline is the first one still in the future *on the chief's clock* (exchanged inside the
            # tick) -- missed deadlines are skipped, never replayed, and no replica decides on its own to run another tick
            # (reference: the chief's timer sleeps the interval after each take_grad, …modified.py:208-215).
            lr = self.lr_schedule(self.local_step)
            res = self.backend.interval_tick(params, self._acc, self._acc_count, lr, self._tick, **self._rule_kw(params))
            chief_now = getattr(self.backend, "last_chief_clock", None)
            nxt = self._tick + 1
            if chief_now is not None and self._t0 is not None:
                nxt = max(nxt, int((chief_now - self._t0) / self.interval_s))
            self._tick = nxt
            self._acc.zero_()
            self._acc_count = 0
            if res.applied:
                info = res
                self._account(res)
        self.last_info = info
        return info
