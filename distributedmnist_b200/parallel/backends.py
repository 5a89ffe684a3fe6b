"""Gradient-aggregation backends: who moves the bytes and applies the update.

The *policy* (K-of-N / full barrier / interval, SURVEY §2.3) lives in
``aggregators.py``; a backend implements the mechanics for one transport:

* :class:`LocalBackend`  -- one replica, no communication.
* :class:`GlooBackend`   -- CPU, multi-process; commit protocol over the c10d
  store, masked ``all_reduce`` for the mean.  This is the plumbing path that runs
  without a GPU (BASELINE.json config 1).
* :class:`NcclBackend`   -- GPU, ``ncclAllReduce`` + separate scale + SGD
  kernels.  **Baseline only** (what a stock framework does); never the product
  path.
* ``FusedBackend`` (``fused.py``) -- the product path: one sm_100a kernel that
  publishes arrival, polls the commit word, reduces over NVLink peer/multicast
  memory, scales by 1/count and applies SGD (no NCCL call, no separate
  elementwise kernel).

All backends honour the same contract: after ``sync_step`` every replica holds
bit-identical parameters (and optimizer state), the divisor is the number of
accepted gradients, and late/stale gradients are discarded without stalling the
update.  ``rule`` (``optim.UpdateRule``, None = SGD) and ``slots`` (its state
arenas, laid out like ``params``) select and carry the update rule.
"""
from __future__ import annotations

import time
from dataclasses import dataclass
from typing import List, Optional

import torch
import torch.distributed as dist

from ..optim import rule_or_sgd
from .context import ReplicaContext
from .protocol import Decision, StoreCommitBoard


@dataclass
class StepInfo:
    global_step: int        # global step after this call
    accepted: bool          # my gradient was part of the mean
    mask: int               # contributor bitmap
    count: int              # divisor
    stale: bool = False
    applied: bool = True    # False when (interval mode) no update happened in this call


class Backend:
    name = "abstract"

    def __init__(self, ctx: ReplicaContext):
        self.ctx = ctx

    # -- memory -----------------------------------------------------------
    def allocate(self, numel: int) -> torch.Tensor:
        """Arena allocation hook (the fused backend returns symmetric memory)."""
        return torch.zeros(numel, dtype=torch.float32, device=self.ctx.device)

    # -- collectives used outside the hot path ---------------------------------
    def barrier(self) -> None:
        if self.ctx.world_size > 1:
            dist.barrier()

    def broadcast_(self, t: torch.Tensor, src: int = 0) -> None:
        if self.ctx.world_size > 1:
            dist.broadcast(t, src)

    def all_gather_object(self, obj) -> List:
        if self.ctx.world_size == 1:
            return [obj]
        out = [None] * self.ctx.world_size
        dist.all_gather_object(out, obj)
        return out

    # -- hot path -----------------------------------------------------------
    def sync_step(self, params: torch.Tensor, grads: torch.Tensor, lr: float, local_step: int,
                  k: int, delay_s: float = 0.0, rule=None, slots=()) -> StepInfo:
        raise NotImplementedError

    def interval_tick(self, params: torch.Tensor, acc: torch.Tensor, count: int, lr: float,
                      tick: int, rule=None, slots=()) -> StepInfo:
        raise NotImplementedError


class LocalBackend(Backend):
    name = "local"

    def __init__(self, ctx: ReplicaContext):
        super().__init__(ctx)
        self._global_step = 0

    def sync_step(self, params, grads, lr, local_step, k, delay_s=0.0, rule=None, slots=()) -> StepInfo:
        if delay_s > 0:
            time.sleep(delay_s)
        rule_or_sgd(rule).apply(params, grads, 1, lr, slots)
        self._global_step = local_step + 1
        return StepInfo(self._global_step, True, 1, 1)

    def interval_tick(self, params, acc, count, lr, tick, rule=None, slots=()) -> StepInfo:
        if count == 0:
            return StepInfo(self._global_step, False, 0, 0, applied=False)
        rule_or_sgd(rule).apply(params, acc, count, lr, slots)
        self._global_step += 1
        return StepInfo(self._global_step, True, 1, count)


class _CollectiveBackend(Backend):
    """Shared logic of the two ``torch.distributed`` collective backends."""

    def __init__(self, ctx: ReplicaContext, board_prefix: str = "commit_board"):
        super().__init__(ctx)
        self._global_step = 0
        self._board: Optional[StoreCommitBoard] = None
        self._board_prefix = board_prefix

    def _get_board(self, k: int) -> StoreCommitBoard:
        if self._board is None or self._board.k != k:
            assert self.ctx.store is not None, "K-of-N needs the rendezvous store"
            self._board = StoreCommitBoard(self.ctx.store, self.ctx.world_size, k,
                                           prefix="%s/k%d" % (self._board_prefix, k))
        return self._board

    def _decide(self, local_step: int, k: int, delay_s: float) -> Decision:
        n = self.ctx.world_size
        if delay_s > 0:
            time.sleep(delay_s)  # injected straggler: arrive late
        if k >= n:
            full = (1 << n) - 1
            return Decision(local_step, True, False, full, n, local_step + 1)
        d = self._get_board(k).arrive(self.ctx.rank, local_step)
        if self.ctx.rank == 0 and local_step >= 8:
            self._board.gc(local_step - 8)
        return d

    def sync_step(self, params, grads, lr, local_step, k, delay_s=0.0, rule=None, slots=()) -> StepInfo:
        d = self._decide(local_step, k, delay_s)
        # Masked contribution: a late replica joins the collective with zeros, so
        # the sum holds exactly the accepted gradients and everyone divides by the
        # same popcount -- replicas stay bit-identical.
        contrib = grads if d.accepted else torch.zeros_like(grads)
        dist.all_reduce(contrib, op=dist.ReduceOp.SUM)
        rule_or_sgd(rule).apply(params, contrib, d.count, lr, slots)
        self._global_step = d.global_step
        return StepInfo(d.global_step, d.accepted, d.mask, d.count, stale=d.stale)

    def interval_tick(self, params, acc, count, lr, tick, rule=None, slots=()) -> StepInfo:
        cnt = torch.tensor([float(count)], dtype=torch.float32, device=acc.device)
        dist.all_reduce(cnt, op=dist.ReduceOp.SUM)
        total = int(cnt.item())
        flags = self.all_gather_object((int(count > 0), time.monotonic()))
        self.last_chief_clock = flags[0][1]        # replicas of one box share CLOCK_MONOTONIC: the chief's "now" of this tick
        mask = sum(1 << i for i, f in enumerate(flags) if f[0])
        if total == 0:
            return StepInfo(self._global_step, False, 0, 0, applied=False)
        dist.all_reduce(acc, op=dist.ReduceOp.SUM)
        rule_or_sgd(rule).apply(params, acc, total, lr, slots)
        self._global_step += 1
        return StepInfo(self._global_step, count > 0, mask, total)


class GlooBackend(_CollectiveBackend):
    name = "gloo"


class NcclBackend(_CollectiveBackend):
    """Baseline: ``ncclAllReduce`` then separate scale/SGD kernels (torch ops)."""
    name = "nccl"


def make_backend(ctx: ReplicaContext, choice: str = "auto", flags=None) -> Backend:
    """``auto``: fused on GPU, gloo on multi-process CPU, local otherwise.  ``flags`` (optional): ``--sync_timeout_ms``,
    ``--use_nvls`` and ``--debug_sync`` configure the fused backend."""
    if choice == "auto":
        if ctx.on_gpu:
            choice = "fused"
        else:
            choice = "gloo" if ctx.world_size > 1 else "local"
    if choice == "local":
        assert ctx.world_size == 1
        return LocalBackend(ctx)
    if choice == "gloo":
        return GlooBackend(ctx) if ctx.world_size > 1 else LocalBackend(ctx)
    if choice == "nccl":
        return NcclBackend(ctx) if ctx.world_size > 1 else LocalBackend(ctx)
    if choice == "fused":
        from .fused import FusedBackend  # imports the sm_100a extension; fails loudly if missing
        kw = {}
        if flags is not None:
            kw = dict(timeout_ms=float(getattr(flags, "sync_timeout_ms", 30000)),
                      use_nvls=None if getattr(flags, "use_nvls", True) else False,
                      debug_sync=bool(getattr(flags, "debug_sync", False)))
        return FusedBackend(ctx, **kw)
    raise ValueError("unknown backend %r" % choice)
