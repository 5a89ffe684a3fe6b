"""Update rules applied by every aggregation path: plain SGD, momentum and RMSProp, with TF 1.x semantics.

The one host-side owner of the optimizer decision: which rule the flags select, how many fp32 state slots it keeps per
parameter, what they start at, what TF calls them in a checkpoint, and the torch implementation the host backends
(``LocalBackend``, gloo, nccl) apply.  The device twin of :meth:`UpdateRule.apply` is ``dm::Update`` in
``csrc/fused_sync.cuh``; the numeric codes of :data:`RULES` are its ``RULE_*`` constants.

With ``g`` the mean gradient of a committed step and ``lr`` its staircase learning rate:

* ``sgd``       ``w -= lr * g``                                            (``ApplyGradientDescent``)
* ``momentum``  ``a = momentum * a + g;  w -= lr * a``                      (``ApplyMomentum``, no Nesterov; ``a`` starts at 0)
* ``rmsprop``   ``ms += (g * g - ms) * (1 - decay)``
  ``mom = momentum * mom + lr * g / sqrt(ms + eps);  w -= mom``            (``ApplyRMSProp``, not centred; ``ms`` starts at 1,
  as TF initialises its ``rms`` slot with ones, ``mom`` at 0)

State changes once per committed global step and nowhere else.  The defaults are the reference's RMSProp constants
(``RMSPROP_DECAY = 0.9``, ``RMSPROP_MOMENTUM = 0.9``, ``RMSPROP_EPSILON = 1.0``, src/distributed_train.py:102-104).
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Dict, List, Optional, Sequence, Tuple

import torch

RULES = {"sgd": 0, "momentum": 1, "rmsprop": 2}
_SLOTS = {"sgd": (), "momentum": (("Momentum", 0.0),), "rmsprop": (("RMSProp", 1.0), ("RMSProp_1", 0.0))}


def check_hyper(name: str, momentum: float, decay: float, eps: float) -> None:
    """Reject an unknown rule or hyper-parameters outside their domain (ValueError)."""
    if name not in RULES:
        raise ValueError("--optimizer=%r: must be one of %s" % (name, "|".join(RULES)))
    if not 0.0 <= momentum < 1.0:
        raise ValueError("--momentum=%r: must lie in [0, 1)" % momentum)
    if not 0.0 <= decay < 1.0:
        raise ValueError("--rmsprop_decay=%r: must lie in [0, 1)" % decay)
    if not eps > 0.0:
        raise ValueError("--rmsprop_epsilon=%r: must be > 0" % eps)


@dataclass(frozen=True)
class UpdateRule:
    name: str = "sgd"
    momentum: float = 0.9
    decay: float = 0.9
    eps: float = 1.0

    def __post_init__(self) -> None:
        check_hyper(self.name, self.momentum, self.decay, self.eps)

    @classmethod
    def from_flags(cls, flags) -> "UpdateRule":
        return cls(flags.optimizer, float(flags.momentum), float(flags.rmsprop_decay), float(flags.rmsprop_epsilon))

    # ---- inventory ------------------------------------------------------------------------------------------------------
    @property
    def code(self) -> int:
        """``RULE_*`` constant of csrc/fused_sync.cuh."""
        return RULES[self.name]

    @property
    def num_slots(self) -> int:
        return len(_SLOTS[self.name])

    @property
    def slot_names(self) -> Tuple[str, ...]:
        """TF's slot suffixes: a slot of variable ``v`` is saved as ``v/<suffix>``."""
        return tuple(n for n, _ in _SLOTS[self.name])

    @property
    def slot_inits(self) -> Tuple[float, ...]:
        return tuple(v for _, v in _SLOTS[self.name])

    @property
    def hyper(self) -> Tuple[float, float, float]:
        return self.momentum, self.decay, self.eps

    # ---- state ----------------------------------------------------------------------------------------------------------
    def allocate_slots(self, allocate, numel: int) -> List[torch.Tensor]:
        """One fp32 arena per slot from ``allocate(numel)`` (``Backend.allocate``: symmetric memory on the fused backend),
        filled with the slot's initial value."""
        out = []
        for v in self.slot_inits:
            t = allocate(numel)
            t.fill_(v)
            out.append(t)
        return out

    def reset_slots(self, slots: Sequence[torch.Tensor]) -> None:
        for t, v in zip(slots, self.slot_inits):
            t.fill_(v)

    def slots_to_state_dict(self, spec, slots: Sequence[torch.Tensor]) -> Dict[str, torch.Tensor]:
        """``Variable_4/Momentum`` style checkpoint entries (TF layouts), empty for ``sgd``."""
        out: Dict[str, torch.Tensor] = {}
        for suffix, t in zip(self.slot_names, slots):
            for name, v in spec.to_state_dict(t).items():
                out["%s/%s" % (name, suffix)] = v
        return out

    def has_slots(self, spec, state: Dict[str, torch.Tensor]) -> bool:
        return all("%s/%s" % (n, s) in state for n in spec.ckpt_names() for s in self.slot_names)

    def slots_from_state_dict(self, spec, state: Dict[str, torch.Tensor]) -> List[torch.Tensor]:
        """Flat CPU arenas of the checkpointed slots; the padding between tensors holds the slot's initial value."""
        out = []
        for suffix, init in zip(self.slot_names, self.slot_inits):
            flat = torch.full((spec.arena_numel,), float(init), dtype=torch.float32)
            for p in spec.params:
                t = state["%s/%s" % (p.ckpt_name, suffix)]
                if tuple(t.shape) != tuple(p.shape):
                    raise ValueError("checkpoint slot %s/%s has shape %s, model wants %s"
                                     % (p.ckpt_name, suffix, tuple(t.shape), p.shape))
                flat[p.offset:p.offset + p.numel] = t.reshape(-1).to(torch.float32)
            out.append(flat)
        return out

    # ---- the update -----------------------------------------------------------------------------------------------------
    def apply(self, params: torch.Tensor, grad_sum: torch.Tensor, divisor: float, lr: float,
              slots: Sequence[torch.Tensor]) -> None:
        """In place, fp32: ``g = grad_sum / divisor`` then the rule.  For ``sgd`` the divisor is folded into the rate
        (``params -= (lr / divisor) * grad_sum``), exactly as the host backends did before state existed."""
        lr = float(lr)
        if self.name == "sgd":
            params.add_(grad_sum, alpha=-lr / divisor)
            return
        g = grad_sum * (1.0 / float(divisor))
        if self.name == "momentum":
            a, = slots
            a.mul_(self.momentum).add_(g)
            params.add_(a, alpha=-lr)
            return
        ms, mom = slots
        ms.add_((g * g - ms) * (1.0 - self.decay))
        mom.mul_(self.momentum).add_(g * lr / torch.sqrt(ms + self.eps))
        params.sub_(mom)


SGD = UpdateRule()


def rule_or_sgd(rule: Optional[UpdateRule]) -> UpdateRule:
    return SGD if rule is None else rule
