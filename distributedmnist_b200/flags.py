"""Flag system: a small absl/`tf.app.flags` work-alike.

The reference scatters `tf.app.flags.DEFINE_*` calls over three modules and
merges them into one global ``FLAGS`` by import side-effect
(reference: src/distributed_train.py:36-99, src/nn_eval.py:36-45,
src/sync_replicas_optimizer_modified/sync_replicas_optimizer_modified.py:38).
Here every flag lives in one registry with the *same names and defaults*, so
command lines written for the reference keep working, plus a small set of new
flags (model choice, synthetic data, straggler injection, backend selection)
that the single-box B200 design needs.

Accepted syntaxes (same as absl): ``--name=value``, ``--name value``,
``--flag`` / ``--noflag`` for booleans, and ``true/false/1/0/yes/no/t/f`` as
boolean values in any case.
"""
from __future__ import annotations

import sys
from dataclasses import dataclass
from typing import Any, Callable, Dict, List, Optional, Sequence

_TRUE = {"true", "t", "1", "yes", "y"}
_FALSE = {"false", "f", "0", "no", "n"}


class FlagError(ValueError):
    pass


@dataclass
class _Flag:
    name: str
    default: Any
    help: str
    kind: str  # 'boolean' | 'integer' | 'float' | 'string'
    value: Any = None
    present: bool = False  # set on the command line

    def parse(self, text: str) -> Any:
        if self.kind == "boolean":
            low = text.strip().lower()
            if low in _TRUE:
                return True
            if low in _FALSE:
                return False
            raise FlagError("flag --%s: %r is not a boolean" % (self.name, text))
        if self.kind == "integer":
            try:
                return int(text, 0) if isinstance(text, str) else int(text)
            except ValueError:
                raise FlagError("flag --%s: %r is not an integer" % (self.name, text))
        if self.kind == "float":
            try:
                return float(text)
            except ValueError:
                raise FlagError("flag --%s: %r is not a float" % (self.name, text))
        return str(text)


class FlagValues:
    """Registry + attribute access (``FLAGS.batch_size``)."""

    def __init__(self) -> None:
        object.__setattr__(self, "_flags", {})
        object.__setattr__(self, "_parsed", False)
        object.__setattr__(self, "_validators", [])

    # ---- definition -----------------------------------------------------
    def _define(self, kind: str, name: str, default: Any, help: str) -> None:
        flags: Dict[str, _Flag] = self._flags
        if name in flags:
            # Re-definition with identical spec is a no-op (modules may be
            # re-imported by the compat shims); anything else is a bug.
            old = flags[name]
            if old.kind != kind or old.default != default:
                raise FlagError("flag --%s defined twice with different specs" % name)
            return
        flags[name] = _Flag(name=name, default=default, help=help, kind=kind, value=default)

    def DEFINE_boolean(self, name: str, default: bool, help: str = "") -> None:
        self._define("boolean", name, default, help)

    DEFINE_bool = DEFINE_boolean

    def DEFINE_integer(self, name: str, default: int, help: str = "") -> None:
        self._define("integer", name, default, help)

    def DEFINE_float(self, name: str, default: float, help: str = "") -> None:
        self._define("float", name, default, help)

    def DEFINE_string(self, name: str, default: str, help: str = "") -> None:
        self._define("string", name, default, help)

    def register_validator(self, check: Callable[["FlagValues"], None]) -> None:
        """``check(flags)`` runs after every :meth:`parse`; a ``ValueError`` it raises becomes a :class:`FlagError`."""
        self._validators.append(check)

    # ---- access ---------------------------------------------------------
    def __getattr__(self, name: str) -> Any:
        flags = object.__getattribute__(self, "_flags")
        if name in flags:
            return flags[name].value
        raise AttributeError("unknown flag %r" % name)

    def __setattr__(self, name: str, value: Any) -> None:
        flags = self._flags
        if name not in flags:
            raise AttributeError("unknown flag %r" % name)
        f = flags[name]
        f.value = f.parse(value) if isinstance(value, str) and f.kind != "string" else value

    def __contains__(self, name: str) -> bool:
        return name in self._flags

    def is_present(self, name: str) -> bool:
        return self._flags[name].present

    def flag_values_dict(self) -> Dict[str, Any]:
        return {k: f.value for k, f in self._flags.items()}

    def defaults_dict(self) -> Dict[str, Any]:
        return {k: f.default for k, f in self._flags.items()}

    def reset(self) -> None:
        for f in self._flags.values():
            f.value = f.default
            f.present = False
        object.__setattr__(self, "_parsed", False)

    # ---- parsing --------------------------------------------------------
    def parse(self, argv: Optional[Sequence[str]] = None, known_only: bool = False) -> List[str]:
        """Parse ``argv`` (without the program name). Returns leftover positionals.

        Unknown ``--flags`` raise unless ``known_only`` (then they are returned).
        """
        flags: Dict[str, _Flag] = self._flags
        args = list(sys.argv[1:] if argv is None else argv)
        rest: List[str] = []
        i = 0
        while i < len(args):
            a = args[i]
            i += 1
            if a == "--":
                rest.extend(args[i:])
                break
            if not a.startswith("-") or a == "-":
                rest.append(a)
                continue
            body = a.lstrip("-")
            if "=" in body:
                name, text = body.split("=", 1)
                has_value = True
            else:
                name, text, has_value = body, "", False
            name = name.replace("-", "_")
            if name not in flags:
                if name.startswith("no") and name[2:] in flags and flags[name[2:]].kind == "boolean" and not has_value:
                    f = flags[name[2:]]
                    f.value, f.present = False, True
                    continue
                if known_only:
                    rest.append(a)
                    continue
                raise FlagError("unknown flag --%s" % name)
            f = flags[name]
            if not has_value:
                if f.kind == "boolean":
                    # `--flag` alone means true; `--flag false` is also accepted.
                    if i < len(args) and args[i].strip().lower() in (_TRUE | _FALSE):
                        text = args[i]
                        i += 1
                    else:
                        text = "true"
                else:
                    if i >= len(args):
                        raise FlagError("flag --%s needs a value" % name)
                    text = args[i]
                    i += 1
            # Strip one level of shell-style quotes that survive cfg templating
            # (the reference wraps host lists in single quotes, cfg/*:79-80).
            if len(text) >= 2 and text[0] == text[-1] and text[0] in "'\"":
                text = text[1:-1]
            f.value = f.parse(text)
            f.present = True
        for check in self._validators:
            try:
                check(self)
            except ValueError as e:
                raise FlagError(str(e)) from None
        object.__setattr__(self, "_parsed", True)
        return rest

    def usage(self) -> str:
        lines = []
        for name in sorted(self._flags):
            f = self._flags[name]
            lines.append("  --%s (%s, default %r)\n      %s" % (name, f.kind, f.default, f.help))
        return "\n".join(lines)


FLAGS = FlagValues()


def define_reference_flags(F: FlagValues = FLAGS) -> FlagValues:
    """Every flag of the reference, same name and default (SURVEY §2.2)."""
    # reference: src/distributed_train.py:36-39
    F.DEFINE_boolean("worker_times_cdf_method", False, "Track worker times cdf (full-barrier mode with timing capture)")
    F.DEFINE_boolean("interval_method", False, "Use the fixed wall-clock interval aggregation method")
    F.DEFINE_boolean("should_summarize", False, "Whether the chief should write summaries")
    F.DEFINE_boolean("timeline_logging", False, "Dump a chrome-trace timeline json per step")
    # reference: src/distributed_train.py:40-48
    F.DEFINE_string("job_name", "", 'One of "ps", "worker"')
    F.DEFINE_string("ps_hosts", "", "Comma-separated hostname:port list of parameter servers (accepted for "
                    "compatibility; the B200 engine has no parameter server)")
    F.DEFINE_string("worker_hosts", "", "Comma-separated hostname:port list of workers; its length is the "
                    "number of replicas when WORLD_SIZE is not set")
    # reference: src/distributed_train.py:50-63
    F.DEFINE_string("train_dir", "/tmp/imagenet_train", "Directory for checkpoints, timelines and .npy results")
    F.DEFINE_integer("rpc_port", 1235, "Port of the timing/ready control plane (rendezvous store port here)")
    F.DEFINE_integer("save_results_period", 1000, "Period (global steps) of saving worker<id>_time_acc.npy")
    F.DEFINE_integer("max_steps", 1000000, "Number of batches to run")
    F.DEFINE_boolean("drop_connect", False, "Multiply gradients by a Bernoulli mask before aggregation")
    F.DEFINE_integer("batch_size", 128, "Batch size per replica")
    F.DEFINE_string("subset", "train", 'Either "train" or "validation" (unused, kept for compatibility)')
    F.DEFINE_boolean("log_device_placement", False, "Log which device every kernel runs on")
    # reference: src/distributed_train.py:68-78
    F.DEFINE_integer("task_id", 0, "Replica index; replica 0 is the chief")
    F.DEFINE_integer("num_replicas_to_aggregate", -1, "Gradients to collect before updating (K of N); -1 = all")
    F.DEFINE_float("save_interval_secs", 20, "Checkpoint interval in seconds (chief); fractions allowed: a B200 step is ~0.1 ms")
    F.DEFINE_integer("save_summaries_secs", 300, "Summary interval in seconds (chief)")
    # reference: src/distributed_train.py:92-98
    F.DEFINE_float("initial_learning_rate", 0.1, "Initial learning rate")
    F.DEFINE_float("num_epochs_per_decay", 2.0, "Epochs after which the learning rate decays")
    F.DEFINE_float("learning_rate_decay_factor", 0.999, "Learning rate decay factor")
    F.DEFINE_float("drop_connect_probability", 0.9, "Keep probability of gradient drop-connect")
    # reference: sync_replicas_optimizer_modified.py:38
    F.DEFINE_integer("interval_ms", 1000, "Aggregation period of the interval method, milliseconds")
    # reference: src/nn_eval.py:36-45
    F.DEFINE_string("eval_dir", "/tmp/imagenet_eval", "Directory where the evaluator writes its event log")
    F.DEFINE_string("checkpoint_dir", "/tmp/imagenet_train", "Directory the evaluator polls for checkpoints")
    F.DEFINE_float("eval_interval_secs", 1, "How often the evaluator polls (seconds, fractions allowed)")
    F.DEFINE_boolean("run_once", False, "Evaluate once and exit")
    return F


def define_engine_flags(F: FlagValues = FLAGS) -> FlagValues:
    """New flags of the B200 engine (no analogue in the reference)."""
    F.DEFINE_string("model", "lenet", "lenet | mlp2 | mlp3")
    F.DEFINE_integer("mlp_hidden", 1024, "Hidden width of the MLP models")
    F.DEFINE_string("data_dir", "MNIST-data", "Directory with the four MNIST IDX .gz files (never downloaded)")
    F.DEFINE_boolean("synthetic_data", True, "Generate MNIST-shaped synthetic data when the IDX files are absent")
    F.DEFINE_boolean("fake_data", False, "Constant all-ones images / label 0 (reference mnist_data.py fake_data)")
    F.DEFINE_integer("seed", 66478, "Base RNG seed (per-replica streams are derived from it)")
    F.DEFINE_string("compute_dtype", "bf16", "bf16 | fp32 (activations / tensor-core operand type)")
    F.DEFINE_string("backend", "auto", "auto | fused (sm_100a kernels + symmetric memory) | nccl | gloo")
    F.DEFINE_string("inject_straggler", "", "rank:prob:usec[,rank:prob:usec...] device-side delay injection")
    F.DEFINE_integer("sync_timeout_ms", 30000, "Watchdog for device-side arrival polling")
    F.DEFINE_boolean("use_cuda_graph", True, "Capture the training step in a CUDA graph")
    F.DEFINE_boolean("use_nvls", True, "Use NVLS multimem reductions when the multicast object binds")
    F.DEFINE_boolean("debug_sync", False, "Dump the aggregation control block (arrival / done words, bitmap, commit ring) "
                                          "when a device-side watchdog fires (reference: the optimizer's debug Print ops)")
    F.DEFINE_boolean("pipeline_steps", True, "GPU path: enqueue step i+1 before reading step i's loss / status words "
                                             "(page-locked result buffers, background batch packer)")
    F.DEFINE_integer("log_every", 1, "Log every n-th local iteration (1 = reference behaviour)")
    F.DEFINE_float("dropout_keep_prob", 0.5, "Keep probability of the fc1 dropout (reference mnist.py:139)")
    # update rule of every aggregation path (distributedmnist_b200/optim.py); the defaults are the reference's otherwise
    # unused RMSProp constants (src/distributed_train.py:102-104)
    F.DEFINE_string("optimizer", "sgd", "sgd | momentum | rmsprop (TF 1.x ApplyGradientDescent / ApplyMomentum / ApplyRMSProp)")
    F.DEFINE_float("momentum", 0.9, "Momentum of --optimizer=momentum and of RMSProp's momentum term, in [0, 1)")
    F.DEFINE_float("rmsprop_decay", 0.9, "RMSProp decay of the mean square, in [0, 1)")
    F.DEFINE_float("rmsprop_epsilon", 1.0, "RMSProp epsilon, > 0")
    if _check_optimizer_flags not in F._validators:
        F.register_validator(_check_optimizer_flags)
    return F


def _check_optimizer_flags(F: FlagValues) -> None:
    from .optim import check_hyper
    check_hyper(F.optimizer, float(F.momentum), float(F.rmsprop_decay), float(F.rmsprop_epsilon))


define_reference_flags()
define_engine_flags()


def app_run(main: Callable[[List[str]], Any], argv: Optional[Sequence[str]] = None) -> None:
    """``tf.app.run`` work-alike: parse flags, call ``main(leftover_argv)``, exit."""
    args = list(sys.argv if argv is None else argv)
    if any(a in ("--help", "-h", "--helpfull") for a in args[1:]):
        print("flags:\n" + FLAGS.usage())
        sys.exit(0)
    rest = FLAGS.parse(args[1:])
    sys.exit(main([args[0]] + rest))
