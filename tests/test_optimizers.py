"""Momentum and RMSProp on the host paths (no GPU): the torch rule against float64 TF formulas, the flags, checkpoint slots,
two gloo replicas under K-of-N masks, and a restart of the training driver from a checkpoint that holds the state."""
import logging
import os

import numpy as np
import pytest
import torch

from distributedmnist_b200 import data as mnist_data
from distributedmnist_b200.checkpoint import Saver
from distributedmnist_b200.flags import FLAGS, FlagError
from distributedmnist_b200.models import get_model
from distributedmnist_b200.optim import SGD, UpdateRule
from distributedmnist_b200.parallel.context import init_context
from distributedmnist_b200.parallel.launcher import run_replicas
from distributedmnist_b200.train import train

from _optim_ref import RefState

HERE = os.path.dirname(os.path.abspath(__file__))
RULES = ["sgd", "momentum", "rmsprop"]


@pytest.fixture
def clean_flags():
    FLAGS.reset()
    saved = {k: os.environ.pop(k) for k in ("RANK", "WORLD_SIZE", "LOCAL_RANK") if k in os.environ}
    yield FLAGS
    FLAGS.reset()
    os.environ.update(saved)


# ---- 1. the torch rule against float64 TF formulas ----------------------------------------------------------------------
@pytest.mark.parametrize("name", RULES)
@pytest.mark.parametrize("divisor", [1, 3])
def test_torch_rule_matches_float64_tf_formulas(name, divisor):
    rule = UpdateRule(name, momentum=0.9, decay=0.9, eps=1.0)
    gen = torch.Generator().manual_seed(7)
    n = 4096
    w = torch.randn(n, generator=gen)
    slots = rule.allocate_slots(lambda k: torch.empty(k), n)
    ref = RefState(name, w.numpy())
    worst = 0.0
    for k in range(50):
        lr = 0.1 * 0.5 ** (k // 10)                                    # staircase
        scale = torch.exp(torch.randn(n, generator=gen) * 2)           # gradients over several decades
        gsum = torch.randn(n, generator=gen) * scale
        rule.apply(w, gsum, divisor, lr, slots)
        ref.step(gsum.numpy(), divisor, lr)
        worst = max(worst, ref.check(w.numpy(), [s.numpy() for s in slots], what="step %d" % k))
    assert worst > 0.0                        # the comparison is not vacuous (fp32 rounding is visible)
    if name != "sgd":
        assert not torch.equal(slots[0], torch.full_like(slots[0], rule.slot_inits[0]))


def test_sgd_rule_is_the_folded_rate_update():
    """``sgd`` is exactly what the host backends computed before state existed: params -= (lr / count) * sum."""
    gen = torch.Generator().manual_seed(3)
    w, g = torch.randn(1000, generator=gen), torch.randn(1000, generator=gen)
    want = w.clone().add_(g, alpha=-0.05 / 3)
    SGD.apply(w, g, 3, 0.05, ())
    assert torch.equal(w, want)


def test_rule_inventory():
    assert (SGD.num_slots, SGD.slot_names) == (0, ())
    m = UpdateRule("momentum")
    assert (m.code, m.slot_names, m.slot_inits) == (1, ("Momentum",), (0.0,))
    r = UpdateRule("rmsprop")
    assert (r.code, r.slot_names, r.slot_inits) == (2, ("RMSProp", "RMSProp_1"), (1.0, 0.0))


# ---- 2. flags -------------------------------------------------------------------------------------------------------------
def test_flag_defaults_are_the_reference_constants(clean_flags):
    FLAGS.parse([])
    assert (FLAGS.optimizer, FLAGS.momentum, FLAGS.rmsprop_decay, FLAGS.rmsprop_epsilon) == ("sgd", 0.9, 0.9, 1.0)
    assert UpdateRule.from_flags(FLAGS) == SGD
    FLAGS.parse(["--optimizer=rmsprop", "--momentum=0.5", "--rmsprop_decay", "0", "--rmsprop_epsilon=1e-10"])
    assert UpdateRule.from_flags(FLAGS) == UpdateRule("rmsprop", 0.5, 0.0, 1e-10)


@pytest.mark.parametrize("argv", [["--optimizer=adam"], ["--optimizer=Momentum"], ["--momentum=1"], ["--momentum=-0.1"],
                                  ["--rmsprop_decay=1.0"], ["--rmsprop_decay=-1e-3"], ["--rmsprop_epsilon=0"],
                                  ["--rmsprop_epsilon=-1"]])
def test_flags_reject_out_of_domain_values_at_parse_time(clean_flags, argv):
    with pytest.raises(FlagError):
        FLAGS.parse(argv)


# ---- 3. checkpoint slots --------------------------------------------------------------------------------------------------
def test_slot_names_round_trip_through_the_saver(tmp_path):
    spec, _ = get_model("lenet")
    rule = UpdateRule("rmsprop")
    gen = torch.Generator().manual_seed(5)
    slots = [torch.rand(spec.arena_numel, generator=gen) for _ in range(2)]
    state = spec.to_state_dict(spec.init_flat(1))
    state.update(rule.slots_to_state_dict(spec, slots))
    assert "Variable_4/RMSProp" in state and "Variable_7/RMSProp_1" in state
    assert len(state) == 3 * len(spec.params)
    Saver().save(str(tmp_path), state, 42)
    back, step = Saver.restore(Saver.latest(str(tmp_path)))
    assert step == 42 and set(back) == set(state)
    assert rule.has_slots(spec, back) and not UpdateRule("momentum").has_slots(spec, back)
    valid = spec.valid_mask()
    for t, flat in zip(slots, rule.slots_from_state_dict(spec, back)):
        assert torch.equal(flat[valid], t[valid])
    assert torch.all(rule.slots_from_state_dict(spec, back)[0][~valid] == 1.0)   # padding holds ms's initial value


def _train(tmp_path, *extra, steps=12, subdir="train"):
    FLAGS.reset()
    FLAGS.parse(["--train_dir=%s" % (tmp_path / subdir), "--batch_size=32", "--max_steps=%d" % steps, "--model=mlp2",
                 "--mlp_hidden=32", "--save_interval_secs=1000", "--initial_learning_rate=0.05", "--fake_data=true"]
                + list(extra))
    ctx = init_context(FLAGS, want_gpu=False)
    ds = mnist_data.load_mnist(FLAGS.data_dir, worker_id=0, n_workers=1, seed=FLAGS.seed, synthetic=True,
                               synthetic_sizes=(256, 64), fake_data=True)
    return train(ctx, ds.train, ds.validation, FLAGS)


def test_sgd_checkpoint_has_no_slot_keys_and_momentum_checkpoint_loads_in_the_evaluator(tmp_path, clean_flags):
    _train(tmp_path, steps=3, subdir="sgd")
    state, _ = Saver.restore(Saver.latest(str(tmp_path / "sgd")))
    assert sorted(state) == sorted(["Variable"] + ["Variable_%d" % i for i in range(1, 4)])
    res = _train(tmp_path, "--optimizer=momentum", steps=3, subdir="mom")
    state, _ = Saver.restore(Saver.latest(str(tmp_path / "mom")))
    assert sorted(k for k in state if "/" in k) == sorted("%s/Momentum" % k for k in state if "/" not in k)
    spec = res["engine"].spec
    flat = spec.from_state_dict(state)                # what the evaluator does (evaluator.py): extra keys are ignored
    assert torch.equal(flat[spec.valid_mask()], res["params"].detach().cpu()[spec.valid_mask()])


# ---- 4. two gloo replicas, K-of-N masks --------------------------------------------------------------------------------
def _run_gloo(tmp_path, extra, n=2, timeout=240):
    out = str(tmp_path / "out")
    argv = ["--model=mlp2", "--mlp_hidden=32", "--batch_size=16", "--backend=gloo", "--initial_learning_rate=0.05",
            "--save_interval_secs=1000", "--train_dir=%s" % (tmp_path / "train_dir"), "--num_epochs_per_decay=0.1",
            "--learning_rate_decay_factor=0.7"] + extra
    worker = os.path.join(HERE, "_optimizer_gloo_worker.py")
    codes = run_replicas(["-c", "import os,sys,runpy; sys.argv=[a.replace('RANK', os.environ['RANK']) for a in sys.argv[1:]];"
                          " runpy.run_path(sys.argv[0], run_name='__main__')", worker, str(tmp_path / "rec_RANK.npz")]
                         + argv, n, timeout=timeout, out_dir=out)
    logs = [open(os.path.join(out, f)).read() for f in sorted(os.listdir(out))]
    assert codes == [0] * n, "\n".join(l[-2000:] for l in logs)
    return [dict(np.load(tmp_path / ("rec_%d.npz" % r))) for r in range(n)]


@pytest.mark.parametrize("name", ["momentum", "rmsprop"])
@pytest.mark.parametrize("k_extra", [["--num_replicas_to_aggregate=2"],
                                     ["--num_replicas_to_aggregate=1", "--inject_straggler=1:1.0:30000"]],
                         ids=["k2", "k1_straggler"])
def test_gloo_replicas_hold_identical_weights_and_state_equal_to_a_float64_replay(tmp_path, name, k_extra):
    a, b = _run_gloo(tmp_path, ["--optimizer=%s" % name, "--max_steps=10"] + k_extra)
    steps = len(a["params"])
    assert steps == len(b["params"]) >= 10
    # bit-identical replicas after every step, weights and state
    assert np.array_equal(a["params"], b["params"]) and np.array_equal(a["slots"], b["slots"])
    assert list(a["mask"]) == list(b["mask"]) and list(a["count"]) == list(b["count"])
    if "--num_replicas_to_aggregate=1" in k_extra:
        assert all(m == 0b01 for m in a["mask"]) and a["accepted"].all() and not b["accepted"].any()
    else:
        assert all(m == 0b11 for m in a["mask"])
    assert len(set(a["lr"])) > 1                               # the staircase moved during the run
    # float64 serial replay of the committed masks
    ref = RefState(name, a["init"])
    for i in range(steps):
        gsum = sum(r["grads"][i].astype(np.float64) for r in (a, b) if r["accepted"][i])
        e_sum = 2 * 2.0 ** -23 * sum(np.abs(r["grads"][i].astype(np.float64)) for r in (a, b) if r["accepted"][i])
        ref.step(gsum, a["count"][i], a["lr"][i], e_sum)
        ref.check(a["params"][i], list(a["slots"][i]), what="step %d" % i)
    init = UpdateRule(name).slot_inits[0]
    assert not np.array_equal(a["slots"][-1][0], np.full_like(a["slots"][-1][0], init))


# ---- 5. restart of the driver from a checkpoint holding the state ----------------------------------------------------------
@pytest.mark.parametrize("name", ["momentum", "rmsprop"])
def test_restart_restores_the_state_and_continues_like_an_uninterrupted_run(tmp_path, clean_flags, caplog, name):
    """fake data: every batch is the same, so a run interrupted by a checkpoint + restart sees exactly the batches an
    uninterrupted run sees -- the two must end bit-identical, which they can only do if the state was restored."""
    whole = _train(tmp_path, "--optimizer=%s" % name, steps=10, subdir="whole")
    first = _train(tmp_path, "--optimizer=%s" % name, steps=5, subdir="split")
    saved, step = Saver.restore(Saver.latest(str(tmp_path / "split")))
    assert step == 6
    rule = UpdateRule(name)
    spec = first["engine"].spec
    valid = spec.valid_mask()
    with caplog.at_level(logging.INFO, logger="dmnist"):
        second = _train(tmp_path, "--optimizer=%s" % name, steps=10, subdir="split")
    assert any("Restored %s optimizer slots" % name in r.getMessage() for r in caplog.records)
    assert second["steps"][0] == 7 and second["final_step"] == whole["final_step"] == 11
    for flat, t in zip(rule.slots_from_state_dict(spec, saved), first["optimizer"].slots):
        assert torch.equal(flat[valid], t[valid])             # the checkpoint holds the state the first run ended with
    assert torch.equal(second["params"], whole["params"])
    for s2, sw in zip(second["optimizer"].slots, whole["optimizer"].slots):
        assert torch.equal(s2[valid], sw[valid])              # (arena padding is not checkpointed: it carries no gradient)


def test_restart_from_a_checkpoint_without_slots_starts_the_state_fresh_and_says_so(tmp_path, clean_flags, caplog):
    _train(tmp_path, steps=3, subdir="mixed")                                   # sgd checkpoint
    with caplog.at_level(logging.INFO, logger="dmnist"):
        res = _train(tmp_path, "--optimizer=momentum", steps=5, subdir="mixed")
    assert any("has no momentum optimizer slots" in r.getMessage() for r in caplog.records)
    assert res["steps"][0] == 5
    state, _ = Saver.restore(Saver.latest(str(tmp_path / "mixed")))
    assert "Variable_3/Momentum" in state
