"""Helper process for tests/test_optimizers.py: runs the real training driver on gloo with a stateful update rule and
records, for every aggregation call, this rank's gradient, its decision, the rate, and the weights and state after it."""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import numpy as np  # noqa: E402
import torch  # noqa: E402

from distributedmnist_b200 import data as mnist_data  # noqa: E402
from distributedmnist_b200.flags import FLAGS  # noqa: E402
from distributedmnist_b200.parallel import backends as B  # noqa: E402
from distributedmnist_b200.parallel.context import init_context, shutdown_context  # noqa: E402
from distributedmnist_b200.train import train  # noqa: E402


def main():
    out = sys.argv[1]
    FLAGS.parse(sys.argv[2:])
    torch.set_num_threads(1)
    ctx = init_context(FLAGS, want_gpu=False)
    rec = {"grads": [], "accepted": [], "mask": [], "count": [], "lr": [], "params": [], "slots": []}
    orig = B._CollectiveBackend.sync_step

    def spy(self, params, grads, lr, local_step, k, delay_s=0.0, rule=None, slots=()):
        g = grads.clone()
        info = orig(self, params, grads, lr, local_step, k, delay_s, rule=rule, slots=slots)
        rec["grads"].append(g.numpy())
        rec["accepted"].append(bool(info.accepted))
        rec["mask"].append(int(info.mask))
        rec["count"].append(int(info.count))
        rec["lr"].append(float(lr))
        rec["params"].append(params.numpy().copy())
        rec["slots"].append(np.stack([s.numpy().copy() for s in slots]))
        return info
    B._CollectiveBackend.sync_step = spy
    ds = mnist_data.load_mnist(FLAGS.data_dir, worker_id=ctx.rank, n_workers=ctx.world_size, seed=FLAGS.seed,
                               synthetic=True, synthetic_sizes=(512, 128))
    res = train(ctx, ds.train, ds.validation, FLAGS)
    init = res["engine"].spec.init_flat(FLAGS.seed).numpy()
    np.savez(out.replace("RANK", str(ctx.rank)), init=init, **{k: np.array(v) for k, v in rec.items()})
    shutdown_context(ctx)


if __name__ == "__main__":
    main()
