"""Worker of tests/test_weight_covariance.py::test_two_rank_full_covariance_equals_single_rank (torch.distributed.run, one rank per
GPU, NCCL): run_iteration(weight_covariance="full") on two ranks -- the exact-Hessian factor travels from the weight-space rank
with (omega_MAP, hess_diag) -- against the same iterations on one rank, cold and with an appended comparison set."""
import datetime
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from ppbo_b200 import iteration, synthetic  # noqa: E402


class _Single(iteration.Shard):
    def __init__(self):
        self.dist, self.group, self.rank, self.world = None, None, 0, 1


def _iterations(shard, prob, d, block, Q0, dev, shares=None):
    m, theta, kernel, S = prob["m"], prob["theta"], prob["kernel"], prob["S"]
    st = iteration.IterationState(kernel, theta, prob["D"], m, Q0 + 1, dev, d["W"], d["b"], shard=shard)
    cold, _, _ = iteration.run_iteration(d, kernel, theta, Q0, m, S, shard=shard, seed=11, state=st, shares=shares,
                                         weight_covariance="full")
    dw = {"block": block, "W": d["W"], "b": d["b"], "grids": d["grids"]}
    warm, _, _ = iteration.run_iteration(dw, kernel, theta, Q0 + 1, m, S, shard=shard, seed=11, state=st, shares=shares,
                                         weight_covariance="full")
    return cold.cpu().numpy(), warm.cpu().numpy()


def main():
    local = int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev, timeout=datetime.timedelta(seconds=90))
    shard = iteration.Shard()
    prob = synthetic.make_problem("levy10d", Q=13, S=4096, P=128, F=256)
    Q0 = 12
    n0 = Q0 * (prob["m"] + 1)
    d = iteration.IterationInputs(prob["X"][:n0], None, prob["W"], prob["b"], None, prob["grids"]).to_device(dev)
    block = torch.from_numpy(prob["X"][n0:]).to(dev)
    results = {tag: _iterations(shard, prob, d, block, Q0, dev, shares)
               for tag, shares in (("default", None), ("rank0_samples", [0.5] + [1.0] * (shard.world - 1)))}
    torch.cuda.synchronize()
    dist.barrier()
    if shard.rank == 0:
        ref = _iterations(_Single(), prob, d, block, Q0, dev)
        for tag, got in results.items():
            for name, g, r in zip(("cold", "warm"), got, ref):
                err = np.abs(g - r).max() / np.abs(r).max()
                assert err <= 1e-12, (tag, name, err)       # same maxima; the sums differ by the order of the partial sums only
                assert int(np.argmax(g[:, 0])) == int(np.argmax(r[:, 0])), (tag, name)
        print("MGPU_FULL_OK world=%d" % shard.world)
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
