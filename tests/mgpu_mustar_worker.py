"""Worker of tests/test_mustar_ascent.py::test_n_rank_incumbent_equals_single_rank (torch.distributed.run, one rank per GPU, NCCL):
run_iteration(incumbent=...) on several ranks, cold and appended, gives every rank the (mu*, x*) of a one-GPU run on the same
inputs, bit for bit (rank 0 runs the search and broadcasts it with mu*)."""
import datetime
import os
import sys

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from ppbo_b200 import iteration, synthetic  # noqa: E402


class _Single(iteration.Shard):
    def __init__(self):
        self.dist, self.group, self.rank, self.world = None, None, 0, 1


def _same_on_all_ranks(t):
    ref = t.clone()
    dist.broadcast(ref, src=0)
    return bool(torch.equal(ref, t))


def main():
    local = int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev, timeout=datetime.timedelta(seconds=90))
    shard = iteration.Shard()
    prob = synthetic.make_problem("levy10d", Q=13, S=4096, P=128, F=256)
    m, D, Qc = prob["m"], prob["D"], 10
    X = torch.from_numpy(prob["X"]).to(dev)
    W, b, grids = (torch.from_numpy(prob[k]).to(dev) for k in ("W", "b", "grids"))
    d0 = {"X": X[:Qc * (m + 1)], "W": W, "b": b, "grids": grids}
    d1 = {"block": X[Qc * (m + 1):], "W": W, "b": b, "grids": grids}
    states = {"many": iteration.IterationState(prob["kernel"], prob["theta"], D, m, prob["Q"], dev, W, b, shard=shard),
              "one": iteration.IterationState(prob["kernel"], prob["theta"], D, m, prob["Q"], dev, W, b, shard=_Single())}
    for d, Q in ((d0, Qc), (d1, prob["Q"])):
        inc = torch.full((D + 1,), float("nan"), dtype=torch.float64, device=dev)
        iteration.run_iteration(d, prob["kernel"], prob["theta"], Q, m, prob["S"], shard=shard, seed=11, state=states["many"],
                                incumbent=inc)
        one = torch.empty(D + 1, dtype=torch.float64, device=dev)
        iteration.run_iteration(d, prob["kernel"], prob["theta"], Q, m, prob["S"], shard=_Single(), seed=11, state=states["one"],
                                incumbent=one)
        assert _same_on_all_ranks(inc), (shard.rank, Q)
        assert torch.equal(inc, one), (shard.rank, Q, inc, one)
    torch.cuda.synchronize()
    dist.barrier()
    if shard.rank == 0:
        print("MGPU_MUSTAR_OK world=%d" % shard.world)
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
