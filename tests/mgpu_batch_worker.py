"""Worker of tests/test_batch_queries.py::test_n_rank_batch_equals_single_rank (torch.distributed.run, one rank per GPU, NCCL):
greedy batch selection over sharded samples.  Injected dyadic maxima (exact sums in any order): every rank's picks equal the
one-rank picks on the whole sample set, rank 0 holding no samples in the default partition.  run_iteration(batch=q): the same
picks on every rank."""
import datetime
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from ppbo_b200 import iteration, synthetic  # noqa: E402
from test_batch_queries import batch_qei_greedy  # noqa: E402


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
    B, S, q = 37, 4099, 6
    f = np.random.RandomState(4).randint(-511, 512, (B, S)) / 8.0
    mustar = torch.tensor([0.25], dtype=torch.float64, device=dev)
    ref_idx, ref_qei = batch_qei_greedy(f, 0.25, q)
    for shares in (None, [0.5] + [1.0] * (shard.world - 1)):
        lo, hi = shard.sample_bounds(S, shares)
        fmax = torch.from_numpy(np.ascontiguousarray(f[:, lo:hi])).to(dev) if hi > lo else None
        idx, qei = iteration.select_batch(fmax, mustar, q, B, shard=shard)
        assert np.array_equal(idx.cpu().numpy(), ref_idx), (shard.rank, shares)
        assert np.array_equal(qei.cpu().numpy(), ref_qei), (shard.rank, shares)
    one_idx, one_qei = iteration.select_batch(torch.from_numpy(f).to(dev), mustar, q, B, shard=_Single())
    assert np.array_equal(one_idx.cpu().numpy(), ref_idx) and np.array_equal(one_qei.cpu().numpy(), ref_qei)

    prob = synthetic.make_problem("levy10d", Q=13, S=4096, P=128, F=256)
    d = iteration.IterationInputs(prob["X"], None, prob["W"], prob["b"], None, prob["grids"]).to_device(dev)
    for cov in ("diag", "full"):
        _, _, _, (idx, qei) = iteration.run_iteration(d, prob["kernel"], prob["theta"], prob["Q"], prob["m"], prob["S"], shard=shard,
                                                      seed=11, weight_covariance=cov, batch=4)
        assert _same_on_all_ranks(idx) and _same_on_all_ranks(qei), (shard.rank, cov)
        assert len(set(idx.cpu().numpy().tolist())) == 4
    torch.cuda.synchronize()
    dist.barrier()
    if shard.rank == 0:
        print("MGPU_BATCH_OK world=%d" % shard.world)
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
