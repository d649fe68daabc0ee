"""One rank of the multi-process check of the chain diagnostics (tests/test_chain_diagnostics_gpu.py::
test_two_ranks_agree_with_one_process).  Every rank runs on the GPU `--device` (two ranks may share one GPU, as in
fused_rank_worker.py), the process group is gloo: the fused run's all-reduce goes through the peer mailboxes, nested
R-hat's combination through torch.distributed.all_gather on CPU tensors."""
import argparse
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rank", type=int, required=True)
    ap.add_argument("--world", type=int, required=True)
    ap.add_argument("--port", type=int, required=True)
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("--out", required=True)
    ap.add_argument("--P", type=int, default=8192)
    ap.add_argument("--S", type=int, default=24)
    ap.add_argument("--M", type=int, default=4)
    a = ap.parse_args()
    import torch
    import torch.distributed as dist

    import physicsbasedbayesianinference_b200 as E
    from physicsbasedbayesianinference_b200.parallel import shard_range

    torch.cuda.set_device(a.device)
    dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{a.port}", rank=a.rank, world_size=a.world)
    KB = 1.380649e-23
    D, L = 10, 6
    lo, hi = shard_range(a.P, a.rank, a.world)
    ens = E.Ensemble(D, hi - lo, dtype=np.float32, device=f"cuda:{a.device}", seed=9, particleOffset=lo)
    ens.setPosition(2.0, superchainSize=a.M)  # Philox ids are global: the same starts as one process
    hmc = E.HMC(ens, L * 0.05 + 1e-9, 0.05, None, potential=E.FunnelPotential(D, 3.0), seed=9, bugCompat=False)
    r = hmc.run(a.S, 1 / KB, adapt=True, targetAccept=0.8, adaptIterations=a.S // 2, keepNumSteps=True, fused=True,
                group=dist.group.WORLD if a.world > 1 else None, adaptLag=2, chainDiagnostics=True,
                superchainSize=a.M)
    torch.cuda.synchronize()
    np.savez(a.out, rhat=r["rhat"].numpy(), rhatBetween=r["rhatBetween"].numpy(), rhatWithin=r["rhatWithin"].numpy(),
             chainMean=r["chainMean"].cpu().numpy(), chainVar=r["chainVar"].cpu().numpy(), lo=lo, hi=hi)
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
