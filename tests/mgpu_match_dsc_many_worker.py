"""Worker of tests/test_multi_gpu_match_dsc_many.py: run under torchrun, one rank per GPU, NCCL.

Checks, on every rank, that parallel.match_dsc_many_sharded returns what pipeline.match_dsc_many returns on this rank's
GPU alone, bit for bit (torch.equal tables, np.array_equal clouds), on: the pair fixtures against several structures
(one without pairs), the C2 map against its six components (cc 0.65), a batch with fewer pairs than ranks, and one
without pairs.  Prints "MGPU-DSC-MANY-OK <world>" on rank 0."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [REPO, os.path.join(REPO, "oracle"), os.path.join(REPO, "tests")]


def main():
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    import dsc_cases as D
    import helpers as H
    from mad_b200 import pipeline as P
    from mad_b200 import parallel as par

    lo, hi = D.pair_tables(P)
    few = D.rows_of(P, lo, [3, 40, 41])
    none = P.FeatureTable(torch.zeros((4, 1024), dtype=torch.int16, device=dev), lo.meta_host[:4, 0], lo.meta_host[:4, 1],
                          lo.meta_host[:4, 2], lo.meta_host[:4, 3], lo.subv_host[:4])
    c2_lo, c2_his = D.c2_tables(P)
    cc = float(H.golden("pair_match")["cc"])
    cases = {"fixtures": (lo, [hi, none, few, hi], 4, cc), "dense": (lo, [few, hi], 6.5, 0.5), "c2": (c2_lo, c2_his, 4, 0.65),
             "few_pairs": (lo, [none, few], 4, 0.999), "no_pairs": (lo, [hi, few], 4, 1.0)}
    for name, (l, hs, dist_, c) in cases.items():
        ref = P.match_dsc_many(l, hs, dist_, c)
        got = par.match_dsc_many_sharded(l, hs, dist_, c)
        assert len(got) == len(ref) == len(hs)
        for (t, lc, hc), (rt, rl, rh) in zip(got, ref):
            assert torch.equal(t, rt) and np.array_equal(lc, rl) and np.array_equal(hc, rh), \
                "%s: sharded match_dsc_many differs from the 1-GPU result" % name
        n = sum(t.shape[0] for t, _, _ in ref)
        if name == "few_pairs":
            assert 0 < n < 8, "few_pairs: %d pairs" % n
        if name == "no_pairs":
            assert n == 0
    dist.barrier()
    if rank == 0:
        print("MGPU-DSC-MANY-OK %d" % world, flush=True)
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
