"""Worker of tests/test_multi_gpu_match_dsc.py: run under torchrun, one rank per GPU, NCCL.

Checks, on every rank, that parallel.match_dsc_sharded and parallel.match_dsc_lists_sharded return what
pipeline.match_dsc / match_dsc_lists return on this rank's GPU alone, bit for bit (torch.equal tables, np.array_equal
clouds), on: the reference pair fixture at its cc (0.6), the dense case (6.5 A, cc 0.5), one C2 component against the C2
map (cc 0.65), a case with fewer pairs than ranks, and one without pairs.  Prints "MGPU-DSC-OK <world>" on rank 0."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [REPO, os.path.join(REPO, "oracle"), os.path.join(REPO, "tests")]


def _features(P, t):
    """DensityFeature list of a FeatureTable (the call shape of MaD._match_dsc)."""
    from mad_b200.DensityFeature import DensityFeature
    d = t.set.dsc.cpu().numpy()
    out = []
    for i in range(t.set.rows):
        df = DensityFeature()
        df.set_detector_info(int(t.meta_host[i, 0]), int(t.meta_host[i, 1]), [0, 0, 0], None, t.subv_host[i], 0.0)
        df.main_bin, df.sec_bin, df.lin_ar_subeqsp = int(t.meta_host[i, 2]), int(t.meta_host[i, 3]), d[i]
        out.append(df)
    return out


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
    c2_lo, c2_his = D.c2_tables(P)
    cases = {"reference": (lo, hi, 4, float(H.golden("pair_match")["cc"])), "dense": (lo, hi, 6.5, 0.5),
             "c2_component": (c2_lo, c2_his[0], 4, 0.65), "few_pairs": (lo, D.rows_of(P, lo, [3, 40, 41]), 4, 0.999),
             "no_pairs": (lo, hi, 4, 1.0)}
    for name, (l, h, dist_, cc) in cases.items():
        ref, rlo, rhi = P.match_dsc(l, h, dist_, cc)
        got, glo, ghi = par.match_dsc_sharded(l, h, dist_, cc)
        assert torch.equal(got, ref) and np.array_equal(glo, rlo) and np.array_equal(ghi, rhi), \
            "%s: sharded match_dsc differs from the 1-GPU result" % name
        if name == "few_pairs":
            assert 0 < ref.shape[0] < 8, "few_pairs: %d pairs" % ref.shape[0]
        if name == "no_pairs":
            assert ref.shape[0] == 0
        if name in ("reference", "few_pairs", "no_pairs"):
            fl, fh = _features(P, l), _features(P, h)
            r1, l1, h1 = P.match_dsc_lists(fl, fh, dist_, cc)
            r2, l2, h2 = par.match_dsc_lists_sharded(fl, fh, dist_, cc)
            assert len(r1) == len(r2) and all(np.array_equal(a, b) for a, b in zip(r1, r2)) and np.array_equal(l1, l2) \
                and np.array_equal(h1, h2), "%s: match_dsc_lists_sharded differs from match_dsc_lists" % name
    dist.barrier()
    if rank == 0:
        print("MGPU-DSC-OK %d" % world, flush=True)
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
