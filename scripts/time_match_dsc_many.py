"""Times pipeline.match_dsc_many (parallel.match_dsc_many_sharded under torchrun) against one match_dsc call per
structure (parallel.match_dsc_sharded under torchrun), at config C2 sizes.

    python scripts/time_match_dsc_many.py --out DIR                                  # one GPU
    torchrun --nproc-per-node 8 scripts/time_match_dsc_many.py --out DIR             # N GPUs

Inputs: the C2 map and its six components described on the device (synth.c2_inputs(0)), matched at cc 0.65 (MaD's
default): the six components (G = 6), then the same six repeated four times (G = 24), so that the amortisation over G
shows.  Each repetition times both forms, alternating: "separate" = G match_dsc calls, the phases summed over the calls;
"batched" = one match_dsc_many call.  Device events split each call into threshold matching (for the batch: with the
stacking of the descriptor sets), anchor clouds + lo grids (with the small read-back), counts (this rank's share),
the all-gather of the counts (N > 1) and the rows; the median of --reps after --warmup, every phase the max over ranks.
Every batched result is checked against its own structure's match_dsc inside the run (torch.equal, clouds
np.array_equal).  Rank 0 writes DIR/match_dsc_many_n<N>.json with the card's name and power limit (read only)."""
import argparse
import json
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(HERE)
sys.path[:0] = [REPO, os.path.join(REPO, "oracle"), os.path.join(REPO, "tests"), HERE]

from time_match_dsc import PHASES, _card, one_call  # noqa: E402


def batched_call(P, par, lo, his, dist_, cc, rank, world):
    """(per-structure results, DscMatchMany, {phase: ms}) of one batched call (world 1: the 1-GPU path's pieces)."""
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(len(PHASES) + 1)]
    ev[0].record()
    pairs = P.match_threshold(P.stack_sets(his), lo.set, cc)
    ev[1].record()
    m = P.DscMatchMany(lo, his, dist_, cc, pairs=pairs)
    ev[2].record()
    if m.p == 0:
        raise SystemExit("no pairs at cc %g" % cc)
    bounds = par.shard_bounds_weighted(m.pair_off, m.hi_n, world)
    local = m.counts(*bounds[rank])
    ev[3].record()
    counts = par.gather_pair_counts(local, m.p, int(m.hi_row_off[-1]), lo.set.rows, bounds=bounds, n_structures=m.G)
    ev[4].record()
    table = m.rows(counts)
    ev[5].record()
    torch.cuda.synchronize()
    return m.results(table), m, {ph: ev[i].elapsed_time(ev[i + 1]) for i, ph in enumerate(PHASES)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--reps", type=int, default=7)
    args = ap.parse_args()
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank, local_rank = int(os.environ.get("RANK", "0")), int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    import dsc_cases as D
    from mad_b200 import pipeline as P
    from mad_b200 import parallel as par

    lo, comps = D.c2_tables(P)
    cc, dist_ = 0.65, 4
    out = {"world": world, "warmup": args.warmup, "reps": args.reps, "lo_rows": lo.set.rows, "anchor_dist_thresh": dist_,
           "cc": cc, "cases": []}
    for name, his in (("c2_six_components", comps), ("c2_six_components_x4", comps * 4)):
        refs = [P.match_dsc(lo, h, dist_, cc) for h in his]                  # this rank's 1-GPU per-structure results
        sep, bat, equal = [], [], True
        for i in range(args.warmup + args.reps):
            ms_sep = dict.fromkeys(PHASES, 0.0)
            for h in his:
                _, _, ms = one_call(P, par, lo, h, dist_, cc, rank, world)
                for ph in PHASES:
                    ms_sep[ph] += ms[ph]
            res, m, ms_bat = batched_call(P, par, lo, his, dist_, cc, rank, world)
            if i >= args.warmup:
                sep.append([ms_sep[ph] for ph in PHASES] + [sum(ms_sep.values())])
                bat.append([ms_bat[ph] for ph in PHASES] + [sum(ms_bat.values())])
        for (t, lc, hc), (rt, rl, rh) in zip(res, refs):
            equal = equal and bool(torch.equal(t, rt) and np.array_equal(lc, rl) and np.array_equal(hc, rh))
        t = torch.tensor([sep, bat], dtype=torch.float64, device=dev)
        ok = torch.tensor([1 if equal else 0], dtype=torch.int32, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)                     # per call and phase: the slowest rank
            dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        med = np.median(t.cpu().numpy(), axis=1)
        rec = {"case": name, "G": len(his), "pairs": m.p, "pairs_per_structure": np.diff(m.pair_off).tolist(),
               "H": m.hi_n.tolist(), "L": m.lo_clouds.n.tolist(), "lo_grid_cells_total": m.lo_clouds.cells,
               "lo_cloud_sort_keys": len(his) * lo.set.rows, "batched_equal_to_per_structure": bool(ok.item()),
               "ms_median_separate": {ph: round(float(v), 4) for ph, v in zip(PHASES + ["total"], med[0])},
               "ms_median_batched": {ph: round(float(v), 4) for ph, v in zip(PHASES + ["total"], med[1])},
               "ms_total_all_reps_separate": [round(float(v), 4) for v in t[0, :, -1].tolist()],
               "ms_total_all_reps_batched": [round(float(v), 4) for v in t[1, :, -1].tolist()]}
        out["cases"].append(rec)
        if rank == 0:
            print(json.dumps(rec), flush=True)
        assert rec["batched_equal_to_per_structure"], "%s: a batched result differs from its match_dsc call" % name
    if rank == 0:
        out["card"] = _card(dev)
        out["cuda_visible_devices"] = os.environ.get("CUDA_VISIBLE_DEVICES")
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "match_dsc_many_n%d.json" % world), "w") as f:
            json.dump(out, f, indent=1)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
