"""Times MaD._match_dsc (pipeline.match_dsc; parallel.match_dsc_sharded under torchrun) at config C2 sizes.

    python scripts/time_match_dsc.py --out DIR                                  # one GPU
    torchrun --nproc-per-node 8 scripts/time_match_dsc.py --out DIR             # N GPUs

Inputs: the C2 map and its six components described on the device (synth.c2_inputs(0)); every component against the map
at cc 0.65 (MaD's default) and the stacked 43 643 component rows against the map at cc 0.6.  Per call, device events split
the time into threshold matching, anchor clouds (+ lo grid, including the one small read-back), counts (this rank's share
of the pairs), the all-gather of the counts (N > 1) and the row expansion; the median of --reps calls after --warmup calls.
Under torchrun every phase is the max over ranks, and every rank checks its sharded table against its own 1-GPU
match_dsc (torch.equal, clouds np.array_equal) inside the run.  Rank 0 writes DIR/match_dsc_n<N>.json with the card's
name and power limit (nvidia-smi --query-gpu, read only)."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch
import torch.distributed as dist

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [REPO, os.path.join(REPO, "oracle"), os.path.join(REPO, "tests")]

PHASES = ["threshold", "clouds", "counts", "gather", "rows"]


def _card(device):
    """Name, power limit and max SM clock of the card torch calls ``device``, found by its PCI address (the CUDA index
    and nvidia-smi's differ under CUDA_VISIBLE_DEVICES)."""
    pr = torch.cuda.get_device_properties(device)
    q = "pci.bus_id,name,power.limit,clocks.max.sm"
    r = subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader"], stdout=subprocess.PIPE,
                       stderr=subprocess.STDOUT, text=True)
    for line in r.stdout.splitlines():
        bus = line.split(",")[0].strip()                        # e.g. 00000000:1B:00.0 (domain:bus:device.function)
        try:
            dom, b, dv = bus.split(":")[0], bus.split(":")[1], bus.split(":")[2].split(".")[0]
            if (int(dom, 16), int(b, 16), int(dv, 16)) == (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id):
                return {"query": q, "value": line.strip()}
        except (IndexError, ValueError):
            continue
    return {"query": q, "value": None, "nvidia_smi": r.stdout.strip(), "pci": [pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id]}


def one_call(P, par, lo, hi, dist_, cc, rank, world):
    """(table, clouds, {phase: ms}, P, H, L) of one sharded match_dsc call (world 1: the 1-GPU path's pieces)."""
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(len(PHASES) + 1)]
    ev[0].record()
    pairs = P.match_threshold(hi.set, lo.set, cc)
    ev[1].record()
    m = P.DscMatch(lo, hi, dist_, cc, pairs=pairs)
    ev[2].record()
    if m.p == 0:
        raise SystemExit("no pairs at cc %g" % cc)
    local = par.match_dsc_local(m, rank, world)
    ev[3].record()
    counts = par.gather_pair_counts(local, m.p, hi.set.rows, lo.set.rows)
    ev[4].record()
    table = m.rows(counts)
    ev[5].record()
    torch.cuda.synchronize()
    ms = {ph: ev[i].elapsed_time(ev[i + 1]) for i, ph in enumerate(PHASES)}
    return table, m, ms


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--reps", type=int, default=5)
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
    cases = [("comp%d" % i, c, 0.65) for i, c in enumerate(comps)] + [("stacked", D.stack_tables(P, comps), 0.6)]
    out = {"world": world, "warmup": args.warmup, "reps": args.reps, "lo_rows": lo.set.rows, "anchor_dist_thresh": 4,
           "cases": []}
    for name, hi, cc in cases:
        ref, rlo, rhi = P.match_dsc(lo, hi, 4, cc)                        # this rank's 1-GPU result
        for _ in range(args.warmup):
            one_call(P, par, lo, hi, 4, cc, rank, world)
        runs = []
        for _ in range(args.reps):
            table, m, ms = one_call(P, par, lo, hi, 4, cc, rank, world)
            runs.append([ms[ph] for ph in PHASES] + [sum(ms.values())])
        equal = bool(torch.equal(table, ref) and np.array_equal(m.lo_cloud.host(), rlo) and np.array_equal(m.hi_cloud.host(), rhi))
        t = torch.tensor(runs, dtype=torch.float64, device=dev)
        ok = torch.tensor([1 if equal else 0], dtype=torch.int32, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)                     # per call and phase: the slowest rank
            dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        med = np.median(t.cpu().numpy(), axis=0)
        rec = {"case": name, "cc": cc, "hi_rows": hi.set.rows, "pairs": m.p, "H": m.hi_cloud.n, "L": m.lo_cloud.n,
               "grid_dims": [int(v) for v in m.lo_cloud.dims], "equal_to_1gpu": bool(ok.item()),
               "ms_median": {ph: round(float(v), 4) for ph, v in zip(PHASES + ["total"], med)},
               "ms_total_all_reps": [round(float(v), 4) for v in t[:, -1].tolist()]}
        out["cases"].append(rec)
        if rank == 0:
            print(json.dumps(rec), flush=True)
        assert rec["equal_to_1gpu"], "%s: the sharded result differs from the 1-GPU result" % name
    if rank == 0:
        out["card"] = _card(dev)
        out["cuda_visible_devices"] = os.environ.get("CUDA_VISIBLE_DEVICES")
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "match_dsc_n%d.json" % world), "w") as f:
            json.dump(out, f, indent=1)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
