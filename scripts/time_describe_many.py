"""Times pipeline.describe_many against the two ways of describing a batch of small maps that existed before it: G
describe_struct calls on one stream ("serial") and MapBatch(streams=4) (four host threads, one CUDA stream each).

    python scripts/time_describe_many.py --out DIR          # writes DIR/describe_many_n1.json

Inputs: the C4 snapshots (synth.c4_snapshot, 96^3), resident on the device before timing (no uploads, results stay on
the device), G = 8 and G = 64.  Each repetition runs the three forms in turn, rotating which one goes first; a form's
time is the host clock around the call up to a device synchronise.  Reported: the median, min and max over --reps after
--warmup.  A separate profiled pass (per-kernel CUDA events of the library, which slow the host) gives the device time
per stage of one serial pass and one describe_many call.  Every batched result is checked equal (torch.equal) to its
own describe_struct call inside the run, and the peak device memory of one describe_many call is recorded.  The card's
name, power limit and clocks are read (read only) in the same run, and scripts/res_usage.py's rows for the orientation /
description kernels and the batch kernels are kept."""
import argparse
import collections
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(HERE)
sys.path[:0] = [REPO, os.path.join(REPO, "oracle"), HERE]

import synth  # noqa: E402
from time_match_dsc import _card  # noqa: E402

STAGE = {"pad3d_kernel": "a1-a4 dense", "spline_up": "a1-a4 dense", "log_pass": "a1-a4 dense",
         "detect_": "a5-a6 detect", "gradient_m": "gradient tiles", "gradient_flags": "gradient tiles",
         "orient_kernel": "a7-a10 orient", "describe_kernel": "a11-a12 describe"}


def stage_of(name):
    for k, v in STAGE.items():
        if name.startswith(k):
            return v
    return "sort / compact / offsets"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--reps", type=int, default=9)
    args = ap.parse_args()
    from mad_b200 import pipeline as P
    dev = torch.device("cuda", torch.cuda.current_device())
    base = synth.random_walk_atoms(9000, 85.0, 1)
    maps = [torch.from_numpy(synth.c4_snapshot(i, base)).to(dev) for i in range(synth.C4_MAPS)]
    mb = P.MapBatch(streams=4)
    forms = {"serial": lambda gs: [P.describe_struct(g) for g in gs],
             "mapbatch4": lambda gs: mb.run(gs, download=False),
             "describe_many": lambda gs: P.describe_many(gs)}
    out = {"maps": "synth.c4_snapshot 0..G-1, 96^3 float32, device-resident", "warmup": args.warmup, "reps": args.reps,
           "cases": []}
    for G in (8, 64):
        gs = maps[:G]
        got = P.describe_many(gs)
        equal = True
        for g, grid in enumerate(gs):
            _, kp, ori, dsc = P.describe_struct(grid)
            equal &= bool(torch.equal(got.kp[g].table[:len(kp)], kp.table[:len(kp)]) and
                          torch.equal(got.ori[g].table[:len(ori)], ori.table[:len(ori)]) and torch.equal(got.dsc[g], dsc))
        assert equal, "G=%d: a batched result differs from its describe_struct call" % G
        del got
        times = collections.defaultdict(list)
        names = list(forms)
        for i in range(args.warmup + args.reps):
            order = names[i % 3:] + names[:i % 3]
            for f in order:
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                res = forms[f](gs)
                torch.cuda.synchronize()
                dt = (time.perf_counter() - t0) * 1e3
                del res
                if i >= args.warmup:
                    times[f].append(dt)
        stages = {}
        for f in ("serial", "describe_many"):
            P.profile_enable(True)
            forms[f](gs)
            torch.cuda.synchronize()
            acc = collections.defaultdict(float)
            recs = P.profile_records()
            P.profile_enable(False)
            for n, ms in recs:
                acc[stage_of(n)] += ms
            stages[f] = {k: round(v, 4) for k, v in sorted(acc.items())}
            stages[f]["launches"] = len(recs)
        torch.cuda.empty_cache()
        torch.cuda.reset_peak_memory_stats(dev)
        before = torch.cuda.memory_allocated(dev)
        got = P.describe_many(gs)
        torch.cuda.synchronize()
        peak = torch.cuda.max_memory_allocated(dev) - before
        rec = {"G": G, "features": int(got.counts[:, 1].sum()), "keypoints": int(got.counts[:, 0].sum()),
               "batched_equal_to_describe_struct": equal,
               "ms_median": {f: round(float(np.median(v)), 3) for f, v in times.items()},
               "ms_min": {f: round(float(np.min(v)), 3) for f, v in times.items()},
               "ms_max": {f: round(float(np.max(v)), 3) for f, v in times.items()},
               "ms_all": {f: [round(x, 3) for x in v] for f, v in times.items()},
               "device_ms_per_stage_profiled": stages,
               "describe_many_peak_bytes_above_inputs": int(peak)}
        del got
        out["cases"].append(rec)
        print(json.dumps({k: rec[k] for k in ("G", "ms_median", "ms_min", "ms_max", "describe_many_peak_bytes_above_inputs")}),
              flush=True)
    out["card"] = _card(dev)
    q = "name,power.limit,clocks.sm,clocks.mem,clocks.max.sm"
    out["clocks"] = {"query": q, "value": subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader"],
                                                         stdout=subprocess.PIPE, text=True).stdout.strip()}
    lib = os.path.join(REPO, "mad_b200", "libmad_b200.so")
    ru = subprocess.run([sys.executable, os.path.join(HERE, "res_usage.py"), lib], stdout=subprocess.PIPE, text=True).stdout
    out["res_usage"] = [ln for ln in ru.splitlines() if ln.split()[:1] != ["#"] and
                        any(k in ln for k in ("orient_kernel", "describe_kernel", "_many_kernel", "feature_meta_kernel",
                                              "cand_offsets_kernel"))]
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "describe_many_n1.json"), "w") as f:
        json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
