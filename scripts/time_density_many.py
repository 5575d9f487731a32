"""Times PDB.density_many (and the stages behind it) against the per-structure calls it replaces.

    python scripts/time_density_many.py --out DIR          # writes DIR/density_many_n1.json

(a) C4 from atoms: 64 snapshots as synth.c4_snapshot draws them (the C1 walk plus N(0, 1.5 A) per atom), 4 A, 1 A per
    voxel, without fit_to_cube.  Forms: 64 x structure_to_density_device against one density_many; 64 x
    (structure_to_density_device + describe_struct) against density_many + describe_many.
(b) Refinement candidates: P = 8 and 32 rigid poses of one C2 component (synth.assembly_atoms with the C2 parameters),
    scored against that component's simulated map.  Forms: P x (structure_to_density_device + get_CCC_with_grid)
    against density_many + get_CCC_with_grids.
Both forms of a comparison get the same inputs, PDB objects, so both look every atom's mass up from its element record
(PDB._masses, a Python loop over the atoms) once per structure.  The same run times that lookup alone ("masses_only")
so that its share of each form is known, and times density_many given one shared mass array ("..._shared_masses": the
refine_poses hand-off, which skips the lookup by design; it is not compared with the per-structure form).
Each repetition runs the forms of a case in turn, rotating which goes first; a form's time is the host clock around it
up to a device synchronise (atoms start on the host, results stay on the device).  Reported: median, min and
max over --reps after --warmup, and the peak device memory of the batched form.  Inside the run, every batched map is
checked against the single path (one float32 ulp of its maximum; the single path splats with atomics) and every batched
score for equality against get_CCC_with_grid on the batch's own grids.  A separate profiled pass (per-kernel CUDA events
of the library, which slow the host) gives the device time per kernel of each form.  The card's name, power limit and
clocks are read (read only) in the same run."""
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


def _pdb(xyz):
    """A PDB object of carbon atoms at xyz (what the reader builds from a file)."""
    from mad_b200.PDB import PDB
    p = PDB.__new__(PDB)
    p.coords = np.ascontiguousarray(xyz, dtype=np.float64)
    p.info = [[i, "CA", "ALA", "A", i, "C", "ATOM"] for i in range(len(xyz))]
    return p


def _time(forms, warmup, reps):
    times = collections.defaultdict(list)
    names = list(forms)
    for i in range(warmup + reps):
        order = names[i % len(names):] + names[:i % len(names)]
        for f in order:
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            res = forms[f]()
            torch.cuda.synchronize()
            dt = (time.perf_counter() - t0) * 1e3
            del res
            if i >= warmup:
                times[f].append(dt)
    return {"ms_median": {f: round(float(np.median(v)), 3) for f, v in times.items()},
            "ms_min": {f: round(float(np.min(v)), 3) for f, v in times.items()},
            "ms_max": {f: round(float(np.max(v)), 3) for f, v in times.items()},
            "ms_all": {f: [round(x, 3) for x in v] for f, v in times.items()}}


def _profile(P, forms):
    out = {}
    for f, fn in forms.items():
        torch.cuda.synchronize()
        P.profile_enable(True)
        res = fn()
        torch.cuda.synchronize()
        recs = P.profile_records()
        P.profile_enable(False)
        del res
        acc, cnt = collections.defaultdict(float), collections.Counter()
        for n, ms in recs:
            acc[n] += ms
            cnt[n] += 1
        out[f] = {"device_ms": {k: round(v, 4) for k, v in sorted(acc.items(), key=lambda kv: -kv[1])},
                  "launches": dict(cnt), "total_device_ms": round(sum(acc.values()), 4), "n_launches": len(recs)}
    return out


def _peak(dev, fn):
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    torch.cuda.reset_peak_memory_stats(dev)
    before = torch.cuda.memory_allocated(dev)
    res = fn()
    torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated(dev) - before
    del res
    return int(peak)


def _maps_close(batch, singles):
    """Largest |batch - single| over the batch, in units of one float32 ulp of the maximum (1.0 after normalisation)."""
    worst = 0.0
    for g, (dens, dxi, dyi, dzi) in enumerate(singles):
        assert batch.grids[g].shape == dens.shape, g
        assert tuple(batch.origins[g]) == (dxi, dyi, dzi), g
        worst = max(worst, float((batch.grids[g] - dens).abs().max()) / float(np.spacing(np.float32(1.0))))
    return worst


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--reps", type=int, default=9)
    args = ap.parse_args()
    from mad_b200 import PDB as PD
    from mad_b200 import pipeline as P
    from mad_b200.Dmap import Dmap
    from mad_b200.math_utils import euler_rod_mat
    dev = torch.device("cuda", torch.cuda.current_device())
    out = {"warmup": args.warmup, "reps": args.reps, "cases": []}

    # (a) C4 from atoms
    base = synth.random_walk_atoms(9000, 85.0, 1)
    snaps = [base + np.random.default_rng(100 + i).normal(scale=1.5, size=base.shape) for i in range(synth.C4_MAPS)]
    pdbs = [_pdb(x) for x in snaps]
    carbon = np.full(len(base), 12.011)
    res, vs = 4.0, 1.0
    batch = PD.density_many(pdbs, res, vs)
    singles = [p.structure_to_density_device(res, vs) for p in pdbs]
    ulps = _maps_close(batch, singles)
    assert ulps <= 1.0, ulps
    del singles
    forms = {"serial_density": lambda: [p.structure_to_density_device(res, vs) for p in pdbs],
             "density_many": lambda: PD.density_many(pdbs, res, vs),
             "masses_only": lambda: [p._masses() for p in pdbs],
             "density_many_shared_masses": lambda: PD.density_many(snaps, res, vs, masses=carbon)}
    rec = {"case": "c4_from_atoms_density", "G": len(snaps), "atoms": len(base), "map_shape": list(batch.grids[0].shape),
           "max_abs_diff_vs_single_in_f32_ulps_of_max": ulps}
    rec.update(_time(forms, args.warmup, args.reps))
    rec["profiled"] = _profile(P, {f: forms[f] for f in ("serial_density", "density_many")})
    rec["density_many_peak_bytes"] = _peak(dev, forms["density_many"])
    out["cases"].append(rec)
    print(json.dumps({k: rec[k] for k in ("case", "G", "ms_median", "ms_min", "ms_max")}), flush=True)

    forms = {"serial_density_describe": lambda: [P.describe_struct(p.structure_to_density_device(res, vs)[0]) for p in pdbs],
             "density_many_describe_many": lambda: P.describe_many(PD.density_many(pdbs, res, vs).grids)}
    got = forms["density_many_describe_many"]()
    rec = {"case": "c4_from_atoms_density_describe", "G": len(snaps), "features": int(got.counts[:, 1].sum())}
    del got
    rec.update(_time(forms, args.warmup, args.reps))
    rec["profiled"] = _profile(P, forms)
    rec["batched_peak_bytes"] = _peak(dev, forms["density_many_describe_many"])
    out["cases"].append(rec)
    print(json.dumps({k: rec[k] for k in ("case", "G", "ms_median", "ms_min", "ms_max")}), flush=True)
    del batch

    # (b) refinement candidates of one C2 component
    cfg = synth.C2
    comp = synth.assembly_atoms(cfg["n"], cfg["voxelsp"], cfg["n_sub"], cfg["atoms_per_sub"], cfg["seed0"], cfg["box"])[0]
    grid, org = synth.simulate_density(comp, cfg["resolution"], cfg["voxelsp"])
    target = Dmap.from_array(np.asarray(grid, dtype=np.float32), cfg["voxelsp"], origin=tuple(float(x) for x in org))
    cen = comp.mean(0)
    cmass = np.full(len(comp), 12.011)
    rng = np.random.default_rng(7)
    res, vs = cfg["resolution"], cfg["voxelsp"]
    for n_poses in (8, 32):
        poses = [np.dot(comp - cen, euler_rod_mat(rng.normal(size=3), 0.05)) + cen + rng.normal(scale=1.0, size=3)
                 for _ in range(n_poses)]
        ppdbs = [_pdb(x) for x in poses]
        batch = PD.density_many(ppdbs, res, vs)
        ulps = _maps_close(batch, [p.structure_to_density_device(res, vs) for p in ppdbs])
        assert ulps <= 1.0, ulps
        scores = target.get_CCC_with_grids(batch.grids, batch.origins)
        one = np.array([target.get_CCC_with_grid(batch.grids[g], *batch.origins[g]) for g in range(n_poses)])
        assert np.array_equal(scores, one), (scores, one)

        def serial():
            out_ = []
            for p in ppdbs:
                dens, dxi, dyi, dzi = p.structure_to_density_device(res, vs)
                out_.append(target.get_CCC_with_grid(dens, dxi, dyi, dzi))
            return out_

        def batched():
            b = PD.density_many(ppdbs, res, vs)
            return target.get_CCC_with_grids(b.grids, b.origins)

        def batched_shared():
            b = PD.density_many(poses, res, vs, masses=cmass)
            return target.get_CCC_with_grids(b.grids, b.origins)
        forms = {"serial_density_score": serial, "density_many_scores": batched,
                 "masses_only": lambda: [p._masses() for p in ppdbs], "density_many_scores_shared_masses": batched_shared}
        rec = {"case": "refinement_candidates", "P": n_poses, "atoms": len(comp), "map_shape": list(batch.grids[0].shape),
               "max_abs_diff_vs_single_in_f32_ulps_of_max": ulps, "scores_equal_to_get_CCC_with_grid": True,
               "scores": [float(s) for s in scores]}
        del batch
        rec.update(_time(forms, args.warmup, args.reps))
        rec["profiled"] = _profile(P, {f: forms[f] for f in ("serial_density_score", "density_many_scores")})
        rec["batched_peak_bytes"] = _peak(dev, batched)
        out["cases"].append(rec)
        print(json.dumps({k: rec[k] for k in ("case", "P", "ms_median", "ms_min", "ms_max")}), flush=True)

    out["card"] = _card(dev)
    q = "name,power.limit,clocks.sm,clocks.mem,clocks.max.sm"
    out["clocks"] = {"query": q, "value": subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader"],
                                                         stdout=subprocess.PIPE, text=True).stdout.strip()}
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "density_many_n1.json"), "w") as f:
        json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
