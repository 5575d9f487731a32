#!/usr/bin/env python
"""bench.py -- throughput of the MaD local-feature hot path on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload all|c2|c4|c5]
                    [--dump-outputs DIR]

Headline (`value`, `e2e`, `roofline`): one *step* = one pass of the hot path over one synthetic map of BASELINE.json
configs[1] (C2): a 256^3 assembly map (8 A, 2 A/voxel, 6 random-walk components) through
    zero-pad -> 2x spline upsample + presmooth -> LoG/Gauss (both octaves) -> 3x3x3 maxima + Newton refinement
    -> gradient tiles around the keypoints -> EQSP orientations -> int16[1024] descriptors
    -> cosine matching (threshold 0.6) of all six components' descriptors against the map's
all in libmad_b200.so (hand-written sm_100a CUDA) through the C ABI.  `value` = input voxels (256^3 per map) per
second with the map resident in HBM; `e2e` = the same through the host-buffer API pipeline.MapStream (pinned host
grid in, host descriptor / keypoint / pair tables out, copies inside the timed region).  N > 1 (torchrun, one rank per
GPU): rank r describes its own C2 map, no data-path collective, "weak" scaling.

`sharded` (same JSON line, measured at EVERY N including 1 so that efficiencies can be computed from the per-N lines):
the two paths that shard (SURVEY.md 8e), total work fixed ("strong"):
  c5  all-pairs matching, 100 000 x 100 000 descriptors, top-8: lo axis cut into N shards, NCCL all_gather + merge;
  c4  64 conformational-snapshot maps of 96^3: map i -> rank i mod N, tables collected over NCCL (all-gather-v).
`verified` (N > 1): the N-GPU results are compared inside the run with the 1-GPU results of the same inputs.

`--impl reference` times the CPU restatement of the reference (oracle/mad_oracle.py, NumPy/SciPy -- the reference is
pure Python and not part of this repository) on a bounded, STAGE-WISE sample of the same C2 map,
one process per host core (see cpu_stage_sample).

`--dump-outputs DIR` (rank 0): after each workload's timed steps, what its last timed step returned goes to DIR/<name>.npy
(see OutputDump), so that two builds can be compared output for output on the same seeded inputs.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

REPO = os.path.dirname(os.path.abspath(__file__))
for _p in (REPO, os.path.join(REPO, "oracle")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import numpy as np  # noqa: E402

import synth  # noqa: E402  (oracle/synth.py: input generators only)

C2 = synth.C2
# sizes of the C2 workload (fixed by the seeds; pinned against the unmodified reference by tests/test_bench_parity.py)
C2_K, C2_D, C2_M = 7907, 40230, 43643
METRIC = "voxels/sec scale-space+detect+describe(+match)"
UNIT = "voxels/s"


def workload_name():
    return ("C2: 256^3 synthetic assembly map, 8 A, 2 A/voxel, 6 components x 40000 atoms; "
            "describe map + threshold-match each component's descriptors against it")


# ---------------------------------------------------------------------------------------------
# CPU side (oracle port of the reference) -- used by cpu_baseline and --impl reference only
# ---------------------------------------------------------------------------------------------
CPU_CROP = 80            # side of the sampled sub-volume (padded to 98^3 / upsampled to 195^3 by build_space)
CPU_KP = 48              # keypoints of the crop that go through orient
CPU_OF = 160             # oriented features of the crop that go through describe
CPU_MATCH = (1024, 4096)  # hi x lo block of the matching lines


CPU_PRESETS = {      # (crop side, keypoints, oriented features, hi rows of the matching block): ~12 / 6 / 3 s per step on 16 cores
    "full": (CPU_CROP, CPU_KP, CPU_OF, CPU_MATCH[0]), "half": (64, 24, 80, 512), "quarter": (48, 12, 40, 256)}


def _cpu_stage_worker(job):
    """One process: the five stages of the path on samples sized in the stage's own unit; returns seconds per unit."""
    crop, voxelsp, n_kp, n_of, n_hi = job
    import mad_oracle as mo
    pc = time.perf_counter
    t0 = pc()
    sp = mo.build_space(crop)
    t_build = pc() - t0
    v1 = int(np.prod(sp["grid_list"][1].shape))
    t0 = pc()
    kp = mo.detect(sp["map_space"], [voxelsp / 2, voxelsp], np.zeros(3))
    t_detect = pc() - t0
    nk = min(n_kp, len(kp["oct"]))
    kp_s = {k: v[:nk] for k, v in kp.items()}
    t0 = pc()
    ori, tab = mo.orient(sp["grad_list"], kp_s)
    t_orient = pc() - t0
    nf = min(n_of, len(ori["kp"]))
    ori_s = {k: v[:nf] for k, v in ori.items()}
    t0 = pc()
    dsc = mo.describe(sp["grad_list"], kp_s, ori_s, tab)
    t_describe = pc() - t0
    rng = np.random.default_rng(0)
    base = dsc if len(dsc) else np.ones((1, 1024), dtype=np.int16)
    hi = base[rng.integers(0, len(base), n_hi)]
    lo = base[rng.integers(0, len(base), CPU_MATCH[1])]
    t0 = pc()
    mo.match_threshold(hi, lo, 0.6)
    t_match = pc() - t0
    return dict(build_per_voxel=t_build / v1, detect_per_voxel=t_detect / v1, orient_per_kp=t_orient / max(nk, 1),
                describe_per_feature=t_describe / max(nf, 1), match_per_pair=t_match / (n_hi * CPU_MATCH[1]),
                crop_keypoints=int(len(kp["oct"])), seconds=t_build + t_detect + t_orient + t_describe + t_match)


def cpu_crops(grid, n_crops, side):
    """n_crops sub-cubes with occupancy closest to the whole map's (first = the most representative)."""
    occ = grid > 0.05
    target = float(occ.mean())
    cands = []
    step = side // 2
    for x in range(0, grid.shape[0] - side + 1, step):
        for y in range(0, grid.shape[1] - side + 1, step):
            for z in range(0, grid.shape[2] - side + 1, step):
                cands.append((abs(float(occ[x:x + side, y:y + side, z:z + side].mean()) - target), x, y, z))
    cands.sort()
    return [np.ascontiguousarray(grid[x:x + side, y:y + side, z:z + side]) for _, x, y, z in cands[:n_crops]]


def cpu_stage_sample(grid, voxelsp, procs, steps, warmup, v1_full, K=C2_K, D=C2_D, M=C2_M, n_vox=None, preset="full"):
    """The reference's CPU path on the C2 map, sampled STAGE BY STAGE in each stage's own unit and scaled to the whole map:
    build_space + find_anchors per padded base voxel (an 80^3 occupancy-matched crop), assign_orientations per keypoint
    (48 keypoints of the crop), generate_descriptors per oriented feature (160 of them), the two matching lines per scored
    pair (a 1024 x 4096 block).  T(map) = t_build V1 + t_detect V1 + t_orient K + t_describe D + t_match M D with the
    workload's V1 = 274^3, K = 7907, D = 40230, M = 43643 (pinned by tests/test_bench_parity.py).  Every step all `procs`
    processes run such a sample concurrently (one map per process is the reference's many-core form, SURVEY 8d), so
    memory-bandwidth contention between the processes is inside the measurement.
    Returns (voxels/s of `procs` maps in flight, seconds per step, per-unit costs of the last step)."""
    import multiprocessing as mp
    side, n_kp, n_of, n_hi = CPU_PRESETS[preset]
    crops = cpu_crops(grid, procs, side)
    while len(crops) < procs:
        crops.append(crops[len(crops) % max(len(crops), 1)])
    jobs = [(c, voxelsp, n_kp, n_of, n_hi) for c in crops]
    ctx = mp.get_context("fork")
    res = None
    with ctx.Pool(procs) as pool:
        for _ in range(warmup):
            pool.map(_cpu_stage_worker, jobs)
        t0 = time.perf_counter()
        for _ in range(steps):
            res = pool.map(_cpu_stage_worker, jobs)
        dt = (time.perf_counter() - t0) / max(steps, 1)
    unit = {k: float(np.mean([r[k] for r in res])) for k in res[0] if k != "seconds"}
    t_map = (unit["build_per_voxel"] * v1_full + unit["detect_per_voxel"] * v1_full + unit["orient_per_kp"] * K +
             unit["describe_per_feature"] * D + unit["match_per_pair"] * M * D)
    unit["seconds_per_map_one_process"] = t_map
    unit["stage_seconds_per_map"] = {"build_space": unit["build_per_voxel"] * v1_full, "find_anchors": unit["detect_per_voxel"] * v1_full,
                                     "assign_orientations": unit["orient_per_kp"] * K,
                                     "generate_descriptors": unit["describe_per_feature"] * D,
                                     "match": unit["match_per_pair"] * M * D}
    return procs * (n_vox if n_vox else C2["n"] ** 3) / t_map, dt, unit


def cpu_sample_text(preset="full"):
    side, n_kp, n_of, n_hi = CPU_PRESETS[preset]
    return ("stage-wise sample of the C2 map per process: build_space + find_anchors on an %d^3 occupancy-matched crop "
            "(scaled per padded base voxel), assign_orientations on %d keypoints, generate_descriptors on %d oriented "
            "features, the matching lines on a %d x %d block; scaled to the map's V1 = 274^3, K = %d, D = %d, M = %d; "
            "oracle/mad_oracle.py = vectorised NumPy/SciPy port, bit-exact with the reference on the fixtures and 1.5x "
            "faster than it (this map, one thread, build container: the reference 374 s, the port 253 s)"
            % (side, n_kp, n_of, n_hi, CPU_MATCH[1], C2_K, C2_D, C2_M))


CPU_SAMPLE_TEXT = cpu_sample_text("full")


def host_procs():
    return max(1, min(os.cpu_count() or 1, 32))


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    grid = synth.assembly_map(**C2)
    procs = host_procs()
    v1 = (C2["n"] + 18) ** 3
    # the sample shrinks with the number of steps so that the whole run stays near three minutes (per-unit costs do not
    # depend on the sample size, only their noise does)
    per_step = 170.0 / max(1, args.steps + args.warmup)
    preset = "full" if per_step >= 12.0 else ("half" if per_step >= 6.0 else "quarter")
    value, s_per_step, unit = cpu_stage_sample(grid, C2["voxelsp"], procs, args.steps, args.warmup, v1, preset=preset)
    unit["sample_preset"] = preset
    sample_text = cpu_sample_text(preset)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": s_per_step * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32 grids, f64 line accumulation (SciPy)",
        "data": "synthetic", "config": {"workload": workload_name(), "sample": sample_text},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": procs, "kind": "port", "sample": sample_text,
                         "per_unit_seconds": unit},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ---------------------------------------------------------------------------------------------
# clocks sampler (nvidia-smi during the timed region)
# ---------------------------------------------------------------------------------------------
class ClockSampler(object):
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows = []
        self.proc = None
        self.index = index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.rows.append((time.perf_counter(), ln.strip()))

    def stop(self):
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except Exception:
                self.proc.kill()

    def summary(self, t0, t1):
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for t, ln in self.rows:
            if t < t0 or t > t1 + 0.15:
                continue
            f = [x.strip() for x in ln.split(",")]
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except Exception:
                continue
            for nm, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                "samples": len(sm)}


# ---------------------------------------------------------------------------------------------
# shared plumbing
# ---------------------------------------------------------------------------------------------
class Ctx(object):
    """Process-group / device context of one rank."""

    def __init__(self):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        if self.world > 1:
            # NCCL's log (NCCL_DEBUG is left to the caller) goes to a file or stderr, never to stdout: rank 0 prints ONE JSON line
            os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
            dist.init_process_group("nccl", device_id=self.dev)
        peaks = {}
        pk_path = os.path.join(REPO, "MEASURED_PEAKS.json")
        if os.path.exists(pk_path):
            peaks = json.load(open(pk_path))
        self.hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
        self.hbm_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback (B200_PROFILING.md 6.65 TB/s)"
        # uint8 x uint8 -> int32 tcgen05.mma.kind::i8: measured issue-bound rate of this part (scripts/ubench/i8_mma_rate.cu,
        # profiles/r02_i8_mma_rate.json) when present, else the nominal dense 8-bit figure of the B200 (4.5 POP/s)
        self.i8_peak, self.i8_src = 4500.0, "nominal dense 8-bit rate of the B200 (4.5 POP/s)"
        p = os.path.join(REPO, "profiles", "r02_i8_mma_rate.json")
        if os.path.exists(p):
            try:
                self.i8_peak = float(json.load(open(p))["tops"])
                self.i8_src = "measured tcgen05.mma.kind::i8 issue rate (profiles/r02_i8_mma_rate.json)"
            except Exception:
                pass
        self.traffic = {}
        tr_path = os.path.join(REPO, "profiles", "ncu_traffic.json")
        if os.path.exists(tr_path):
            self.traffic = json.load(open(tr_path))

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, *vals):
        if self.world == 1:
            return [float(v) for v in vals]
        t = self.torch.tensor(list(vals), dtype=self.torch.float64, device=self.dev)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return [float(x) for x in t]

    def all_true(self, flag):
        if self.world == 1:
            return bool(flag)
        t = self.torch.tensor([1 if flag else 0], dtype=self.torch.int32, device=self.dev)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MIN)
        return bool(int(t[0]))


def timed(ctx, fn, steps):
    """K calls of fn between barrier + synchronize on both sides, CUDA events on the current stream -> (ms, what the
    last call returned).  Only the last call's result is held, so every earlier step frees its outputs as before."""
    torch = ctx.torch
    ctx.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps - 1):
        fn()
    last = fn()
    e1.record()
    ctx.barrier()
    return e0.elapsed_time(e1), last


class OutputDump(object):
    """--dump-outputs DIR: arrays a caller of a timed path receives, as DIR/<name>.npy.  Integer and float32 fields are
    stored as float32 (exact: every index and count here is below 2^24), float64 scores as float64.  Tables too large
    for the 64 MB budget are stored as a fixed, seeded sample of rows (``rows``), identical from run to run."""
    LIMIT = 64 * 10 ** 6

    def __init__(self, path):
        self.path = path
        self.nbytes = 0
        os.makedirs(path, exist_ok=True)

    @staticmethod
    def rows(n, k, seed):
        """k of n row positions (all when n <= k) in ascending order, fixed by the seed."""
        if n <= k:
            return np.arange(n)
        return np.sort(np.random.default_rng(seed).choice(n, size=k, replace=False))

    def put(self, name, a, dtype=np.float32):
        a = np.ascontiguousarray(a, dtype=dtype)
        self.nbytes += a.nbytes
        if self.nbytes > self.LIMIT:
            raise RuntimeError("--dump-outputs: %s takes the dump past %d bytes" % (name, self.LIMIT))
        np.save(os.path.join(self.path, name + ".npy"), a)

    def sample(self, t, k, seed):
        """A seeded sample of k rows of the device tensor t (its first axis)."""
        import torch
        return t[torch.from_numpy(self.rows(int(t.shape[0]), k, seed)).to(t.device)]

    def put_rows(self, name, t, k, seed, dtype=np.float32):
        self.put(name, self.sample(t, k, seed).cpu().numpy(), dtype)

    def put_keypoints(self, name, table):
        """MadKeypoint rows (int32 [K, 12] on the device): vox[3], oct, off[3], val, peak[3], accepted."""
        a = table.cpu().numpy()
        out = a.astype(np.float32)
        out[:, 4:8] = a[:, 4:8].view(np.float32)
        self.put(name, out)

    def put_oriented(self, name, table):
        """MadOriented rows (int32 [D, 2] on the device) as (keypoint, main bin, secondary bin)."""
        from mad_b200._lib import ORIENTED_DTYPE
        a = np.ascontiguousarray(table.cpu().numpy()).view(ORIENTED_DTYPE).reshape(-1)
        self.put(name, np.stack([a["kp"], a["main"], a["sec"]], 1))


# ---------------------------------------------------------------------------------------------
# C2: the headline
# ---------------------------------------------------------------------------------------------
def c2_stages(V0, V1, K, D):
    """stage -> (kernels, SURVEY 8(d) algorithmic bytes): every logical array read once / written once in float32."""
    VV = V0 + V1
    return {
        "upsample+presmooth": (("pad3d_kernel", "spline_up_z_kernel", "spline_up_x_kernel", "spline_up_y_kernel"), 4 * V1 + 4 * V0),
        "LoG+Gauss": (("log_pass_x_kernel", "log_pass_y_kernel", "log_pass_z_kernel", "log_pass_yz_kernel"), 12 * VV),
        "gradient": (("gradient_kernel", "gradient_masked_kernel", "gradient_mark_kernel", "gradient_flags_done_kernel"), 16 * VV),
        "detect": (("detect_peaks_kernel", "detect_refine_kernel", "cub_merge_sort_pairs", "build_keys_kernel", "scatter_kernel",
                    "flags_kernel"), 4 * VV),
        "orient": (("orient_kernel", "compact_oriented_kernel", "cub_exclusive_sum"), 58956 * K),
        "describe": (("describe_kernel",), 51200 * D),
    }


def dump_c2(dump, sp, kp, ori, dsc, pairs):
    """One C2 step: the counts (keypoints, oriented features, pairs), the keypoint and oriented-feature tables, and seeded
    samples of the descriptor rows, of the pair list (hi row, lo row, score) and of both octaves' LoG grids."""
    ph, pl, sc = pairs
    dump.put("c2_counts", [len(kp), len(ori), int(ph.numel())], np.float64)
    dump.put_keypoints("c2_keypoints", kp.table[:len(kp)])
    dump.put_oriented("c2_oriented", ori.table[:len(ori)])
    dump.put_rows("c2_descriptors", dsc, 2048, 1)
    dump.put_rows("c2_pair_hi", ph, 1 << 19, 2)
    dump.put_rows("c2_pair_lo", pl, 1 << 19, 2)
    dump.put_rows("c2_pair_score", sc, 1 << 19, 2, np.float64)
    for o in range(2):
        dump.put_rows("c2_log%d" % o, sp.logs[o].reshape(-1), 1 << 19, 3 + o)


def bench_c2(ctx, args):
    torch = ctx.torch
    from mad_b200 import pipeline as P
    dev = ctx.dev
    grid_h, comps_h = synth.c2_inputs(ctx.rank)
    n_vox = int(grid_h.size)
    grid_pin = torch.from_numpy(grid_h).pin_memory()
    grid_d = grid_pin.to(dev)
    exact = bool(args.exact)

    # component descriptor sets: resident in HBM before the timed region (MaD caches them: dsc_db/).  All components are
    # stacked into ONE hi set, so one matching launch per step serves the six subunits.
    comp_sets = []
    for c in comps_h:
        _, _, _, dsc = P.describe_struct(c, exact_f64=exact)
        comp_sets.append(P.DescriptorSet(dsc))
    hi_all, comp_offs = P.concat_sets(comp_sets)
    torch.cuda.synchronize()

    def step_device():
        sp, kp, ori, dsc = P.describe_struct(grid_d, exact_f64=exact)
        lo = P.DescriptorSet(dsc)
        pairs = P.match_threshold(hi_all, lo, 0.6, impl=args.match_impl)
        return sp, kp, ori, dsc, pairs

    # e2e uses the compact wire format (uint8 descriptors, (hi, lo, exact dot) pairs + norms; the host widens / recomputes
    # the float64 scores bit for bit: tests/test_gpu_parity.py::test_map_stream_compact_format)
    stream_api = P.MapStream(hi=hi_all, cc=0.6, exact_f64=exact, match_impl=args.match_impl, compact=not args.full_format)

    def run_e2e(n_steps):
        prev, out = None, None
        nxt = stream_api.upload(grid_pin)
        for s_i in range(n_steps):
            cur = nxt
            nxt = stream_api.upload(grid_pin) if s_i + 1 < n_steps else None
            ticket = stream_api.submit(cur)
            if prev is not None:
                out = stream_api.result(prev)
            prev = ticket
        out = stream_api.result(prev)
        return out

    for _ in range(args.warmup):
        res = step_device()
    sp, kp, ori, dsc, pairs = res
    K, D = len(kp), len(ori)
    n_pairs = int(pairs[0].numel())
    dims = sp.dims
    V0 = dims[0][0] * dims[0][1] * dims[0][2]
    V1 = dims[1][0] * dims[1][1] * dims[1][2]
    grad_frac = [float((f == 2).float().mean().item()) if f is not None else 1.0 for f in sp.grad_flags]
    del res, sp, kp, ori, dsc, pairs

    sampler = ClockSampler(ctx.local)
    if ctx.rank == 0:
        sampler.start()
        time.sleep(0.3)

    # ---- timed region: K steps, device-resident input
    P.profile_enable(True)
    l0 = P.launch_count()
    t_wall0 = time.perf_counter()
    ms, last = timed(ctx, step_device, args.steps)
    t_wall1 = time.perf_counter()
    launches = P.launch_count() - l0
    recs = P.profile_records()
    P.profile_enable(False)
    if args.dump is not None:
        dump_c2(args.dump, *last)
    del last

    # ---- e2e: host buffers in and out
    out = run_e2e(2)
    d2h = int(sum(t.numel() * t.element_size() for t in out.values()))
    d2h_detail = {k: int(t.numel() * t.element_size()) for k, t in out.items()}
    ms_e2e, _ = timed(ctx, lambda: run_e2e(args.steps), 1)
    clocks = sampler.summary(t_wall0, t_wall1) if ctx.rank == 0 else None
    if ctx.rank == 0:
        sampler.stop()
    ms, ms_e2e = ctx.max_over_ranks(ms, ms_e2e)
    if ctx.rank != 0:
        return None

    by_name = {}
    for nm, t in recs:
        by_name.setdefault(nm, []).append(t)
    total_kernel_ms = sum(sum(v) for v in by_name.values())
    kernels = sorted(((nm, sum(v), len(v)) for nm, v in by_name.items()), key=lambda x: -x[1])
    per_step = {nm: t / args.steps for nm, t, _ in kernels}

    # ---- stages with the SURVEY 8(d) byte convention; roofline = the stage with the largest share of the step
    stages = c2_stages(V0, V1, K, D)
    per_stage = {}
    for name, (kns, nbytes) in stages.items():
        t_ms = sum(per_step.get(k, 0.0) for k in kns)
        if t_ms <= 0:
            continue
        gbs = nbytes / (t_ms * 1e-3) / 1e9
        top = max(kns, key=lambda k: per_step.get(k, 0.0))
        tr = ctx.traffic.get(top)
        per_stage[name] = {"ms": round(t_ms, 4), "algorithmic_bytes": int(nbytes), "achieved": round(gbs, 1), "unit": "GB/s",
                           "frac": round(gbs / ctx.hbm_peak, 4), "dominant_kernel": top, "traffic": tr,
                           # the dominant kernel's OWN DRAM bytes (ncu) over its own time: how close it runs to the memory system
                           "own_traffic_frac": round(tr / (per_step[top] * 1e-3) / 1e9 / ctx.hbm_peak, 4) if tr and per_step.get(top) else None}
    M_hi = hi_all.rows
    match_kernels = [k for k in per_step if "match" in k or "pairs" in k or k in ("cub_radix_sort_pairs", "dsc_prepare_kernel",
                                                                                  "publish_small_kernel", "zero_u64_kernel")]
    match_ms = sum(per_step[k] for k in match_kernels)
    describe_ms = total_kernel_ms / args.steps - match_ms
    mk = per_step.get("match_u8_pairs_kernel")
    ops = 2.0 * M_hi * D * 1024
    matching = None
    if mk:
        matching = {"bound": "tensor", "kernel": "match_u8_pairs_kernel", "ops_per_launch": ops, "avg_launch_ms": mk,
                    "achieved": ops / (mk * 1e-3) / 1e12, "peak": ctx.i8_peak, "unit": "TOP/s",
                    "frac": ops / (mk * 1e-3) / 1e12 / ctx.i8_peak, "peak_source": ctx.i8_src,
                    "stage_ms_incl_sort_and_finish": match_ms, "pairs_found": n_pairs,
                    "traffic": ctx.traffic.get("match_u8_pairs_kernel")}
    dom = max(per_stage, key=lambda s: per_stage[s]["ms"])
    ds = per_stage[dom]
    n_l = {nm: n // args.steps for nm, _, n in kernels}
    roofline = {"bound": "hbm", "stage": dom, "kernel": ds["dominant_kernel"], "achieved": ds["achieved"], "peak": ctx.hbm_peak,
                "unit": "GB/s", "frac": ds["frac"], "traffic": ds["traffic"], "peak_source": ctx.hbm_src,
                "algorithmic_bytes_per_step": ds["algorithmic_bytes"], "ms_per_step": ds["ms"],
                "launches_per_step": int(sum(n_l.get(k, 0) for k in stages[dom][0])),
                "avg_launch_ms": per_step.get(ds["dominant_kernel"], 0.0) / max(1, n_l.get(ds["dominant_kernel"], 1)),
                "share_of_kernel_time": ds["ms"] / (total_kernel_ms / args.steps),
                "note": "SURVEY 8(d) convention: the stage's logical arrays read once / written once in f32 over ALL launches of "
                        "the stage; `traffic` = ncu dram bytes of the stage's dominant kernel (profiles/ncu_traffic.json)"}
    if dom == "LoG+Gauss" and exact:
        # SciPy's float64 line accumulation: 26 (X) + 43 (Y, computed for 128 columns per 112 kept) + 60 (Z) FP64 operations
        # per voxel against the measured DFMA / DADD / DMUL issue rate (scripts/ubench/fp64_rate.cu: 18.3 T lane-ops/s)
        opsv = (26.0 + 43.0 * 128.0 / 112.0 + 60.0) * (V0 + V1)
        roofline["fp64_issue"] = {"lane_ops_per_voxel": round(opsv / (V0 + V1), 1), "achieved": opsv / (ds["ms"] * 1e-3) / 1e12,
                                  "peak": 18.3, "unit": "T lane-ops/s", "frac": opsv / (ds["ms"] * 1e-3) / 1e12 / 18.3}
    map_bytes = 36 * (V0 + V1) + 58956 * K + 51200 * D
    step_ms = ms / args.steps
    line = {
        "metric": METRIC, "value": ctx.world * n_vox / (step_ms * 1e-3), "unit": UNIT, "n_gpus": ctx.world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": step_ms, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32 grids, f64 line accumulation, u8 x u8 -> s32 matching" if exact else "f32",
        "data": "synthetic",
        "config": {"workload": workload_name(), "grids": {"up": list(dims[0]), "base": list(dims[1])},
                   "keypoints": K, "oriented_features": D, "component_descriptors": M_hi, "pairs": n_pairs,
                   "parallelism": "1 map per GPU, no collective (sharded paths: see `sharded`)" if ctx.world > 1 else "1 GPU",
                   "l2": "no explicit flush: per-step working set %.1f GB >> 126 MB L2" % (28.0 * (V0 + V1) / 1e9),
                   "exact_f64": exact, "gradient_tiles_computed": {"up": round(grad_frac[0], 4), "base": round(grad_frac[1], 4)}},
        "e2e": {"value": ctx.world * n_vox / (ms_e2e / args.steps * 1e-3), "unit": UNIT,
                "h2d_bytes_per_step": int(grid_pin.numel() * 4), "d2h_bytes_per_step": d2h, "d2h_detail": d2h_detail,
                "d2h_format": "full (int16 descriptors, float64 scores)" if args.full_format else
                              "compact (uint8 descriptors; pairs as per-hi-row counts + lo index + int32 dot, + int32 squared norms; indices / scores rebuilt on the host bit for bit)",
                "ms_per_step": ms_e2e / args.steps},
        "gpu_launches": int(launches),
        "clocks": clocks,
        "roofline": roofline,
        "path_roofline": {"algorithmic_bytes_per_map": map_bytes, "describe_kernels_ms": describe_ms,
                          "achieved": map_bytes / (describe_ms * 1e-3) / 1e9, "peak": ctx.hbm_peak, "unit": "GB/s",
                          "frac": map_bytes / (describe_ms * 1e-3) / 1e9 / ctx.hbm_peak,
                          "note": "HEADLINE roofline fraction: all of a1-a12 against SURVEY 8(d)'s 36 (V0+V1) + 58956 K + 51200 D bytes"},
        "per_stage": per_stage,
        "matching": matching,
        "describe_voxels_per_s": ctx.world * n_vox / (describe_ms * 1e-3),
        "matches_per_s": ctx.world * M_hi * D / (match_ms * 1e-3 + 1e-12),
        "kernels_ms_per_step": {nm: round(t, 4) for nm, t in per_step.items()},
    }
    if not args.no_cpu_baseline and ctx.world == 1:
        procs = host_procs()
        v, s_per, unit = cpu_stage_sample(grid_h, C2["voxelsp"], procs, 1, 0, V1)
        line["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": procs, "kind": "port", "sample": CPU_SAMPLE_TEXT,
                                "seconds": s_per, "per_unit_seconds": unit}
    return line


# ---------------------------------------------------------------------------------------------
# C5: all-pairs matching, lo axis sharded (SURVEY 8e), NCCL all_gather + merge
# ---------------------------------------------------------------------------------------------
def bench_c5(ctx, args):
    torch = ctx.torch
    from mad_b200 import pipeline as P
    from mad_b200 import parallel as par
    dev, world, rank = ctx.dev, ctx.world, ctx.rank
    M = N = int(os.environ.get("MAD_C5_ROWS", "100000"))
    k = 8
    hi_h, lo_h = synth.c5_descriptor_sets(M, N)                # identical inputs on every rank (same seeds)
    # rank grid: the reference (lo) axis is always cut; for larger worlds part of the factor goes to the hi axis, because
    # cutting lo alone leaves every rank with all 782 CTAs and their fixed start-up (parallel.pick_topk_grid)
    grid = tuple(int(x) for x in os.environ["MAD_C5_GRID"].split("x")) if "MAD_C5_GRID" in os.environ else par.pick_topk_grid(M, N, world)
    gh, gl = grid
    bh, bl = par.grid_coords(rank, gh, gl)
    hs, he = par.shard_bounds(M, gh)[bh]
    s, e = par.shard_bounds(N, gl)[bl]
    hi_pin = torch.from_numpy(np.ascontiguousarray(hi_h[hs:he])).pin_memory()
    lo_pin = torch.from_numpy(np.ascontiguousarray(lo_h[s:e])).pin_memory()
    hi = P.DescriptorSet(hi_pin.to(dev))
    lo = P.DescriptorSet(lo_pin.to(dev))
    stage = P.HostStage()
    hi_up = torch.empty(tuple(hi_pin.shape), dtype=torch.int16, device=dev)
    lo_up = torch.empty(tuple(lo_pin.shape), dtype=torch.int16, device=dev)

    def step_device():
        return par.match_topk_grid_sets(hi, lo, k, M, s, grid)

    def step_e2e():                                             # per rank: its hi block and its lo shard over PCIe
        hi_up.copy_(hi_pin, non_blocking=True)
        lo_up.copy_(lo_pin, non_blocking=True)
        idx, sc = par.match_topk_grid_sets(P.DescriptorSet(hi_up), P.DescriptorSet(lo_up), k, M, s, grid)
        out = [stage.fetch("idx", idx), stage.fetch("sc", sc)]
        stage.sync()
        return out

    steps = args.steps
    for _ in range(max(args.warmup, 3)):
        idx, sc = step_device()
    # ---- parity inside the run: sampled hi rows against the whole lo set on ONE GPU (the same kernel, unsharded)
    verified = None
    if world > 1:
        rows = np.sort(np.random.default_rng(5).choice(M, size=2048, replace=False))
        full = P.DescriptorSet(torch.from_numpy(lo_h).to(dev))
        sub = P.DescriptorSet(torch.from_numpy(np.ascontiguousarray(hi_h[rows])).to(dev))
        i1, s1 = P.match_topk(sub, full, k)
        rows_d = torch.from_numpy(rows).to(dev)
        verified = ctx.all_true(torch.equal(i1, idx[rows_d]) and torch.equal(s1, sc[rows_d]))
        del full, sub
    P.profile_enable(True)
    l0 = P.launch_count()
    ms, last = timed(ctx, step_device, steps)
    launches = P.launch_count() - l0
    recs = P.profile_records()
    P.profile_enable(False)
    if args.dump is not None:
        args.dump.put("c5_topk_index", last[0].cpu().numpy())
        args.dump.put("c5_topk_score", last[1].cpu().numpy(), np.float64)
    del last
    out = step_e2e()
    d2h = int(sum(t.numel() * t.element_size() for t in out))
    ms_e2e, _ = timed(ctx, step_e2e, steps)
    ms, ms_e2e = ctx.max_over_ranks(ms, ms_e2e)
    kms = [t for nm, t in recs if nm == "match_u8_topk_kernel"]
    # device time of the matching kernel per step (a step may take two launches: the full waves and the tail rows)
    avg = float(np.sum(kms)) / steps if kms else float("nan")
    (avg,) = ctx.max_over_ranks(avg)
    n_launch = len(kms) // steps if kms else 0
    if rank != 0:
        return None
    ops = 2.0 * (he - hs) * (e - s) * 1024
    step_ms = ms / steps
    res = {
        "metric": "descriptor matches/sec (all-pairs cosine + top-8)", "value": M * N / (step_ms * 1e-3), "unit": "pairs/s",
        "n_gpus": world, "steps": steps, "ms_per_step": step_ms, "scaling": "strong",
        "config": {"workload": "C5: %d x %d int16[1024] descriptors, top-%d, rank grid %d hi blocks x %d lo (reference-axis) shards, NCCL "
                               "all_gather of the per-rank [rows, k] lists + k-way merge over the lo shards" % (M, N, k, gh, gl),
                   "grid": {"hi_blocks": gh, "lo_shards": gl},
                   "l2": "operands %.0f MB per rank > 126 MB L2" % ((he - hs + e - s) * 1024 / 1e6)},
        "e2e": {"value": M * N / (ms_e2e / steps * 1e-3), "unit": "pairs/s",
                "h2d_bytes_per_step": int(hi_pin.numel() * 2 + lo_pin.numel() * 2), "d2h_bytes_per_step": d2h,
                "note": "per rank: its hi block and its lo shard over PCIe, the merged [M, k] lists back",
                "ms_per_step": ms_e2e / steps},
        "gpu_launches": int(launches),
        "roofline": {"bound": "tensor", "kernel": "match_u8_topk_kernel", "achieved": ops / (avg * 1e-3) / 1e12,
                     "peak": ctx.i8_peak, "unit": "TOP/s", "frac": ops / (avg * 1e-3) / 1e12 / ctx.i8_peak,
                     "traffic": ctx.traffic.get("match_u8_topk_kernel") if world == 1 else None,
                     "peak_source": ctx.i8_src, "kernel_ms_per_step": avg, "launches_per_step": n_launch,
                     "avg_launch_ms": avg / max(n_launch, 1), "ops_per_step": ops},
        "verified_equal_to_1gpu": verified,
    }
    if not args.no_cpu_baseline and world == 1:
        import mad_oracle as mo
        blk = 256
        t0 = time.perf_counter()
        mo.match_topk(hi_h[:blk], lo_h, k)
        dt = time.perf_counter() - t0
        res["cpu_baseline"] = {"value": blk * N / dt, "unit": "pairs/s", "cores": os.cpu_count(), "kind": "port",
                               "sample": "%d hi rows x all %d lo rows: the reference's two lines (mad/MaD.py:416-420, float64 "
                                         "np.dot on OpenBLAS threads) + stable argsort top-%d, row-blocked" % (blk, N, k),
                               "seconds": dt}
    return res


# ---------------------------------------------------------------------------------------------
# C4: a batch of 64 snapshot maps, map i -> rank i mod N (SURVEY 8e)
# ---------------------------------------------------------------------------------------------
def dump_c4(dump, res):
    """One C4 step (this rank's maps, in order): per map (keypoints, oriented features), and seeded samples of the rows of
    the maps' keypoint, oriented-feature and descriptor tables put end to end (keypoint indices stay per map)."""
    import torch
    dump.put("c4_counts", [[r["n_kp"], r["n_dsc"]] for r in res], np.float64)
    dump.put_keypoints("c4_keypoints", dump.sample(torch.cat([r["kp"] for r in res]), 1 << 16, 4))
    dump.put_oriented("c4_oriented", dump.sample(torch.cat([r["ori"] for r in res]), 1 << 17, 5))
    dump.put_rows("c4_descriptors", torch.cat([r["dsc"] for r in res]), 1024, 6)


def bench_c4(ctx, args):
    torch = ctx.torch
    from mad_b200 import pipeline as P
    from mad_b200 import parallel as par
    dev, world, rank = ctx.dev, ctx.world, ctx.rank
    n_maps = int(os.environ.get("MAD_C4_MAPS", str(synth.C4_MAPS)))
    base = synth.random_walk_atoms(9000, 85.0, 1)
    mine = par.assign_units(n_maps, rank, world)
    grids = [synth.c4_snapshot(i, base) for i in mine]
    pins = [torch.from_numpy(g).pin_memory() for g in grids]
    devs = [p.to(dev) for p in pins]
    n_vox_total = n_maps * 96 ** 3
    batch = P.MapBatch(streams=int(os.environ.get("MAD_C4_STREAMS", "4")), compact=not args.full_format)
    like = torch.empty((0, 1024), dtype=torch.int16, device=dev)

    def step(host):
        res = batch.run(pins if host else devs, download=host)
        # result collection: per-map descriptor counts of every rank (all-gather); with host=True the tables themselves
        # have gone to pinned host memory on each rank (rank-local write, SURVEY 8e; uint8 descriptors unless --full-format)
        counts = torch.tensor([int(r["n_dsc"]) for r in res], dtype=torch.int64, device=dev).reshape(-1, 1)
        return res, par.gather_varlen(counts)

    for _ in range(max(args.warmup, 3)):
        res, counts = step(False)
    verified = None
    if world > 1:
        # maps 0 and n_maps-1 as described by their owners (tables over NCCL) == described here on this rank's GPU
        tabs = par.collect_units([r["dsc"] for r in res], n_maps, like=like)
        ok = True
        for u in (0, n_maps - 1):
            _, _, _, d1 = P.describe_struct(torch.from_numpy(synth.c4_snapshot(u, base)).to(dev))
            ok = ok and torch.equal(d1, tabs[u])
        verified = ctx.all_true(ok)
        del tabs
    steps = args.steps
    P.profile_enable(True)
    l0 = P.launch_count()
    ms, last = timed(ctx, lambda: step(False), steps)
    launches = P.launch_count() - l0
    recs = P.profile_records()
    P.profile_enable(False)
    if args.dump is not None:
        dump_c4(args.dump, last[0])
    del last
    step(True)
    ms_e2e, _ = timed(ctx, lambda: step(True), steps)
    ms, ms_e2e = ctx.max_over_ranks(ms, ms_e2e)
    K_tot = float(sum(int(r["n_kp"]) for r in res))
    D_tot = float(sum(int(r["n_dsc"]) for r in res))
    if world > 1:
        t = torch.tensor([K_tot, D_tot], dtype=torch.float64, device=dev)
        ctx.dist.all_reduce(t)
        K_tot, D_tot = float(t[0]), float(t[1])
    if rank != 0:
        return None
    sp0 = P.build_space(devs[0], full_gradient=False)
    V0 = int(np.prod(sp0.dims[0]))
    V1 = int(np.prod(sp0.dims[1]))
    step_ms = ms / steps
    kern_ms = sum(t for _, t in recs) / steps                    # rank 0's kernels (its share of the maps), summed over streams
    bytes_batch = n_maps * 36.0 * (V0 + V1) + 58956.0 * K_tot + 51200.0 * D_tot
    res_line = {
        "metric": "voxels/sec scale-space+detect+describe (batch of maps)", "value": n_vox_total / (step_ms * 1e-3),
        "unit": "voxels/s", "n_gpus": world, "steps": steps, "ms_per_step": step_ms, "scaling": "strong",
        "config": {"workload": "C4: %d snapshot maps of 96^3 (9000 atoms, 4 A, sigma 1.5 A displacements), map i -> rank i mod %d, "
                               "no collective on the data path, counts all-gathered; %d host threads / CUDA streams per rank"
                               % (n_maps, world, batch.nw),
                   "keypoints_total": int(K_tot), "oriented_features_total": int(D_tot),
                   "l2": "a map's working set (~0.6 GB) exceeds the 126 MB L2"},
        "e2e": {"value": n_vox_total / (ms_e2e / steps * 1e-3), "unit": "voxels/s",
                "h2d_bytes_per_step": int(sum(p.numel() * 4 for p in pins)), "d2h_bytes_per_step": int(batch.last_d2h_bytes),
                "ms_per_step": ms_e2e / steps},
        "gpu_launches": int(launches),
        "roofline": {"bound": "hbm", "stage": "whole path a1-a12 over the batch", "kernel": "all kernels of the path",
                     "achieved": bytes_batch / (step_ms * 1e-3) / 1e9 / world,
                     "peak": ctx.hbm_peak, "unit": "GB/s per GPU", "frac": bytes_batch / (step_ms * 1e-3) / 1e9 / ctx.hbm_peak / world,
                     "algorithmic_bytes_per_step": bytes_batch, "peak_source": ctx.hbm_src,
                     "rank0_kernel_ms_per_step": kern_ms, "traffic": None},
        "verified_equal_to_1gpu": verified,
    }
    if not args.no_cpu_baseline and world == 1:
        procs = host_procs()
        k_map, d_map = K_tot / n_maps, D_tot / n_maps
        v, s_per, unit = cpu_stage_sample(grids[0], 1.0, procs, 1, 0, V1, K=k_map, D=d_map, M=0, n_vox=96 ** 3)
        res_line["cpu_baseline"] = {"value": v, "unit": "voxels/s", "cores": procs, "kind": "port", "seconds": s_per,
                                    "sample": "stage-wise sample of one snapshot map per process (as for C2: %d^3 crop, %d keypoints, %d oriented "
                                              "features) scaled to a map's V1 = 114^3, K = %.0f, D = %.0f; one map per process on all host cores"
                                              % (CPU_CROP, CPU_KP, CPU_OF, k_map, d_map),
                                    "per_unit_seconds": unit}
    return res_line


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="all", choices=["all", "c2", "c4", "c5"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--match-impl", type=int, default=None, help="default: product (uint8 tcgen05 one-pass); 1 = SIMT check, 2 = fp16 tcgen05")
    ap.add_argument("--exact", type=int, default=1, help="1 = float64 line accumulation (bit-exact with SciPy)")
    ap.add_argument("--full-format", action="store_true", help="e2e downloads int16 descriptors and float64 scores instead of the compact format")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step of each workload returned to DIR/<name>.npy (at most 64 MB); "
                         "under torchrun rank 0 writes its own results only")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes what the GPU path computes (--impl ours)")
    args.dump = OutputDump(args.dump_outputs) if args.dump_outputs and int(os.environ.get("RANK", "0")) == 0 else None
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        return run_reference(args)
    ctx = Ctx()
    line = None
    if args.workload in ("all", "c2"):
        line = bench_c2(ctx, args)
    sharded = {}
    if args.workload in ("all", "c5"):
        sharded["c5"] = bench_c5(ctx, args)
    if args.workload in ("all", "c4"):
        sharded["c4"] = bench_c4(ctx, args)
    if ctx.rank == 0:
        if line is None:                                            # a sharded workload on its own: it is the headline
            key = "c5" if "c5" in sharded else "c4"
            line = dict(sharded.pop(key))
            line.update(warmup=args.warmup, higher_is_better=True, vs_baseline=None, data="synthetic",
                        dtype="u8 x u8 -> s32 (exact), f64 scores" if key == "c5" else "f32 grids, f64 line accumulation")
        if sharded:
            line["sharded"] = sharded
            if ctx.world > 1:
                line["verified"] = {k: v.get("verified_equal_to_1gpu") for k, v in sharded.items()}
        print(json.dumps(line))
    if ctx.world > 1:
        ctx.dist.destroy_process_group()


if __name__ == "__main__":
    main()
