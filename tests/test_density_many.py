"""PDB.density_many (G structures simulated in one batch) and Dmap.get_CCC_with_grids (G grids scored in one batch).

CPU: the host layout (box dims, minimum corners, origins) against the oracle's restatement of the reference, and the
refusals that come before any device work.  GPU: the exactness contract --
  1. the batched float64 splat equals the reference's sequential loop bit for bit;
  2. given that splat, the maps equal the single-path kernels (mad_normalise_f64, three mad_conv_full_f64,
     mad_grid_max, mad_threshold_normalise) bit for bit;
  3. a structure's map does not depend on the batch around it, nor on the run;
  4. against structure_to_density_device (float64 atomics) and the reference fixture: one float32 ulp of the maximum;
  5. get_CCC_with_grids equals get_CCC_with_grid on the same grids exactly --
plus no synchronisation inside density_many, launches that do not grow with G, one host read per scored batch, and the
hand-offs to describe_many and from refine_poses."""
import ctypes as C
import os

import numpy as np
import pytest

import density_oracle as do
import helpers as H
import synth

CASES = (("a", dict(resolution=8.0, voxelsp=2.0)), ("b", dict(resolution=4.0, voxelsp=1.0, isovalue=0.2)),
         ("c", dict(resolution=5.0, voxelsp=2.0, isovalue=0.2, pad=1)))
MASS = {"C": 12.011, "N": 14.0067, "O": 15.9994}


def _golden_atoms():
    g = H.golden("density")
    coords, masses = [], []
    for line in bytes(g["pdb_text"]).decode().splitlines():
        if line[:6].strip() in ("ATOM", "HETATM"):
            coords.append([float(line[30:38]), float(line[38:46]), float(line[46:54])])
            masses.append(MASS.get(line[76:78].strip().upper(), 12.011))
    return np.array(coords), np.array(masses)


def _random_structures():
    """Random structures, some with every coordinate on a lattice multiple, some entirely negative, one single atom."""
    rng = np.random.default_rng(5)
    out = []
    for k in range(6):
        n = int(rng.integers(1, 40)) if k else 1
        xyz = rng.normal(scale=6.0, size=(n, 3)) + rng.uniform(-30, 30, size=3)
        if k == 2:
            xyz = np.round(xyz / 2.0) * 2.0                       # on the 2 A lattice
        if k == 3:
            xyz = -np.abs(xyz) - 0.5
        out.append((xyz, rng.uniform(1.0, 30.0, size=n)))
    return out


class _NoDivide(object):
    """numpy, except that np.divide returns its first operand: the oracle's loop then yields the splat before its
    division by the maximum (mad/PDB.py:287)."""

    def __getattr__(self, name):
        return getattr(np, name)

    @staticmethod
    def divide(a, b):
        return a


def _oracle_splat(monkeypatch, xyz, m, voxelsp, pad):
    with monkeypatch.context() as mp:
        mp.setattr(do, "np", _NoDivide())
        grid, px, py, pz, *mins = do.interpolate_to_grid_massweighted(xyz, m, voxelsp, pad)
    return np.reshape(grid, (px, py, pz), order="F"), mins


# ---- CPU ---------------------------------------------------------------------------------------------------------------
def test_host_layout_equals_the_oracle():
    from mad_b200 import PDB as P
    structures = [(_golden_atoms(), kw) for _, kw in CASES] + [(s, dict(resolution=6.0, voxelsp=2.0, pad=p))
                                                                for p, s in enumerate(_random_structures())]
    for (xyz, m), kw in structures:
        vs, pad = kw["voxelsp"], kw.get("pad", 0)
        r, _ = P._gauss_1d(kw["resolution"], vs)
        boxes, totals, origins = P._density_layout([xyz], vs, r, 2 + pad)
        _, px, py, pz, minx, miny, minz = do.interpolate_to_grid_massweighted(xyz, m, vs, pad)
        assert tuple(boxes[0].dims) == (px, py, pz)
        assert tuple(boxes[0].min) == (minx, miny, minz)
        grid, dxi, dyi, dzi = do.structure_to_density(xyz, m, kw["resolution"], vs, kw.get("isovalue", 0.0), pad)
        assert tuple(origins[0]) == (dxi, dyi, dzi)
        assert totals[4] == grid.size and tuple(d + 2 * r for d in boxes[0].dims) == grid.shape


def test_refusals_before_device_work():
    from mad_b200 import PDB as P
    from mad_b200 import _lib
    xyz, m = _golden_atoms()
    with pytest.raises(_lib.MadError, match="no structures"):
        P.density_many([], 4.0, 1.0)
    with pytest.raises(_lib.MadError, match="structure 1 has no atoms"):
        P.density_many([xyz, np.zeros((0, 3))], 4.0, 1.0, masses=[m, np.zeros(0)])
    bad = xyz.copy()
    bad[7, 1] = np.nan
    with pytest.raises(_lib.MadError, match="structure 2 has non-finite"):
        P.density_many([xyz, xyz, bad], 4.0, 1.0, masses=m)
    with pytest.raises(_lib.MadError, match="structure 1 has 300 atoms and 299 masses"):
        P.density_many([xyz, xyz], 4.0, 1.0, masses=[m, m[1:]])
    with pytest.raises(_lib.MadError, match="structure 0 is a coordinate array"):
        P.density_many([xyz], 4.0, 1.0)
    # a box of 2^32 + 5 voxels along x would wrap to a small int32 dim: refused by name, not truncated
    wide = np.array([[0.0, 0.0, 0.0], [float(1 << 32), 1.0, 1.0]])
    with pytest.raises(_lib.MadError, match="structure 1 spans a box"):
        P.density_many([xyz, wide], 4.0, 1.0, masses=[m, np.ones(2)])
    near = np.array([[0.0, 0.0, 0.0], [float((1 << 30) - 11), 1.0, 1.0]])     # + 2 margins + 1 + 2r (r = 3) = 2^30
    with pytest.raises(_lib.MadError, match="structure 0 spans a box"):
        P.density_many([near], 4.0, 1.0, masses=np.ones(2))
    with pytest.raises(_lib.MadError, match="at most 65535"):
        P.density_many([xyz[:1]] * 65536, 4.0, 1.0, masses=m[:1])
    # the C ABI: an empty structure, a non-positive dim, more than 2^31 - 1 corner contributions
    L = _lib.lib
    boxes = (_lib.MadDensityBox * 2)()
    for b in boxes:
        b.n_atoms, b.margin = 10, 2
        b.dims[:] = (8, 8, 8)
    totals = (C.c_longlong * 5)()
    assert L.mad_density_layout(boxes, 2, 3, totals) == 0 and totals[0] == 20 and totals[1] == 1024
    assert L.mad_density_splat_many(None, None, boxes, 2, None, C.c_double(1.0), None, None, 0, None) == -1
    boxes[1].n_atoms = 0
    assert L.mad_density_layout(boxes, 2, 3, totals) == -1
    boxes[1].n_atoms, boxes[1].dims[2] = 10, 0
    assert L.mad_density_layout(boxes, 2, 3, totals) == -1
    boxes[1].dims[2] = 8
    boxes[0].n_atoms, boxes[1].n_atoms = 1 << 27, 1 << 27
    assert L.mad_density_layout(boxes, 2, 3, totals) == -1
    assert b"bad argument" in L.mad_last_error_string()
    boxes[1].n_atoms = (1 << 27) - 1
    assert L.mad_density_layout(boxes, 2, 3, totals) == 0


# ---- GPU ---------------------------------------------------------------------------------------------------------------
def _cuda():
    torch = pytest.importorskip("torch")
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch


@pytest.fixture(scope="module")
def golden_pdb(tmp_path_factory):
    _cuda()
    from mad_b200.PDB import PDB
    path = os.path.join(str(tmp_path_factory.mktemp("pdb")), "case.pdb")
    open(path, "wb").write(bytes(H.golden("density")["pdb_text"]))
    return PDB(path)


def _batch_splat(torch, xyzs, ms, voxelsp, pad):
    """The batch's float64 splat read at the C-ABI stage (before the division), one host array per structure."""
    from mad_b200 import PDB as P
    from mad_b200 import _lib
    boxes, totals, _ = P._density_layout(xyzs, voxelsp, 0, 2 + pad)
    dev = torch.device("cuda")
    d_xyz = torch.from_numpy(np.concatenate(xyzs)).to(dev)
    d_mass = torch.from_numpy(np.concatenate(ms).astype(np.float64)).to(dev)
    d_boxes = torch.from_numpy(np.frombuffer(bytearray(boxes), dtype=np.uint8).copy()).to(dev)
    ws = torch.empty(int(_lib.lib.mad_density_splat_many_workspace_bytes(int(totals[0]))), dtype=torch.uint8, device=dev)
    grid = torch.empty(totals[1], dtype=torch.float64, device=dev)
    _lib.call("mad_density_splat_many", P._ptr(d_xyz), P._ptr(d_mass), boxes, len(xyzs), P._ptr(d_boxes), C.c_double(voxelsp),
              P._ptr(grid), P._ptr(ws), ws.numel(), P._stream())
    flat = grid.cpu().numpy()
    return [flat[b.off[0]:b.off[0] + b.dims[0] * b.dims[1] * b.dims[2]].reshape(tuple(b.dims)) for b in boxes]


def _single_chain(torch, splat, resolution, voxelsp, isovalue):
    """structure_to_density_device after its splat: the single-path kernels on one structure's grid."""
    from mad_b200 import PDB as P
    from mad_b200 import _lib
    call, ptr, st, dev = _lib.call, P._ptr, P._stream(), torch.device("cuda")
    grid = torch.from_numpy(np.ascontiguousarray(splat)).to(dev)
    pxb, pyb, pzb = grid.shape
    scratch = torch.empty(1, dtype=torch.int64, device=dev)
    call("mad_normalise_f64", ptr(grid), grid.numel(), ptr(scratch), st)
    r, w = P._gauss_1d(resolution, voxelsp)
    w = torch.from_numpy(w).to(dev)
    a = torch.empty((pxb + 2 * r, pyb, pzb), dtype=torch.float64, device=dev)
    call("mad_conv_full_f64", ptr(grid), 1, pxb, pyb * pzb, ptr(w), r, ptr(a), 0, st)
    b = torch.empty((pxb + 2 * r, pyb + 2 * r, pzb), dtype=torch.float64, device=dev)
    call("mad_conv_full_f64", ptr(a), pxb + 2 * r, pyb, pzb, ptr(w), r, ptr(b), 0, st)
    dens = torch.empty((pxb + 2 * r, pyb + 2 * r, pzb + 2 * r), dtype=torch.float32, device=dev)
    call("mad_conv_full_f64", ptr(b), (pxb + 2 * r) * (pyb + 2 * r), pzb, 1, ptr(w), r, ptr(dens), 1, st)
    mx = torch.zeros(1, dtype=torch.int32, device=dev)
    call("mad_grid_max", ptr(dens), dens.numel(), ptr(mx), st)
    vmax = float(_lib.lib.mad_grid_max_decode(C.c_uint(int(mx.item()) & 0xFFFFFFFF)))
    call("mad_threshold_normalise", ptr(dens), dens.numel(), C.c_float(-np.inf), C.c_float(vmax), 1, st)
    if isovalue:
        call("mad_threshold_normalise", ptr(dens), dens.numel(), C.c_float(isovalue), C.c_float(1.0), 0, st)
    return dens


def _mixed():
    """One-atom structure, atoms on lattice points, very different sizes, and the golden structure."""
    rng = np.random.default_rng(11)
    xyz0, m0 = _golden_atoms()
    big = synth.random_walk_atoms(6000, 60.0, 3)
    lattice = np.round(rng.uniform(-20, 20, size=(50, 3)))
    return [(xyz0, m0), (np.array([[1.25, -3.5, 7.0]]), np.array([14.0067])), (lattice, rng.uniform(1, 20, 50)),
            (big, np.full(len(big), 12.011)), (xyz0 + 0.37, m0)]


def _check_contract(torch, monkeypatch, structs, resolution, voxelsp, isovalue=0.0, pad=0):
    from mad_b200 import PDB as P
    xyzs, ms = [s[0] for s in structs], [s[1] for s in structs]
    batch = P.density_many(xyzs, resolution, voxelsp, isovalue, pad, masses=list(ms))
    splats = _batch_splat(torch, xyzs, ms, voxelsp, pad)
    for g, (xyz, m) in enumerate(structs):
        ref, mins = _oracle_splat(monkeypatch, xyz, m, voxelsp, pad)                        # 1
        assert splats[g].shape == ref.shape and splats[g].tobytes() == ref.tobytes(), g
        assert torch.equal(batch.grids[g], _single_chain(torch, splats[g], resolution, voxelsp, isovalue)), g   # 2
        r = P._gauss_1d(resolution, voxelsp)[0]
        assert tuple(batch.origins[g]) == tuple(mn - (r + 2 + pad) * voxelsp for mn in mins)
        assert batch.grids[g].shape == tuple(d + 2 * r for d in ref.shape)
    return batch


@pytest.mark.gpu
@pytest.mark.parametrize("tag,kw", CASES)
def test_golden_structure_contract(monkeypatch, golden_pdb, tag, kw):
    torch = _cuda()
    from mad_b200 import PDB as P
    xyz, m = _golden_atoms()
    batch = _check_contract(torch, monkeypatch, [(xyz, m)], **kw)
    # 4: against the reference fixture and the atomics path, one float32 ulp of the maximum (near-cut voxels may flip)
    g = H.golden("density")
    ref = g[tag + "_grid"]
    grid, dxi, dyi, dzi = batch.host(0)
    assert grid.shape == ref.shape and grid.dtype == np.float32 and grid.max() == 1.0
    assert np.array_equal([dxi, dyi, dzi], g[tag + "_origin"])
    iso = kw.get("isovalue", 0.0)
    for other in (ref, golden_pdb.structure_to_density(**kw)[0]):
        near_cut = np.abs(np.where(other == 0, grid, other) - iso) <= 2.4e-7 if iso else np.zeros(ref.shape, bool)
        assert np.abs(grid - other)[~near_cut].max() <= 1.2e-7
        assert near_cut.sum() <= 2
    # PDB objects take their masses from the elements
    again = P.density_many([golden_pdb], **kw)
    assert torch.equal(again.grids[0], batch.grids[0])


@pytest.mark.gpu
def test_mixed_batch_contract(monkeypatch):
    torch = _cuda()
    structs = _mixed()
    _check_contract(torch, monkeypatch, structs, 4.0, 1.0)
    _check_contract(torch, monkeypatch, structs, 6.0, 2.0, isovalue=0.3, pad=2)


@pytest.mark.gpu
def test_map_does_not_depend_on_the_batch():
    torch = _cuda()
    from mad_b200 import PDB as P
    a, b = _mixed()[0], _mixed()[3]
    kw = dict(resolution=5.0, voxelsp=1.5, isovalue=0.1, pad=1)

    def run(structs):
        return P.density_many([s[0] for s in structs], masses=[s[1] for s in structs], **kw)
    ref = run([a])
    for batch, idx in ((run([a, b]), (0,)), (run([b, a]), (1,)), (run([a, a]), (0, 1)), (run([a]), (0,))):
        for i in idx:
            assert torch.equal(batch.grids[i], ref.grids[0])
            assert np.array_equal(batch.origins[i], ref.origins[0])
    assert torch.equal(run([b, a]).grids[0], run([b]).grids[0])


@pytest.mark.gpu
def test_no_synchronisation_and_launches_do_not_grow_with_g():
    torch = _cuda()
    from mad_b200 import PDB as P
    from mad_b200 import pipeline
    base = synth.random_walk_atoms(3000, 50.0, 1)
    rng = np.random.default_rng(0)
    snaps = [base + rng.normal(scale=1.5, size=base.shape) for _ in range(16)]
    m = np.full(len(base), 12.011)
    P.density_many(snaps[:2], 4.0, 1.0, masses=m)                   # warm-up (module load, CUB tuning)
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        batch = P.density_many(snaps, 4.0, 1.0, masses=m)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    assert len(batch) == 16
    counts = {}
    for G in (1, 4, 16):
        n0 = pipeline.launch_count()
        P.density_many(snaps[:G], 4.0, 1.0, masses=m)
        counts[G] = pipeline.launch_count() - n0
    assert counts[1] == counts[4] == counts[16], counts


@pytest.mark.gpu
def test_description_hand_off():
    torch = _cuda()
    from mad_b200 import PDB as P
    from mad_b200 import pipeline
    from mad_b200.Descriptor import Descriptor
    from mad_b200.Detector import Detector
    from mad_b200.MapSpace import MapSpace
    from mad_b200.Orientator import Orientator
    base = synth.random_walk_atoms(2500, 45.0, 2)
    rng = np.random.default_rng(1)
    v, pad_map = 1.0, 9
    batch = P.density_many([base, base + rng.normal(scale=1.5, size=base.shape)], 4.0, v, masses=np.full(len(base), 12.011))
    tables = pipeline.describe_many(batch.grids).feature_tables([[v / 2, v]] * len(batch),
                                                                [batch.origins[g] - pad_map * v for g in range(len(batch))])
    for g in range(len(batch)):
        ms = MapSpace.from_grid(batch.grids[g].clone(), v, tuple(batch.origins[g]))
        ms.build_space()
        ref = pipeline.FeatureTable.from_features(
            Descriptor().generate_descriptors(ms, Orientator().assign_orientations(ms, Detector().find_anchors(ms))))
        assert ref.meta.shape[0] > 0
        assert torch.equal(tables[g].meta, ref.meta), g
        assert tables[g].subv.cpu().numpy().tobytes() == ref.subv.cpu().numpy().tobytes(), g
        assert torch.equal(tables[g].set.dsc, ref.set.dsc), g


def _target_and_poses(n_poses):
    """A C2-style component, its map as the target, and n_poses rigid poses of it."""
    from mad_b200.Dmap import Dmap
    from mad_b200.math_utils import euler_rod_mat
    cfg = synth.C2
    atoms = synth.assembly_atoms(cfg["n"] // 4, cfg["voxelsp"], 2, 4000, cfg["seed0"], 40.0)[0]
    grid, org = synth.simulate_density(atoms, cfg["resolution"], cfg["voxelsp"])
    target = lambda: Dmap.from_array(np.asarray(grid, dtype=np.float32), cfg["voxelsp"], origin=tuple(float(x) for x in org))
    cen = atoms.mean(0)
    rng = np.random.default_rng(4)
    poses = np.stack([np.dot(atoms - cen, euler_rod_mat(rng.normal(size=3), 0.05 * p)) + cen + rng.normal(scale=1.5, size=3)
                      for p in range(n_poses)])
    return target, poses, np.full(len(atoms), 12.011), cfg


@pytest.mark.gpu
@pytest.mark.parametrize("isovalue", [0.0, 0.15])
def test_scores_equal_the_per_structure_calls(isovalue):
    torch = _cuda()
    from mad_b200 import PDB as P
    target, poses, m, cfg = _target_and_poses(6)
    batch = P.density_many(poses, cfg["resolution"], cfg["voxelsp"], masses=m)
    far = batch.origins.copy()
    far[2] += 1e4                                                   # pose 2 lies far away: a disjoint box
    tgt = target()
    got = tgt.get_CCC_with_grids(batch.grids, far, isovalue)
    assert got.dtype == np.float64 and got.shape == (6,) and got[2] == 0
    assert (got[[0, 1, 3, 4, 5]] > 0.5).all(), got
    for g in range(6):
        assert got[g] == tgt.get_CCC_with_grid(batch.grids[g], *far[g], isovalue), g
    # the isovalue cut happened in place, on the target and on every grid
    if isovalue:
        assert all(float(x[(x > 0)].min()) >= isovalue for x in batch.grids)
    # a NumPy grid is uploaded and scored the same way
    host = batch.host(1)[0]
    assert tgt.get_CCC_with_grids([host], far[1:2], isovalue)[0] == got[1]


def _counting_reads(monkeypatch):
    from mad_b200 import pipeline as P
    calls = []
    orig = P._Readback.read.__func__

    def read(cls, *tensors):
        calls.append(len(tensors))
        return orig(cls, *tensors)
    monkeypatch.setattr(P._Readback, "read", classmethod(read))
    return calls


@pytest.mark.gpu
def test_one_host_read_and_mismatch_refusal(monkeypatch):
    torch = _cuda()
    from mad_b200 import PDB as P
    from mad_b200.Dmap import Dmap
    target, poses, m, cfg = _target_and_poses(5)
    batch = P.density_many(poses, cfg["resolution"], cfg["voxelsp"], masses=m)
    tgt = target()
    calls = _counting_reads(monkeypatch)
    tgt.get_CCC_with_grids(batch.grids, batch.origins)
    assert len(calls) == 1, calls
    # a half-voxel offset whose two common-box extents round differently: refused, naming the structure, before any work
    vs = tgt.voxsp
    o1, s1 = [tgt.xi / vs, tgt.yi / vs, tgt.zi / vs], [tgt.xb, tgt.yb, tgt.zb]
    bad = None
    for shift in np.arange(-40.5, 40.5, 1.0):
        for n in range(5, 60):
            try:
                Dmap._common_box(o1, s1, [o1[0] + shift, o1[1], o1[2]], [n, tgt.yb, tgt.zb])
            except ValueError:
                bad = (shift, n)
                break
        if bad:
            break
    assert bad is not None
    odd = torch.zeros((bad[1], tgt.yb, tgt.zb), dtype=torch.float32, device="cuda")
    before = tgt.device_grid().clone()
    with pytest.raises(ValueError, match="structure 1"):
        tgt.get_CCC_with_grids([batch.grids[0], odd], [batch.origins[0], [tgt.xi + bad[0] * vs, tgt.yi, tgt.zi]], 0.5)
    assert torch.equal(tgt.device_grid(), before)                   # nothing was cut


@pytest.mark.gpu
def test_refined_poses_to_scores():
    torch = _cuda()
    from mad_b200 import PDB as P
    from mad_b200.structure_utils import RefineField, refine_poses
    target, poses, m, cfg = _target_and_poses(8)
    coords, conv, step, bad = refine_poses(RefineField(target()), poses, n_steps=200, max_step_size=1, min_step_size=0.1)
    assert not bad.any()
    batch = P.density_many(coords, cfg["resolution"], cfg["voxelsp"], masses=m)
    tgt = target()
    got = tgt.get_CCC_with_grids(batch.grids, batch.origins)
    for g in range(len(coords)):
        one = P.density_many([coords[g]], cfg["resolution"], cfg["voxelsp"], masses=m)
        assert torch.equal(one.grids[0], batch.grids[g])
        assert got[g] == tgt.get_CCC_with_grid(batch.grids[g], *batch.origins[g])
