"""MaD._match_dsc (mad/MaD.py:414-453) in pieces, on one GPU: the anchor clouds and the lo grid built on the device
against the host construction they replace (np.unique + a NumPy grid, kept below as the reference), the per-pair counts
over sub-ranges of the pairs, the row expansion, and the sharded form's per-rank steps for simulated worlds joined on
one device.  The collectives themselves: tests/test_match_dsc_gloo.py (CPU) and tests/test_multi_gpu_match_dsc.py."""
import numpy as np
import pytest

import dsc_cases as D
import helpers as H

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")


@pytest.fixture(scope="module")
def P():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from mad_b200 import pipeline
    return pipeline


@pytest.fixture(scope="module")
def par():
    from mad_b200 import parallel
    return parallel


def host_cloud_grid(cloud, cell):
    """The host construction the device builder replaces: uniform grid (cell size = the distance threshold) over the
    cloud: cell-sorted points, cell_start, and the bitmap of cells whose 27-cell neighbourhood holds a point."""
    org = cloud.min(0) - cell
    dims = (np.floor((cloud.max(0) - org) / cell).astype(np.int64) + 2)
    cidx = np.floor((cloud - org) / cell).astype(np.int64)
    lin = (cidx[:, 0] * dims[1] + cidx[:, 1]) * dims[2] + cidx[:, 2]
    order = np.argsort(lin, kind="stable")
    ncell = int(dims.prod())
    cell_start = np.zeros(ncell + 1, dtype=np.int32)
    np.cumsum(np.bincount(lin, minlength=ncell), out=cell_start[1:])
    occ = np.zeros(tuple(dims), dtype=bool)
    occ[cidx[:, 0], cidx[:, 1], cidx[:, 2]] = True
    near = np.zeros_like(occ)
    p = np.pad(occ, 1)
    for dx in range(3):
        for dy in range(3):
            for dz in range(3):
                near |= p[dx:dx + dims[0], dy:dy + dims[1], dz:dz + dims[2]]
    bits = np.packbits(near.reshape(-1), bitorder="little")
    bits = np.concatenate([bits, np.zeros((-len(bits)) % 4, dtype=np.uint8)]).view(np.uint32)
    return np.ascontiguousarray(cloud[order]), cell_start, bits, org.astype(np.float64), dims.astype(np.int32)


def _bits(a):
    """Bytes of a float64 array with -0.0 taken as +0.0 (np.unique keeps either of two rows it treats as equal)."""
    return (np.ascontiguousarray(a, dtype=np.float64) + 0.0).tobytes()


def _check_cloud(P, subv, used, cell):
    subv = np.ascontiguousarray(subv, dtype=np.float64).reshape(-1, 3)
    used = np.asarray(used, dtype=bool)
    ref_cloud = np.unique(subv[used], axis=0)
    ref = host_cloud_grid(ref_cloud, cell)
    c = P.anchor_cloud(torch.from_numpy(subv).cuda(), torch.from_numpy(used.astype(np.uint8)).cuda(), cell)
    cloud = c.host()
    assert cloud.shape == ref_cloud.shape and np.array_equal(cloud, ref_cloud) and _bits(cloud) == _bits(ref_cloud)
    assert _bits(c.sorted.cpu().numpy()) == _bits(ref[0]), "lo_sorted"
    assert np.array_equal(c.cell_start.cpu().numpy(), ref[1]), "cell_start"
    assert np.array_equal(c.near_bits.cpu().numpy().view(np.uint32), ref[2]), "near_bits"
    assert c.org.tobytes() == ref[3].tobytes() and np.array_equal(c.dims, ref[4]), "org / dims"
    return c


def _adversarial():
    rng = np.random.default_rng(5)
    out = {}
    out["all_equal"] = np.tile([[1.25, -3.5, 7.0]], (300, 1))
    out["one_row"] = np.array([[12.3, 45.6, -7.8]])
    base = rng.normal(scale=20.0, size=(5, 3))
    out["many_duplicates"] = base[rng.integers(0, 5, size=2000)]
    # on org + k cell: every coordinate a multiple of the cell, so (c - org) / cell lands exactly on integers
    out["on_cell_edges"] = 4.0 * rng.integers(-6, 7, size=(400, 3)).astype(np.float64)
    out["negative"] = -np.abs(rng.normal(scale=30.0, size=(500, 3))) - 100.0
    z = np.array([[0.0, 1.0, 2.0], [-0.0, 1.0, 2.0], [3.0, -0.0, 0.0], [3.0, 0.0, -0.0], [-0.0, -0.0, -0.0],
                  [0.0, 0.0, 0.0], [-1e-300, 0.0, 5e-324]])
    out["signed_zeros"] = z[rng.integers(0, len(z), size=64)]
    out["far_apart"] = np.array([[0.0, 0.0, 0.0], [400.0, 3.0, 800.0]])
    out["ties_in_x"] = np.stack([np.full(600, 2.0), rng.integers(0, 4, 600), rng.integers(0, 4, 600)], 1).astype(np.float64)
    return out


@pytest.mark.parametrize("cell", [4.0, 6.5])
@pytest.mark.parametrize("case", sorted(_adversarial()))
def test_device_cloud_equals_host_on_adversarial_sets(P, case, cell):
    subv = _adversarial()[case]
    _check_cloud(P, subv, np.ones(len(subv), dtype=bool), cell)
    rng = np.random.default_rng(len(subv))
    used = rng.random(len(subv)) < 0.5
    used[0] = True
    _check_cloud(P, subv, used, cell)                      # unused rows (sorted behind the used ones) drop out


@pytest.mark.parametrize("name", ["pair_hi", "pair_lo"])
def test_device_cloud_equals_host_on_pair_fixtures(P, name):
    subv = H.golden(name)["of_subv_map_coords"]
    for cell in (4.0, 6.5):
        _check_cloud(P, subv, np.ones(len(subv), dtype=bool), cell)
        _check_cloud(P, subv, np.arange(len(subv)) % 3 == 1, cell)


def test_device_cloud_equals_host_on_c2_components(P):
    gc = H.golden("c2_comp")
    rng = np.random.default_rng(3)
    subs = [gc["comp%d_of_subv_map_coords" % i] for i in range(6)]
    for s in subs:
        _check_cloud(P, s, rng.random(len(s)) < 0.3, 4.0)
    stacked = np.concatenate(subs)
    _check_cloud(P, stacked, np.ones(len(stacked), dtype=bool), 4.0)


def test_non_finite_coordinates_are_refused(P):
    from mad_b200._lib import MadError
    subv = np.array([[1.0, 2.0, 3.0], [4.0, np.nan, 6.0], [7.0, 8.0, np.inf]])
    for bad in (1, 2):
        used = np.zeros(3, dtype=bool)
        used[[0, bad]] = True
        with pytest.raises(MadError, match="non-finite"):
            P.anchor_cloud(torch.from_numpy(subv).cuda(), torch.from_numpy(used.astype(np.uint8)).cuda(), 4.0)
    _check_cloud(P, subv, np.array([True, False, False]), 4.0)          # an unused non-finite row is no concern


def test_grid_of_2_31_cells_is_refused(P):
    from mad_b200._lib import MadError
    # dims = floor((5160 + 4) / 4) + 2 = 1293 per axis: 2.16e9 cells >= 2^31, refused before anything of that size exists
    subv = torch.tensor([[0.0, 0.0, 0.0], [5160.0, 5160.0, 5160.0]], dtype=torch.float64, device="cuda")
    used = torch.ones(2, dtype=torch.uint8, device="cuda")
    c, = P.read_clouds(P.AnchorCloud(subv, used, 4.0))
    assert c.dims.tolist() == [1293] * 3
    with pytest.raises(MadError, match="bad argument"):
        c.build_grid()
    with pytest.raises(MadError, match="bad argument"):
        P.anchor_cloud(subv * 1e200, used, 4.0)            # dims far beyond int64 range (clamped on the device)


def _cases(P):
    lo, hi = D.pair_tables(P)
    gm = H.golden("pair_match")
    few_hi = D.rows_of(P, lo, [3, 40, 41])           # exact copies of lo rows: a handful of pairs at cc 0.999
    return {"reference": (lo, hi, 4, float(gm["cc"])), "dense": (lo, hi, 6.5, 0.5), "few_pairs": (lo, few_hi, 4, 0.999),
            "no_pairs": (lo, hi, 4, 1.0)}


def test_counts_over_ranges_and_rows_equal_match_dsc(P):
    for name, (lo, hi, dist, cc) in _cases(P).items():
        m = P.DscMatch(lo, hi, dist, cc)
        ref, lo_cloud, hi_cloud = P.match_dsc(lo, hi, dist, cc)
        assert m.p == ref.shape[0], name
        if m.p == 0:
            assert name == "no_pairs" and lo_cloud.shape == (0, 3) and hi_cloud.shape == (0, 3)
            continue
        full = m.counts(0, m.p)
        for p0, p1 in [(0, 0), (0, 1), (1, min(17, m.p)), (m.p // 3, m.p // 2), (max(m.p - 5, 0), m.p), (m.p, m.p), (0, m.p)]:
            part = m.counts(p0, p1)
            assert part.shape == (p1 - p0,) and torch.equal(part, full[p0:p1]), (name, p0, p1)
        assert torch.equal(m.rows(full), ref), name                      # counts + rows == mad_repeatability
        assert torch.equal(m.table(), ref), name
        assert np.array_equal(m.lo_cloud.host(), lo_cloud) and np.array_equal(m.hi_cloud.host(), hi_cloud)
        if name == "few_pairs":
            assert 0 < m.p < 8                                          # fewer pairs than ranks in a world of 8


def test_match_dsc_clouds_equal_reference_fixture(P):
    """The clouds match_dsc returns, now built on the device, against the reference's own (np.unique) clouds."""
    lo, hi = D.pair_tables(P)
    gm = H.golden("pair_match")
    _, lo_cloud, hi_cloud = P.match_dsc(lo, hi, 4, float(gm["cc"]))
    assert _bits(lo_cloud) == _bits(gm["lo_cloud"]) and _bits(hi_cloud) == _bits(gm["hi_cloud"])


@pytest.mark.parametrize("world", [2, 3, 8])
def test_sharded_steps_of_simulated_worlds_equal_match_dsc(P, par, world):
    for name, (lo, hi, dist, cc) in _cases(P).items():
        ref, lo_cloud, hi_cloud = P.match_dsc(lo, hi, dist, cc)
        m = P.DscMatch(lo, hi, dist, cc)
        if m.p == 0:
            got = par.match_dsc_sharded(lo, hi, dist, cc)             # no process group: the world of one
            assert got[0].shape == (0, 23) and got[1].shape == (0, 3) and got[2].shape == (0, 3)
            continue
        shares = [par.pad_counts(par.match_dsc_local(m, r, world), m.p, world) for r in range(world)]
        assert len({s.numel() for s in shares}) == 1
        joined = par.join_counts(torch.stack(shares), m.p)
        assert torch.equal(joined, m.counts(0, m.p)), (name, world)
        assert torch.equal(m.rows(joined), ref), (name, world)
        got, glo, ghi = par.match_dsc_sharded(lo, hi, dist, cc)
        assert torch.equal(got, ref) and np.array_equal(glo, lo_cloud) and np.array_equal(ghi, hi_cloud)
