"""pipeline.match_dsc_many (one map against G structures in one batch) on one GPU: every structure's result equals its own
match_dsc call bit for bit; the segmented clouds and grids equal the single-structure device builders (and through them
the host construction of tests/test_match_dsc_sharded.py); the refusals name the structure; counts over sub-ranges that
cross structure boundaries; and the per-rank steps of match_dsc_many_sharded for simulated worlds, joined on one device.
The collectives: tests/test_match_dsc_many_cpu.py (gloo) and tests/test_multi_gpu_match_dsc_many.py (NCCL)."""
import numpy as np
import pytest

import dsc_cases as D
import helpers as H
from test_match_dsc_sharded import _adversarial, _bits, host_cloud_grid

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


def _table(P, dsc, meta, subv):
    return P.FeatureTable(dsc, meta[:, 0], meta[:, 1], meta[:, 2], meta[:, 3], subv)


def _no_pairs(P, lo, n=5):
    """A structure whose rows are zero descriptors: cosine 0, no pair above any cc >= 0."""
    return _table(P, torch.zeros((n, 1024), dtype=torch.int16, device="cuda"), lo.meta_host[:n], lo.subv_host[:n] + 1.0)


def _check_equal(P, lo, his, dist, cc):
    got = P.match_dsc_many(lo, his, dist, cc)
    assert len(got) == len(his)
    for g, h in enumerate(his):
        ref = P.match_dsc(lo, h, dist, cc)
        t, lc, hc = got[g]
        assert t.shape == ref[0].shape and t.dtype == ref[0].dtype and torch.equal(t, ref[0]), (g, t.shape, ref[0].shape)
        for a, b in ((lc, ref[1]), (hc, ref[2])):
            assert a.shape == b.shape and np.array_equal(a, b) and a.tobytes() == b.tobytes(), g
    return got


def _fixture_batch(P):
    lo, hi = D.pair_tables(P)
    few_hi = D.rows_of(P, lo, [3, 40, 41])
    subset = D.rows_of(P, hi, np.arange(1, hi.set.rows, 3))
    return lo, hi, few_hi, subset, _no_pairs(P, lo)


@pytest.mark.parametrize("where", [0, 2, 4])
def test_pair_fixtures_equal_match_dsc(P, where):
    lo, hi, few_hi, subset, none = _fixture_batch(P)
    his = [hi, few_hi, subset, hi]
    his.insert(where, none)
    got = _check_equal(P, lo, his, 4, float(H.golden("pair_match")["cc"]))
    assert got[where][0].shape == (0, 23) and got[where][1].shape == (0, 3) and got[where][2].shape == (0, 3)
    assert all(got[g][0].shape[0] > 0 for g in range(len(his)) if g != where)


def test_one_structure_and_no_structure(P):
    lo, hi, few_hi, subset, none = _fixture_batch(P)
    _check_equal(P, lo, [hi], 4, float(H.golden("pair_match")["cc"]))
    _check_equal(P, lo, [few_hi], 4, 0.999)
    _check_equal(P, lo, [none], 4, 0.6)
    _check_equal(P, lo, [hi, subset], 4, 1.0)                     # no pair at all
    assert P.match_dsc_many(lo, [], 4, 0.6) == []


def test_dense_case_equals_match_dsc(P):
    lo, hi, few_hi, subset, none = _fixture_batch(P)
    _check_equal(P, lo, [hi, none, few_hi, subset], 6.5, 0.5)


def test_c2_components_equal_match_dsc(P):
    lo, comps = D.c2_tables(P)
    got = _check_equal(P, lo, comps, 4, 0.65)
    assert all(t.shape[0] > 0 for t, _, _ in got)


def _check_segments(P, subvs, useds, cell):
    subvs = [np.ascontiguousarray(s, dtype=np.float64).reshape(-1, 3) for s in subvs]
    useds = [np.asarray(u, dtype=bool) for u in useds]
    c = P.anchor_clouds([torch.from_numpy(s).cuda() for s in subvs], [torch.from_numpy(u.astype(np.uint8)).cuda() for u in useds],
                        cell)
    for g, (s, u) in enumerate(zip(subvs, useds)):
        cloud = c.cloud_of(g).cpu().numpy()
        if not u.any():
            assert c.n[g] == 0 and cloud.shape == (0, 3)
            assert all(t.numel() == (1 if k == 1 else 0) for k, t in enumerate(c.grid_of(g)))
            continue
        ref_cloud = np.unique(s[u], axis=0)
        assert cloud.shape == ref_cloud.shape and np.array_equal(cloud, ref_cloud) and _bits(cloud) == _bits(ref_cloud), g
        one = P.anchor_cloud(torch.from_numpy(s).cuda(), torch.from_numpy(u.astype(np.uint8)).cuda(), cell)
        assert cloud.tobytes() == one.host().tobytes(), g
        srt, cs, nb = c.grid_of(g)
        assert srt.cpu().numpy().tobytes() == one.sorted.cpu().numpy().tobytes(), g
        assert torch.equal(cs, one.cell_start) and torch.equal(nb, one.near_bits), g
        assert c.org[g].tobytes() == one.org.tobytes() and np.array_equal(c.dims64[g], one.dims64), g
        ref = host_cloud_grid(ref_cloud, cell)
        assert np.array_equal(cs.cpu().numpy(), ref[1]) and np.array_equal(nb.cpu().numpy().view(np.uint32), ref[2]), g
    return c


@pytest.mark.parametrize("cell", [4.0, 6.5])
def test_segmented_clouds_equal_single_builders_on_adversarial_sets(P, cell):
    sets = _adversarial()
    names = sorted(sets)
    rng = np.random.default_rng(11)
    subvs, useds = [], []
    for name in names:
        s = sets[name]
        subvs.append(s)
        useds.append(np.ones(len(s), dtype=bool))
        u = rng.random(len(s)) < 0.5
        u[0] = True
        subvs.append(s)
        useds.append(u)
    _check_segments(P, subvs, useds, cell)
    _check_segments(P, subvs[::-1], useds[::-1], cell)


def test_identical_rows_in_two_structures_stay_apart(P):
    s = _adversarial()["many_duplicates"]
    c = _check_segments(P, [s, s, s[:7]], [np.ones(len(s), dtype=bool)] * 2 + [np.ones(7, dtype=bool)], 4.0)
    assert c.n[0] == c.n[1] == len(np.unique(s, axis=0))


def test_signed_zeros_and_structures_without_used_rows(P):
    z = _adversarial()["signed_zeros"]
    none = np.zeros(len(z), dtype=bool)
    _check_segments(P, [z, z, z, -z], [none, np.ones(len(z), dtype=bool), none, np.arange(len(z)) % 2 == 0], 4.0)
    _check_segments(P, [z, z], [np.ones(len(z), dtype=bool), none], 4.0)


def test_non_finite_used_coordinate_is_refused_naming_the_structure(P):
    from mad_b200._lib import MadError
    good = np.array([[1.0, 2.0, 3.0], [4.0, 5.0, 6.0]])
    bad = np.array([[1.0, 2.0, 3.0], [4.0, np.nan, 6.0], [7.0, 8.0, np.inf]])
    on = np.ones(2, dtype=bool)
    with pytest.raises(MadError, match="structure 1: 1 used feature"):
        _check_segments(P, [good, bad, good], [on, np.array([True, True, False]), on], 4.0)
    with pytest.raises(MadError, match="structure 2: 2 used feature"):
        _check_segments(P, [good, good, bad], [on, on, np.ones(3, dtype=bool)], 4.0)
    _check_segments(P, [good, bad, good], [on, np.array([True, False, False]), on], 4.0)   # unused: no concern
    # through match_dsc_many: a non-finite coordinate on a row that pairs, and on one that does not
    lo, hi, few_hi, subset, none = _fixture_batch(P)
    dsc = torch.cat([few_hi.set.dsc, torch.zeros((1, 1024), dtype=torch.int16, device="cuda")])
    meta = np.concatenate([few_hi.meta_host, few_hi.meta_host[:1]])
    subv = np.concatenate([few_hi.subv_host, [[np.nan, 0.0, 0.0]]])
    nan_unused = _table(P, dsc, meta, subv)
    _check_equal(P, lo, [hi, nan_unused], 4, 0.999)
    subv_used = few_hi.subv_host.copy()
    subv_used[0, 2] = np.inf
    with pytest.raises(MadError, match="structure 1: 1 used feature"):
        P.match_dsc_many(lo, [few_hi, _table(P, few_hi.set.dsc, few_hi.meta_host, subv_used)], 4, 0.999)


def test_grid_of_2_31_cells_is_refused_naming_the_structure(P):
    from mad_b200._lib import MadError
    small = np.array([[0.0, 0.0, 0.0], [8.0, 8.0, 8.0]])
    big = np.array([[0.0, 0.0, 0.0], [5160.0, 5160.0, 5160.0]])        # 1293^3 cells >= 2^31
    on = np.ones(2, dtype=bool)
    with pytest.raises(MadError, match=r"structure 1: a lo grid of 2161700757 cells \(>= 2\^31"):
        _check_segments(P, [small, big, small], [on, on, on], 4.0)


def test_grids_that_fit_alone_but_not_together_run(P):
    """Two lo grids of 1100^3 = 1.33e9 cells each: 2.66e9 together, beyond int32, addressed with int64 offsets."""
    lo, hi = D.pair_tables(P)
    subv = np.zeros_like(lo.subv_host)
    subv[40] = 4390.0                                                  # dims = floor((4390 + 4) / 4) + 2 = 1100
    lo_far = _table(P, lo.set.dsc, lo.meta_host, subv)
    his = [D.rows_of(P, lo_far, [3, 40]), D.rows_of(P, lo_far, [40, 3])]
    m = P.DscMatchMany(lo_far, his, 4, 0.999)
    assert [list(d) for d in m.lo_clouds.dims64] == [[1100] * 3] * 2
    assert m.lo_clouds.cells == 2 * 1100 ** 3 > 1 << 31
    del m
    _check_equal(P, lo_far, his, 4, 0.999)


def test_counts_over_ranges_across_structures_and_rows_checks(P):
    from mad_b200._lib import MadError
    lo, hi, few_hi, subset, none = _fixture_batch(P)
    m = P.DscMatchMany(lo, [few_hi, hi, none, subset, few_hi], 4, float(H.golden("pair_match")["cc"]))
    full = m.counts(0, m.p)
    cuts = sorted({int(v) for v in m.pair_off} | {int(v) + d for v in m.pair_off for d in (-1, 1)})
    cuts = [c for c in cuts if 0 <= c <= m.p]
    for p0 in cuts:
        for p1 in cuts:
            if p1 >= p0:
                assert torch.equal(m.counts(p0, p1), full[p0:p1]), (p0, p1)
    table = m.rows(full)
    for g, h in enumerate(m.his):
        a, b = m.pair_off[g], m.pair_off[g + 1]
        ref = P.DscMatch(lo, h, 4, float(H.golden("pair_match")["cc"]))
        if ref.p:
            assert torch.equal(full[a:b], ref.counts(0, ref.p)) and torch.equal(table[a:b], ref.table()), g
    for bad in (full[:-1], full.to(torch.int64), full.cpu()):
        with pytest.raises(MadError, match="DscMatchMany.rows"):
            m.rows(bad)


@pytest.mark.parametrize("world", [2, 3, 8])
def test_weighted_shares_of_simulated_worlds_equal_match_dsc_many(P, par, world):
    lo, hi, few_hi, subset, none = _fixture_batch(P)
    cc = float(H.golden("pair_match")["cc"])
    for his, dist, c in (([hi, none, subset, few_hi], 4, cc), ([none, few_hi], 4, 0.999), ([hi, few_hi], 6.5, 0.5)):
        ref = P.match_dsc_many(lo, his, dist, c)
        m = P.DscMatchMany(lo, his, dist, c)
        bounds = par.shard_bounds_weighted(m.pair_off, m.hi_n, world)
        shares = [par.pad_counts(par.match_dsc_many_local(m, r, world), m.p, world, bounds) for r in range(world)]
        assert [s.numel() for s in shares] == [max(e - s for s, e in bounds)] * world
        joined = par.join_counts(torch.stack(shares), m.p, bounds)
        assert torch.equal(joined, m.counts(0, m.p)), world
        table = m.rows(joined)
        got = par.match_dsc_many_sharded(lo, his, dist, c)                 # no process group: the world of one
        for g in range(len(his)):
            a, b = m.pair_off[g], m.pair_off[g + 1]
            assert torch.equal(table[a:b], ref[g][0]) and torch.equal(got[g][0], ref[g][0])
            assert np.array_equal(got[g][1], ref[g][1]) and np.array_equal(got[g][2], ref[g][2])
        if his[1] is few_hi and dist == 4 and c == 0.999:
            assert 0 < m.p < 8                                            # fewer pairs than ranks in a world of 8


def test_batch_of_more_than_64_structures(P):
    """70 structures: the per-structure records (64 bytes each, per side) pass 4096 bytes and still come home in the
    batch's one read-back."""
    lo, hi, few_hi, subset, none = _fixture_batch(P)
    his = [few_hi] * 35 + [none] + [D.rows_of(P, lo, [40, 3])] * 35
    got = _check_equal(P, lo, his, 4, 0.999)
    assert len(got) == 71 and got[35][0].shape == (0, 23) and all(got[g][0].shape[0] > 0 for g in range(71) if g != 35)
    z = _adversarial()["signed_zeros"]
    rng = np.random.default_rng(2)
    _check_segments(P, [z] * 80, [rng.random(len(z)) < 0.5 for _ in range(80)], 4.0)
