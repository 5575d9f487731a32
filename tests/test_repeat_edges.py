"""The per-pair repeatability kernels (mad_repeat_counts / mad_repeat_rows / mad_repeatability and the batched forms)
against the exact host reference tests/repeat_ref.py, bit for bit, at the edges of the lo grid and of the distance test.

Every case chooses the pairs, both clouds and the rotations itself: DscMatch / DscMatchMany get ``pairs=`` and a
substituted rotation table (``m.tb``), and ``match_dsc_many`` runs with the same pairs and table put in place of the
threshold matching and of the orientation tables."""
import numpy as np
import pytest

import repeat_ref as rr
from test_repeat_ref import exact_case, grid_counts

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")


@pytest.fixture(scope="module")
def P():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from mad_b200 import pipeline
    return pipeline


class Tables(object):
    """What DscMatch reads of the device tables: rf, rf_inv [zones * zones, 9] and ori_zones."""

    def __init__(self, rf, rf_inv, zones):
        self.rf_host = np.ascontiguousarray(rf, dtype=np.float64).reshape(-1, 9)
        self.rf_inv_host = np.ascontiguousarray(rf_inv, dtype=np.float64).reshape(-1, 9)
        self.rf = torch.from_numpy(self.rf_host).cuda()
        self.rf_inv = torch.from_numpy(self.rf_inv_host).cuda()
        self.ori_zones = int(zones)


def identity_tables():
    return Tables(np.eye(3)[None], np.eye(3)[None], 1)


def eqsp_tables():
    from mad_b200 import tables
    ot = tables.orientation_tables(112)
    return Tables(ot.rf, ot.rf_inv, 112)


def _table(P, subv, meta):
    subv = np.ascontiguousarray(subv, dtype=np.float64).reshape(-1, 3)
    meta = np.asarray(meta, dtype=np.int64).reshape(-1, 4)
    return P.FeatureTable(np.zeros((len(subv), 1024), dtype=np.int16), meta[:, 0], meta[:, 1], meta[:, 2], meta[:, 3], subv)


def _meta(n, zones, rng):
    return np.stack([np.arange(n), np.zeros(n, int), rng.integers(0, zones, n), rng.integers(0, zones, n)], 1)


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).tobytes()


def _ref(case, ph, pl, sc, hi_subv, hi_meta, hi_cloud, lo_cloud):
    tb = case["tb"]
    return rr.repeat(ph, pl, sc, hi_subv, case["lo_subv"], hi_meta, case["lo_meta"], tb.rf_host, tb.rf_inv_host, tb.ori_zones,
                     hi_cloud, lo_cloud, case["dist"])


def check_single(P, case):
    """DscMatch with the case's pairs and table: counts over sub-ranges, rows and table() against the reference; returns
    the reference counts."""
    ph, pl = np.asarray(case["pair_hi"], dtype=np.int64), np.asarray(case["pair_lo"], dtype=np.int64)
    sc = np.random.default_rng(len(ph)).random(len(ph))
    lo, hi = _table(P, case["lo_subv"], case["lo_meta"]), _table(P, case["hi_subv"], case["hi_meta"])
    pairs = (torch.from_numpy(ph.astype(np.int32)).cuda(), torch.from_numpy(pl.astype(np.int32)).cuda(),
             torch.from_numpy(sc).cuda())
    m = P.DscMatch(lo, hi, case["dist"], pairs=pairs)
    m.tb = case["tb"]
    hi_cloud, lo_cloud = m.hi_cloud.host(), m.lo_cloud.host()
    assert np.array_equal(hi_cloud, np.unique(np.asarray(case["hi_subv"], dtype=np.float64)[ph], axis=0))
    assert np.array_equal(lo_cloud, np.unique(np.asarray(case["lo_subv"], dtype=np.float64)[pl], axis=0))
    counts, rows = _ref(case, ph, pl, sc, case["hi_subv"], case["hi_meta"], hi_cloud, lo_cloud)
    full = m.counts(0, m.p)
    assert full.cpu().numpy().tolist() == counts.tolist()
    p = m.p
    for p0, p1 in [(0, 1), (p // 3, p // 2 + 1), (max(p - 3, 0), p)]:
        assert m.counts(p0, p1).cpu().numpy().tolist() == counts[p0:p1].tolist(), (p0, p1)
    assert _bits(m.rows(full).cpu().numpy()) == _bits(rows), "rows"
    assert _bits(m.table().cpu().numpy()) == _bits(rows), "table"
    return counts


def check_batch(P, monkeypatch, case, structures):
    """DscMatchMany over ``structures`` [(hi_subv, hi_meta, pair_hi, pair_lo)] against one lo side: counts over
    ranges that start and end inside structures and on their boundaries, rows and match_dsc_many, each structure
    against the reference with its own clouds."""
    his, ph, pl, offs = [], [], [], [0]
    for hs, hm, sh, sl in structures:
        his.append(_table(P, hs, hm))
        order = np.lexsort((np.asarray(sl), np.asarray(sh)))
        ph.append(np.asarray(sh, dtype=np.int64)[order] + offs[-1])
        pl.append(np.asarray(sl, dtype=np.int64)[order])
        offs.append(offs[-1] + len(hs))
    ph, pl = np.concatenate(ph), np.concatenate(pl)
    sc = np.random.default_rng(len(ph)).random(len(ph))
    lo = _table(P, case["lo_subv"], case["lo_meta"])
    pairs = (torch.from_numpy(ph.astype(np.int32)).cuda(), torch.from_numpy(pl.astype(np.int32)).cuda(),
             torch.from_numpy(sc).cuda())
    m = P.DscMatchMany(lo, his, case["dist"], pairs=pairs)
    m.tb = case["tb"]
    want_counts, want_rows = [], []
    for g, (hs, hm, _, _) in enumerate(structures):
        a, b = int(m.pair_off[g]), int(m.pair_off[g + 1])
        if a == b:
            continue
        hi_cloud = m.hi_clouds.cloud_of(g).cpu().numpy()
        lo_cloud = m.lo_clouds.cloud_of(g).cpu().numpy()
        c, r = _ref(case, ph[a:b] - offs[g], pl[a:b], sc[a:b], hs, hm, hi_cloud, lo_cloud)
        want_counts.append(c)
        want_rows.append(r)
    want_counts, want_rows = np.concatenate(want_counts), np.concatenate(want_rows)
    full = m.counts(0, m.p)
    assert full.cpu().numpy().tolist() == want_counts.tolist()
    cuts = sorted({int(v) + d for v in m.pair_off for d in (-1, 0, 1) if 0 <= int(v) + d <= m.p})
    for p0, p1 in zip(cuts[:-1], cuts[1:]):
        assert m.counts(p0, p1).cpu().numpy().tolist() == want_counts[p0:p1].tolist(), (p0, p1)
    if len(cuts) >= 4:
        assert m.counts(cuts[1], cuts[-2]).cpu().numpy().tolist() == want_counts[cuts[1]:cuts[-2]].tolist()
    rows = m.rows(full).cpu().numpy()
    assert _bits(rows) == _bits(want_rows), "rows"
    # match_dsc_many: the same pairs and rotation table in place of the threshold matching and the EQSP tables
    monkeypatch.setattr(P, "match_threshold", lambda *a, **k: pairs)
    monkeypatch.setattr(P, "device_tables", lambda dev: case["tb"])
    got = P.match_dsc_many(lo, his, case["dist"])
    monkeypatch.undo()
    for g in range(len(his)):
        a, b = int(m.pair_off[g]), int(m.pair_off[g + 1])
        assert _bits(got[g][0].cpu().numpy()) == _bits(rows[a:b]), g
    return want_counts, m.pair_off


# ---------------------------------------------------------------------------------------------
# the grid's borders: found by a seeded search, in one dimension (y = z = 0), identity rotation, both pair rows at the
# origin (so q is the hi anchor itself)
# ---------------------------------------------------------------------------------------------
def _ulps(x, k):
    """x moved k (an int array) ulps up."""
    return x + k * np.abs(np.spacing(x))


def border_configs(kind, dist, n, seed):
    """Up to n (lo xs, hi x) configurations, found by a seeded search, in which a lo point l lies within dist of the hi
    anchor q by the device's arithmetic (|RN(l - q)| < dist), or just not (low border).  The lo cloud holds the minimum
    m far below, the origin (the pair's lo row, which the origin hi anchor hits) and l; no other lo point is within
    reach of q.  With org = RN(m - dist) and cell coordinate RN(RN(x - org) / dist):
      interior: l < 0 near a cell edge, q just over dist below it, where a grid of cell dist puts l two cells above q;
      high:     l > 0 the maximum, just under a cell edge, q just under dist above it, where a grid of cell dist puts q
                in cell dims, outside the grid;
      low:      q around m - dist (l = m), a border a grid of cell dist already gets right."""
    rng = np.random.default_rng(seed)
    N = 200000
    m = -rng.uniform(20 * dist, 100 * dist, N)
    if kind == "interior":
        # l - org near k dist, where (k - 1) dist is near a power of two half the time: there the ulp of x - org
        # doubles between q's cell edge and l's, and a dist that is not a power of two adds the division's rounding
        k = np.where(rng.random(N) < 0.5, np.round(2.0 ** rng.integers(4, 9, N) / dist) + 1, rng.integers(5, 90, N))
        m = -(k * dist + rng.uniform(2.5 * dist, 10 * dist, N)) + dist
        org = m - dist
        l = _ulps(org + k * dist, -rng.integers(0, 10, N))
        q = _ulps(l - dist, rng.integers(-1, 4, N))
        keep = (np.abs(l - q) < dist) & (np.floor((l - org) / dist) - np.floor((q - org) / dist) >= 2)
    elif kind == "high":
        org = m - dist
        k = np.floor((rng.uniform(2.5 * dist, 10 * dist, N) - org) / dist) + 1
        l = _ulps(org + k * dist, -rng.integers(1, 7, N))
        q = _ulps(l + dist, -rng.integers(0, 5, N))
        keep = (np.abs(l - q) < dist) & (np.floor((q - org) / dist) >= np.floor((l - org) / dist) + 2)
    else:
        org = m - dist
        l = m
        q = _ulps(m - dist, rng.integers(-2, 4, N))
        keep = np.ones(N, dtype=bool)
    out = []
    for i in np.nonzero(keep)[0][:n]:
        lo = [m[i], 0.0, l[i]] if kind != "low" else [m[i], 0.0]
        if kind != "low":                       # the miss, restated with the device's +-1 search over a grid of cell dist
            pts = np.array([[x, 0.0, 0.0] for x in lo])
            assert grid_counts(np.array([[q[i], 0.0, 0.0], [0.0, 0.0, 0.0]]), pts, dist, dist) == 1
        out.append((lo, float(q[i])))
    return out


def _case(tb, lo_subv, lo_meta, dist, **kw):
    return dict(tb=tb, lo_subv=np.asarray(lo_subv, dtype=np.float64).reshape(-1, 3), lo_meta=lo_meta, dist=dist, **kw)


def _all_pairs(n_hi, n_lo):
    ph, pl = np.meshgrid(np.arange(n_hi), np.arange(n_lo), indexing="ij")
    return ph.ravel(), pl.ravel()


def _line(xs):
    return np.array([[x, 0.0, 0.0] for x in xs])


@pytest.mark.parametrize("dist", [4.0, 6.5, 4.1, 0.37])
@pytest.mark.parametrize("kind", ["interior", "high", "low"])
def test_grid_borders_equal_reference(P, monkeypatch, kind, dist):
    """Lo points within dist of an anchor two cells away (interior) or beyond the last cell (high) on a grid of cell
    dist, and anchors around min - dist (low).  A grid of cell dist counted one hit too few on the first two."""
    configs = border_configs(kind, dist, 6, seed=int(dist * 100) + len(kind))
    assert len(configs) == 6                                   # the search found its cases: the test is not vacuous
    tb = identity_tables()
    zero = np.zeros((1, 4), dtype=int)
    for lo_x, q in configs:
        lo_subv = _line(lo_x)
        hi_subv = _line([0.0, q])
        lo_meta, hi_meta = np.repeat(zero, len(lo_subv), 0), np.repeat(zero, 2, 0)
        ph, pl = _all_pairs(2, len(lo_subv))
        case = _case(tb, lo_subv, lo_meta, dist, hi_subv=hi_subv, hi_meta=hi_meta, pair_hi=ph, pair_lo=pl)
        counts = check_single(P, case)
        origin = list(zip(ph, pl)).index((0, 1))             # both pair rows at the origin: q is the anchor itself
        if kind != "low":
            assert counts[origin] == 2, (lo_x, q)
        other = (_line([1.5, 0.25]), np.repeat(zero, 2, 0), [0, 1, 1], [0, 0, 1])
        got, off = check_batch(P, monkeypatch, case, [other, (hi_subv, hi_meta, ph, pl)])
        assert got[int(off[1]):].tolist() == counts.tolist()


@pytest.mark.parametrize("dist, leg", [(5.0, (3.0, 4.0, 0.0)), (3.0, (2.0, 2.0, 1.0)), (5.0, (0.0, 3.0, 4.0))])
def test_distance_edges_on_dyadic_lattices(P, monkeypatch, dist, leg):
    """Anchors at exactly dist from a lo point (not counted), one ulp inside (counted), at distance 0, and at a distance
    whose exact value is below dist but whose computed value rounds to dist (not counted)."""
    lo = np.array([[0.0, 0.0, 0.0], [32.0, 0.0, 0.0], [0.0, -32.0, 16.0], [32.0, 32.0, 32.0]])
    leg = np.array(leg)
    inside = np.nextafter(dist, 0.0)
    anchors = [lo[0]]                                                   # distance 0 (the pair rows: q = anchor)
    for l in lo:
        for sgn in ([1, 1, 1], [-1, 1, -1], [1, -1, 1]):
            anchors.append(l + leg * sgn)                               # exactly dist
            anchors.append(l + np.roll(leg, 1) * sgn)
    anchors += [lo[0] + [inside, 0, 0], lo[0] - [0, inside, 0], lo[0] + [0, 0, inside],      # one ulp inside
                lo[0] + [np.nextafter(dist, 9.0), 0, 0]]                                    # one ulp outside
    below = np.nextafter(1.0, 0.0)
    anchors.append(lo[0] + [2.0, 2.0, below] if dist == 3.0 else lo[0] + [3.0, 4.0 * below, 0.0])
    hi = np.array(anchors)
    zero = np.zeros((1, 4), dtype=int)
    hi_meta, lo_meta = np.repeat(zero, len(hi), 0), np.repeat(zero, len(lo), 0)
    case = _case(identity_tables(), lo, lo_meta, dist, hi_subv=hi, hi_meta=hi_meta)
    # hi row 0 (the origin) against every lo row, every other hi row against the origin: both clouds complete
    case["pair_hi"] = np.r_[np.zeros(len(lo), dtype=int), np.arange(1, len(hi))]
    case["pair_lo"] = np.r_[np.arange(len(lo)), np.zeros(len(hi) - 1, dtype=int)]
    counts = check_single(P, case)
    h, _ = rr.anchor_hits(hi, lo, dist)
    assert counts[0] == 1 + 3 == np.count_nonzero(h)                    # origin + three one-ulp-inside anchors
    check_batch(P, monkeypatch, case, [(hi[:1], hi_meta[:1], [0], [1]), (hi, hi_meta, case["pair_hi"], case["pair_lo"])])


@pytest.mark.parametrize("dist", [4.0, 5.0, 3.0, 1.5])
def test_exact_arithmetic_equals_ckdtree_restatement(P, monkeypatch, dist):
    """Dyadic coordinates and signed-permutation rotation tables: every operation is exact, so the counts also equal
    the reference loop's (cKDTree) with no flips."""
    rng = np.random.default_rng(int(dist * 10))
    c = exact_case(rng, dist=dist)
    case = _case(Tables(c["rf"], c["rf_inv"], c["zones"]), c["lo_subv"], c["lo_meta"], dist, hi_subv=c["hi_subv"],
                 hi_meta=c["hi_meta"], pair_hi=c["pair_hi"], pair_lo=c["pair_lo"])
    counts = check_single(P, case)
    assert counts.tolist() == rr.ckdtree_counts(**c).tolist()
    assert 0 < counts.sum() < len(counts) * len(c["hi_cloud"])
    half = len(c["hi_subv"]) // 2
    sel = c["pair_hi"] >= half
    check_batch(P, monkeypatch, case, [(c["hi_subv"][:half], c["hi_meta"][:half], c["pair_hi"][~sel], c["pair_lo"][~sel]),
                                       (c["hi_subv"][half:], c["hi_meta"][half:], c["pair_hi"][sel] - half, c["pair_lo"][sel])])


@pytest.mark.parametrize("dist", [4.0, 6.5, 4.1, 0.37, 1e3])
def test_general_rotations_on_random_clouds(P, monkeypatch, dist):
    """The EQSP orientation tables, random clouds of 1 to about 2000 anchors; dist 0.37 makes many cells, 1e3 a 3x3x3
    grid."""
    tb = eqsp_tables()
    rng = np.random.default_rng(int(dist * 100))
    for n_hi, n_lo, scale in ((1, 1, 10.0), (7, 30, 8.0), (2000, 40, 15.0), (300, 600, 25.0)):
        lo = rng.normal(scale=scale, size=(n_lo, 3))
        hi = rng.normal(scale=scale, size=(n_hi, 3))
        # every hi row in one pair (the hi cloud is the used hi rows), a few rows in two
        ph = np.sort(np.r_[np.arange(n_hi), rng.integers(0, n_hi, 5)])
        pl = rng.integers(0, n_lo, len(ph))
        case = _case(tb, lo, _meta(n_lo, 112, rng), dist, hi_subv=hi, hi_meta=_meta(n_hi, 112, rng), pair_hi=ph, pair_lo=pl)
        counts = check_single(P, case)
        if n_hi > 100 and dist >= 4:
            assert counts.max() > 0
    n_hi = 60
    hi = rng.normal(scale=12.0, size=(n_hi, 3))
    lo = rng.normal(scale=12.0, size=(200, 3))
    hm = _meta(n_hi, 112, rng)
    case = _case(tb, lo, _meta(200, 112, rng), dist)
    check_batch(P, monkeypatch, case, [(hi[:20], hm[:20], np.arange(20), rng.integers(0, 200, 20)),
                                       (hi[20:21], hm[20:21], [0, 0, 0], [5, 6, 7]),                   # one-anchor hi cloud
                                       (hi[21:30], hm[21:30], [], []),                                   # no pairs
                                       (hi[30:], hm[30:], np.arange(30) % 30, rng.integers(0, 200, 30))])


def test_degenerate_grids(P, monkeypatch):
    """One lo point; a lo cloud flat along one axis; hi anchors that move far outside the grid (up to 1e15 A)."""
    rng = np.random.default_rng(9)
    tb = eqsp_tables()
    zero = np.zeros((1, 4), dtype=int)
    # one lo point, anchors around it
    one = _case(identity_tables(), [[3.0, -2.0, 7.5]], zero, 4.0, hi_subv=np.r_[[[0.0, 0.0, 0.0]], rng.normal(size=(50, 3)) * 3],
                hi_meta=np.repeat(zero, 51, 0), pair_hi=np.arange(51), pair_lo=np.zeros(51, dtype=int))
    assert check_single(P, one).max() > 0
    # flat along z
    lo = rng.normal(scale=10.0, size=(400, 3))
    lo[:, 2] = 1.25
    hi = rng.normal(scale=10.0, size=(300, 3))
    hi[:, 2] = rng.choice([1.25, 1.25 + 3.9, 1.25 - 4.2], 300)
    flat = _case(tb, lo, _meta(400, 112, rng), 4.0, hi_subv=hi, hi_meta=_meta(300, 112, rng), pair_hi=np.arange(300),
                 pair_lo=rng.integers(0, 400, 300))
    assert check_single(P, flat).max() > 0
    # far outside: anchors 1e3 .. 1e15 away from the pair's hi row
    far = np.r_[rng.normal(size=(20, 3)), np.outer(10.0 ** np.arange(3, 16), [1.0, -0.5, 0.25]),
                -np.outer(10.0 ** np.arange(3, 16), [0.3, 1.0, -1.0])]
    n = len(far)
    far_case = _case(tb, lo, _meta(400, 112, rng), 4.0, hi_subv=far, hi_meta=_meta(n, 112, rng), pair_hi=np.arange(n),
                     pair_lo=rng.integers(0, 400, n))
    check_single(P, far_case)
    check_batch(P, monkeypatch, far_case, [(hi[:5], flat["hi_meta"][:5], np.arange(5), np.arange(5)),
                                           (far, far_case["hi_meta"], far_case["pair_hi"], far_case["pair_lo"])])


def test_grid_just_below_2_31_cells(P):
    """A lo grid of dims (3, 3, 238609294), 2^31 - 2 cells, at the grid cell the repeatability uses; anchors hit and miss
    lo points in its last cells.  Needs about 9 GB of device memory, freed at the end."""
    cell = P.repeat_grid_cell(4.0)
    top = 238609291.5 * cell                                   # floor((top + cell) / cell) + 2 = 238609294
    lo = np.array([[0.0, 0.0, 0.0], [0.0, 0.0, top], [1.0, 2.0, top - 3.0], [3.0, 3.0, top - 10.0]])
    hi = np.array([[0.0, 0.0, 0.0], [0.0, 0.0, top + 3.99], [0.0, 0.0, top + 4.0], [1.0, 2.0, top - 6.5],
                   [2.5, 2.5, top - 10.0], [0.0, 0.0, top + 40.0], [0.0, 0.0, top - 20.0]])
    zero = np.zeros((1, 4), dtype=int)
    case = _case(identity_tables(), lo, np.repeat(zero, 4, 0), 4.0, hi_subv=hi, hi_meta=np.repeat(zero, len(hi), 0),
                 pair_hi=np.r_[np.zeros(4, dtype=int), np.arange(1, len(hi))], pair_lo=np.r_[np.arange(4), np.zeros(len(hi) - 1, dtype=int)])
    try:
        lo_t, hi_t = _table(P, lo, case["lo_meta"]), _table(P, hi, case["hi_meta"])
        m = P.DscMatch(lo_t, hi_t, 4.0, pairs=(torch.from_numpy(case["pair_hi"].astype(np.int32)).cuda(),
                                               torch.from_numpy(case["pair_lo"].astype(np.int32)).cuda(),
                                               torch.zeros(len(case["pair_hi"]), dtype=torch.float64, device="cuda")))
        assert m.lo_cloud.dims.tolist() == [3, 3, 238609294]
        del m
        counts = check_single(P, case)
        assert counts[0] == 4                                  # the origin, top + 3.99, top - 6.5 (to top - 3), top - 10
    finally:
        torch.cuda.empty_cache()
