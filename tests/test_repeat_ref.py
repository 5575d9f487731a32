"""The exact host reference of the per-pair repeatability (tests/repeat_ref.py) on its own, without a device: its fused
operation against exact rational rounding, its counts against a cKDTree restatement of the reference loop where every
operation is exact, and the grid miss it exists to catch."""
from fractions import Fraction

import numpy as np

import repeat_ref as rr


def _exact_fma(a, b, c):
    return float(Fraction(a) * Fraction(b) + Fraction(c))


def test_fma_is_exact_rational_rounding():
    rng = np.random.default_rng(0)
    n = 4000
    a = rng.normal(size=n) * 10.0 ** rng.integers(-12, 13, n)
    b = rng.normal(size=n) * 10.0 ** rng.integers(-12, 13, n)
    ab = a * b
    cases = {
        "random": rng.normal(size=n) * 10.0 ** rng.integers(-12, 13, n),
        "cancelling": -ab,                                                 # the result is the rounding error of a b
        "nearly_cancelling": -ab * (1 + rng.integers(-8, 9, n) * 2.0 ** -52),
        "one_ulp_off": np.nextafter(-ab, np.where(rng.random(n) < 0.5, np.inf, -np.inf)),
        "tiny_addend": ab * 2.0 ** -60 * rng.normal(size=n),               # decides a tie or near-tie of a b alone
        "zeros": np.where(rng.random(n) < 0.5, 0.0, -0.0),
    }
    for name, c in cases.items():
        got = rr.fma(a, b, c)
        want = np.array([_exact_fma(x, y, z) for x, y, z in zip(a, b, c)])
        assert np.array_equal(got, want), name
    # exact zeros keep IEEE's sign: -0 only for (-0) + (-0)
    z = np.array([0.0, -0.0, 1.0, -1.0])
    za, zb, zc = (g.ravel() for g in np.meshgrid(z, z, [0.0, -0.0], indexing="ij"))
    want = np.array([float(np.float64(x) * np.float64(y)) + w for x, y, w in zip(za, zb, zc)])
    assert rr.fma(za, zb, zc).tobytes() == want.tobytes()
    assert rr.fma(np.array([3.0]), np.array([0.5]), np.array([-1.5])).tobytes() == np.array([0.0]).tobytes()
    # products with long exact expansions and addends far below their last bit, of either sign
    h = (1.0 + rng.integers(1, 1 << 20, n) * 2.0 ** -26)
    got = rr.fma(h, h, np.full(n, 2.0 ** -80))
    want = np.array([_exact_fma(x, x, 2.0 ** -80) for x in h])
    assert np.array_equal(got, want)
    got = rr.fma(h, h, np.full(n, -2.0 ** -80))
    want = np.array([_exact_fma(x, x, -2.0 ** -80) for x in h])
    assert np.array_equal(got, want)


def signed_permutations(zones, rng):
    """rf [zones * zones, 3, 3] of random signed permutation matrices and rf_inv = their transposes (exact inverses)."""
    perms = [(0, 1, 2), (0, 2, 1), (1, 0, 2), (1, 2, 0), (2, 0, 1), (2, 1, 0)]
    rf = np.zeros((zones * zones, 3, 3))
    for k in range(zones * zones):
        p = perms[rng.integers(0, 6)]
        rf[k, [0, 1, 2], p] = rng.choice([-1.0, 1.0], 3)
    return rf, np.ascontiguousarray(rf.transpose(0, 2, 1))


def exact_case(rng, zones=3, n_hi=40, n_lo=50, dist=4.0):
    """Dyadic inputs on which every operation of the sequence is exact: coordinates are multiples of 1/4 below 2^6,
    rotations signed permutations, so R, q, e and e e are exact, and a squared distance below dist^2 lies at least 1/16
    below it (its square root then more than an ulp below dist)."""
    hi_subv = rng.integers(-64, 64, size=(n_hi, 3)) / 4.0
    lo_subv = rng.integers(-64, 64, size=(n_lo, 3)) / 4.0
    hi_meta = np.stack([np.arange(n_hi), np.zeros(n_hi, int), rng.integers(0, zones, n_hi), rng.integers(0, zones, n_hi)], 1)
    lo_meta = np.stack([np.arange(n_lo), np.zeros(n_lo, int), rng.integers(0, zones, n_lo), rng.integers(0, zones, n_lo)], 1)
    rf, rf_inv = signed_permutations(zones, rng)
    pairs = sorted({(int(h), int(l)) for h, l in zip(rng.integers(0, n_hi, 150), rng.integers(0, n_lo, 150))})
    ph, pl = np.array(pairs).T
    return dict(pair_hi=ph, pair_lo=pl, pair_score=rng.random(len(ph)), hi_subv=hi_subv, lo_subv=lo_subv, hi_meta=hi_meta,
                lo_meta=lo_meta, rf=rf, rf_inv=rf_inv, zones=zones, hi_cloud=np.unique(hi_subv[ph], axis=0),
                lo_cloud=np.unique(lo_subv[pl], axis=0), dist=dist)


def test_counts_equal_ckdtree_restatement_where_everything_is_exact():
    rng = np.random.default_rng(1)
    for dist in (4.0, 5.0, 3.0, 1.5):
        case = exact_case(rng, dist=dist)
        counts, rows = rr.repeat(**case)
        assert np.array_equal(counts, rr.ckdtree_counts(**case)), dist
        assert 0 < counts.sum() < len(counts) * len(case["hi_cloud"]), dist     # neither all misses nor all hits
        assert np.array_equal(rows[:, 1], 100 * counts / len(case["hi_cloud"]))


def grid_counts(q, lo_cloud, dist, cell):
    """NumPy restatement of the device's search: the grid of cell ``cell`` over the lo cloud (org = min - cell,
    dims = floor((max - org) / cell) + 2), the cell of q by the same formulas, the cells at +-1 of it."""
    org = lo_cloud.min(0) - cell
    dims = np.floor((lo_cloud.max(0) - org) / cell).astype(np.int64) + 2
    cl = np.floor((lo_cloud - org) / cell).astype(np.int64)
    n = 0
    for x in q:
        c = np.floor((x - org) / cell).astype(np.int64)
        if (c < 0).any() or (c >= dims).any():
            continue
        near = (np.abs(cl - c) <= 1).all(1)
        n += bool((rr.distance(lo_cloud[near] - x) < dist).any())
    return n


def test_reference_finds_the_neighbour_a_grid_of_cell_dist_misses():
    """cell = dist = 4, identity rotation, both pair rows at the origin (so q is the hi anchor): p - q =
    3.999999999999999 < 4, but q falls in cell 15 and p in cell 17."""
    lo = np.array([[-71.53692888964844, 0, 0], [-7.5369288896484425, 0, 0], [0.0, 0, 0]])
    hi = np.array([[-11.536928889648442, 0, 0], [0.0, 0, 0]])
    eye = np.eye(3)[None]
    meta = np.zeros((1, 4), dtype=int)
    kw = dict(hi_subv=np.zeros((1, 3)), lo_subv=np.zeros((1, 3)), hi_meta=meta, lo_meta=meta, rf=eye, rf_inv=eye, zones=1,
              hi_cloud=hi, lo_cloud=lo, dist=4.0)
    counts, rows = rr.repeat([0], [0], [1.0], **kw)
    assert counts.tolist() == [2] and rows[0, 1] == 100.0
    assert rr.ckdtree_counts([0], [0], [1.0], **kw).tolist() == [2]
    assert grid_counts(hi, lo, 4.0, 4.0) == 1                           # the +-1 search over a grid of cell dist
    assert grid_counts(hi, lo, 4.0, 4.0 * (1 + 2.0 ** -16)) == 2        # the cell the repeatability grid now uses
    q = hi[0, 0]
    org = lo[:, 0].min() - 4.0
    assert np.floor((q - org) / 4.0) == 15 and np.floor((lo[1, 0] - org) / 4.0) == 17


def test_anchor_hits_band_matches_the_fused_sum_everywhere():
    """The plain pass decides only outside the band; inside and outside, the verdicts equal the fused sum's on every
    (anchor, lo point), on general coordinates with distances clustered around dist."""
    rng = np.random.default_rng(2)
    lo = rng.normal(scale=50.0, size=(300, 3))
    dirs = rng.normal(size=(300, 3))
    dirs /= np.sqrt((dirs * dirs).sum(1))[:, None]
    for dist in (4.0, 6.5, 0.37):
        q = lo + dirs * dist * (1 + rng.integers(-4, 5, size=(300, 1)) * 2.0 ** -52)
        hit, nearest = rr.anchor_hits(q, lo, dist)
        full = rr.distance(lo[None, :, :] - q[:, None, :])
        assert np.array_equal(hit, (full < dist).any(1)), dist
        band = np.abs(nearest - dist) <= rr.BAND * dist
        assert np.array_equal(nearest[band], full.min(1)[band]) and band.sum() > 200, dist
