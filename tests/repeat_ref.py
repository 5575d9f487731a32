"""Exact host reference of the per-pair repeatability (csrc/repeat.cu: mad_repeat_counts, mad_repeat_rows and the
batched forms).  No grid: every transformed hi anchor is compared with the whole lo cloud.

It evaluates the float64 sequence include/mad_b200.h states, with the fused operations rounded once:
    R[i][j] = fma(A[i][2], B[2][j], fma(A[i][1], B[1][j], A[i][0] B[0][j]))        A = inv(Rfinal_lo), B = Rfinal_hi
    d = p - subv_hi,   q[i] = fma(d[2], R[i][2], fma(d[1], R[i][1], d[0] R[i][0])) + subv_lo[i]
    e = l - q,         hit  = sqrt(fma(e[2], e[2], fma(e[1], e[1], e[0] e[0]))) < dist
    row[1] = (100 count) / H
so the counts and the 23-column rows it returns are those of the device bit for bit.

``fma`` is correctly rounded (tests/test_repeat_ref.py checks it against exact rational rounding): an error-free
product (Dekker), an error-free sum (Knuth) and Boldo and Melquiond's emulation with a sum rounded to odd.  It is exact
for operands whose product is zero or above 2^-960 in magnitude and whose values stay below 2^995 (no underflow or
overflow in the splitting); the tests stay far inside that range.

The distance test runs a plain float64 pass first.  Its e = RN(l - q) is the device's own, bit for bit (q is the exact
sequence's); only the three-term sum differs, NumPy's (e0 e0 + e1 e1) + e2 e2 against the fused chain.  Both are sums of
the same three non-negative products with at most three roundings each, so the two sums agree to a relative 4u and the
two rounded square roots to 8u (u = 2^-53), whatever the coordinates, as long as e e neither underflows nor overflows
(|e| between 2^-500 and 2^500, or 0: true for every coordinate in the tests, up to 1e15).  A distance of the plain pass
more than 2^-40 dist away from dist (2^13 times that bound) is therefore on the same side of dist as the device's; only
the few (anchor, lo point) candidates inside that band are evaluated again with the fused sum.
"""
import numpy as np

_SPLIT = 134217729.0                      # 2^27 + 1
BAND = 2.0 ** -40                         # relative half-width of the band of re-evaluated distances


def two_sum(a, b):
    """s + e == a + b exactly, s = RN(a + b)."""
    s = a + b
    bb = s - a
    return s, (a - (s - bb)) + (b - bb)


def _split(a):
    c = _SPLIT * a
    hi = c - (c - a)
    return hi, a - hi


def two_prod(a, b):
    """p + e == a b exactly, p = RN(a b)."""
    p = a * b
    ah, al = _split(a)
    bh, bl = _split(b)
    return p, ((ah * bh - p) + ah * bl + al * bh) + al * bl


def add_round_odd(a, b):
    """a + b rounded to odd: exact if representable, else the neighbour whose last significand bit is 1."""
    s, e = two_sum(a, b)
    even = (np.asarray(s).view(np.int64) & 1) == 0
    move = (e != 0) & even
    return np.where(move, np.nextafter(s, np.where(e > 0, np.inf, -np.inf)), s)


def fma(a, b, c):
    """RN(a b + c) with one rounding: the emulated FMA of Boldo and Melquiond, "Emulation of FMA and correctly rounded
    sums: proved algorithms using rounding to odd", IEEE Trans. Computers 57(4), 2008."""
    a, b, c = (np.asarray(v, dtype=np.float64) for v in (a, b, c))
    uh, ul = two_prod(a, b)
    th, tl = two_sum(c, uh)
    v = add_round_odd(tl, ul)
    r = th + v
    return np.where(r == 0, uh + c, r)            # an exact zero takes the sign IEEE gives a b + c (uh = a b then)


def pair_rotations(A, B):
    """R [P, 3, 3] of the pairs from A = inv(Rfinal_lo) [P, 3, 3] and B = Rfinal_hi [P, 3, 3]."""
    A, B = np.asarray(A, dtype=np.float64), np.asarray(B, dtype=np.float64)
    R = np.empty(np.broadcast(A, B).shape)
    for i in range(3):
        for j in range(3):
            R[..., i, j] = fma(A[..., i, 2], B[..., 2, j], fma(A[..., i, 1], B[..., 1, j], A[..., i, 0] * B[..., 0, j]))
    return R


def transform(cloud, shi, R, slo):
    """q [H, 3] of the hi cloud [H, 3] under the pair (shi, R, slo)."""
    d = np.asarray(cloud, dtype=np.float64) - shi
    return np.stack([fma(d[:, 2], R[i, 2], fma(d[:, 1], R[i, 1], d[:, 0] * R[i, 0])) + slo[i] for i in range(3)], 1)


def distance(e):
    """The device's distance of difference vectors e [..., 3] (e = l - q)."""
    return np.sqrt(fma(e[..., 2], e[..., 2], fma(e[..., 1], e[..., 1], e[..., 0] * e[..., 0])))


def anchor_hits(q, lo_cloud, dist, chunk=1 << 22):
    """(hit bool [H], nearest float64 [H]) of the transformed anchors q against the whole lo cloud.  nearest = the
    smallest computed distance; it is the device's value wherever it lies within the band around dist (elsewhere the
    plain pass's, within 8u of it)."""
    lo_cloud = np.asarray(lo_cloud, dtype=np.float64)
    H, L = len(q), len(lo_cloud)
    hit = np.zeros(H, dtype=bool)
    nearest = np.full(H, np.inf)
    lo_b, hi_b = dist * (1 - BAND), dist * (1 + BAND)
    step = max(1, chunk // max(L, 1))
    for a in range(0, H, step):
        qa = q[a:a + step]
        e = lo_cloud[None, :, :] - qa[:, None, :]
        plain = np.sqrt((e[..., 0] * e[..., 0] + e[..., 1] * e[..., 1]) + e[..., 2] * e[..., 2])
        band = (plain >= lo_b) & (plain <= hi_b)
        if band.any():
            plain[band] = distance(e[band])
        hit[a:a + step] = (plain < dist).any(1)
        nearest[a:a + step] = plain.min(1) if L else np.inf
    return hit, nearest


def repeat(pair_hi, pair_lo, pair_score, hi_subv, lo_subv, hi_meta, lo_meta, rf, rf_inv, zones, hi_cloud, lo_cloud, dist,
           detail=False):
    """(counts int64 [P], rows float64 [P, 23]) of the pairs (pair_hi, pair_lo, pair_score) of one structure, as
    mad_repeat_counts + mad_repeat_rows compute them: hi_subv / lo_subv float64 [D, 3], hi_meta / lo_meta int [D, 4]
    (index, oct_scale, main_bin, sec_bin), rf / rf_inv float64 [zones * zones, 9] (or [.., 3, 3]), hi_cloud [H, 3],
    lo_cloud [L, 3].  detail=True also returns per pair the (hit, nearest) arrays of ``anchor_hits``."""
    ph, pl = np.asarray(pair_hi, dtype=np.int64), np.asarray(pair_lo, dtype=np.int64)
    hi_meta, lo_meta = np.asarray(hi_meta, dtype=np.int64), np.asarray(lo_meta, dtype=np.int64)
    hi_subv, lo_subv = np.asarray(hi_subv, dtype=np.float64), np.asarray(lo_subv, dtype=np.float64)
    rf, rf_inv = np.asarray(rf, dtype=np.float64).reshape(-1, 3, 3), np.asarray(rf_inv, dtype=np.float64).reshape(-1, 3, 3)
    hi_cloud = np.asarray(hi_cloud, dtype=np.float64).reshape(-1, 3)
    P, H = len(ph), len(hi_cloud)
    R = pair_rotations(rf_inv[lo_meta[pl, 2] * zones + lo_meta[pl, 3]], rf[hi_meta[ph, 2] * zones + hi_meta[ph, 3]])
    counts = np.zeros(P, dtype=np.int64)
    details = []
    for k in range(P):
        q = transform(hi_cloud, hi_subv[ph[k]], R[k], lo_subv[pl[k]])
        hit, nearest = anchor_hits(q, lo_cloud, dist)
        counts[k] = np.count_nonzero(hit)
        if detail:
            details.append((hit, nearest))
    rows = np.empty((P, 23))
    rows[:, 0] = pair_score
    rows[:, 1] = (100 * counts).astype(np.float64) / np.float64(H) if P else 0
    rows[:, 2:5] = lo_meta[pl, :3]
    rows[:, 5:8] = hi_meta[ph, :3]
    rows[:, 8:11] = hi_subv[ph]
    rows[:, 11:14] = lo_subv[pl]
    rows[:, 14:] = R.reshape(P, 9)
    return (counts, rows, details) if detail else (counts, rows)


def ckdtree_counts(pair_hi, pair_lo, pair_score, hi_subv, lo_subv, hi_meta, lo_meta, rf, rf_inv, zones, hi_cloud, lo_cloud,
                   dist):
    """The counts as the reference loop computes them (mad/MaD.py:431-447, oracle/mad_oracle.py match_dsc): R from np.dot,
    the cloud moved with np.dot, cKDTree.query with distance_upper_bound and ``distances < dist``.  Equal to ``repeat``'s
    where every operation is exact; elsewhere a count may differ where a distance is within ulps of dist."""
    from scipy.spatial import cKDTree
    rf, rf_inv = np.asarray(rf, dtype=np.float64).reshape(-1, 3, 3), np.asarray(rf_inv, dtype=np.float64).reshape(-1, 3, 3)
    hi_meta, lo_meta = np.asarray(hi_meta), np.asarray(lo_meta)
    hi_subv, lo_subv = np.asarray(hi_subv, dtype=np.float64), np.asarray(lo_subv, dtype=np.float64)
    tree = cKDTree(np.asarray(lo_cloud, dtype=np.float64))
    out = []
    for h, l in zip(pair_hi, pair_lo):
        R = np.dot(rf_inv[lo_meta[l, 2] * zones + lo_meta[l, 3]], rf[hi_meta[h, 2] * zones + hi_meta[h, 3]])
        cur = np.dot(np.asarray(hi_cloud, dtype=np.float64) - hi_subv[h], R.T) + lo_subv[l]
        d, _ = tree.query(cur, distance_upper_bound=dist)
        out.append(np.count_nonzero(d < dist))
    return np.array(out, dtype=np.int64)
