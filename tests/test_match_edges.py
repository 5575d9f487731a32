"""Descriptor matching at its edges, against an exact host reference of the matching contract.

The contract (include/mad_b200.h, a15): score(i, j) = dot(hi_i, lo_j) / sqrt(|hi_i|^2 |lo_j|^2) in float64 from the exact
integer dot product and squared norms (multiply, sqrt, divide: each correctly rounded), 0 if either row is zero.
Threshold mode: every (i, j) with score > cc in row-major order.  Top-k mode: per hi row the k best lo rows by (score
descending, index ascending), -1 / -inf padded.  The reference below computes exactly that, independently of every kernel,
and each check asserts identity: indices, order and float64 scores bit for bit.

The inputs are built to hit what random descriptors never do: scores exactly on cc, exact ties and one-ulp near-ties
(lo rows b and m b have the same cosine with any hi row, but their float64 scores may differ by one ulp) straddling the
k-th place, zero rows, entries at 255 and dot products up to 66 585 600, entries beyond what the uint8 and fp16 kernels
can take, and shapes at tile, CTA-pair and segment edges.
"""
import os

import numpy as np
import pytest

torch = pytest.importorskip("torch")

gpu = pytest.mark.gpu
IMPLS = (0, 1, 2)
L = 1024


@pytest.fixture(scope="module")
def P():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from mad_b200 import pipeline
    return pipeline


# ---------------------------------------------------------------------------------------------
# exact host reference
# ---------------------------------------------------------------------------------------------
def ref_scores(hi, lo):
    """float64 scores of every (hi, lo) pair.  The float64 product is exact: integer terms whose partial sums stay below
    2^53 (true for any int16 set whose squared norms fit int32)."""
    dot = hi.astype(np.float64) @ lo.astype(np.float64).T
    n_hi = (hi.astype(np.int64) ** 2).sum(1).astype(np.float64)
    n_lo = (lo.astype(np.int64) ** 2).sum(1).astype(np.float64)
    p = n_hi[:, None] * n_lo[None, :]
    out = np.zeros_like(dot)
    nz = p > 0.0
    out[nz] = dot[nz] / np.sqrt(p[nz])
    return out


def ref_threshold(s, cc):
    ph, pl = np.nonzero(s > cc)
    return ph.astype(np.int32), pl.astype(np.int32), s[ph, pl]


def ref_topk(s, k, base=0):
    m, n = s.shape
    idx = np.full((m, k), -1, dtype=np.int32)
    sc = np.full((m, k), -np.inf)
    kk = min(k, n)
    for r0 in range(0, m, 2048):
        blk = s[r0:r0 + 2048]
        order = np.argsort(-blk, axis=1, kind="stable")[:, :kk]      # stable: equal scores keep ascending index
        idx[r0:r0 + 2048, :kk] = order + base
        sc[r0:r0 + 2048, :kk] = np.take_along_axis(blk, order, 1)
    return idx, sc


def fp16_exact(hi, lo):
    """The fp16 kernel's fp32 sums are exact for entries in [0, 2048] with max |hi|^2 max |lo|^2 <= 2^48 (every dot
    product <= 2^24 by Cauchy-Schwarz); it refuses other sets."""
    n2 = lambda x: int((x.astype(np.int64) ** 2).sum(1).max()) if len(x) else 0
    return min(hi.min(), lo.min()) >= 0 and max(hi.max(), lo.max()) <= 2048 and n2(hi) * n2(lo) <= 1 << 48


def impls_for(P, hi, lo, dh, dl):
    """The implementations that accept the pair of sets; where the fp16 kernel does not, check that it refuses."""
    if fp16_exact(hi, lo):
        return IMPLS
    from mad_b200._lib import MadError
    with pytest.raises(MadError):
        P.match_threshold(dh, dl, 0.6, impl=2)
    with pytest.raises(MadError):
        P.match_topk(dh, dl, 8, impl=2)
    return (0, 1)


def assert_pairs(got, want):
    ph, pl, sc = (t.cpu().numpy() for t in got)
    assert np.array_equal(ph, want[0]) and np.array_equal(pl, want[1]), "pair lists differ (%d vs %d pairs)" % (len(ph), len(want[0]))
    assert np.array_equal(sc.view(np.int64), want[2].view(np.int64)), "scores differ"


def assert_topk(got, want):
    gi, gs = (t.cpu().numpy() for t in got)
    bad = np.nonzero((gi != want[0]).any(1) | (gs.view(np.int64) != want[1].view(np.int64)).any(1))[0]
    assert len(bad) == 0, "%d rows differ, first %d: got %s %s, want %s %s" % (
        len(bad), bad[0], gi[bad[0]], gs[bad[0]], want[0][bad[0]], want[1][bad[0]])


def assert_ordered(idx, sc):
    """Every row non-increasing in score, ascending index among equal scores, padding last."""
    idx, sc = idx.cpu().numpy().astype(np.int64), sc.cpu().numpy()
    a, b = sc[:, :-1], sc[:, 1:]
    ia, ib = idx[:, :-1], idx[:, 1:]
    ok = (a > b) | ((a == b) & ((ib < 0) | ((ia >= 0) & (ia < ib))))
    assert ok.all()


# ---------------------------------------------------------------------------------------------
# inputs
# ---------------------------------------------------------------------------------------------
def noise(rng, n, vmax=255):
    """Rows of mixed density and range: sparse ones score near 0 with everything, dense ones near 0.75."""
    out = np.zeros((n, L), dtype=np.int16)
    for r in range(n):
        dens = rng.choice([0.02, 0.1, 1.0])
        top = int(rng.choice([3, 64, vmax]))
        m = rng.random(L) < dens
        out[r, m] = rng.integers(0, top + 1, m.sum())
    return out


def tie_sets(rng, m, n):
    """lo: multiples m b (entries <= 255) of a few base rows b, duplicates, zero rows, rows orthogonal to everything
    else, interleaved with noise; hi: noisy copies of the bases, exact bases and a zero row.  Every hi row built on a
    base has a run of exactly tied / one-ulp apart scores at the top of its list."""
    nb = 6
    base = np.zeros((nb, L), dtype=np.int16)
    for b in range(nb):
        sup = rng.choice(L - 64, 200, replace=False)                  # last 64 columns stay free for the orthogonal rows
        base[b, sup] = rng.integers(1, 37, 200)                         # 7 * 36 = 252
    group = [(b, mul) for b in range(nb) for mul in (1, 2, 3, 5, 6, 7, 4, 1)]      # (b, 1) twice: a duplicate
    lo = noise(rng, n, 64)
    slots = rng.permutation(n)
    for t, (b, mul) in enumerate(group):
        if t < n:
            lo[slots[t]] = base[b] * mul
    for t in range(len(group), min(len(group) + 6, n)):
        lo[slots[t]] = 0
    for t in range(len(group) + 6, min(len(group) + 12, n)):
        lo[slots[t]] = 0
        lo[slots[t], L - 64 + (t % 64)] = 200                           # orthogonal to every base
    hi = noise(rng, m, 64)
    for r in range(m):
        kind = r % 4
        if kind < 2:
            b = base[r % nb].astype(np.int32)
            hi[r] = np.clip(b + rng.integers(-2, 3, L) * (b > 0), 0, 255) if kind == 0 else b
    hi[m // 2] = 0
    return hi, lo


_REF = {}


def cached(key, fn):
    if key not in _REF:
        _REF[key] = fn()
    return _REF[key]


def sets(P, hi, lo):
    return P.DescriptorSet(hi), P.DescriptorSet(lo)


# ---------------------------------------------------------------------------------------------
# A. the threshold boundary
# ---------------------------------------------------------------------------------------------
def boundary_pairs():
    """(hi row, lo row) whose float64 score is known exactly: 3-4-5 (0.6, the default cc), (1,1,1,1).(1,0,0,0) = 0.5, and
    pairs of small integer vectors from a seeded search (their scores s are what the kernels must put exactly on cc)."""
    out = []
    a = np.zeros(L, np.int16); a[:2] = (3, 4)
    b = np.zeros(L, np.int16); b[0] = 1
    out.append((a, b))
    a = np.zeros(L, np.int16); a[:4] = 1
    out.append((a, b.copy()))
    rng = np.random.default_rng(1234)
    while len(out) < 6:
        u = np.zeros(L, np.int16); v = np.zeros(L, np.int16)
        u[:8] = rng.integers(0, 12, 8)
        v[:8] = rng.integers(0, 12, 8)
        if u.any() and v.any():
            out.append((u, v))
    return out


HI_AT = (0, 127, 128, 255, 256)
LO_AT = (0, 31, 32, 127, 128, 255, 256)


def boundary_case(j, m=300, n=300):
    a, b = boundary_pairs()[j]
    rng = np.random.default_rng(100 + j)
    hi, lo = noise(rng, m), noise(rng, n)
    for r in HI_AT + (m - 1,):
        hi[r] = a
    for c in LO_AT + (n - 1,):
        lo[c] = b
    s = float(ref_scores(a[None], b[None])[0, 0])
    return hi, lo, s


@gpu
@pytest.mark.parametrize("j", range(6))
def test_threshold_on_the_boundary(P, j):
    hi, lo, s = boundary_case(j)
    if j == 0:
        assert s == 0.6
    if j == 1:
        assert s == 0.5
    ref = ref_scores(hi, lo)
    dh, dl = sets(P, hi, lo)
    impls = impls_for(P, hi, lo, dh, dl)
    for cc in (s, np.nextafter(s, -np.inf), np.nextafter(s, np.inf)):
        want = ref_threshold(ref, cc)
        assert (ref[HI_AT[0], LO_AT[0]] > cc) == (cc < s)             # the planted pairs sit exactly on the boundary
        for impl in impls:
            assert_pairs(P.match_threshold(dh, dl, float(cc), impl=impl), want)
        # compact form: exact int32 dots, host scores with the device's operations
        ph, pl, dot = P.match_threshold(dh, dl, float(cc), impl=0, want="dot")
        ph, pl = ph.cpu().numpy(), pl.cpu().numpy()
        sc = P.scores_from_dots(ph, pl, dot.cpu().numpy(), dh.norm2.cpu().numpy(), dl.norm2.cpu().numpy())
        assert np.array_equal(ph, want[0]) and np.array_equal(pl, want[1])
        assert np.array_equal(sc.view(np.int64), want[2].view(np.int64))


# ---------------------------------------------------------------------------------------------
# B. cc at its edges: negative, zero, one, just below one
# ---------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("m,n", [(200, 300), (100, 130)])
def test_threshold_cc_edge_values(P, m, n):
    rng = np.random.default_rng(m + n)
    hi, lo = noise(rng, m), noise(rng, n)
    hi[[0, 57, m - 1]] = 0                                          # zero rows on both sides score 0 with everything
    lo[[0, 33, n - 1]] = 0
    hi[5], hi[130 % m] = lo[7], lo[n - 2]                             # identical rows: score exactly 1.0
    hi[9] = np.minimum(lo[7].astype(np.int32) * 2, 255)              # a multiple of lo[7] except where it clips
    ref = ref_scores(hi, lo)
    assert ref[5, 7] == 1.0 and ref[0, 0] == 0.0
    dh, dl = sets(P, hi, lo)
    impls = impls_for(P, hi, lo, dh, dl)
    for cc in (-0.5, 0.0, 1.0, np.nextafter(1.0, 0.0)):
        want = ref_threshold(ref, cc)
        for impl in impls:
            assert_pairs(P.match_threshold(dh, dl, float(cc), impl=impl), want)


# ---------------------------------------------------------------------------------------------
# C. exact ties and one-ulp near-ties at the k-th place
# ---------------------------------------------------------------------------------------------
TIE_K = (1, 2, 3, 7, 8, 9, 16, 31, 32)


@gpu
@pytest.mark.parametrize("m,n", [(100, 1500), (300, 2000)])
@pytest.mark.parametrize("local", [None, "0"])
def test_topk_ties(P, m, n, local):
    """local: the top-8 kernel keeps the first tiles of a sweep in thread-local lists and hands later ones to its drain
    warps; "0" sends every tile through the drain warps (both insertion sites have their own near-tie branch)."""
    hi, lo = tie_sets(np.random.default_rng(m), m, n)
    ref = cached(("ties", m, n), lambda: ref_scores(hi, lo))
    srt = np.sort(ref, 1)[:, ::-1]
    # the inputs do what they are for: exact ties and one-ulp neighbours at the top of the lists
    assert (srt[:, 0] == srt[:, 1]).sum() > m // 4
    assert (np.abs(srt[:, :8] - srt[:, 1:9]) <= np.spacing(srt[:, :8]) * 1.01).sum() > m
    dh, dl = sets(P, hi, lo)
    assert fp16_exact(hi, lo)
    old = os.environ.get("MAD_TOPK_LOCAL")
    if local is not None:
        os.environ["MAD_TOPK_LOCAL"] = local
    try:
        for k in TIE_K:
            want = ref_topk(ref, k)
            for impl in (IMPLS if local is None else (0,)):
                got = P.match_topk(dh, dl, k, impl=impl)
                assert_ordered(*got)
                assert_topk(got, want)
    finally:
        if local is not None:
            if old is None:
                del os.environ["MAD_TOPK_LOCAL"]
            else:
                os.environ["MAD_TOPK_LOCAL"] = old


# ---------------------------------------------------------------------------------------------
# D. shape x k sweep (one-CTA kernel vs CTA pairs, N < k, several lo segments, the tail wave)
# ---------------------------------------------------------------------------------------------
SWEEP_M = (1, 127, 128, 129, 255, 256, 257, 383)
SWEEP_N = (1, 7, 8, 9, 127, 128, 129, 255, 256, 257, 4099)
SWEEP_K = (1, 3, 8, 9, 32)


@gpu
@pytest.mark.parametrize("m", SWEEP_M)
def test_shape_sweep(P, m):
    rng = np.random.default_rng(7000 + m)
    hi_all, lo_all = tie_sets(rng, m, max(SWEEP_N))
    ref_all = cached(("sweep", m), lambda: ref_scores(hi_all, lo_all))
    dh = P.DescriptorSet(hi_all)
    for n in SWEEP_N:
        lo = np.ascontiguousarray(lo_all[-n:])                      # the last n rows: ties and zero rows at varying places
        ref = ref_all[:, -n:]
        dl = P.DescriptorSet(lo)
        want = ref_threshold(ref, 0.6)
        for impl in IMPLS:
            assert_pairs(P.match_threshold(dh, dl, 0.6, impl=impl), want)
        for k in SWEEP_K:
            for base in (0, 123457):
                want = ref_topk(ref, k, base)
                for impl in IMPLS:
                    assert_topk(P.match_topk(dh, dl, k, lo_index_base=base, impl=impl), want)


@gpu
def test_topk_tail_wave(P):
    """74 full CTA pairs + 300 rows: the rows of the poorly filled last wave get a launch of their own, with the lo axis
    cut into segments; the full waves keep one segment, so their later tiles go through the drain warps."""
    m, n = 74 * 256 + 300, 3000
    rng = np.random.default_rng(99)
    hi0, lo = tie_sets(rng, 2048, n)
    hi = np.concatenate([np.roll(hi0, 5 * r, axis=0) for r in range((m + 2047) // 2048)])[:m]
    hi[m - 5] = 0
    ref = cached("tail", lambda: ref_scores(hi, lo))
    want = ref_topk(ref, 3, 11)
    dh, dl = sets(P, hi, lo)
    for impl in IMPLS:
        assert_topk(P.match_topk(dh, dl, 3, lo_index_base=11, impl=impl), want)


# ---------------------------------------------------------------------------------------------
# E. entry range
# ---------------------------------------------------------------------------------------------
@gpu
def test_entries_at_255(P):
    """All-255 rows (|.|^2 = dot = 66 585 600, the largest the uint8 path sees: 27-bit |lo|^2 field and dot << 35 of the
    top-8 staging, fp32 pre-filter at its largest values) and rows with a single 255."""
    rng = np.random.default_rng(255)
    m, n = 260, 700
    hi, lo = noise(rng, m), noise(rng, n)
    for r in (0, 3, 128, 200, m - 1):
        hi[r] = 255
    for c in (1, 2, 128, 255, 256, 300, 600, n - 1):
        lo[c] = 255
    for r in (4, 129):
        hi[r] = 0
        hi[r, r] = 255
    for c in (5, 6, 400, 401, 640):
        lo[c] = 0
        lo[c, c % L] = 255
    lo[7] = 254
    lo[8] = 0
    lo[8, 1::2] = 255                                               # half the entries 255: cosine 1/sqrt(2) with all-255
    ref = ref_scores(hi, lo)
    assert ref[0, 1] == 1.0
    dh, dl = sets(P, hi, lo)
    impls = impls_for(P, hi, lo, dh, dl)
    for cc in (0.6, float(ref[0, 8]), float(np.nextafter(ref[0, 8], 0.0))):
        want = ref_threshold(ref, cc)
        for impl in impls:
            assert_pairs(P.match_threshold(dh, dl, cc, impl=impl), want)
    for k in (1, 8, 9):
        want = ref_topk(ref, k)
        for impl in impls:
            assert_topk(P.match_topk(dh, dl, k, impl=impl), want)


@gpu
@pytest.mark.parametrize("kind", ["dense", "sparse"])
def test_entries_above_255(P, kind):
    """Entries of 256..2048.  dense: odd entries of about 260-300 in every position, dot products near 8e7 > 2^24 -- the
    fp32 sums of the fp16 kernel would round them, so the product must not use it and impl 2 must refuse.  sparse: a few
    entries up to 2048 with every dot product <= 2^24, where the fp16 kernel is exact.  The product path (impl None) must
    equal the reference."""
    from mad_b200._lib import MadError
    rng = np.random.default_rng(300)
    m, n = 150, 400
    if kind == "dense":
        hi = (rng.integers(130, 150, (m, L)) * 2 + 1).astype(np.int16)
        lo = (rng.integers(130, 150, (n, L)) * 2 + 1).astype(np.int16)
        lo[:50] = hi[:50]
    else:
        hi, lo = np.zeros((m, L), np.int16), np.zeros((n, L), np.int16)
        for a in (hi, lo):
            for r in range(len(a)):
                c = rng.choice(L, 4, replace=False)
                a[r, c] = rng.integers(1, 2049, 4)
        lo[:50] = hi[:50]
    ref = ref_scores(hi, lo)
    dh, dl = sets(P, hi, lo)
    for cc in (0.6, 0.95):
        want = ref_threshold(ref, cc)
        for impl in (None, 1, 2):
            try:
                got = P.match_threshold(dh, dl, cc, impl=impl)
            except MadError:
                assert impl == 2 and not fp16_exact(hi, lo)
                continue
            assert impl != 2 or fp16_exact(hi, lo)
            assert_pairs(got, want)
    for k in (3, 8, 9):
        want = ref_topk(ref, k)
        for impl in (None, 1, 2):
            try:
                got = P.match_topk(dh, dl, k, impl=impl)
            except MadError:
                assert impl == 2 and not fp16_exact(hi, lo)
                continue
            assert impl != 2 or fp16_exact(hi, lo)
            assert_topk(got, want)
    # fresh sets: the product path's first call does not know the maxima yet (optimistic uint8 launch, then re-dispatch)
    assert_pairs(P.match_threshold(hi, lo, 0.6), ref_threshold(ref, 0.6))
    assert_topk(P.match_topk(hi, lo, 8), ref_topk(ref, 8))


@gpu
@pytest.mark.parametrize("kind", ["negative", "norm"])
def test_non_descriptor_sets_are_refused(P, kind):
    """A negative entry, or a squared norm >= 2^31 (int32 norms and dot products would overflow), is not a descriptor
    set: every path raises."""
    from mad_b200._lib import MadError
    rng = np.random.default_rng(5)
    good = noise(rng, 40)
    bad = noise(rng, 30)
    if kind == "negative":
        bad[3, 17] = -1
    else:
        bad[3] = 1500                                                 # 1024 * 1500^2 = 2.3e9 >= 2^31
    for hi, lo in ((bad, good), (good, bad)):
        for impl in (None, 0, 1, 2):
            with pytest.raises(MadError):
                P.match_threshold(hi, lo, 0.6, impl=impl)
            with pytest.raises(MadError):
                P.match_topk(hi, lo, 8, impl=impl)


# ---------------------------------------------------------------------------------------------
# F. merge of per-shard lists: padding, equal scores across shards, the incomplete-list sentinel
# ---------------------------------------------------------------------------------------------
def merge_inputs():
    ninf = -np.inf
    idx = np.array([
        [[-1, -1, -1, -1], [4, 1, -1, -1], [7, 8, 9, 10], [3, -1, -1, -1]],
        [[-1, -1, -1, -1], [0, 2, 3, -1], [-2, -2, -2, -2], [12, 11, -1, -1]],
        [[-1, -1, -1, -1], [5, 6, 7, 8], [1, 2, 3, 4], [20, -1, -1, -1]],
    ], dtype=np.int32)
    sc = np.array([
        [[ninf] * 4, [0.5, 0.25, ninf, ninf], [0.9, 0.8, 0.7, 0.6], [0.0, ninf, ninf, ninf]],
        [[ninf] * 4, [0.5, 0.5, 0.25, ninf], [ninf] * 4, [0.0, 0.0, ninf, ninf]],
        [[ninf] * 4, [0.5, 0.25, 0.25, 0.1], [0.95, 0.9, 0.1, 0.0], [1.0, ninf, ninf, ninf]],
    ])
    want_i = np.array([[-1, -1, -1, -1], [0, 2, 4, 5], [-2, -2, -2, -2], [20, 3, 11, 12]], dtype=np.int32)
    want_s = np.array([[ninf] * 4, [0.5, 0.5, 0.5, 0.5], [ninf] * 4, [1.0, 0.0, 0.0, 0.0]])
    return idx, sc, want_i, want_s


@gpu
def test_topk_merge_padding_ties_and_incomplete_lists(P):
    idx, sc, want_i, want_s = merge_inputs()
    mi, ms = P.topk_merge(torch.from_numpy(idx).cuda(), torch.from_numpy(sc).cuda())
    assert np.array_equal(mi.cpu().numpy(), want_i)
    assert np.array_equal(ms.cpu().numpy(), want_s)


def test_host_merge_padding_ties_and_incomplete_lists():
    """The CPU twin of mad_topk_merge (gloo path) follows the same rule."""
    from mad_b200.parallel import _merge_lists_host
    idx, sc, want_i, want_s = merge_inputs()
    mi, ms = _merge_lists_host(torch.from_numpy(idx), torch.from_numpy(sc))
    assert np.array_equal(mi.numpy(), want_i)
    assert np.array_equal(ms.numpy(), want_s)
