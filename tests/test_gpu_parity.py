"""Parity of the CUDA path (through the C ABI of libmad_b200.so) with the reference's results.

Every test here needs a B200.  Dense stages are compared bit-for-bit (SHA-256 of the arrays the
UNMODIFIED reference produced, tests/golden/*.npz), sparse stages element by element against the
goldens and against the oracle (oracle/mad_oracle.py) on seeded inputs; at benchmark sizes the
checks are size-independent properties (exact power-of-two linearity, sharded == unsharded,
threshold/top-k consistency).

Tolerances (BASELINE.json north_star): voxel indices / match index lists bit-exact; sub-voxel
positions within 1e-4 relative (here: <= 1e-6 A absolute, float32 Newton arithmetic as NumPy 2);
descriptors are integers and must be identical.
"""
import numpy as np
import pytest

import helpers as H

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")


@pytest.fixture(scope="module")
def P():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from mad_b200 import pipeline
    return pipeline


def _run_case(P, name):
    import synth
    g = H.golden(name)
    grid = synth.dequantise_u16(g["input_q"])
    sp, kp, ori, dsc = P.describe_struct(grid, keep_gauss=True)
    return g, sp, kp, ori, dsc


_CASES = {}


def run_case(P, name):
    if name not in _CASES:
        _CASES[name] = _run_case(P, name)
    return _CASES[name]


@pytest.mark.parametrize("case", ["tiny", "small", "pair_hi", "pair_lo", "c1"])
def test_scale_space_bit_exact(P, case):
    """a1-a4: up grid, LoG, Gaussian, gradient equal the reference's arrays bit for bit
    (every value with |v| >= 1e-10; smaller ones -- the spline's decaying tails in the zero
    padding -- are flushed on both sides, see helpers.flushed), plus the sampled values."""
    g, sp, kp, ori, dsc = run_case(P, case)
    arrays = {"up_grid": sp.grids[0].cpu().numpy()}
    for o in range(2):
        arrays["log%d" % o] = sp.logs[o].cpu().numpy()
        arrays["gauss%d" % o] = sp.gauss[o].cpu().numpy()
        arrays["grad%d" % o] = np.ascontiguousarray(sp.grad4[o].cpu().numpy()[..., :3])
        assert not sp.grad4[o][..., 3].any()
    for key, a in arrays.items():
        assert H.sha_flushed(a) == str(g[key + "_sha256_flushed"]), key
        pos = g[key + "_pos"]
        assert H.equal_flushed(a[pos[:, 0], pos[:, 1], pos[:, 2]], g[key + "_val"]), key


@pytest.mark.parametrize("case", ["tiny", "small", "pair_hi", "pair_lo", "c1"])
def test_keypoints_equal_reference(P, case):
    """a5/a6: same keypoints in the same (canonical) order; sub-voxel positions within tolerance."""
    g, sp, kp, ori, dsc = run_case(P, case)
    hk = kp.host()
    assert len(kp) == len(g["kp_oct"])
    assert np.array_equal(hk["oct"], g["kp_oct"])
    assert np.array_equal(hk["vox"], g["kp_coords"])
    assert np.array_equal(hk["val"], g["kp_val"])
    v = float(g["voxelsp"])
    vs = np.where(hk["oct"] == 0, v / 2, v)[:, None]
    org = np.asarray(g["ms_origin"], dtype=np.float64)
    sub = (hk["vox"].astype(np.float64) + hk["off"].astype(np.float64)) * vs + org
    ref = g["kp_subv_map_coords"]
    assert np.abs(sub - ref).max() <= 1e-6                      # Angstrom; 1e-4 relative allowed
    mc = hk["vox"].astype(np.float64) * vs + org
    assert np.array_equal(mc, g["kp_map_coords"])


@pytest.mark.parametrize("case", ["tiny", "small", "pair_hi", "pair_lo", "c1"])
def test_orientations_and_descriptors_equal_reference(P, case):
    """a7-a12: identical (index, main, sec) triples in emission order, identical int16 descriptors."""
    g, sp, kp, ori, dsc = run_case(P, case)
    ho = ori.host()
    assert len(ori) == len(g["of_index"])
    assert np.array_equal(ho["kp"], g["of_index"])              # keypoint row == reference index
    assert np.array_equal(ho["main"], g["of_main"])
    assert np.array_equal(ho["sec"], g["of_sec"])
    d = dsc.cpu().numpy()
    assert d.dtype == np.int16 and d.shape == (len(ori), 1024)
    if "dsc" in g:
        assert np.array_equal(d, g["dsc"])
    assert np.array_equal(H.crc_rows(d), g["dsc_crc32"])
    assert np.array_equal(d.sum(1, dtype=np.int64), g["dsc_rowsum"])
    assert H.sha(d) == str(g["dsc_sha256"])


@pytest.mark.parametrize("case", ["tiny", "small", "pair_lo", "c1"])
def test_masked_gradient_path_equals_full_field_path(P, case):
    """The product path computes the gradient only on the 8^3 tiles around the keypoints (mad_gradient_mark /
    mad_gradient_masked): same keypoints, orientations and descriptors as with the whole field, the computed tiles hold
    the reference's values, and ``full_gradient`` afterwards completes the field bit for bit."""
    import synth
    g, sp, kp, ori, dsc = run_case(P, case)
    grid = synth.dequantise_u16(g["input_q"])
    sp2, kp2, ori2, dsc2 = P.describe_struct(grid)
    assert sp2.grad_flags[0] is not None and sp.grad_flags[0] is None
    assert torch.equal(kp.table[:len(kp)], kp2.table[:len(kp2)]) and torch.equal(ori.table[:len(ori)], ori2.table[:len(ori2)])
    assert torch.equal(dsc, dsc2)
    for o in range(2):
        fl = sp2.grad_flags[o].clone()
        assert int((fl == 1).sum()) == 0 and int((fl == 2).sum()) > 0
        nx, ny, nz = sp2.dims[o]
        t = fl.view((nx + 7) // 8, (ny + 7) // 8, (nz + 7) // 8)
        done = t.repeat_interleave(8, 0).repeat_interleave(8, 1).repeat_interleave(8, 2)[:nx, :ny, :nz] == 2
        assert torch.equal(sp2.grad4[o][done], sp.grad4[o][done])
    P.full_gradient(sp2)
    for o in range(2):
        assert sp2.grad_flags[o] is None and torch.equal(sp2.grad4[o], sp.grad4[o])


def test_stages_against_oracle_inputs(P):
    """Stage isolation: orient/describe fed with the ORACLE's keypoints reproduce the oracle."""
    grid, osp, okp, oori, odsc, tab_o = H.oracle_case("small")
    sp = P.build_space(grid)
    k = np.zeros(len(okp["oct"]), dtype=P.KEYPOINT_DTYPE)
    k["vox"], k["oct"], k["peak"], k["accepted"] = okp["coords"], okp["oct"], okp["coords"], 1
    kp = P.keypoints_from_host(k, sp.grad4[0].device)
    ori = P.orient(sp, kp)
    ho = ori.host()
    assert np.array_equal(ho["kp"], oori["kp"]) and np.array_equal(ho["main"], oori["main"])
    assert np.array_equal(ho["sec"], oori["sec"])
    o = np.zeros(len(oori["kp"]), dtype=P.ORIENTED_DTYPE)
    o["kp"], o["main"], o["sec"] = oori["kp"], oori["main"], oori["sec"]
    dsc = P.describe(sp, kp, P.oriented_from_host(o, sp.grad4[0].device))
    assert np.array_equal(dsc.cpu().numpy(), odsc)


@pytest.mark.parametrize("shape", [(64, 70, 76), (65, 71, 77), (66, 72, 78), (67, 73, 79), (68, 74, 80), (69, 75, 81)])
def test_spline_line_lengths(P, shape):
    """a2 on lines of every length class (n mod 16 = 0..15, both sides of the look-ahead boundaries): the long-line
    control flow of the spline kernels (head / interior chunks / one final sweep / compact tail) gives the very bits of
    the generic chunk loop, and both equal the oracle's interp1d + gaussian_filter (mad/MapSpace.py:137-146)."""
    import os
    import mad_oracle as mo
    from scipy import ndimage as ndi
    rng = np.random.default_rng(sum(shape))
    g = ndi.gaussian_filter(rng.random(shape), 1.5).astype(np.float32)
    g[rng.random(shape) < 0.3] = 0.0                                   # maps are zero over most of the box
    fast = P.build_space(g, map_padding=0, oct_mode="up", full_gradient=False).grids[0].clone()
    os.environ["MAD_SPLINE_GENERIC"] = "1"
    try:
        slow = P.build_space(g, map_padding=0, oct_mode="up", full_gradient=False).grids[0].clone()
    finally:
        del os.environ["MAD_SPLINE_GENERIC"]
    assert torch.equal(fast, slow)
    want = ndi.gaussian_filter(mo.upsample2(g), sigma=1).astype(np.float32)
    assert tuple(fast.shape) == want.shape
    assert H.equal_flushed(fast.cpu().numpy(), want)


@pytest.mark.parametrize("shape", [(20, 22, 24), (31, 17, 23)])
def test_ragged_and_empty_maps(P, shape):
    """Non-cubic maps and an all-zero map (no keypoints, no descriptors) -- reference edge cases."""
    import mad_oracle as mo
    z = np.zeros(shape, dtype=np.float32)
    sp, kp, ori, dsc = P.describe_struct(z)
    assert len(kp) == 0 and len(ori) == 0 and tuple(dsc.shape) == (0, 1024)
    assert not sp.logs[0].any() and not sp.logs[1].any()
    rng = np.random.default_rng(5)
    blob = np.zeros(shape, dtype=np.float32)
    c = np.array(shape) // 2
    x, y, zc = np.meshgrid(*[np.arange(s) for s in shape], indexing="ij")
    for _ in range(6):
        p = c + rng.integers(-4, 5, size=3)
        blob += np.exp(-((x - p[0]) ** 2 + (y - p[1]) ** 2 + (zc - p[2]) ** 2) / 6.0).astype(np.float32)
    blob /= blob.max()
    sp, kp, ori, dsc = P.describe_struct(blob, keep_gauss=True)
    osp = mo.build_space(blob)
    assert H.equal_flushed(sp.grids[0].cpu().numpy(), osp["grid_list"][0])
    for o in range(2):
        assert H.equal_flushed(sp.logs[o].cpu().numpy(), osp["map_space"][o])
        assert H.equal_flushed(sp.gauss[o].cpu().numpy(), osp["gauss_list"][o])
        assert H.equal_flushed(sp.grad4[o].cpu().numpy()[..., :3], osp["grad_list"][o])
    okp = mo.detect(osp["map_space"], [0.5, 1.0], [0, 0, 0])
    assert np.array_equal(kp.host()["vox"], okp["coords"])
    oori, tab = mo.orient(osp["grad_list"], okp)
    assert np.array_equal(ori.host()["main"], oori["main"]) and np.array_equal(ori.host()["sec"], oori["sec"])
    assert np.array_equal(dsc.cpu().numpy(), mo.describe(osp["grad_list"], okp, oori, tab))


def test_patch_sizes(P):
    """patch_size 12 and 20 (MaD_notebook_instructions.ipynb uses 12..24) against the oracle."""
    import mad_oracle as mo
    grid, osp, okp, _, _, _ = H.oracle_case("small")
    sp = P.build_space(grid)
    kp = P.detect(sp)
    for patch in (12, 20):
        r = patch // 2
        ori = P.orient(sp, kp, r)
        dsc = P.describe(sp, kp, ori, r)
        tab_o = mo.OrientTables(patch)
        oori, _ = mo.orient(osp["grad_list"], okp, patch, tab_o)
        assert np.array_equal(ori.host()["kp"], oori["kp"])
        assert np.array_equal(ori.host()["main"], oori["main"]) and np.array_equal(ori.host()["sec"], oori["sec"])
        odsc = mo.describe(osp["grad_list"], okp, oori, tab_o, patch, mo.DescribeTables(patch))
        assert np.array_equal(dsc.cpu().numpy(), odsc)


def test_float32_accumulation_mode_is_within_tolerance(P):
    """exact_f64=False (float32 line accumulation) is NOT the parity mode; it must stay within
    the stated tolerance: same keypoints, dense arrays within 1e-6 of max."""
    g, sp, kp, ori, dsc = run_case(P, "small")
    import synth
    grid = synth.dequantise_u16(g["input_q"])
    sp32, kp32, ori32, dsc32 = P.describe_struct(grid, exact_f64=False, keep_gauss=True)
    for o in range(2):
        a, b = sp32.logs[o].cpu().numpy(), sp.logs[o].cpu().numpy()
        assert np.abs(a - b).max() <= 1e-6 * np.abs(b).max()
    assert np.array_equal(kp32.host()["vox"], kp.host()["vox"])


# ---------------------------------------------------------------------------------------------
# properties at benchmark size (no oracle: too slow on the CPU)
# ---------------------------------------------------------------------------------------------
def test_full_size_power_of_two_linearity(P):
    """256^3 (BASELINE config 2 size): scaling the input by 1/2 scales every linear stage by
    exactly 1/2 (power-of-two scaling commutes with IEEE rounding), so keypoint VOXELS with value
    above twice the threshold, their orientations and descriptors must be identical."""
    import synth
    grid = synth.assembly_map(256, 8.0, 2.0, 6, 8000, 10)
    a = P.describe_struct(grid, keep_gauss=True)
    b = P.describe_struct(grid * np.float32(0.5), keep_gauss=True)

    def halves(x, y):
        # exact where float32 is normal; the spline's decaying tails reach the denormal range
        big = x.abs() > 1e-30
        return torch.equal(x[big] * 0.5, y[big]) and float((x * 0.5 - y).abs().max()) <= 1e-37

    for o in range(2):
        assert halves(a[0].grids[o], b[0].grids[o])
        assert halves(a[0].logs[o], b[0].logs[o])
        assert halves(a[0].grad4[o], b[0].grad4[o])
    ka, kb = a[1].host(), b[1].host()
    assert len(ka) > 1000
    # threshold 0.05 on the halved map == 0.1 on the original; Newton offsets are scale-free
    keep = ka["val"] * np.float32(0.5) > np.float32(0.05)
    assert keep.sum() == len(kb)
    assert np.array_equal(ka["oct"][keep], kb["oct"]) and np.array_equal(ka["vox"][keep], kb["vox"])
    assert np.array_equal(ka["off"][keep], kb["off"])
    # descriptors of the common oriented features are identical (gradient directions unchanged)
    def keyed(res):
        k, o, d = res[1].host(), res[2].host(), res[3].cpu().numpy()
        keys = np.c_[k["oct"][o["kp"]], k["vox"][o["kp"]], o["main"], o["sec"]]
        return {tuple(r): d[i] for i, r in enumerate(keys)}
    da, db = keyed(a), keyed(b)
    common = set(da) & set(db)
    assert len(common) > 1000
    # Normalised gradient directions are unchanged by the exact halving, so a vote can only be LOST
    # (never moved or gained) on the halved map: where the halved magnitude drops below the 1e-5
    # cut-off of mad/Descriptor.py:190.  Hence db <= da bin by bin, and few votes are lost overall.
    lost = 0
    total = 0
    for c in common:
        assert np.all(db[c] <= da[c])
        lost += int((da[c].astype(np.int64) - db[c]).sum())
        total += int(da[c].sum())
    assert lost <= 0.05 * total


# ---------------------------------------------------------------------------------------------
# a15 matching
# ---------------------------------------------------------------------------------------------
IMPLS = [1, 2, 0]   # 1 = SIMT integer kernel (check), 2 = fp16 tcgen05 kernel, 0 = uint8 tcgen05 kernel (the product)


@pytest.mark.parametrize("impl", IMPLS)
def test_match_threshold_equals_reference_pairs(P, impl):
    ghi, glo, gm = H.golden("pair_hi"), H.golden("pair_lo"), H.golden("pair_match")
    ph, pl, sc = P.match_threshold(ghi["dsc"], glo["dsc"], float(gm["cc"]), impl=impl)
    pairs = np.stack([ph.cpu().numpy(), pl.cpu().numpy()], 1)
    assert np.array_equal(pairs, gm["pairs"])                   # row-major order of np.where
    assert np.abs(sc.cpu().numpy() - gm["scores"]).max() < 1e-14


@pytest.mark.parametrize("impl", IMPLS)
def test_match_topk_equals_oracle(P, impl):
    ghi, glo, gm = H.golden("pair_hi"), H.golden("pair_lo"), H.golden("pair_match")
    idx, sc = P.match_topk(ghi["dsc"], glo["dsc"], 8, impl=impl)
    import mad_oracle as mo
    preds = mo.match_scores(ghi["dsc"], glo["dsc"])
    got = idx.cpu().numpy()
    # the oracle's stable argsort works on dgemm scores (ties differ from exact ties at 1e-16):
    # compare the score multiset exactly-ish and the indices wherever scores are not tied
    ref_sc = np.take_along_axis(preds, gm["topk8_idx"], 1)
    assert np.abs(sc.cpu().numpy() - ref_sc).max() < 1e-14
    same = got == gm["topk8_idx"]
    tied = np.zeros_like(same)
    tied[:, 1:] |= np.abs(ref_sc[:, 1:] - ref_sc[:, :-1]) < 1e-14
    tied[:, :-1] |= np.abs(ref_sc[:, 1:] - ref_sc[:, :-1]) < 1e-14
    nineth = np.sort(preds, 1)[:, -9]
    tied |= np.abs(ref_sc - nineth[:, None]) < 1e-14
    assert np.all(same | tied)


@pytest.mark.parametrize("impl", IMPLS)
@pytest.mark.parametrize("m,n", [(1, 1), (3, 130), (129, 257), (300, 77)])
def test_match_ragged_sizes_against_oracle(P, impl, m, n):
    import mad_oracle as mo
    import synth
    lo = synth.synthetic_descriptors(n, 3)
    hi = synth.synthetic_descriptors(m, 4, noisy_copy_of=lo)
    hi[0] = 0                                                   # zero descriptor: scores 0 with all
    pairs, scores = mo.match_threshold(hi, lo, 0.6)
    ph, pl, sc = P.match_threshold(hi, lo, 0.6, impl=impl)
    assert np.array_equal(np.stack([ph.cpu().numpy(), pl.cpu().numpy()], 1), pairs)
    k = min(8, n)
    idx, tsc = P.match_topk(hi, lo, k, impl=impl)
    oi, osc = mo.match_topk(hi, lo, k)
    assert np.abs(tsc.cpu().numpy() - osc).max() < 1e-14
    assert (idx.cpu().numpy()[0] == np.arange(k)).all()          # all-tied row: lowest indices win


@pytest.mark.parametrize("impl", IMPLS)
def test_match_empty_sets(P, impl):
    e = np.zeros((0, 1024), dtype=np.int16)
    a = np.ones((5, 1024), dtype=np.int16)
    for hi, lo in ((e, a), (a, e), (e, e)):
        ph, pl, sc = P.match_threshold(hi, lo, 0.6, impl=impl)
        assert ph.numel() == 0 and pl.numel() == 0 and sc.numel() == 0


@pytest.mark.parametrize("impl", IMPLS)
def test_match_properties_at_size(P, impl):
    """8192 x 8192 (no CPU oracle): tcgen05 == SIMT is covered elsewhere; here size-independent
    properties: self-match contains the diagonal, pairs(hi,lo) == swapped pairs(lo,hi),
    threshold and top-k agree, sharded top-k merge == unsharded."""
    import synth
    n = 8192 if impl != 1 else 2048
    lo = synth.synthetic_descriptors(n, 7)
    hi = synth.synthetic_descriptors(n, 8, noisy_copy_of=lo)
    dl, dh = P.DescriptorSet(lo), P.DescriptorSet(hi)
    ph, pl, sc = P.match_threshold(dl, dl, 0.6, impl=impl)
    ph, pl = ph.cpu().numpy(), pl.cpu().numpy()
    diag = ph == pl
    assert diag.sum() == n and np.all(sc.cpu().numpy()[diag] == 1.0)
    a = P.match_threshold(dh, dl, 0.6, impl=impl)
    b = P.match_threshold(dl, dh, 0.6, impl=impl)
    sa = np.stack([a[0].cpu().numpy(), a[1].cpu().numpy()], 1)
    sb = np.stack([b[1].cpu().numpy(), b[0].cpu().numpy()], 1)
    assert len(sa) > n // 4
    assert np.array_equal(sa, sb[np.lexsort((sb[:, 1], sb[:, 0]))])
    assert np.all(np.diff(sa[:, 0].astype(np.int64) * n + sa[:, 1]) > 0)       # row-major, strictly increasing
    idx, tsc = P.match_topk(dh, dl, 8, impl=impl)
    best = np.full(n, -1.0)
    np.maximum.at(best, sa[:, 0], a[2].cpu().numpy())
    has = best > 0
    assert np.array_equal(tsc.cpu().numpy()[has, 0], best[has])
    # reference axis sharded in 4 unequal shards + merge == unsharded
    cuts = [0, 1000, 1000 + n // 3, n - 5, n]
    parts = [P.match_topk(dh, P.DescriptorSet(lo[s:e]), 8, lo_index_base=s, impl=impl) for s, e in zip(cuts, cuts[1:])]
    mi, ms = P.topk_merge(torch.stack([p[0] for p in parts]), torch.stack([p[1] for p in parts]))
    assert torch.equal(mi, idx) and torch.equal(ms, tsc)


def test_tcgen05_equals_simt_exactly(P):
    import synth
    lo = synth.synthetic_descriptors(1500, 11)
    hi = synth.synthetic_descriptors(700, 12, noisy_copy_of=lo)
    r1 = P.match_threshold(hi, lo, 0.55, impl=1)
    t1 = P.match_topk(hi, lo, 16, impl=1)
    for impl in (0, 2):
        r0 = P.match_threshold(hi, lo, 0.55, impl=impl)
        for x, y in zip(r0, r1):
            assert torch.equal(x, y)
        t0 = P.match_topk(hi, lo, 16, impl=impl)
        assert torch.equal(t0[0], t1[0]) and torch.equal(t0[1], t1[1])


def test_topk_last_wave_split_equals_simt(P):
    """mad_match_topk gives the rows of a poorly filled last wave (here 74 full CTA pairs + 300 rows) a second, segmented
    launch: the stitched result must equal the SIMT integer kernel's bit for bit, and the unsplit launch's."""
    import os
    import synth
    lo = synth.synthetic_descriptors(3000, 51)
    m = 74 * 256 + 300
    base = synth.synthetic_descriptors(2048, 52, noisy_copy_of=lo)
    hi = np.concatenate([np.roll(base, 7 * r, axis=1) for r in range((m + 2047) // 2048)])[:m]
    hi[m - 5] = 0
    dh, dl = P.DescriptorSet(hi), P.DescriptorSet(lo)
    a = P.match_topk(dh, dl, 8, lo_index_base=11, impl=0)
    b = P.match_topk(dh, dl, 8, lo_index_base=11, impl=1)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
    os.environ["MAD_TOPK_NO_TAIL"] = "1"
    try:
        c = P.match_topk(dh, dl, 8, lo_index_base=11, impl=0)
    finally:
        del os.environ["MAD_TOPK_NO_TAIL"]
    assert torch.equal(a[0], c[0]) and torch.equal(a[1], c[1])


def test_onepass_candidate_overflow_and_dense_hits(P):
    """The one-pass matcher's candidate list: a too-small first buffer is repeated with room;
    very dense hits (a set against itself at a low threshold) overflow the per-warp staging and
    take the direct path.  Both must give exactly the SIMT kernel's pairs."""
    import synth
    lo = synth.synthetic_descriptors(900, 21)
    P._PAIR_CAP[(900, 900)] = 64                                 # force the overflow / repeat path
    a = P.match_threshold(lo, lo, 0.05, impl=0)                  # nearly every pair passes
    b = P.match_threshold(lo, lo, 0.05, impl=1)
    assert a[0].numel() > 400000
    for x, y in zip(a, b):
        assert torch.equal(x, y)


def test_entries_above_255_use_the_fp16_kernel(P):
    """Descriptor entries > 255 (patch sizes > 24) do not fit the uint8 operand: the product picks
    the fp16 tensor-core kernel, and asking for the uint8 one fails loudly."""
    import synth
    from mad_b200._lib import MadError
    lo = synth.synthetic_descriptors(300, 31)
    hi = synth.synthetic_descriptors(200, 32, noisy_copy_of=lo)
    lo[:, :16] *= 9                                              # entries of 16-bin blocks reach ~40: up to ~360
    hi[:, :16] *= 9
    assert P.DescriptorSet(lo).max_entry > 255
    r = P.match_threshold(hi, lo, 0.5)
    r1 = P.match_threshold(hi, lo, 0.5, impl=1)
    for x, y in zip(r, r1):
        assert torch.equal(x, y)
    with pytest.raises(MadError):
        P.match_threshold(hi, lo, 0.5, impl=0)


def test_stacked_hi_sets_equal_separate_matches(P):
    """concat_sets: one launch over the stacked hi sets returns exactly the per-set pair lists
    (global hi row = offset + local row), in the same order."""
    import synth
    lo = synth.synthetic_descriptors(700, 41)
    his = [synth.synthetic_descriptors(m, 42 + i, noisy_copy_of=lo) for i, m in enumerate((130, 1, 257))]
    sets = [P.DescriptorSet(h) for h in his]
    allset, offs = P.concat_sets(sets)
    dl = P.DescriptorSet(lo)
    ph, pl, sc = [t.cpu().numpy() for t in P.match_threshold(allset, dl, 0.55)]
    for i, s in enumerate(sets):
        a = [t.cpu().numpy() for t in P.match_threshold(s, dl, 0.55)]
        sel = (ph >= offs[i]) & (ph < offs[i + 1])
        assert np.array_equal(ph[sel] - offs[i], a[0]) and np.array_equal(pl[sel], a[1]) and np.array_equal(sc[sel], a[2])


def test_host_stage_roundtrip(P):
    st = P.HostStage()
    x = torch.arange(1000, dtype=torch.int32, device="cuda").reshape(100, 10)
    a = st.fetch("x", x)
    b = st.fetch("y", x.double() * 0.5, overlap=True)
    st.sync()
    assert np.array_equal(a.numpy(), x.cpu().numpy()) and np.array_equal(b.numpy(), x.cpu().numpy() * 0.5)


def test_map_stream_equals_separate_calls(P):
    """MapStream (uploads / downloads of neighbouring maps overlapped with the kernels) returns for every map exactly what
    describe_struct + match_threshold return for it, whatever the interleaving."""
    import synth
    grids = [synth.dequantise_u16(H.golden(n)["input_q"]) for n in ("pair_lo", "pair_hi", "small", "pair_lo")]
    _, _, _, hi_dsc = P.describe_struct(grids[1])
    hi = P.DescriptorSet(hi_dsc)
    want = []
    for g in grids:
        sp, kp, ori, dsc = P.describe_struct(g)
        ph, pl, sc = P.match_threshold(hi, P.DescriptorSet(dsc), 0.6)
        want.append((dsc.cpu().numpy(), kp.host(), ori.host(), ph.cpu().numpy(), pl.cpu().numpy(), sc.cpu().numpy()))
    ms = P.MapStream(hi=hi, cc=0.6)
    pinned = [torch.from_numpy(g).pin_memory() for g in grids]
    got, prev = [], None
    nxt = ms.upload(pinned[0])
    for i in range(len(grids)):
        cur = nxt
        nxt = ms.upload(pinned[i + 1]) if i + 1 < len(grids) else None
        ticket = ms.submit(cur)
        if prev is not None:
            got.append({k: v.numpy().copy() for k, v in ms.result(prev).items()})
        prev = ticket
    got.append({k: v.numpy().copy() for k, v in ms.result(prev).items()})
    for w, g in zip(want, got):
        assert np.array_equal(w[0], g["dsc"])
        assert w[1].tobytes() == g["kp"].tobytes() and w[2].tobytes() == g["ori"].tobytes()
        assert np.array_equal(w[3], g["pair_hi"]) and np.array_equal(w[4], g["pair_lo"]) and np.array_equal(w[5], g["score"])
    assert len(got[0]["pair_hi"]) == len(H.golden("pair_match")["pairs"])


def test_map_stream_compact_format(P):
    """MapStream(compact=True): uint8 descriptors and (hi, lo, exact dot) pairs + norms carry exactly the information of the
    full format -- widened descriptors and recomputed float64 scores are bit-identical."""
    import synth
    grids = [synth.dequantise_u16(H.golden(n)["input_q"]) for n in ("pair_lo", "small")]
    _, _, _, hi_dsc = P.describe_struct(synth.dequantise_u16(H.golden("pair_hi")["input_q"]))
    hi = P.DescriptorSet(hi_dsc)
    ms = P.MapStream(hi=hi, cc=0.6, compact=True)
    for g in grids:
        sp, kp, ori, dsc = P.describe_struct(g)
        ph, pl, sc = P.match_threshold(hi, P.DescriptorSet(dsc), 0.6)
        out = ms.result(ms.submit(ms.upload(torch.from_numpy(g).pin_memory())))
        assert out["dsc_u8"].dtype == torch.uint8 and np.array_equal(out["dsc_u8"].numpy().astype(np.int16), dsc.cpu().numpy())
        pair_hi = P.pair_hi_from_counts(out["pair_hi_counts"].numpy())
        assert np.array_equal(pair_hi, ph.cpu().numpy()) and np.array_equal(out["pair_lo"].numpy(), pl.cpu().numpy())
        got = P.scores_from_dots(pair_hi, out["pair_lo"].numpy(), out["pair_dot"].numpy(), hi.norm2.cpu().numpy(),
                                 out["lo_norm2"].numpy())
        assert np.array_equal(got, sc.cpu().numpy())


def test_c3_size_scale_space_linearity(P):
    """BASELINE config 3 size (512^3 -> 530^3 + 1059^3 grids, ~50 GB of device arrays): the stencil
    chain runs at that size and is exactly linear under power-of-two scaling; detection on the
    halved map equals detection on the original with the threshold doubled."""
    g = torch.Generator(device="cuda").manual_seed(3)
    n = 512
    coarse = torch.rand((1, 1, 20, 20, 20), device="cuda", generator=g)
    grid = torch.nn.functional.interpolate(coarse, size=(n, n, n), mode="trilinear", align_corners=True)[0, 0]
    grid = (grid - 0.45).clamp_(min=0).contiguous()
    grid /= grid.max()
    a = P.build_space(grid, keep_gauss=False)
    ka = P.detect(a).host().copy()
    la = [t.clone() for t in a.logs]
    ga = a.grad4[1][::7, ::5, ::3].clone()
    del a
    torch.cuda.empty_cache()
    b = P.build_space(grid * 0.5, keep_gauss=False)
    kb = P.detect(b).host()
    for o in range(2):
        big = la[o].abs() > 1e-30
        assert torch.equal(la[o][big] * 0.5, b.logs[o][big])
    assert torch.equal(ga * 0.5, b.grad4[1][::7, ::5, ::3])
    keep = ka["val"] * np.float32(0.5) > np.float32(0.05)
    assert len(ka) > 100 and keep.sum() == len(kb)
    assert np.array_equal(ka["vox"][keep], kb["vox"]) and np.array_equal(ka["off"][keep], kb["off"])


# ---------------------------------------------------------------------------------------------
# next component: the per-pair loop of MaD._match_dsc (mad/MaD.py:426-453)
# ---------------------------------------------------------------------------------------------
def _feature_table(P, g):
    return P.FeatureTable(g["dsc"], g["of_index"], g["of_oct"], g["of_main"], g["of_sec"], g["of_subv_map_coords"])


def test_match_dsc_loop_equals_reference_results(P):
    """results[P, 23] of MaD._match_dsc: score, repeatability, (index, octave, main bin) of both features, both
    sub-voxel coordinates and R = inv(Rfinal_lo) . Rfinal_hi -- against the table the reference produced."""
    ghi, glo, gm = H.golden("pair_hi"), H.golden("pair_lo"), H.golden("pair_match")
    res, lo_cloud, hi_cloud = P.match_dsc(_feature_table(P, glo), _feature_table(P, ghi), 4, float(gm["cc"]))
    res = res.cpu().numpy()
    ref = gm["results"]
    assert np.array_equal(lo_cloud, gm["lo_cloud"]) and np.array_equal(hi_cloud, gm["hi_cloud"])
    assert res.shape == ref.shape
    assert np.array_equal(res[:, 1], ref[:, 1])                            # repeatability: exact counts
    assert np.array_equal(res[:, 2:14], ref[:, 2:14])                      # bookkeeping and coordinates
    assert np.abs(res[:, 0] - ref[:, 0]).max() < 1e-14
    assert np.abs(res[:, 14:] - ref[:, 14:]).max() < 1e-14                 # rotation (dgemm vs plain sums)


def test_match_dsc_loop_against_oracle_on_a_denser_case(P):
    """A lower threshold gives thousands of pairs and larger clouds (oracle = cKDTree restatement)."""
    import mad_oracle as mo
    ghi, glo = H.golden("pair_hi"), H.golden("pair_lo")
    res, lo_cloud, hi_cloud = P.match_dsc(_feature_table(P, glo), _feature_table(P, ghi), 6.5, 0.5)
    res = res.cpu().numpy()

    def fd(g):
        rf = {(int(a), int(b)): m for (a, b), m in zip(g["rfinal_ab"], g["rfinal_mat"])}
        return dict(dsc=g["dsc"], subv=g["of_subv_map_coords"], index=g["of_index"], oct=g["of_oct"], main=g["of_main"],
                    sec=g["of_sec"], Rfinal=np.array([rf[(int(a), int(b))] for a, b in zip(g["of_main"], g["of_sec"])]))
    ores, olo, ohi = mo.match_dsc(fd(glo), fd(ghi), 6.5, 0.5)
    assert len(ores) > 5000 and res.shape == ores.shape
    assert np.array_equal(lo_cloud, olo) and np.array_equal(hi_cloud, ohi)
    flips = np.nonzero(res[:, 1] != ores[:, 1])[0]
    assert len(flips) <= 1e-3 * len(ores)                                   # a distance within ulps of the bound may flip
    assert np.array_equal(res[:, 2:14], ores[:, 2:14])
    # the device equals the exact reference of its own arithmetic (tests/repeat_ref.py), rotation bits included; a pair
    # the oracle counts differently differs only through anchors whose distance lies within a few ulps of dist
    import repeat_ref as rr
    from scipy.spatial import cKDTree
    from mad_b200 import tables
    ot = tables.orientation_tables(112)
    ph, pl = np.nonzero(mo.match_scores(ghi["dsc"], glo["dsc"]) > 0.5)
    meta = [np.stack([g["of_index"], g["of_oct"], g["of_main"], g["of_sec"]], 1) for g in (ghi, glo)]
    _, rows, detail = rr.repeat(ph, pl, res[:, 0], ghi["of_subv_map_coords"], glo["of_subv_map_coords"], meta[0], meta[1],
                                ot.rf, ot.rf_inv, 112, hi_cloud, lo_cloud, 6.5, detail=True)
    assert rows.tobytes() == res.tobytes()
    few = 16 * np.spacing(max(6.5, np.abs(lo_cloud).max(), np.abs(hi_cloud).max()))
    tree = cKDTree(lo_cloud)
    hi_rf, lo_rf = fd(ghi)["Rfinal"], fd(glo)["Rfinal"]
    for k in flips:                                                          # the oracle's loop, per anchor
        R = np.dot(np.linalg.inv(lo_rf[pl[k]]), hi_rf[ph[k]])
        d, _ = tree.query(np.dot(hi_cloud - ghi["of_subv_map_coords"][ph[k]], R.T) + glo["of_subv_map_coords"][pl[k]],
                          distance_upper_bound=6.5)
        hit, nearest = detail[k]
        differ = np.nonzero((d < 6.5) != hit)[0]
        assert len(differ) and (np.abs(nearest[differ] - 6.5) <= few).all(), (k, nearest[differ] - 6.5)


def test_match_dsc_lists_is_a_drop_in(P):
    """Same call shape as the reference: lists of DensityFeature in, (list of 23-vectors, clouds) out."""
    from mad_b200.DensityFeature import DensityFeature
    ghi, glo, gm = H.golden("pair_hi"), H.golden("pair_lo"), H.golden("pair_match")

    def feats(g):
        out = []
        for i in range(len(g["of_index"])):
            df = DensityFeature()
            df.set_detector_info(int(g["of_index"][i]), int(g["of_oct"][i]), list(g["of_coords"][i]), None,
                                 g["of_subv_map_coords"][i], 0.0)
            df.main_bin, df.sec_bin, df.lin_ar_subeqsp = int(g["of_main"][i]), int(g["of_sec"][i]), g["dsc"][i]
            out.append(df)
        return out
    results, lo_cloud, hi_cloud = P.match_dsc_lists(feats(glo), feats(ghi), cc_threshold=float(gm["cc"]))
    assert len(results) == len(gm["results"]) and np.array_equal(np.array(results)[:, 1], gm["results"][:, 1])
