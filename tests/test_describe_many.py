"""pipeline.describe_many (G maps described in one batch) on one GPU: every map's keypoint table, oriented table and
descriptors equal its own describe_struct call (torch.equal) for mixed shapes, repeated maps, maps without keypoints or
without oriented features, patch sizes 12 / 16 / 24, exact_f64=False and an overflowing candidate region; two host reads
per batch for any G (three with an overflow); sparse-stage launches that do not grow with G; FeatureTable.from_device
against from_features of the reference-shaped classes, and match_dsc_many on either kind of table; the refusals."""
import numpy as np
import pytest

import helpers as H
import synth

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")


@pytest.fixture(scope="module")
def P():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from mad_b200 import pipeline
    return pipeline


@pytest.fixture(scope="module")
def c4():
    base = synth.random_walk_atoms(9000, 85.0, 1)
    return [synth.c4_snapshot(i, base) for i in range(synth.C4_MAPS)]


def _golden(name):
    return synth.dequantise_u16(H.golden(name)["input_q"])


def _blob(n=32, sigma=2.5):
    """One isotropic Gaussian blob: it is detected, but its gradient directions spread evenly over the sphere, so more
    than six zones pass the 80 % rule and no orientation survives."""
    x = np.arange(n, dtype=np.float64) - (n - 1) / 2.0
    r2 = x[:, None, None] ** 2 + x[None, :, None] ** 2 + x[None, None, :] ** 2
    return np.exp(-r2 / (2 * sigma * sigma)).astype(np.float32)


def _no_oriented_map(P):
    for n, sigma in ((32, 2.5), (32, 3.0), (28, 2.0), (36, 4.0)):
        g = _blob(n, sigma)
        _, kp, ori, _ = P.describe_struct(g)
        if len(kp) > 0 and len(ori) == 0:
            return g
    raise AssertionError("no blob map with keypoints and no oriented features")


def _check(P, grids, **kw):
    got = P.describe_many(grids, **kw)
    assert len(got) == len(grids)
    single = {k: v for k, v in kw.items() if k != "cap"}
    for g, grid in enumerate(grids):
        _, kp, ori, dsc = P.describe_struct(grid, **single)
        k, o, d = got.kp[g], got.ori[g], got.dsc[g]
        assert len(k) == len(kp) and len(o) == len(ori), (g, len(k), len(kp), len(o), len(ori))
        assert torch.equal(k.table[:len(k)], kp.table[:len(kp)]), g
        assert torch.equal(o.table[:len(o)], ori.table[:len(ori)]), g
        assert d.dtype == torch.int16 and torch.equal(d, dsc), g
        assert tuple(got.counts[g]) == (len(kp), len(ori))
    return got


def test_mixed_shapes_equal_describe_struct(P, c4):
    grids = [_golden("tiny"), _golden("small"), _golden("c1"), c4[0], c4[31], c4[63]]
    got = _check(P, grids)
    assert all(got.counts[:, 1] > 0)
    # CUDA tensors of any shape are taken in place
    _check(P, [torch.from_numpy(g).cuda() for g in grids[:3]])


def test_one_map_and_the_same_map_twice(P, c4):
    _check(P, [c4[5]])
    got = _check(P, [c4[7], c4[7]])
    assert torch.equal(got.dsc[0], got.dsc[1]) and torch.equal(got.ori[0].table, got.ori[1].table)


def test_maps_without_keypoints_or_without_oriented_features(P, c4):
    zero = np.zeros((30, 30, 30), dtype=np.float32)
    blob = _no_oriented_map(P)
    got = _check(P, [c4[1], zero, c4[2]])
    assert tuple(got.counts[1]) == (0, 0) and got.dsc[1].shape == (0, 1024)
    got = _check(P, [c4[3], blob, zero, c4[4]])
    assert got.counts[1, 0] > 0 and got.counts[1, 1] == 0
    got = _check(P, [zero])
    assert got.dsc_table.shape == (0, 1024)
    _check(P, [blob, zero])


@pytest.mark.parametrize("patch_size", [12, 16, 24])
def test_patch_sizes(P, c4, patch_size):
    _check(P, [_golden("small"), c4[10], c4[11]], patch_size=patch_size)


def test_float32_log(P, c4):
    _check(P, [_golden("tiny"), c4[12], c4[13]], exact_f64=False)


def _counting_reads(P, monkeypatch):
    calls = []
    orig = P._Readback.read.__func__

    def read(cls, *tensors):
        calls.append(len(tensors))
        return orig(cls, *tensors)
    monkeypatch.setattr(P._Readback, "read", classmethod(read))
    return calls


def test_overflow_redoes_detection_with_room(P, c4, monkeypatch):
    grids = [_golden("small"), c4[20], c4[21]]
    n0 = len(P.describe_struct(c4[20])[1])
    calls = _counting_reads(P, monkeypatch)
    _check(P, grids, cap=8)
    ref_reads = len(calls) - 3 * len(grids)                # (each describe_struct of _check reads three times)
    assert n0 > 8 and ref_reads == 3, calls


@pytest.mark.parametrize("G", [1, 6, 64])
def test_two_host_reads_per_batch(P, c4, monkeypatch, G):
    calls = _counting_reads(P, monkeypatch)
    got = P.describe_many(c4[:G])
    assert len(calls) == 2 and got.counts[:, 1].sum() > 0, calls


def _names(P, fn):
    P.profile_enable(True)
    try:
        fn()
        torch.cuda.synchronize()
        return [n for n, _ in P.profile_records()]
    finally:
        P.profile_enable(False)


def test_sparse_launches_do_not_grow_with_g(P, c4):
    grid = c4[0]

    def dense_one():
        sp = P.build_space(grid, keep_gauss=False, full_gradient=False)
        cand = torch.empty((1 << 16, 12), dtype=torch.int32, device="cuda")
        cnt = torch.zeros(1, dtype=torch.int32, device="cuda")
        for o, (lg, (gx, gy, gz)) in enumerate(zip(sp.logs, sp.dims)):
            P.call("mad_detect", P._ptr(lg), gx, gy, gz, o, 12, P.C.c_float(5e-2), P._ptr(cand), 1 << 16, P._ptr(cnt), P._stream())
        for o, (gx, gy, gz) in enumerate(sp.dims):
            P.call("mad_gradient_masked", P._ptr(sp._gauss[o]), gx, gy, gz, P._ptr(sp.grad4[o]), P._ptr(sp.grad_flags[o]),
                   P._stream())
    dense = _names(P, dense_one)
    per_map = {n: dense.count(n) for n in set(dense)}
    sparse = {}
    for G in (1, 6, 64):
        names = _names(P, lambda: P.describe_many(c4[:G]))
        for n, c in per_map.items():
            assert names.count(n) == G * c, (G, n)
        sparse[G] = sorted(n for n in names if n not in per_map)
    assert sparse[1] == sparse[6] == sparse[64], sparse
    assert "orient_kernel" in sparse[1] and "describe_kernel" in sparse[1]


def _feature_lists(grid, voxelsp, origin):
    from mad_b200.Descriptor import Descriptor
    from mad_b200.Detector import Detector
    from mad_b200.MapSpace import MapSpace
    from mad_b200.Orientator import Orientator
    ms = MapSpace.from_grid(grid, voxelsp, origin)
    ms.build_space()
    df = Descriptor().generate_descriptors(ms, Orientator().assign_orientations(ms, Detector().find_anchors(ms)))
    return ms, df


def test_feature_tables_from_device_equal_from_features(P, c4):
    maps = [(_golden("c1"), float(H.golden("c1")["voxelsp"]), tuple(H.golden("c1")["origin"])),
            (c4[40], 1.0, (-3.25, 7.5, 0.1)), (_golden("small"), 0.7, (1e3, -2.0, 0.3))]
    got = P.describe_many([m[0] for m in maps])
    spaces, refs = [], []
    for grid, vs, org in maps:
        ms, df = _feature_lists(grid, vs, org)
        spaces.append(ms)
        refs.append(P.FeatureTable.from_features(df))
    tables = got.feature_tables([ms.voxelsp_list for ms in spaces], [(ms.xi, ms.yi, ms.zi) for ms in spaces])
    for g, (t, ref, ms) in enumerate(zip(tables, refs, spaces)):
        one = P.FeatureTable.from_device(got.kp[g], got.ori[g], got.dsc[g], ms.voxelsp_list, (ms.xi, ms.yi, ms.zi))
        for tab in (t, one):
            assert torch.equal(tab.meta, ref.meta), g
            assert tab.subv.shape == ref.subv.shape
            assert tab.subv.cpu().numpy().tobytes() == ref.subv.cpu().numpy().tobytes(), g
            assert torch.equal(tab.set.dsc, ref.set.dsc), g
    # the hand-off to matching stays on the device: the same results as from the host-built tables
    lo = tables[0]
    for dev_t, host_t in zip(P.match_dsc_many(lo, tables[1:] + tables[:1]), P.match_dsc_many(refs[0], refs[1:] + refs[:1])):
        assert torch.equal(dev_t[0], host_t[0])
        assert np.array_equal(dev_t[1], host_t[1]) and np.array_equal(dev_t[2], host_t[2])
    assert P.match_dsc_many(lo, [tables[0]])[0][0].shape[0] > 0


def test_refusals(P, c4):
    with pytest.raises(P._lib.MadError):
        P.describe_many([])
    with pytest.raises(P._lib.MadError):
        P.describe_many([c4[0], np.zeros((30, 30), dtype=np.float32)])
    for mode in ("up", "base"):
        with pytest.raises(P._lib.MadError):
            P.describe_many([c4[0]], oct_mode=mode)
