"""Descriptor cache round trip (mad/MaD.py:846-873): the four datasets with the reference's dtypes."""
import os

import numpy as np

import helpers as H


def test_descriptor_cache_round_trip(tmp_path):
    from mad_b200 import cache
    from mad_b200.DensityFeature import DensityFeature
    g = H.golden("tiny")
    rf = {(int(a), int(b)): m for (a, b), m in zip(g["rfinal_ab"], g["rfinal_mat"])}
    feats = []
    for i in range(len(g["of_index"])):
        df = DensityFeature()
        df.set_detector_info(int(g["of_index"][i]), int(g["of_oct"][i]), g["of_coords"][i].astype(np.float64),
                             g["of_subv_map_coords"][i] * 0 + 1.5, g["of_subv_map_coords"][i], 0.0)
        df.eqsp_size, df.subeqsp_size = 112, 16
        df.main_bin, df.sec_bin = int(g["of_main"][i]), int(g["of_sec"][i])
        df.Rfinal = rf[(df.main_bin, df.sec_bin)]
        df.lin_ar_subeqsp = g["dsc"][i]
        feats.append(df)
    path = os.path.join(str(tmp_path), "dsc_cache.h5")
    cache.save_descriptors(feats, path)
    with np.load(path) as z:
        assert sorted(z.files) == ["coords", "dsc", "info", "rot"]
        assert z["info"].dtype == np.uint16 and z["info"].shape == (len(feats), 6)
        assert z["dsc"].dtype == np.int16 and z["coords"].shape == (len(feats), 3, 3) and z["rot"].shape == (len(feats), 3, 3)
    back = cache.load_descriptors(path)
    assert len(back) == len(feats)
    for a, b in zip(feats, back):
        assert (a.index, a.main_bin, a.sec_bin, a.oct_scale) == (b.index, b.main_bin, b.sec_bin, b.oct_scale)
        assert (b.eqsp_size, b.subeqsp_size) == (112, 16)
        assert np.array_equal(a.lin_ar_subeqsp, b.lin_ar_subeqsp) and np.array_equal(a.Rfinal, b.Rfinal)
        assert np.array_equal(a.subv_map_coords, b.subv_map_coords) and np.array_equal(a.coords, b.coords)


def _plain(v):
    return v.tolist() if isinstance(v, np.ndarray) else v


def test_density_feature_record_equals_the_reference_record():
    """Every attribute our record carries has the reference's value after the same constructor / setter calls
    (mad/DensityFeature.py:6-84); the reference's extra attributes are its per-feature scratch arrays.
    tests/golden/density_feature_record.json holds, per call sequence below, the reference record's attributes outside
    those scratch arrays (vars() of the reference's DensityFeature, values as plain lists / numbers); the reference
    creates lin_ar_subeqsp only when a descriptor is set (mad/Descriptor.py:198, set_from_file_dsc)."""
    import json
    from mad_b200.DensityFeature import DensityFeature
    rf = np.arange(9.0).reshape(3, 3)
    calls = [
        [],
        [("set_detector_info", (7, 1, [3, 4, 5], [1.0, 2.0, 3.0], [1.1, 2.1, 3.1], 0.25))],
        [("set_detector_info", (7, 0, [3, 4, 5], [1.0, 2.0, 3.0], [1.1, 2.1, 3.1], 0.25)), ("set_orientator_info", (112, 8))],
        [("set_orientator_info", (112, 8)), ("set_descriptor_info", (16, 10))],
        [("set_from_file_ori", (3, 5, 17, 1, 112, [1, 2, 3], [4.0, 5.0, 6.0], [4.5, 5.5, 6.5], rf, np.arange(112)))],
        [("set_from_file_dsc", (3, 5, 17, 0, 112, 16, [1, 2, 3], [4.0, 5.0, 6.0], [4.5, 5.5, 6.5], rf, np.arange(1024)))],
    ]
    with open(os.path.join(H.GOLD, "density_feature_record.json")) as f:
        reference = json.load(f)
    assert len(reference) == len(calls)
    scratch = {"grad_box", "magn_box", "ar_magn", "ar_count", "norm_zone_counts", "interp_grad_box", "ar_subcount",
               "lin_magn_sudo", "step_ar_counts", "step_v_counts"}
    for seq, theirs in zip(calls, reference):
        ours = DensityFeature()
        for name, args in seq:
            getattr(ours, name)(*args)
        mine = vars(ours)
        for k, v in mine.items():
            if k == "lin_ar_subeqsp" and k not in theirs:      # the reference creates it in step06 only (mad/Descriptor.py:198)
                assert v == []
                continue
            assert k in theirs, k
            assert _plain(v) == theirs[k], (seq, k)
        missing = set(theirs) - set(mine) - scratch
        assert not missing, missing
