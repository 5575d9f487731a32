"""The C-ABI shared library loads and exports every symbol include/mad_b200.h declares; argument
validation answers before any device work (no compute calls here: runs without a GPU)."""
import ctypes as C
import os
import re

import pytest

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_symbols():
    text = open(os.path.join(REPO, "include", "mad_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(mad_[a-z0-9_]+)\s*\(", text)))


@pytest.fixture(scope="module")
def lib():
    from mad_b200 import build
    build.build()
    from mad_b200 import _lib
    return _lib


def test_library_exports_every_declared_symbol(lib):
    names = header_symbols()
    assert len(names) >= 25
    for n in names:
        assert hasattr(lib.lib, n), "libmad_b200.so does not export %s" % n
    # and the ctypes binding lists exactly the header's entry points
    assert sorted(lib.SIGNATURES) == names


def test_struct_layouts_match_the_header(lib):
    assert lib.KEYPOINT_DTYPE.itemsize == 48          # MadKeypoint
    assert lib.ORIENTED_DTYPE.itemsize == 8           # MadOriented
    assert C.sizeof(lib.MadZoneTable) == 40
    assert C.sizeof(lib.MadDscSet) == 56          # 5 pointers + 4 int32


def test_bad_arguments_are_rejected_without_touching_the_device(lib):
    L = lib.lib
    assert L.mad_pad3d(None, 4, 4, 4, 1, None, None) == -1
    assert b"bad argument" in L.mad_last_error_string()
    assert L.mad_upsample_presmooth(None, 8, 8, 8, None, 0, None, None, 0, None) == -1
    assert L.mad_log_gauss(None, 8, 8, 8, None, None, 8, 4.0, None, None, None, 0, 1, None) == -1
    assert L.mad_match_topk(None, None, 8, 0, None, None, None, 0, 0, None) == -1
    assert L.mad_topk_merge(None, None, 0, 1, 8, None, None, None) == -1
    with pytest.raises(lib.MadError):
        lib.call("mad_gradient", None, 1, 1, 1, None, None)
    assert L.mad_version() >= 100
    assert L.mad_upsample_workspace_bytes(10, 10, 10) >= 10 * 10 * 19 * 8 + 19 * 10 * 19 * 8


def test_product_path_has_no_cpu_fallback(lib):
    import torch
    from mad_b200 import pipeline
    import numpy as np
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(lib.MadError):
        pipeline.build_space(np.zeros((8, 8, 8), dtype=np.float32))
    with pytest.raises(lib.MadError):
        pipeline.DescriptorSet(np.zeros((2, 1024), dtype=np.int16))


def test_product_never_imports_the_oracle():
    pkg = os.path.join(REPO, "mad_b200")
    for root, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(root, f)).read()
                assert not re.search(r"^\s*(import|from)\s+(mad_oracle|synth|ref_shims|oracle)\b", src, flags=re.M), f


def test_scores_from_dots_is_the_device_formula():
    """pipeline.scores_from_dots (host side of the compact pair format) against the reference's own lines on unit rows
    (mad/MaD.py:416-420): the exact integer dot over sqrt(n_hi n_lo) agrees with the float64 dgemm score to 1e-14, and zero
    descriptors score 0."""
    import numpy as np
    import synth
    import mad_oracle as mo
    from mad_b200.pipeline import scores_from_dots
    lo = synth.synthetic_descriptors(60, 3)
    hi = synth.synthetic_descriptors(40, 4, noisy_copy_of=lo)
    hi[3] = 0
    ph, pl = np.meshgrid(np.arange(40), np.arange(60), indexing="ij")
    ph, pl = ph.ravel(), pl.ravel()
    dot = (hi.astype(np.int64) @ lo.astype(np.int64).T).ravel()
    n_hi, n_lo = (hi.astype(np.int64) ** 2).sum(1), (lo.astype(np.int64) ** 2).sum(1)
    got = scores_from_dots(ph, pl, dot, n_hi, n_lo).reshape(40, 60)
    assert np.abs(got - mo.match_scores(hi, lo)).max() < 1e-14 and not got[3].any()
