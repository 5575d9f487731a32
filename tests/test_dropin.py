"""The ``mad`` drop-in package (SURVEY.md 8b: "run_MaD.py and the notebooks drop in unchanged"): the reference's module
names bound to mad_b200, and the reference's own orchestrator file loaded on top of them (mad/MaD.py of this repo).

CPU: name binding, the loader's error without the orchestrator file, and -- when MAD_REFERENCE_MAD_PY names the
reference's mad/MaD.py, which is not part of this repository -- that it executes on top of the package with every
hot-path name resolved to mad_b200 (no compute).  GPU: the call sequences of ``MaD._describe_struct``
(mad/MaD.py:358-368) and ``MaD._match_dsc`` (mad/MaD.py:414-453) written against the ``mad.*`` names, on config C1 and
the matching fixtures."""
import importlib
import os
import sys

import numpy as np
import pytest

import helpers as H

REF_MAD_PY = os.environ.get("MAD_REFERENCE_MAD_PY", "")


def test_reference_module_names_are_bound_to_mad_b200():
    import mad_b200.MapSpace, mad_b200.Detector, mad_b200.Orientator, mad_b200.Descriptor, mad_b200.Dmap, mad_b200.PDB  # noqa: E401
    for name in ("MapSpace", "Detector", "Orientator", "Descriptor", "Dmap", "PDB", "DensityFeature"):
        m = importlib.import_module("mad." + name)
        assert getattr(m, name) is getattr(importlib.import_module("mad_b200." + name), name)
    su = importlib.import_module("mad.structure_utils")
    assert all(hasattr(su, n) for n in ("move_copy_structure", "refine_pdb", "get_overlap"))           # mad/MaD.py:20
    mu = importlib.import_module("mad.math_utils")
    assert all(hasattr(mu, n) for n in ("get_rototrans_SVD", "euler_rod_mat", "unit_vector"))          # mad/MaD.py:21
    from mad.eqsp.eqsp import EQSP_Sphere                                                               # mad/MaD.py:22
    assert EQSP_Sphere().size == 112


def test_orchestrator_is_not_shipped(monkeypatch):
    monkeypatch.delenv("MAD_REFERENCE_MAD_PY", raising=False)
    sys.modules.pop("mad.MaD", None)
    with pytest.raises(ImportError, match="MAD_REFERENCE_MAD_PY"):
        importlib.import_module("mad.MaD")


@pytest.mark.skipif(not os.path.isfile(REF_MAD_PY), reason="needs the reference's mad/MaD.py (MAD_REFERENCE_MAD_PY)")
def test_reference_orchestrator_loads_on_top_of_the_package(monkeypatch, tmp_path):
    """run_MaD.py:63-76 up to the first compute call: ``MaD.MaD()``, ``add_map``, ``add_subunit``."""
    import ref_shims
    ref_shims.install()                                           # h5py / matplotlib are not in this image (I/O and plots only)
    monkeypatch.setenv("MAD_REFERENCE_MAD_PY", REF_MAD_PY)
    sys.modules.pop("mad.MaD", None)
    M = importlib.import_module("mad.MaD")
    import mad_b200.MapSpace, mad_b200.Descriptor, mad_b200.structure_utils   # noqa: E401
    assert M.MapSpace is mad_b200.MapSpace.MapSpace and M.Descriptor is mad_b200.Descriptor.Descriptor
    assert M.refine_pdb is mad_b200.structure_utils.refine_pdb
    assert M.MaD._match_dsc.__doc__.startswith("mad/MaD.py:414-453 on the device")
    m = M.MaD()
    p = tmp_path / "map.mrc"
    p.write_bytes(b"")
    s = tmp_path / "sub.pdb"
    s.write_text("")
    m.add_map(str(p), 8)
    m.add_subunit(str(s), n_copies=2)
    assert m.input_map == str(p) and list(m.input_subunits.values())[0] == [str(s), 2]
    sys.modules.pop("mad.MaD", None)


@pytest.mark.gpu
def test_describe_struct_sequence_through_the_mad_names_at_c1(tmp_path):
    torch = pytest.importorskip("torch")
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import synth
    from mad_b200 import mrc
    from mad.MapSpace import MapSpace
    from mad.Detector import Detector
    from mad.Orientator import Orientator
    from mad.Descriptor import Descriptor
    g = H.golden("c1")
    grid = synth.dequantise_u16(g["input_q"])
    path = os.path.join(str(tmp_path), "c1.mrc")
    mrc.write_mrc(path, grid.transpose(2, 1, 0), float(g["voxelsp"]), origin=tuple(g["origin"]))
    # the body of MaD._describe_struct, mad/MaD.py:358-368 (patch_size = 16: MaD.run's default)
    ms = MapSpace(path, resolution=4.0, voxelsp=float(g["voxelsp"]), sig_init=2, sig_presmooth=1)
    ms.build_space()
    det = Detector()
    anchors = det.find_anchors(ms)
    ori = Orientator(ori_radius=16)
    oriented_anchors = ori.assign_orientations(ms, anchors)
    dsc = Descriptor(dsc_radius=16)
    dsc_list = dsc.generate_descriptors(ms, oriented_anchors)
    assert len(anchors) == len(g["kp_oct"]) and len(dsc_list) == len(g["of_index"])
    assert np.array_equal(np.array([a.coords for a in anchors]), g["kp_coords"])
    assert np.array_equal([d.index for d in dsc_list], g["of_index"])
    assert np.array_equal([d.main_bin for d in dsc_list], g["of_main"]) and np.array_equal([d.sec_bin for d in dsc_list], g["of_sec"])
    d = np.array([f.lin_ar_subeqsp for f in dsc_list], dtype=np.int16)
    assert np.array_equal(H.crc_rows(d), g["dsc_crc32"])
    # what MaD.get_solutions reads off the features afterwards (mad/MaD.py:416-451)
    f = dsc_list[0]
    assert np.asarray(f.Rfinal).shape == (3, 3) and len(f.subv_map_coords) == 3 and f.oct_scale in (0, 1)
