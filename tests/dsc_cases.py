"""Inputs of the match_dsc tests and of scripts/time_match_dsc.py: FeatureTables of the pair fixtures and of config C2
(the map and its six components, described on the device; their feature bookkeeping comes from the fixtures the
reference produced, whose row order the device path reproduces: tests/test_bench_parity.py)."""
import numpy as np
import torch

import helpers as H


def feature_table(P, g, prefix="", dsc=None):
    return P.FeatureTable(g[prefix + "dsc"] if dsc is None else dsc, g[prefix + "of_index"], g[prefix + "of_oct"],
                          g[prefix + "of_main"], g[prefix + "of_sec"], g[prefix + "of_subv_map_coords"])


def pair_tables(P):
    """(lo, hi) FeatureTables of the reference's pair fixture."""
    return feature_table(P, H.golden("pair_lo")), feature_table(P, H.golden("pair_hi"))


def c2_tables(P):
    """(map FeatureTable, [six component FeatureTables]) of config C2 (synth.c2_inputs(0))."""
    import synth
    grid, comps = synth.c2_inputs(0)
    g, gc = H.golden("c2"), H.golden("c2_comp")
    _, _, _, dsc = P.describe_struct(grid)
    assert dsc.shape[0] == len(g["of_index"])
    lo = feature_table(P, g, dsc=dsc)
    his = []
    for i, c in enumerate(comps):
        _, _, _, cdsc = P.describe_struct(c)
        assert cdsc.shape[0] == len(gc["comp%d_of_index" % i])
        his.append(feature_table(P, gc, "comp%d_" % i, dsc=cdsc))
    return lo, his


def stack_tables(P, tables):
    """One FeatureTable with the rows of several (the stacked subunits of an assembly)."""
    dsc = torch.cat([t.set.dsc for t in tables])
    m = np.concatenate([t.meta_host for t in tables])
    return P.FeatureTable(dsc, m[:, 0], m[:, 1], m[:, 2], m[:, 3], np.concatenate([t.subv_host for t in tables]))


def rows_of(P, t, rows):
    """FeatureTable of some rows of ``t``."""
    rows = np.asarray(rows)
    m = t.meta_host[rows]
    return P.FeatureTable(t.set.dsc[rows.tolist()].contiguous(), m[:, 0], m[:, 1], m[:, 2], m[:, 3], t.subv_host[rows])
