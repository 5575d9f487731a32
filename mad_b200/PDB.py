"""PDB with the part of the reference's interface that sits in front of the hot path
(mad/PDB.py:8-80, 131-209, 215-292): fixed-column coordinate reader and ``structure_to_density``.

The density simulation (mass-weighted trilinear splat, Gaussian of sigma = resolution / (pi sqrt 2) /
voxelsp truncated at 3 sigma, max normalisation, isovalue cut) runs in libmad_b200.so; the result can stay
on the device (``structure_to_density_device``) so that ``MapSpace`` in PDB mode starts from HBM.
The manipulation helpers of the reference's class (rotate_atoms, translate_atoms, rmsd, write_pdb; mad/PDB.py:80-128)
are host glue with the reference's semantics, used by ``structure_utils``.
"""
import ctypes as C
import os
import sys
from math import ceil, floor, sqrt

import numpy as np
import torch

from . import _lib
from . import mrc as _mrc
from ._lib import call

MASS = {"H": 1.00797, "BE": 9.01218, "C": 12.011, "N": 14.0067, "O": 15.9994, "F": 18.998403, "S": 32.06, "P": 30.97376,
        "MG": 24.305, "CL": 35.453, "K": 39.0983, "CA": 40.078, "MN": 54.9380, "FE": 55.847, "NI": 58.70, "CU": 63.546,
        "ZN": 65.38, "SE": 78.96}                                        # mad/PDB.py:220-221


def _ptr(t):
    return C.c_void_p(t.data_ptr())


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def write_situs(outname, grid, voxelsp, dxi, dyi, dzi):
    """Situs text map exactly as the reference writes it (mad/PDB.py:165-179): header line, blank line, then the voxels
    x-fastest, a line break before every 10th value."""
    dxb, dyb, dzb = grid.shape
    with open(outname, "w") as f:
        f.write("%f %f %f %f %i %i %i\n\n" % (voxelsp, dxi, dyi, dzi, dxb, dyb, dzb))
        voxi = 0
        for z in range(dzb):
            for y in range(dyb):
                for x in range(dxb):
                    if (voxi + 1) % 10 == 0:
                        f.write("\n")
                    f.write("   %6.6f   " % grid[x][y][z])
                    voxi += 1


def _splat_box(xyz, voxelsp, margin):
    """Lattice-registered minimum corner and splat box dims of atoms xyz [n][3] (host scalars, mad/PDB.py:236-254)."""
    minx = voxelsp * floor(np.amin(xyz[:, 0]) / voxelsp)
    maxx = voxelsp * ceil(np.amax(xyz[:, 0]) / voxelsp)
    miny = voxelsp * floor(np.amin(xyz[:, 1]) / voxelsp)
    maxy = voxelsp * ceil(np.amax(xyz[:, 1]) / voxelsp)
    minz = voxelsp * floor(np.amin(xyz[:, 2]) / voxelsp)
    maxz = voxelsp * ceil(np.amax(xyz[:, 2]) / voxelsp)
    pxb = ceil((maxx - minx) / voxelsp) + 2 * margin + 1
    pyb = ceil((maxy - miny) / voxelsp) + 2 * margin + 1
    pzb = ceil((maxz - minz) / voxelsp) + 2 * margin + 1
    return (minx, miny, minz), (pxb, pyb, pzb)


def _gauss_1d(resolution, voxelsp):
    """(r, w): radius and float64 weights [2r + 1] of the 1-D factor of the Gaussian, mad/PDB.py:138-150 (the 3-D kernel
    exp(-(x^2+y^2+z^2) / 2 sig^2) / sum is a product of 1-D kernels)."""
    sig = resolution / (np.pi * sqrt(2)) / voxelsp
    r = int(ceil(3.0 * sig))
    t = np.arange(-r, r + 1)
    g1 = np.exp(-(t * t) / (2.0 * sig ** 2))
    return r, np.ascontiguousarray(g1 / g1.sum())


def _pinned_to(a, dev):
    """One asynchronous host -> device copy through pinned memory (the caching host allocator keeps the pinned block until
    the copy has run)."""
    return torch.from_numpy(np.ascontiguousarray(a)).pin_memory().to(dev, non_blocking=True)


MAX_BATCH = 65535          # structures per batch: the batched kernels run one CTA row (grid y) per structure
MAX_DIM = 1 << 30          # a map's extent per axis (splat box + 2r), as mad_density_layout bounds it


def _batch_atoms(structures, masses):
    """(xyz [g] float64 [n_g][3], mass [g] float64 [n_g]) of density_many's inputs, checked on the host."""
    if not structures:
        raise _lib.MadError("density_many: no structures")
    if len(structures) > MAX_BATCH:
        raise _lib.MadError("density_many: %d structures; a batch holds at most %d (split it)" % (len(structures), MAX_BATCH))
    per_structure = isinstance(masses, (list, tuple))
    if per_structure and len(masses) != len(structures):
        raise _lib.MadError("density_many: %d mass arrays for %d structures" % (len(masses), len(structures)))
    xyzs, ms = [], []
    for g, s in enumerate(structures):
        if isinstance(s, PDB):                                    # density_many refuses masses next to PDB objects
            xyz = np.asarray(s.coords, dtype=np.float64)
            m = s._masses()
        else:
            xyz = np.asarray(s, dtype=np.float64)
            if masses is None:
                raise _lib.MadError("density_many: structure %d is a coordinate array and no masses were given" % g)
            m = masses[g] if per_structure else masses
        m = np.ascontiguousarray(m, dtype=np.float64).reshape(-1)
        if xyz.ndim != 2 or xyz.shape[1] != 3 or xyz.shape[0] == 0:
            raise _lib.MadError("density_many: structure %d has no atoms (coordinates of shape %s)" % (g, xyz.shape))
        if not np.isfinite(xyz).all():
            raise _lib.MadError("density_many: structure %d has non-finite coordinates" % g)
        if len(m) != len(xyz):
            raise _lib.MadError("density_many: structure %d has %d atoms and %d masses" % (g, len(xyz), len(m)))
        xyzs.append(np.ascontiguousarray(xyz))
        ms.append(m)
    return xyzs, ms


def _density_layout(xyzs, voxelsp, r, margin):
    """The batch's MadDensityBox table laid out by mad_density_layout, the totals, and the map origins [G][3] (host)."""
    G = len(xyzs)
    boxes = (_lib.MadDensityBox * G)()
    origins = np.empty((G, 3), dtype=np.float64)
    for g, xyz in enumerate(xyzs):
        mins, dims = _splat_box(xyz, voxelsp, margin)
        if any(d + 2 * r >= MAX_DIM for d in dims):
            raise _lib.MadError("density_many: structure %d spans a box of %s voxels (+ %d per axis for the Gaussian); "
                                "each axis must stay below %d" % (g, list(dims), 2 * r, MAX_DIM))
        b = boxes[g]
        b.min[:] = mins
        b.dims[:] = dims
        b.n_atoms = len(xyz) if len(xyz) < (1 << 31) else -1
        b.margin = margin
        origins[g] = [mn - (r + margin) * voxelsp for mn in mins]
    totals = (C.c_longlong * 5)()
    call("mad_density_layout", boxes, G, r, totals)
    return boxes, list(totals), origins


class DensityBatch(object):
    """The simulated maps of a batch: ``grids[g]`` = float32 CUDA view [x][y][z] of structure g's map in one flat buffer,
    ``origins`` [G][3] = its (dxi, dyi, dzi) (host float64), ``voxelsp``."""

    def __init__(self, maps, grids, origins, voxelsp):
        self.maps = maps
        self.grids = grids
        self.origins = origins
        self.voxelsp = voxelsp

    def __len__(self):
        return len(self.grids)

    def host(self, g):
        """What ``structure_to_density`` returns for structure g: (grid float32 [x][y][z], dxi, dyi, dzi)."""
        dxi, dyi, dzi = (float(v) for v in self.origins[g])
        return self.grids[g].cpu().numpy().astype(np.float32), dxi, dyi, dzi


def density_many(structures, resolution, voxelsp, isovalue=0.0, pad=0, masses=None):
    """``structure_to_density_device`` for G structures in one batch, with no host read and no device synchronisation.

    ``structures``: ``PDB`` objects (masses from their elements; ``masses`` must then be None) or coordinate arrays
    [n_g][3]; for arrays, ``masses`` is one array shared by every structure (poses of one structure) or a list / tuple of
    one array per structure.  Every structure's float64 splat equals the reference's sequential loop (mad/PDB.py:278-285)
    bit for bit (sorted contributions instead of atomics), and the map does not depend on the rest of the batch.  The
    later stages are those of the single path.  Raises ``MadError`` naming the structure, before any device work, for an
    empty list, a structure without atoms, non-finite coordinates, a mass count that does not match, or a box of 2^30
    voxels or more along an axis.  A batch holds at most 65535 structures (one CTA row each); a longer list is refused,
    not split."""
    structures = list(structures)
    if masses is not None and any(isinstance(s, PDB) for s in structures):
        raise _lib.MadError("density_many: masses are taken from the PDB objects' elements")
    xyzs, ms = _batch_atoms(structures, masses)
    margin = 2 + pad
    r, w = _gauss_1d(resolution, voxelsp)
    boxes, totals, origins = _density_layout(xyzs, voxelsp, r, margin)
    if not torch.cuda.is_available():
        raise _lib.MadError("mad_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
    G = len(xyzs)
    dev = torch.device("cuda", torch.cuda.current_device())
    st = _stream()
    d_xyz = _pinned_to(np.concatenate(xyzs), dev)
    d_mass = _pinned_to(np.concatenate(ms), dev)
    d_w = _pinned_to(w, dev)
    d_boxes = _pinned_to(np.frombuffer(bytearray(boxes), dtype=np.uint8), dev)
    ws = torch.empty(max(1, int(_lib.lib.mad_density_splat_many_workspace_bytes(int(totals[0])))), dtype=torch.uint8, device=dev)
    splat = torch.empty(totals[1], dtype=torch.float64, device=dev)
    call("mad_density_splat_many", _ptr(d_xyz), _ptr(d_mass), boxes, G, _ptr(d_boxes), C.c_double(voxelsp), _ptr(splat),
         _ptr(ws), ws.numel(), st)
    del ws, d_xyz, d_mass
    scratch = torch.empty(G, dtype=torch.int64, device=dev)
    call("mad_normalise_f64_many", _ptr(splat), boxes, G, _ptr(d_boxes), _ptr(scratch), st)
    xpass = torch.empty(totals[2], dtype=torch.float64, device=dev)
    call("mad_conv_full_f64_many", _ptr(splat), boxes, G, _ptr(d_boxes), 0, _ptr(d_w), r, _ptr(xpass), st)
    del splat
    ypass = torch.empty(totals[3], dtype=torch.float64, device=dev)
    call("mad_conv_full_f64_many", _ptr(xpass), boxes, G, _ptr(d_boxes), 1, _ptr(d_w), r, _ptr(ypass), st)
    del xpass
    maps = torch.empty(totals[4], dtype=torch.float32, device=dev)
    call("mad_conv_full_f64_many", _ptr(ypass), boxes, G, _ptr(d_boxes), 2, _ptr(d_w), r, _ptr(maps), st)
    del ypass
    call("mad_map_normalise_many", _ptr(maps), boxes, G, _ptr(d_boxes), r, C.c_float(isovalue), _ptr(scratch), st)
    grids = []
    for g in range(G):
        shape = tuple(int(d) + 2 * r for d in boxes[g].dims)
        o = int(boxes[g].off[3])
        grids.append(maps[o:o + shape[0] * shape[1] * shape[2]].view(shape))
    return DensityBatch(maps, grids, origins, voxelsp)


class PDB(object):
    def __init__(self, pdb_file):
        self.pdb_file = pdb_file
        self.coords = []
        self.info = []
        if not os.path.exists(self.pdb_file):
            print("PDB> File not found: %s" % self.pdb_file)
            sys.exit(1)
        self.CA_idx = []
        self.BB_idx = []
        c = 0
        at_num = res_num = 0
        at_name = res_name = chain_id = element_symbol = ""
        x = y = z = 0.0
        with open(self.pdb_file, "r") as pdb:
            for line in pdb:
                line_type = line[0:6].strip()
                if line_type in ["ATOM", "HETATM"]:
                    try:                                                  # mad/PDB.py:46-58 (a bad line repeats the previous values)
                        at_num = int(line[6:11].strip())
                        at_name = line[12:16].strip()
                        res_name = line[17:20]
                        chain_id = line[21]
                        res_num = int(line[22:26].strip())
                        x = float(line[30:38])
                        y = float(line[38:46])
                        z = float(line[46:54])
                        element_symbol = line[76:78].strip()
                    except Exception:
                        pass
                    self.info.append([at_num, at_name, res_name, chain_id, res_num, element_symbol, line_type])
                    self.coords.append([x, y, z])
                    if at_name == "CA":
                        self.CA_idx.append(c)
                    if at_name in ["C", "CA", "N", "O"]:
                        self.BB_idx.append(c)
                    c += 1
        self.coords = np.array(self.coords)
        self.CA_idx = tuple(self.CA_idx)
        self.n_atoms = len(self.coords)
        self.n_CA = len(self.CA_idx)
        self.minx, self.maxx = np.amin(self.coords[:, 0]), np.amax(self.coords[:, 0])
        self.miny, self.maxy = np.amin(self.coords[:, 1]), np.amax(self.coords[:, 1])
        self.minz, self.maxz = np.amin(self.coords[:, 2]), np.amax(self.coords[:, 2])

    def get_coords(self):
        return self.coords

    def set_coords(self, coords):
        self.coords = coords.copy()

    def rotate_atoms(self, rot_mat):
        self.coords = np.dot(self.coords, rot_mat)                         # mad/PDB.py:109-110

    def translate_atoms(self, trans_vec):
        self.coords += np.array(trans_vec)                                 # mad/PDB.py:112-113

    def get_rmsd_with(self, pdb):
        d2 = np.square(self.coords - pdb.coords)                           # mad/PDB.py:115-117
        return np.sqrt(np.sum(d2, axis=(0, 1)) / d2.shape[0])

    def get_rmsdCA_with(self, pdb):
        if not len(self.CA_idx):                                           # mad/PDB.py:119-128
            print("PDB> No alpha carbons detected; returning all-atom RMSD instead.")
            return self.get_rmsd_with(pdb)
        d2 = np.square(self.coords[self.CA_idx, :] - pdb.coords[pdb.CA_idx, :])
        return np.sqrt(np.sum(d2, axis=(0, 1)) / d2.shape[0])

    def write_pdb(self, outname):
        """Fixed-column ATOM / HETATM records, occupancy 1.00, B 0.00 (mad/PDB.py:80-94): 4-letter atom names start
        one column earlier."""
        with open(outname, "w") as f:
            for rec, (x, y, z) in zip(self.info, self.coords):
                at_num, at_name, res_name, chain_id, res_num, element, line_type = rec
                name = " %-4s " % at_name if len(at_name) == 4 else "  %-3s " % at_name
                f.write("%-6s%5i%s%3s%2s%4s    %8.3f%8.3f%8.3f%6.2f%6.2f          %-2s\n"
                        % (line_type, at_num, name, res_name, chain_id, res_num, x, y, z, 1.0, 0.0, element))

    # ---- density ----------------------------------------------------------------------------------
    def _masses(self):
        out = np.empty(len(self.info), dtype=np.float64)
        for i, rec in enumerate(self.info):
            elem = rec[-2].upper()
            if elem in MASS:
                out[i] = MASS[elem]
            else:
                print("PDB> (dens) Element %s not in dict. Using mass of carbon." % elem)
                out[i] = MASS["C"]
        return out

    def structure_to_density_device(self, resolution, voxelsp, isovalue=0.0, pad=0):
        """(float32 CUDA tensor [x][y][z], dxi, dyi, dzi): mad/PDB.py:131-163 on the device."""
        if not torch.cuda.is_available():
            raise _lib.MadError("mad_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
        dev = torch.device("cuda", torch.cuda.current_device())
        st = _stream()
        xyz = np.ascontiguousarray(self.coords, dtype=np.float64)
        mass = self._masses()
        margin = 2 + pad
        (minx, miny, minz), (pxb, pyb, pzb) = _splat_box(xyz, voxelsp, margin)
        d_xyz = torch.from_numpy(xyz).to(dev)
        d_mass = torch.from_numpy(mass).to(dev)
        grid = torch.empty((pxb, pyb, pzb), dtype=torch.float64, device=dev)
        mins = np.array([minx, miny, minz], dtype=np.float64)
        call("mad_density_splat", _ptr(d_xyz), _ptr(d_mass), len(xyz), mins.ctypes.data_as(C.c_void_p), C.c_double(voxelsp),
             margin, pxb, pyb, pzb, _ptr(grid), st)
        scratch = torch.empty(1, dtype=torch.int64, device=dev)
        call("mad_normalise_f64", _ptr(grid), grid.numel(), _ptr(scratch), st)
        # Gaussian, mad/PDB.py:138-150: the 3-D kernel exp(-(x^2+y^2+z^2) / 2 sig^2) / sum is a product of 1-D kernels
        r, w = _gauss_1d(resolution, voxelsp)
        w = torch.from_numpy(w).to(dev)
        a = torch.empty((pxb + 2 * r, pyb, pzb), dtype=torch.float64, device=dev)
        call("mad_conv_full_f64", _ptr(grid), 1, pxb, pyb * pzb, _ptr(w), r, _ptr(a), 0, st)
        b = torch.empty((pxb + 2 * r, pyb + 2 * r, pzb), dtype=torch.float64, device=dev)
        call("mad_conv_full_f64", _ptr(a), pxb + 2 * r, pyb, pzb, _ptr(w), r, _ptr(b), 0, st)
        dens = torch.empty((pxb + 2 * r, pyb + 2 * r, pzb + 2 * r), dtype=torch.float32, device=dev)
        call("mad_conv_full_f64", _ptr(b), (pxb + 2 * r) * (pyb + 2 * r), pzb, 1, _ptr(w), r, _ptr(dens), 1, st)
        dxi = minx - (r + margin) * voxelsp
        dyi = miny - (r + margin) * voxelsp
        dzi = minz - (r + margin) * voxelsp
        # [0, 1] range, isovalue cut (float32), mad/PDB.py:158-159
        mx = torch.zeros(1, dtype=torch.int32, device=dev)
        call("mad_grid_max", _ptr(dens), dens.numel(), _ptr(mx), st)
        vmax = float(_lib.lib.mad_grid_max_decode(C.c_uint(int(mx.item()) & 0xFFFFFFFF)))
        call("mad_threshold_normalise", _ptr(dens), dens.numel(), C.c_float(-np.inf), C.c_float(vmax), 1, st)
        if isovalue:
            call("mad_threshold_normalise", _ptr(dens), dens.numel(), C.c_float(isovalue), C.c_float(1.0), 0, st)
        return dens, dxi, dyi, dzi

    def structure_to_density(self, resolution, voxelsp, isovalue=0.0, pad=0, outname=""):
        """Reference signature and return value: (grid float32 [x][y][z], dxi, dyi, dzi)."""
        dens, dxi, dyi, dzi = self.structure_to_density_device(resolution, voxelsp, isovalue, pad)
        grid = dens.cpu().numpy()
        if outname != "":
            ext = os.path.splitext(outname)[-1].lower()
            if ext in [".sit", ".situs"]:
                write_situs(outname, grid, voxelsp, dxi, dyi, dzi)
            else:
                _mrc.write_mrc(outname, grid.transpose(2, 1, 0), voxelsp, origin=(dxi, dyi, dzi))
        return grid.astype(np.float32), dxi, dyi, dzi
