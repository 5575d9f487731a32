"""Dmap with the reference's interface (mad/Dmap.py:6-97), the voxel grid resident in HBM.

    dm = Dmap(map_name, isovalue=0.0, normalize=True, pad=0)
    dm.reduce_void(); dm.pad_grid(5); ms = MapSpace.from_grid(dm.device_grid(), dm.voxsp, (dm.xi, dm.yi, dm.zi))

File parsing is host glue as in the reference (Situs text, MRC through mad_b200.mrc); the isovalue
cut, the max normalisation, the bounding box of ``reduce_void`` and crop / zero padding run in
libmad_b200.so on the device grid (row a0 of SURVEY.md section 8).  ``grid3d`` is a lazily synchronised
NumPy copy for Python consumers; ``device_grid()`` hands the CUDA tensor to ``MapSpace.from_grid``
without a host round trip.  The scoring / masking methods (``mask_with``, ``get_CCC_with_grid``,
``get_CCC_with_dmap``; mad/Dmap.py:99-372, SURVEY.md 8f rank 4) are single streaming reductions over the
common box of two device grids (``score.cu``).
"""
import ctypes as C
import os
import sys

import numpy as np
import torch

from . import _lib
from . import mrc as _mrc
from ._lib import call


def _ptr(t):
    return C.c_void_p(t.data_ptr())


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


class Dmap(object):
    def __init__(self, map_name, isovalue=0.0, normalize=True, pad=0):
        if not os.path.isfile(map_name):
            print("Dmap> ERROR: file %s not found" % map_name)
            sys.exit(1)
        ext = os.path.splitext(map_name)[-1]
        if ext.lower() in [".sit", ".situs"]:
            with open(map_name, "r") as f:
                header = f.readline().replace("\n", "").replace("  ", "").split(" ")
                f.readline()
                self.voxsp, self.xi, self.yi, self.zi = [float(x) for x in header[:4]]
                self.xb, self.yb, self.zb = [int(x) for x in header[4:]]
                grid1d = np.array(f.read().split(), dtype=np.float64).astype(np.float32)   # as np.fromstring(...).astype
                grid = np.reshape(grid1d, (self.xb, self.yb, self.zb), order="F")
        elif ext.lower() in [".map", ".mrc"]:
            h, data = _mrc.read_mrc(map_name)
            axis_order = [h.mapc - 1, h.mapr - 1, h.maps - 1]
            self.axis_order = axis_order
            self.voxsp = h.voxel_size[0]
            if np.all([h.nxstart, h.nystart, h.nzstart]):                  # mad/Dmap.py:34-36
                origin = np.array([h.nxstart, h.nystart, h.nzstart], dtype=int)
                self.xi, self.yi, self.zi = [origin[a] * self.voxsp for a in axis_order]
            else:                                                           # int-truncated origin, :38-39
                origin = np.array(h.origin, dtype=int)
                self.xi, self.yi, self.zi = [origin[a] for a in axis_order]
            boxdim = np.array([h.mx, h.my, h.mz], dtype=int)
            self.xb, self.yb, self.zb = [int(boxdim[a]) for a in axis_order]
            grid = np.transpose(data.copy(), axis_order[::-1])
        else:
            print("Dmap> ERROR: incompatible extension for map %s" % map_name)
            return
        self.map_name = map_name
        self.name = map_name.split("/")[-1].split(".")[0]
        self._init_from_array(grid, isovalue, normalize, pad)

    @classmethod
    def from_array(cls, grid, voxsp, origin=(0.0, 0.0, 0.0), isovalue=0.0, normalize=True, pad=0, name="grid"):
        """Array entry point (NumPy or CUDA tensor, float32 [x][y][z]); same post-processing as a file."""
        self = cls.__new__(cls)
        self.voxsp = voxsp
        self.xi, self.yi, self.zi = origin
        self.map_name = name
        self.name = name
        self.xb, self.yb, self.zb = [int(v) for v in grid.shape]
        self._init_from_array(grid, isovalue, normalize, pad)
        return self

    # ---- device side ------------------------------------------------------------------------------
    def _init_from_array(self, grid, isovalue, normalize, pad):
        if not torch.cuda.is_available():
            raise _lib.MadError("mad_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
        if isinstance(grid, np.ndarray):
            grid = torch.from_numpy(np.ascontiguousarray(grid, dtype=np.float32)).cuda()
        self._dev = grid.contiguous().float().clone()
        self._host = None
        vmax = self._max()
        if vmax > isovalue:                                                 # mad/Dmap.py:49-54
            thr = float(isovalue)
        else:
            print("Dmap> WARNING: asked isovalue is larger than maximum density found in file (%f). Considering isovalue=0" % vmax)
            thr = 0.0
            vmax = max(vmax, 0.0)
        call("mad_threshold_normalise", _ptr(self._dev), self._dev.numel(), C.c_float(thr), C.c_float(1.0), 0, _stream())
        if pad:
            self.pad_grid(pad)
        if np.isclose(vmax, 0):
            print("Dmap> WARNING: Max value in map is 0")
        if normalize:                                                       # mad/Dmap.py:66-67
            call("mad_threshold_normalise", _ptr(self._dev), self._dev.numel(), C.c_float(-np.inf), C.c_float(vmax), 1, _stream())

    def _max(self):
        out = torch.zeros(1, dtype=torch.int32, device=self._dev.device)
        call("mad_grid_max", _ptr(self._dev), self._dev.numel(), _ptr(out), _stream())
        return float(_lib.lib.mad_grid_max_decode(C.c_uint(int(out.item()) & 0xFFFFFFFF)))

    def device_grid(self):
        """The float32 [x][y][z] CUDA tensor (no copy)."""
        return self._dev

    @property
    def grid3d(self):
        if self._host is None:
            self._host = self._dev.cpu().numpy()
        return self._host

    @grid3d.setter
    def grid3d(self, value):
        self._dev = torch.from_numpy(np.ascontiguousarray(value, dtype=np.float32)).cuda()
        self._host = None
        self.xb, self.yb, self.zb = [int(v) for v in self._dev.shape]

    def _crop_pad(self, x0, y0, z0, cx, cy, cz, pad):
        nx, ny, nz = [int(v) for v in self._dev.shape]
        out = torch.empty((cx + 2 * pad, cy + 2 * pad, cz + 2 * pad), dtype=torch.float32, device=self._dev.device)
        call("mad_crop_pad3d", _ptr(self._dev), nx, ny, nz, x0, y0, z0, cx, cy, cz, int(pad), _ptr(out), _stream())
        self._dev = out
        self._host = None
        self.xb, self.yb, self.zb = [int(v) for v in out.shape]

    def reduce_void(self, zeros_padding=10):
        """Crop to the bounding box of the non-zero voxels, then zero-pad (mad/Dmap.py:73-90)."""
        nx, ny, nz = [int(v) for v in self._dev.shape]
        bbox = torch.empty(6, dtype=torch.int32, device=self._dev.device)
        call("mad_grid_bbox", _ptr(self._dev), nx, ny, nz, _ptr(bbox), _stream())
        b = [int(v) for v in bbox.tolist()]
        if b[3] < 0:
            raise ValueError("zero-size array to reduction operation minimum which has no identity")   # as np.amin does
        minx, miny, minz, maxx, maxy, maxz = b
        self.xi = self.xi + minx * self.voxsp
        self.yi = self.yi + miny * self.voxsp
        self.zi = self.zi + minz * self.voxsp
        self._crop_pad(minx, miny, minz, maxx - minx + 1, maxy - miny + 1, maxz - minz + 1, 0)
        self.pad_grid(zeros_padding)

    def pad_grid(self, pad):
        """np.pad(grid3d, pad) with the origin moved (mad/Dmap.py:92-97)."""
        nx, ny, nz = [int(v) for v in self._dev.shape]
        self._crop_pad(0, 0, 0, nx, ny, nz, int(pad))
        self.xi -= pad * self.voxsp
        self.yi -= pad * self.voxsp
        self.zi -= pad * self.voxsp

    # ---- scoring on the device (SURVEY.md 8f rank 4) -----------------------------------------------
    @staticmethod
    def _common_box(o1, s1, o2, s2):
        """Bounds of the common box as the reference rounds them (mad/Dmap.py:172-241); origins in voxels.
        Returns [x1, y1, z1, x2, y2, z2, ex, ey, ez] or None when an extent is negative."""
        bounds = []
        for a in range(3):
            i1, i2, b1, b2 = o1[a], o2[a], s1[a], s2[a]
            if i1 > i2:
                mn1, mn2 = 0, int(round(i1 - i2))
            elif i1 < i2:
                mn1, mn2 = int(round(i2 - i1)), 0
            else:
                mn1, mn2 = 0, 0
            if i1 + b1 > i2 + b2:
                mx1, mx2 = int(round(i2 + b2 - i1)), int(round(b2))
            elif i1 + b1 < i2 + b2:
                mx1, mx2 = int(round(b1)), int(round(i1 + b1 - i2))
            else:
                mx1, mx2 = int(round(b1)), int(round(b2))
            bounds.append((mn1, mn2, mx1, mx2))
        if any(mx1 - mn1 < 0 for mn1, _, mx1, _ in bounds):       # mad/Dmap.py:239-241, tested before any slicing
            return None
        lo1, lo2, ext = [], [], []
        for a, (mn1, mn2, mx1, mx2) in enumerate(bounds):
            # NumPy slicing clips both boxes to their arrays; the two extents agree except for rounding at x.5 offsets
            e1 = max(0, min(mx1, s1[a]) - mn1)
            e2 = max(0, min(mx2, s2[a]) - mn2)
            if e1 != e2:
                raise ValueError("operands could not be broadcast together: common boxes differ on axis %d (%d vs %d)" % (a, e1, e2))
            lo1.append(mn1); lo2.append(mn2); ext.append(e1)
        return lo1 + lo2 + ext

    @staticmethod
    def _as_device_grid(grid, dev):
        if isinstance(grid, np.ndarray):
            return torch.from_numpy(np.ascontiguousarray(grid, dtype=np.float32)).to(dev)
        return grid.contiguous()

    def _box_scores(self, g2, xi2, yi2, zi2, isovalue):
        """out8 of mad_box_scores for this map against device grid g2 (host float64 array), or None."""
        voxsp = self.voxsp
        box = self._common_box([self.xi / voxsp, self.yi / voxsp, self.zi / voxsp], [self.xb, self.yb, self.zb],
                               [xi2 / voxsp, yi2 / voxsp, zi2 / voxsp], [int(v) for v in g2.shape])
        if box is None:
            return None
        dev = self._dev.device
        ws = torch.empty(max(1, int(_lib.lib.mad_box_scores_workspace_bytes(box[6], box[7], box[8])) // 8), dtype=torch.float64, device=dev)
        out = torch.empty(8, dtype=torch.float64, device=dev)
        box_c = (C.c_int * 9)(*box)
        n1, n2 = [int(v) for v in self._dev.shape], [int(v) for v in g2.shape]
        call("mad_box_scores", _ptr(self._dev), n1[0], n1[1], n1[2], _ptr(g2), n2[0], n2[1], n2[2], box_c,
             C.c_float(isovalue), _ptr(out), _ptr(ws), ws.numel() * 8, _stream())
        return out.cpu().numpy()

    def _count_gt(self, grid, thr):
        out = torch.zeros(1, dtype=torch.int64, device=grid.device)
        call("mad_grid_count_gt", _ptr(grid), grid.numel(), C.c_float(thr), _ptr(out), _stream())
        return int(out.item())

    def get_CCC_with_grid(self, grid2, xi2, yi2, zi2, isovalue=0):
        """mad/Dmap.py:153-258: cosine of the two maps over their common box.  As in the reference both grids are
        cut at the isovalue IN PLACE first (this map's device grid; ``grid2`` when it is a CUDA tensor -- a NumPy
        ``grid2`` is uploaded and left untouched).  The three sums are float64 (the reference's are float32 BLAS
        dots: agreement ~1e-6 relative)."""
        g2 = self._as_device_grid(grid2, self._dev.device)
        call("mad_threshold_normalise", _ptr(self._dev), self._dev.numel(), C.c_float(isovalue), C.c_float(1.0), 0, _stream())
        call("mad_threshold_normalise", _ptr(g2), g2.numel(), C.c_float(isovalue), C.c_float(1.0), 0, _stream())
        self._host = None
        s = self._box_scores(g2, xi2, yi2, zi2, 0.0)
        if s is None:
            return 0
        return s[0] / np.sqrt(s[1] * s[2])

    def get_CCC_with_grids(self, grids, origins, isovalue=0):
        """``get_CCC_with_grid`` of this map against G grids (e.g. ``PDB.density_many(...).grids``) with origins [G][3]:
        float64 array [G] whose element g equals ``get_CCC_with_grid(grids[g], *origins[g], isovalue)`` exactly.  As there,
        this map and every CUDA grid are cut at the isovalue in place (the G grids in one launch); a NumPy grid is uploaded.
        The common boxes are checked before any device work (``ValueError`` naming the structure); a disjoint box scores 0.
        One host read for the batch.  A batch holds at most 65535 grids (one CTA row each); a longer list is refused
        (``ValueError``, before any device work), not split."""
        from .pipeline import _Readback
        G = len(grids)
        if G > 65535:
            raise ValueError("get_CCC_with_grids: %d grids; a batch holds at most 65535 (split it)" % G)
        origins = np.asarray(origins, dtype=np.float64).reshape(G, 3) if G else np.zeros((0, 3))
        voxsp = self.voxsp
        o1 = [self.xi / voxsp, self.yi / voxsp, self.zi / voxsp]
        boxes = (_lib.MadScoreBox * max(G, 1))()
        disjoint = np.zeros(G, dtype=bool)
        for g in range(G):
            shape = [int(v) for v in grids[g].shape]
            if len(shape) != 3 or (isinstance(grids[g], torch.Tensor) and (not grids[g].is_cuda or grids[g].dtype != torch.float32)):
                raise ValueError("structure %d: a grid must be a float32 CUDA tensor or a NumPy array [x][y][z]" % g)
            xi2, yi2, zi2 = origins[g]
            try:
                box = self._common_box(o1, [self.xb, self.yb, self.zb], [xi2 / voxsp, yi2 / voxsp, zi2 / voxsp], shape)
            except ValueError as e:
                raise ValueError("structure %d: %s" % (g, e))
            disjoint[g] = box is None
            boxes[g].dims[:] = shape
            boxes[g].box[:] = box if box is not None else [0] * 9
        if G == 0:
            return np.zeros(0, dtype=np.float64)
        dev = self._dev.device
        st = _stream()
        g2s = [self._as_device_grid(grid, dev) for grid in grids]
        for g in range(G):
            boxes[g].grid = g2s[g].data_ptr()
        n_partial = C.c_longlong()
        call("mad_box_scores_layout", boxes, G, C.byref(n_partial))
        d_boxes = torch.from_numpy(np.frombuffer(bytearray(boxes), dtype=np.uint8)).pin_memory().to(dev, non_blocking=True)
        call("mad_threshold_normalise", _ptr(self._dev), self._dev.numel(), C.c_float(isovalue), C.c_float(1.0), 0, st)
        call("mad_threshold_many", boxes, G, _ptr(d_boxes), C.c_float(isovalue), st)
        self._host = None
        ws = torch.empty(max(1, n_partial.value) * 8, dtype=torch.float64, device=dev)
        out = torch.empty((G, 8), dtype=torch.float64, device=dev)
        n1 = [int(v) for v in self._dev.shape]
        call("mad_box_scores_many", _ptr(self._dev), n1[0], n1[1], n1[2], boxes, G, _ptr(d_boxes), C.c_float(0.0), _ptr(out),
             _ptr(ws), ws.numel() * 8, st)
        s = np.array(_Readback.read(out.view(torch.int64)), dtype=np.int64).view(np.float64).reshape(G, 8)
        res = np.zeros(G, dtype=np.float64)
        for g in range(G):
            if not disjoint[g]:
                res[g] = s[g][0] / np.sqrt(s[g][1] * s[g][2])
        return res

    def get_CCC_with_dmap(self, m2, isovalue=0):
        """mad/Dmap.py:260-372: overlap-normalised score against another Dmap."""
        if self.voxsp != m2.voxsp:
            print("ERROR: voxsp differ (%f vs %f)" % (self.voxsp, m2.voxsp))
        g2 = m2.device_grid() if isinstance(m2, Dmap) else self._as_device_grid(m2.grid3d, self._dev.device)
        s = self._box_scores(g2, m2.xi, m2.yi, m2.zi, float(isovalue))
        if s is None:
            return 0
        nonzero_vox = min(self._count_gt(self._dev, float(isovalue)), self._count_gt(g2, float(isovalue)))
        common_vox = int(s[5])
        if not common_vox or not nonzero_vox:
            return 0
        return s[0] / (np.sqrt(s[3]) * np.sqrt(s[4])) * (common_vox / nonzero_vox)

    def mask_with(self, mask_map):
        """mad/Dmap.py:99-151: voxels outside ``mask_map``'s box, or where it is < 1e-8, become 0 in this map."""
        if not np.isclose(self.voxsp, mask_map.voxsp):
            print("ERROR: voxsp do not match! %f vs %f" % (self.voxsp, mask_map.voxsp))
            sys.exit(1)
        voxsp = self.voxsp
        g2 = mask_map.device_grid() if isinstance(mask_map, Dmap) else self._as_device_grid(mask_map.grid3d, self._dev.device)
        o1 = [self.xi / voxsp, self.yi / voxsp, self.zi / voxsp]
        o2 = [mask_map.xi / voxsp, mask_map.yi / voxsp, mask_map.zi / voxsp]
        n1, n2 = [int(v) for v in self._dev.shape], [int(v) for v in g2.shape]
        shift = [int(round(o2[a] - o1[a])) for a in range(3)]
        lo = [min(shift[a], n1[a]) if shift[a] > 0 else 0 for a in range(3)]
        hi = [max(lo[a], min(n1[a], n2[a] + shift[a])) for a in range(3)]
        call("mad_mask_with", _ptr(self._dev), n1[0], n1[1], n1[2], _ptr(g2), n2[0], n2[1], n2[2],
             (C.c_int * 3)(*shift), (C.c_int * 3)(*lo), (C.c_int * 3)(*hi), _stream())
        self._host = None

    def gradient_device(self):
        """np.gradient of the grid as a float4-per-voxel CUDA tensor [x][y][z][4] (mad/structure_utils.py:79)."""
        nx, ny, nz = [int(v) for v in self._dev.shape]
        grad = torch.empty((nx, ny, nz, 4), dtype=torch.float32, device=self._dev.device)
        call("mad_gradient", _ptr(self._dev), nx, ny, nz, _ptr(grad), _stream())
        return grad

    def write_to_mrc(self, outname):
        """mad/Dmap.py:392-415: data as [z][y][x], nstart 0, origin = (xi, yi, zi), cella = box * voxsp."""
        _mrc.write_mrc(outname, self.grid3d.transpose(2, 1, 0), float(self.voxsp), origin=(self.xi, self.yi, self.zi))
