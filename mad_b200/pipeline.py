"""Array-level host API of the B200 hot path: device memory and streams come from PyTorch, all
arithmetic happens in libmad_b200.so (hand-written sm_100a CUDA) through the C ABI.

    space = build_space(grid)                 # a1-a4  (mad/MapSpace.py:116-189)
    kp    = detect(space)                     # a5-a6  (mad/Detector.py:18-128)
    ori   = orient(space, kp)                 # a7-a10 (mad/Orientator.py:68-343)
    dsc   = describe(space, kp, ori)          # a11-a12 (mad/Descriptor.py:106-202)
    pairs = match_threshold(hi_dsc, lo_dsc)   # a15    (mad/MaD.py:416-424)

The reference-shaped classes (MapSpace, Detector, Orientator, Descriptor) are thin wrappers over
these functions.  Nothing here computes on the CPU: without a CUDA device every call raises.
"""
import ctypes as C
import math
import os

import numpy as np
import torch

from . import _lib
from . import tables
from ._lib import call, KEYPOINT_DTYPE, ORIENTED_DTYPE, MAX_ORI, DSC_LEN

def launch_count():
    """Kernels launched by libmad_b200 in this process so far."""
    return int(_lib.lib.mad_launch_count())


def profile_enable(on=True):
    """Per-kernel CUDA-event timing inside the library (measurement only; adds two events per launch)."""
    call("mad_profile_reset")
    call("mad_profile_enable", 1 if on else 0)


def profile_records():
    """[(kernel name, milliseconds)] for every launch since profile_enable(True); clears the list."""
    out = []
    name = C.c_char_p()
    ms = C.c_float()
    for i in range(_lib.lib.mad_profile_count()):
        call("mad_profile_get", i, C.byref(name), C.byref(ms))
        out.append((name.value.decode(), float(ms.value)))
    call("mad_profile_reset")
    return out


def _require_cuda():
    if not torch.cuda.is_available():
        raise _lib.MadError("mad_b200 needs a CUDA device (sm_100a); there is no CPU fallback")


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


class _Readback(object):
    """Small device -> host reads (counts) through pinned mapped memory written by a kernel (mad_publish_small): a
    cudaMemcpy of 4 bytes would queue behind any large transfer the device -> host copy engine is busy with."""
    _slots = {}

    @classmethod
    def read(cls, *tensors):
        """Values of the given small int32 / int64 device tensors as Python ints (one synchronisation)."""
        dev = tensors[0].device
        key = (dev.index, torch.cuda.current_stream().cuda_stream)
        slot = cls._slots.get(key)
        if slot is None:
            slot = cls._slots[key] = torch.zeros(512, dtype=torch.int64).pin_memory()
        st = _stream()
        off, views = 0, []
        for t in tensors:
            t = t.contiguous().view(-1)
            nbytes = t.numel() * t.element_size()
            assert nbytes % 4 == 0 and off + nbytes <= slot.numel() * 8
            call("mad_publish_small", _ptr(t), C.c_void_p(slot.data_ptr() + off), nbytes, st)
            views.append((off, t.dtype, t.numel()))
            off += (nbytes + 7) // 8 * 8
        torch.cuda.current_stream().synchronize()
        raw = slot.numpy()
        out = []
        for o, dt, n in views:
            a = raw.view(np.uint8)[o:o + n * (8 if dt == torch.int64 else 4)].view(np.int64 if dt == torch.int64 else np.int32)
            out.extend(int(v) for v in a)
        return out


def _dptr(a):
    return a.ctypes.data_as(C.c_void_p)


class _DeviceTables(object):
    """Zone / rotation tables resident on one device."""

    def __init__(self, device, ori_zones=112, dsc_zones=16):
        self.device = device
        self.keep = []
        self.z_ori = self._zone_struct(tables.zone_tables(ori_zones))
        self.z_dsc = self._zone_struct(tables.zone_tables(dsc_zones))
        ot = tables.orientation_tables(ori_zones)
        self.ori_zones = ori_zones
        self.r1 = torch.from_numpy(np.ascontiguousarray(ot.r1.reshape(-1, 9))).to(device)
        self.rf = torch.from_numpy(np.ascontiguousarray(ot.rf.reshape(-1, 9))).to(device)
        self.rf_inv = torch.from_numpy(np.ascontiguousarray(ot.rf_inv.reshape(-1, 9))).to(device)

    def _zone_struct(self, zt):
        b = torch.from_numpy(np.ascontiguousarray(zt.bounds)).to(self.device)
        f = torch.from_numpy(np.ascontiguousarray(zt.belt_first)).to(self.device)
        p = torch.from_numpy(np.ascontiguousarray(zt.belt_phi)).to(self.device)
        self.keep += [b, f, p]
        s = _lib.MadZoneTable()
        s.n_zones, s.n_belts = zt.size, zt.n_belts
        s.bounds, s.belt_first, s.belt_phi = b.data_ptr(), f.data_ptr(), p.data_ptr()
        s.fast = None
        fast = torch.zeros(_lib.ZONE_FAST_BYTES, dtype=torch.uint8, device=self.device)
        with torch.cuda.device(self.device):
            call("mad_zone_fast_build", C.byref(s), _ptr(fast), _stream())
            torch.cuda.current_stream().synchronize()         # other streams may use the tables right away
        self.keep.append(fast)
        s.fast = fast.data_ptr()
        return s


_TABLE_CACHE = {}


def device_tables(device):
    key = (str(device),)
    if key not in _TABLE_CACHE:
        _TABLE_CACHE[key] = _DeviceTables(device)
    return _TABLE_CACHE[key]


class Space(object):
    """Device-resident scale space of one map (both octaves): what MapSpace.build_space makes."""

    def __init__(self):
        self.grids = []      # [up, base]           f32 [x][y][z]
        self.logs = []       # map_space            f32
        self.gauss = []      # gauss_list           f32
        self.grad4 = []      # grad_list as float4  f32 [x][y][z][4]
        self.grad_flags = [] # per octave: None = the whole field is computed; else uint8 tile flags (mad_gradient_masked)
        self.dims = []
        self.n_oct = 2       # 1 for oct_mode "up" / "base": octave slot 1 is a dummy the kernels never touch
        self.n_input_voxels = 0
        self._gauss = []     # Gaussian grids kept while tiles of the gradient may still be requested
        self._grad_done = {}  # (id(keypoint table object), radius) -> that object (kept alive: ids stay unique)

    @property
    def dims_host(self):
        return np.array([d for o in self.dims for d in o], dtype=np.int32)


def gradient_reach(radius):
    """Voxels around a keypoint's voxel the orientation / description stages may read, (up octave, base octave):
    the orientation patch spans +-2r (+-r) voxels (mad/Orientator.py:129-155), the rotated description lattice
    +-(2r - 1) sqrt(3) (+-(r - 0.5) sqrt(3)) before the nearest-voxel rule (mad/Descriptor.py:123-149)."""
    up = max(2 * radius, int(math.ceil((2 * radius - 1) * math.sqrt(3.0))) + 1)
    base = max(radius, int(math.ceil((radius - 0.5) * math.sqrt(3.0))) + 1)
    return up, base


def ensure_gradient(space, kp, radius=8):
    """Computes the gradient tiles within reach of the keypoints ``kp`` (no-op for a fully computed field)."""
    if all(f is None for f in space.grad_flags[:space.n_oct]) or len(kp) == 0:
        return
    key = (id(kp), int(radius))
    if key in space._grad_done:
        return
    st = _stream()
    up, base = gradient_reach(int(radius))
    f0, f1 = space.grad_flags
    if f0 is None or f1 is None:
        raise _lib.MadError("ensure_gradient: octaves must share the gradient mode")
    call("mad_gradient_mark", _ptr(kp.table), len(kp), _dptr(space.dims_host), up, base, _ptr(f0), _ptr(f1), st)
    for o, (gx, gy, gz) in enumerate(space.dims[:space.n_oct]):
        call("mad_gradient_masked", _ptr(space._gauss[o]), gx, gy, gz, _ptr(space.grad4[o]), _ptr(space.grad_flags[o]), st)
    space._grad_done[key] = kp


def full_gradient(space):
    """Materialises the whole gradient field (``MapSpace.grad_list``): every tile not computed yet is requested."""
    st = _stream()
    for o, (gx, gy, gz) in enumerate(space.dims[:space.n_oct]):
        fl = space.grad_flags[o]
        if fl is None:
            continue
        fl[fl == 0] = 1
        call("mad_gradient_masked", _ptr(space._gauss[o]), gx, gy, gz, _ptr(space.grad4[o]), _ptr(fl), st)
        space.grad_flags[o] = None
    space.grad_flags = [None] * len(space.grad_flags)           # (a single-octave space's dummy slot follows)
    return space.grad4


def build_space(grid, map_padding=9, sig_init=2, sig_presmooth=1, exact_f64=True, keep_gauss=True, full_gradient=True,
                oct_mode="both"):
    """a1-a4.  ``grid``: float32 [x][y][z], torch CUDA tensor or NumPy array (copied to the device).
    oct_mode (mad/MapSpace.py:149-163): "both" = [up, base]; "up" / "base" = that grid alone AS OCTAVE 0 -- the later
    stages pick their patch geometry from the octave index (mad/Orientator.py:125, mad/Descriptor.py:131), so a lone base
    grid is sampled with the stride-2 patches of octave 0, exactly as the reference does.
    full_gradient=False: the gradient field is computed later, only on the tiles the keypoints' patches touch
    (``ensure_gradient``, called by ``orient`` / ``describe``) or on demand (``full_gradient``)."""
    _require_cuda()
    if isinstance(grid, np.ndarray):
        grid = torch.from_numpy(np.ascontiguousarray(grid, dtype=np.float32)).cuda()
    grid = grid.contiguous().float()
    dev = grid.device
    st = _stream()
    nx, ny, nz = grid.shape
    sp = Space()
    sp.n_input_voxels = nx * ny * nz
    if map_padding:
        bx, by, bz = nx + 2 * map_padding, ny + 2 * map_padding, nz + 2 * map_padding
        base = torch.empty((bx, by, bz), dtype=torch.float32, device=dev)
        call("mad_pad3d", _ptr(grid), nx, ny, nz, int(map_padding), _ptr(base), st)
    else:
        bx, by, bz = nx, ny, nz
        base = grid
    if oct_mode not in ("both", "up", "base"):
        raise _lib.MadError("build_space: oct_mode %r" % (oct_mode,))
    # a2: 2x upsampled octave
    ux, uy, uz = 2 * bx - 1, 2 * by - 1, 2 * bz - 1
    if oct_mode != "base":
        up = torch.empty((ux, uy, uz), dtype=torch.float32, device=dev)
        ws_bytes = _lib.lib.mad_upsample_workspace_bytes(bx, by, bz)
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        if sig_presmooth:
            rad = tables.gaussian_radius(sig_presmooth)
            gw = np.ascontiguousarray(tables.gaussian_weights(sig_presmooth, 0, rad))
            call("mad_upsample_presmooth", _ptr(base), bx, by, bz, _dptr(gw), rad, _ptr(up), _ptr(ws), ws_bytes, st)
        else:
            call("mad_upsample_presmooth", _ptr(base), bx, by, bz, C.c_void_p(0), 0, _ptr(up), _ptr(ws), ws_bytes, st)
        del ws
    if oct_mode == "both":
        sp.grids = [up, base]
        sp.dims = [(ux, uy, uz), (bx, by, bz)]
    else:
        sp.n_oct = 1
        sp.grids = [up] if oct_mode == "up" else [base]
        sp.dims = [(ux, uy, uz) if oct_mode == "up" else (bx, by, bz)]
    # a3/a4 per octave
    rad = tables.gaussian_radius(sig_init)
    w0 = np.ascontiguousarray(tables.gaussian_weights(sig_init, 0, rad))
    w2 = np.ascontiguousarray(tables.gaussian_weights(sig_init, 2, rad))
    scale = float(np.float32(sig_init ** 2))
    for g, (gx, gy, gz) in zip(sp.grids, sp.dims):
        ws_bytes = _lib.lib.mad_log_gauss_workspace_bytes(gx, gy, gz)
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        lg = torch.empty((gx, gy, gz), dtype=torch.float32, device=dev)
        gs = torch.empty((gx, gy, gz), dtype=torch.float32, device=dev)
        call("mad_log_gauss", _ptr(g), gx, gy, gz, _dptr(w0), _dptr(w2), rad, C.c_float(scale), _ptr(lg), _ptr(gs),
             _ptr(ws), ws_bytes, 1 if exact_f64 else 0, st)
        del ws
        gr = torch.empty((gx, gy, gz, 4), dtype=torch.float32, device=dev)
        if full_gradient:
            call("mad_gradient", _ptr(gs), gx, gy, gz, _ptr(gr), st)
            sp.grad_flags.append(None)
        else:
            sp.grad_flags.append(torch.zeros(_lib.lib.mad_gradient_tiles(gx, gy, gz), dtype=torch.uint8, device=dev))
        sp._gauss.append(gs)
        sp.logs.append(lg)
        sp.gauss.append(gs if keep_gauss else None)
        sp.grad4.append(gr)
    if full_gradient and not keep_gauss:
        sp._gauss = []
    if sp.n_oct == 1:                                        # dummy octave 1: never indexed (no keypoint carries octave 1)
        sp.dims.append((1, 1, 1))
        sp.grad4.append(torch.zeros((1, 1, 1, 4), dtype=torch.float32, device=dev))
        sp.grad_flags.append(None if full_gradient else torch.zeros(1, dtype=torch.uint8, device=dev))
    return sp


class Keypoints(object):
    """Accepted keypoints in canonical order; device table (MadKeypoint[K]) + lazy host copy."""

    def __init__(self, table, count):
        self.table = table          # torch int32 [cap, 12] on the device
        self.count = int(count)
        self._host = None

    def host(self):
        if self._host is None:
            self._host = self.table[:self.count].cpu().numpy().view(KEYPOINT_DTYPE).reshape(-1)
        return self._host

    def __len__(self):
        return self.count


def keypoints_from_host(arr, device):
    arr = np.ascontiguousarray(arr, dtype=KEYPOINT_DTYPE)
    t = torch.from_numpy(arr.view(np.int32).reshape(-1, 12).copy()).to(device)
    k = Keypoints(t, len(arr))
    k._host = arr
    return k


def detect(space, border=12, threshold=5e-2, cap=None):
    """a5/a6 on both octaves, canonical order, accepted keypoints only."""
    _require_cuda()
    dev = space.logs[0].device
    st = _stream()
    if cap is None:
        cap = 1 << 16
    while True:
        cand = torch.empty((cap, 12), dtype=torch.int32, device=dev)
        counter = torch.zeros(1, dtype=torch.int32, device=dev)
        for o, (lg, (gx, gy, gz)) in enumerate(zip(space.logs, space.dims)):      # (logs has n_oct entries)
            call("mad_detect", _ptr(lg), gx, gy, gz, o, int(border), C.c_float(threshold), _ptr(cand), cap,
                 _ptr(counter), st)
        n = _Readback.read(counter)[0]
        if n <= cap:
            break
        cap = int(n * 1.25) + 16        # rare: candidate list overflowed, redo with room
    out = torch.empty((max(n, 1), 12), dtype=torch.int32, device=dev)
    out_count = torch.zeros(1, dtype=torch.int32, device=dev)
    ws_bytes = _lib.lib.mad_sort_keypoints_workspace_bytes(n)
    ws = torch.empty(max(ws_bytes, 1), dtype=torch.uint8, device=dev)
    dims = space.dims_host
    call("mad_sort_keypoints", _ptr(cand), n, _dptr(dims), _ptr(out), _ptr(out_count), _ptr(ws), ws_bytes, st)
    return Keypoints(out, _Readback.read(out_count)[0])


class Oriented(object):
    def __init__(self, table, count):
        self.table = table          # torch int32 [cap, 2] on the device (MadOriented)
        self.count = int(count)
        self._host = None

    def host(self):
        if self._host is None:
            self._host = self.table[:self.count].cpu().numpy().view(ORIENTED_DTYPE).reshape(-1)
        return self._host

    def __len__(self):
        return self.count


def oriented_from_host(arr, device):
    arr = np.ascontiguousarray(arr, dtype=ORIENTED_DTYPE)
    t = torch.from_numpy(arr.view(np.int32).reshape(-1, 2).copy()).to(device)
    o = Oriented(t, len(arr))
    o._host = arr
    return o


def orient(space, kp, radius=8, lim_main=6, lim_sec=6):
    """a7-a10: per keypoint up to 36 (main, sec) pairs, compacted in emission order."""
    _require_cuda()
    dev = space.grad4[0].device
    st = _stream()
    tb = device_tables(dev)
    n = len(kp)
    if n == 0:
        return Oriented(torch.empty((1, 2), dtype=torch.int32, device=dev), 0)
    ensure_gradient(space, kp, radius)
    n_ori = torch.empty(n, dtype=torch.int32, device=dev)
    slots = torch.empty((n, MAX_ORI), dtype=torch.int32, device=dev)
    dims = space.dims_host
    call("mad_orient", _ptr(space.grad4[0]), _ptr(space.grad4[1]), _dptr(dims), _ptr(kp.table), n, int(radius),
         C.byref(tb.z_ori), _ptr(tb.r1), int(lim_main), int(lim_sec), _ptr(n_ori), _ptr(slots), st)
    cap = n * MAX_ORI
    out = torch.empty((cap, 2), dtype=torch.int32, device=dev)
    out_count = torch.zeros(1, dtype=torch.int32, device=dev)
    ws_bytes = _lib.lib.mad_compact_oriented_workspace_bytes(n)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    call("mad_compact_oriented", _ptr(n_ori), _ptr(slots), n, _ptr(out), cap, _ptr(out_count), _ptr(ws), ws_bytes, st)
    return Oriented(out, _Readback.read(out_count)[0])


def describe(space, kp, ori, radius=8):
    """a11/a12: int16 [D, 1024] descriptors on the device."""
    _require_cuda()
    dev = space.grad4[0].device
    st = _stream()
    tb = device_tables(dev)
    d = len(ori)
    dsc = torch.empty((d, DSC_LEN), dtype=torch.int16, device=dev)
    if d == 0:
        return dsc
    ensure_gradient(space, kp, radius)
    dims = space.dims_host
    call("mad_describe", _ptr(space.grad4[0]), _ptr(space.grad4[1]), _dptr(dims), _ptr(kp.table), _ptr(ori.table), d,
         int(radius), C.byref(tb.z_dsc), _ptr(tb.rf), _ptr(tb.rf_inv), tb.ori_zones, _ptr(dsc), st)
    return dsc


def describe_struct(grid, patch_size=16, map_padding=9, sig_init=2, sig_presmooth=1, exact_f64=True,
                    keep_gauss=False, full_gradient=None):
    """The whole a1-a12 chain of ``MaD._describe_struct`` (mad/MaD.py:358-368) on device arrays.
    full_gradient: None = only when the dense arrays are kept for inspection (keep_gauss); the product path computes
    the gradient on the tiles around the keypoints (same descriptors, see ``ensure_gradient``)."""
    r = (patch_size - patch_size % 2) // 2
    if full_gradient is None:
        full_gradient = bool(keep_gauss)
    sp = build_space(grid, map_padding, sig_init, sig_presmooth, exact_f64=exact_f64, keep_gauss=keep_gauss,
                     full_gradient=full_gradient)
    kp = detect(sp)
    ori = orient(sp, kp, r)
    dsc = describe(sp, kp, ori, r)
    return sp, kp, ori, dsc


# ---------------------------------------------------------------------------------------------
# a15 matching
# ---------------------------------------------------------------------------------------------
class DescriptorSet(object):
    """int16 descriptors prepared for matching: exact norms, the uint8 tensor-core operand
    (tcgen05 kind::i8, exact while every entry <= 255) and, on demand, an fp16 copy for the general
    tensor-core kernel (impl 2)."""

    def __init__(self, dsc, need_half=False):
        _require_cuda()
        if isinstance(dsc, np.ndarray):
            dsc = torch.from_numpy(np.ascontiguousarray(dsc, dtype=np.int16)).cuda()
        self.dsc = dsc.contiguous()
        assert self.dsc.dtype == torch.int16 and self.dsc.dim() == 2 and self.dsc.shape[1] == DSC_LEN
        dev = self.dsc.device
        st = _stream()
        self.rows = self.dsc.shape[0]
        self.rows_padded = max((self.rows + 255) // 256 * 256, 256)      # CTA-pair kernel: 256-row lo tiles
        self.norm2 = torch.empty(max(self.rows, 1), dtype=torch.int32, device=dev)
        self.rnorm = torch.empty(self.rows_padded, dtype=torch.float32, device=dev)
        self.u8 = torch.empty((self.rows_padded, DSC_LEN), dtype=torch.uint8, device=dev)
        mx = torch.zeros(2, dtype=torch.int32, device=dev)           # largest entry, largest squared norm
        call("mad_dsc_prepare", _ptr(self.dsc), self.rows, self.rows_padded, _ptr(self.norm2), _ptr(self.rnorm),
             _ptr(self.u8), _ptr(mx), _ptr(mx[1:]), st)
        self._max_dev = mx
        self._max_entry = None
        self._max_norm2 = None
        self.half = None
        s = _lib.MadDscSet()
        s.dsc = self.dsc.data_ptr()
        s.half = 0
        s.norm2 = self.norm2.data_ptr()
        s.u8 = self.u8.data_ptr()
        s.rnorm = self.rnorm.data_ptr()
        s.rows, s.rows_padded = self.rows, self.rows_padded
        s.max_entry = -1
        s.max_norm2 = -1
        self.c = s
        if need_half:
            self.ensure_half()

    @property
    def max_entry(self):
        """Largest descriptor entry (one device->host read, cached); DSC_REFUSED if the set is not a descriptor set."""
        if self._max_entry is None:
            self._set_maxima(*self._max_dev.tolist())
        return self._max_entry

    def _set_maxima(self, max_entry, max_norm2):
        self._max_entry, self._max_norm2 = int(max_entry), int(max_norm2)
        self.c.max_entry, self.c.max_norm2 = self._max_entry, self._max_norm2

    def ensure_half(self):
        if self.half is None:
            self.half = torch.empty((self.rows_padded, DSC_LEN), dtype=torch.float16, device=self.dsc.device)
            call("mad_dsc_to_half", _ptr(self.dsc), self.rows, self.rows_padded, _ptr(self.half), _stream())
            self.c.half = self.half.data_ptr()
        return self


def _as_set(x):
    return x if isinstance(x, DescriptorSet) else DescriptorSet(x)


def _check_descriptors(hi, lo):
    if max(hi._max_entry, lo._max_entry) >= _lib.DSC_REFUSED:
        raise _lib.MadError("mad_match: not a descriptor set (a negative entry, or a squared norm >= 2^31)")


def _exact_impl(hi, lo):
    """Product choice for sets whose maxima are known: the uint8 kernel while every entry is <= 255; else the fp16 kernel
    where its fp32 sums are exact (entries <= 2048 and max |hi|^2 max |lo|^2 <= 2^48, so every dot product is <= 2^24),
    else the SIMT kernel (exact in int32)."""
    _check_descriptors(hi, lo)
    if max(hi._max_entry, lo._max_entry) <= 255:
        return 0
    if max(hi._max_entry, lo._max_entry) <= 2048 and hi._max_norm2 * lo._max_norm2 <= 1 << 48:
        return 2
    return 1


def _pick_impl(hi, lo, impl):
    """impl None = product choice (``_exact_impl``): the uint8 tcgen05 kernel, or, if an entry exceeds 255, a kernel that
    is exact for the set.  Returns (impl, verify).  When the largest entry of a set has not been read back yet, the uint8
    kernel runs optimistically and the check is folded into the read-back the call makes anyway
    (verify = True): a separate 4-byte device-to-host read here would queue behind any large
    copy-out in flight on another stream and stall the matching kernel for its whole duration."""
    verify = False
    if impl is None:
        if hi._max_entry is None or lo._max_entry is None:
            return 0, True
        impl = _exact_impl(hi, lo)
    return _pick_impl_explicit(hi, lo, impl), verify


def _pick_impl_explicit(hi, lo, impl):
    hi.max_entry, lo.max_entry              # noqa: B018  (fills the C structs: the library checks the sets' maxima)
    if impl == 2:
        hi.ensure_half()
        lo.ensure_half()
    return impl


_PAIR_CAP = {}


def scores_from_dots(pair_hi, pair_lo, pair_dot, hi_norm2, lo_norm2):
    """Host side of the compact pair format: float64 cosine scores from the exact integer dot products and squared norms,
    with the operations of the device's mad_score (multiply, sqrt, divide: all correctly rounded), hence bit-identical."""
    p = np.asarray(hi_norm2, dtype=np.float64)[np.asarray(pair_hi)] * np.asarray(lo_norm2, dtype=np.float64)[np.asarray(pair_lo)]
    out = np.zeros(len(p), dtype=np.float64)
    nz = p > 0.0
    out[nz] = np.asarray(pair_dot, dtype=np.float64)[nz] / np.sqrt(p[nz])
    return out


def pair_hi_from_counts(counts):
    """Host side of the compact pair format: the hi index of every pair from the per-hi-row pair counts (the pair list is
    in row-major order, so pair_hi is non-decreasing)."""
    counts = np.asarray(counts)
    return np.repeat(np.arange(len(counts), dtype=np.int32), counts)


def match_threshold(hi, lo, cc=0.6, impl=None, want="score"):
    """Pairs (i, j) with cosine(hi_i, lo_j) > cc in row-major order (mad/MaD.py:420-424).
    Returns (hi index int32 [P], lo index int32 [P], score float64 [P]) as device tensors; want="dot" (uint8 kernel only)
    returns the exact int32 dot products instead of the scores (``scores_from_dots``).
    impl: None/0 = one-pass uint8 tcgen05 kernel + sort (product), 1 = SIMT check kernel,
    2 = fp16 tcgen05 kernel (both two-pass count/fill)."""
    hi, lo = _as_set(hi), _as_set(lo)
    dev = hi.dsc.device
    st = _stream()
    m = hi.rows
    if m == 0 or lo.rows == 0:
        e = torch.empty(0, dtype=torch.int32, device=dev)
        return e, e.clone(), torch.empty(0, dtype=torch.float64, device=dev)
    impl, verify = _pick_impl(hi, lo, impl)
    if impl == 0:
        return _match_threshold_onepass(hi, lo, cc, dev, st, verify, want)
    if want != "score":
        raise _lib.MadError("match_threshold: want='dot' is a format of the uint8 kernel (impl 0)")
    n_seg = int(_lib.lib.mad_match_segments(m, lo.rows, impl))
    seg_count = torch.empty(m * n_seg, dtype=torch.int32, device=dev)
    call("mad_match_count", C.byref(hi.c), C.byref(lo.c), C.c_double(cc), n_seg, _ptr(seg_count), impl, st)
    seg_off = torch.empty(m * n_seg, dtype=torch.int64, device=dev)
    total = torch.zeros(1, dtype=torch.int64, device=dev)
    ws_bytes = _lib.lib.mad_exclusive_scan_workspace_bytes(m * n_seg)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    call("mad_exclusive_scan_i32_to_i64", _ptr(seg_count), m * n_seg, _ptr(seg_off), _ptr(total), _ptr(ws), ws_bytes, st)
    p = int(total.item())
    pair_hi = torch.empty(max(p, 1), dtype=torch.int32, device=dev)
    pair_lo = torch.empty(max(p, 1), dtype=torch.int32, device=dev)
    score = torch.empty(max(p, 1), dtype=torch.float64, device=dev)
    call("mad_match_fill", C.byref(hi.c), C.byref(lo.c), C.c_double(cc), n_seg, _ptr(seg_off), _ptr(pair_hi), _ptr(pair_lo),
         _ptr(score), impl, st)
    return pair_hi[:p], pair_lo[:p], score[:p]


def _read_counts(count, hi, lo):
    """One device->host read: (pairs found, largest entry and squared norm of hi, of lo); caches the maxima."""
    vals = _Readback.read(count, hi._max_dev, lo._max_dev)
    hi._set_maxima(vals[1], vals[2])
    lo._set_maxima(vals[3], vals[4])
    return int(vals[0])


def _match_threshold_onepass(hi, lo, cc, dev, st, verify=False, want="score"):
    key = (hi.rows, lo.rows)
    cap = _PAIR_CAP.get(key, max(1 << 20, 16 * (hi.rows + lo.rows)))
    while True:
        cand_key = torch.empty(cap, dtype=torch.int64, device=dev)
        cand_dot = torch.empty(cap, dtype=torch.int32, device=dev)
        count = torch.empty(1, dtype=torch.int64, device=dev)
        call("mad_match_pairs", C.byref(hi.c), C.byref(lo.c), C.c_double(cc), _ptr(cand_key), _ptr(cand_dot),
             C.c_uint64(cap), _ptr(count), st)
        p = _read_counts(count, hi, lo)
        if p >= (1 << 62):
            raise _lib.MadError("mad_match_pairs: the kernel's internal hand-off timed out (pair list incomplete)")
        if verify and _exact_impl(hi, lo) != 0:
            if want != "score":
                raise _lib.MadError("match_threshold: entries above 255 need the fp16 or SIMT kernel, which have no want='dot' form")
            return match_threshold(hi, lo, cc)              # entries above 255: the kernel that is exact for the sets
        if p <= cap:
            break
        cap = p + p // 8 + 1024            # the candidate list overflowed: repeat with room
    _PAIR_CAP[key] = max(cap, p + p // 4)
    pair_hi = torch.empty(max(p, 1), dtype=torch.int32, device=dev)
    pair_lo = torch.empty(max(p, 1), dtype=torch.int32, device=dev)
    score = torch.empty(max(p, 1), dtype=torch.float64 if want == "score" else torch.int32, device=dev)
    if p:
        ws_bytes = _lib.lib.mad_match_pairs_finish_workspace_bytes(p)
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        if want == "score":
            call("mad_match_pairs_finish", _ptr(cand_key), _ptr(cand_dot), p, hi.rows, lo.rows, _ptr(hi.norm2), _ptr(lo.norm2),
                 _ptr(pair_hi), _ptr(pair_lo), _ptr(score), _ptr(ws), ws_bytes, st)
        else:
            call("mad_match_pairs_finish_dot", _ptr(cand_key), _ptr(cand_dot), p, hi.rows, lo.rows, _ptr(pair_hi), _ptr(pair_lo),
                 _ptr(score), _ptr(ws), ws_bytes, st)
    return pair_hi[:p], pair_lo[:p], score[:p]


HOST_COPY_CTAS = int(os.environ.get("MAD_HOST_COPY_CTAS", "8"))    # 2: copy-bound (12.5 ms per C2 map); 4-8: 9.1-9.6; 16-32: 9.4-9.7


class HostStage(object):
    """Pinned host staging buffers for device -> host results, reused across calls: ``fetch`` starts
    an asynchronous copy on the current stream and returns the CPU view, valid after ``sync()``."""

    def __init__(self):
        self.bufs = {}
        self.copy_stream = None
        self.keep = []

    def fetch(self, name, t, overlap=False):
        """overlap=True: the copy runs on a side stream (after everything queued so far on the
        current stream), so later kernels on the current stream are not held up by the PCIe copy."""
        n = t.numel() * t.element_size()
        buf = self.bufs.get(name)
        if buf is None or buf.numel() < n:
            if buf is not None:
                self.keep.append(buf)      # a copy kernel may still be writing into the old buffer: free it after the wait
            buf = torch.empty(max(n * 5 // 4, 256), dtype=torch.uint8).pin_memory()
            self.bufs[name] = buf
        view = buf[:n].view(t.dtype).view(t.shape)
        if not n:
            return view
        if overlap:
            if self.copy_stream is None:
                self.copy_stream = torch.cuda.Stream()
            self.copy_stream.wait_stream(torch.cuda.current_stream())
            t = t.contiguous()
            if t.data_ptr() % 16 == 0:
                # a few CTAs store straight into the pinned (device-mapped) buffer: the copy engine stays free, so nothing
                # of the next map (CUB's internal memsets, ...) queues behind a multi-millisecond download
                call("mad_copy_to_host", _ptr(t), C.c_void_p(buf.data_ptr()), n, HOST_COPY_CTAS, C.c_void_p(self.copy_stream.cuda_stream))
            else:
                with torch.cuda.stream(self.copy_stream):
                    view.copy_(t, non_blocking=True)
            t.record_stream(self.copy_stream)
            self.keep.append(t)
        else:
            view.copy_(t, non_blocking=True)
        return view

    def sync(self):
        torch.cuda.current_stream().synchronize()
        if self.copy_stream is not None:
            self.copy_stream.synchronize()
        self.keep = []
        self.marks = []

    def mark(self):
        """Records the point after every copy issued so far; ``wait()`` then blocks the host on exactly these copies
        (and not on later work queued on the compute stream)."""
        evs = [torch.cuda.Event()]
        evs[0].record(torch.cuda.current_stream())
        if self.copy_stream is not None:
            evs.append(torch.cuda.Event())
            evs[1].record(self.copy_stream)
        self.marks = evs

    def wait(self):
        for ev in getattr(self, "marks", []):
            ev.synchronize()
        self.marks = []
        self.keep = []


class MapStream(object):
    """Streams maps through the hot path (a1-a12, and a15 against resident descriptor sets) with the PCIe copies of
    neighbouring maps overlapped with the kernels: the upload of the next map runs on a copy stream while the current
    one is on the SMs, and results travel to pinned host buffers on a side stream while the next map computes.

        ms = MapStream(hi=component_sets, cc=0.6)
        up = ms.upload(pinned_grid_0)
        for grid in more_grids:                  # every map: upload -> describe (+ match) -> download
            nxt = ms.upload(grid); ticket = ms.submit(up); ...; res = ms.result(ticket); up = nxt

    ``result`` returns host arrays: dsc int16 [D][1024], kp / ori tables and, with ``hi``, the pair lists."""

    def __init__(self, hi=None, cc=0.6, exact_f64=True, match_impl=None, patch_size=16, depth=2, download=True, compact=False):
        """compact=True: results travel in the compact wire format -- descriptors as the uint8 matching operand
        (``dsc_u8``; entries are vote counts <= 255, widen with ``.astype(np.int16)``), pairs as per-hi-row counts + (lo,
        exact int32 dot) + the map's squared norms (``pair_hi_counts``, ``pair_lo``, ``pair_dot``, ``lo_norm2``;
        ``pair_hi_from_counts`` / ``scores_from_dots`` rebuild the indices and the float64 scores bit for bit):
        70 MB instead of 140 MB per C2 map over PCIe."""
        _require_cuda()
        self.compact = bool(compact)
        self.download = download                        # False: results stay on the device (result() returns CUDA tensors)
        self.hi = _as_set(hi) if hi is not None else None
        self.cc, self.exact, self.impl, self.patch = cc, exact_f64, match_impl, patch_size
        self.up_stream = torch.cuda.Stream()
        self.stages = [HostStage() for _ in range(max(2, depth))]
        self.n = 0
        self.gbuf = [None] * max(2, depth)                 # persistent upload buffers
        self.gfree = [None] * max(2, depth)
        self.n_up = 0

    def upload(self, grid):
        """Starts the host -> device copy of a float32 [x][y][z] grid (pinned CPU tensor for an asynchronous copy) into one
        of ``depth`` persistent device buffers.  (A fresh tensor per map made the caching allocator call cudaMalloc /
        cudaFree in steady state -- a block freed while another stream still uses it cannot be reused at once -- and each
        of those synchronises the device: 16 ms per C2 map instead of 8.3.)"""
        if isinstance(grid, np.ndarray):
            grid = torch.from_numpy(np.ascontiguousarray(grid, dtype=np.float32))
        if self.n_up - self.n >= len(self.gbuf):
            raise _lib.MadError("MapStream.upload: %d uploads are waiting for submit(); the %d upload buffers are all in use"
                                % (self.n_up - self.n, len(self.gbuf)))
        k = self.n_up % len(self.gbuf)
        self.n_up += 1
        dev = torch.device("cuda", torch.cuda.current_device())
        if self.gbuf[k] is None or self.gbuf[k].shape != grid.shape:
            self.gbuf[k] = torch.empty(tuple(grid.shape), dtype=torch.float32, device=dev)
        if self.gfree[k] is not None:
            self.up_stream.wait_event(self.gfree[k])        # the map that used this buffer has been consumed
        with torch.cuda.stream(self.up_stream):
            self.gbuf[k].copy_(grid, non_blocking=True)
            ev = torch.cuda.Event()
            ev.record(self.up_stream)
        return self.gbuf[k], ev, k

    def submit(self, uploaded):
        g, ev, k = uploaded
        cur = torch.cuda.current_stream()
        cur.wait_event(ev)
        stage = self.stages[self.n % len(self.stages)]
        self.n += 1
        stage.wait()                                    # the slot's previous results have left the device
        sp, kp, ori, dsc = describe_struct(g, patch_size=self.patch, exact_f64=self.exact)
        if k is not None:
            self.gfree[k] = torch.cuda.Event()
            self.gfree[k].record(cur)                       # the upload buffer may be overwritten from here on
        get = (lambda name, t: stage.fetch(name, t, overlap=True)) if self.download else (lambda name, t: t)
        out = {"kp": get("kp", kp.table[:len(kp)]), "ori": get("ori", ori.table[:len(ori)])}
        lo = DescriptorSet(dsc) if (self.hi is not None or self.compact) else None
        if self.compact:
            out.update(dsc_u8=get("dsc8", lo.u8[:lo.rows]), lo_norm2=get("n2", lo.norm2[:lo.rows]))
        else:
            out["dsc"] = get("dsc", dsc)
        if self.hi is not None:
            if self.compact:
                ph, pl, dot = match_threshold(self.hi, lo, self.cc, impl=self.impl, want="dot")
                # the list is sorted by hi row: the per-row pair counts (4 B per hi row) carry pair_hi (4 B per PAIR) --
                # ``pair_hi_from_counts`` expands them on the host
                cnt = torch.zeros(self.hi.rows, dtype=torch.int32, device=ph.device)      # (no bincount: it synchronises)
                if ph.numel():
                    cnt.scatter_add_(0, ph.long(), torch.ones_like(ph))
                out.update(pair_hi_counts=get("pc", cnt), pair_lo=get("pl", pl), pair_dot=get("pd", dot))
            else:
                ph, pl, sc = match_threshold(self.hi, lo, self.cc, impl=self.impl)
                out.update(pair_hi=get("ph", ph), pair_lo=get("pl", pl), score=get("sc", sc))
        stage.mark()
        return stage, out

    def result(self, ticket):
        stage, out = ticket
        stage.wait()
        return out


class MapBatch(object):
    """A batch of independent maps (ensemble frames / conformational snapshots: the loops of mad/MaD.py:143-162,178-189)
    through a1-a12.  Small maps are launch- and host-latency bound (a 96^3 map is ~40 launches and 3 count read-backs for
    under a millisecond of GPU work), so ``streams`` host threads, each with its own CUDA stream, persistent upload buffer
    and pinned result stage, work on different maps: one map's host round trips hide behind another map's kernels.

        batch = MapBatch(streams=4)
        results = batch.run(list_of_pinned_grids)          # [{"n_kp", "n_dsc", "dsc", "kp", "ori"}] in input order
    """

    def __init__(self, streams=4, patch_size=16, exact_f64=True, compact=False):
        """compact=True: descriptors come home as uint8 (``dsc_u8``: vote counts <= 255 for every patch size the reference
        uses; checked per map, the int16 table is sent instead if an entry is larger) -- half the bytes over PCIe."""
        _require_cuda()
        from concurrent.futures import ThreadPoolExecutor
        self.compact = bool(compact)
        self.nw = max(1, int(streams))
        self.patch, self.exact = patch_size, exact_f64
        self.device = torch.cuda.current_device()
        self.streams = [torch.cuda.Stream() for _ in range(self.nw)]
        self.stages = [HostStage() for _ in range(self.nw)]
        self.up = [None] * self.nw
        self.pool = ThreadPoolExecutor(self.nw)
        self.last_d2h_bytes = 0
        device_tables(torch.device("cuda", self.device))       # one-time table initialisation before the workers start

    def _work(self, w, grids, download):
        torch.cuda.set_device(self.device)
        out = []
        with torch.cuda.stream(self.streams[w]):
            for j in range(w, len(grids), self.nw):
                g = grids[j]
                if isinstance(g, np.ndarray):
                    g = torch.from_numpy(np.ascontiguousarray(g, dtype=np.float32))
                if not g.is_cuda:                               # persistent upload buffer: no allocator traffic per map
                    if self.up[w] is None or self.up[w].shape != g.shape:
                        self.up[w] = torch.empty(tuple(g.shape), dtype=torch.float32, device="cuda")
                    self.up[w].copy_(g, non_blocking=True)
                    g = self.up[w]
                sp, kp, ori, dsc = describe_struct(g, patch_size=self.patch, exact_f64=self.exact)
                r = {"n_kp": len(kp), "n_dsc": len(ori)}
                if download:
                    st = self.stages[w]
                    r.update(kp=st.fetch("kp%d" % j, kp.table[:len(kp)]), ori=st.fetch("ori%d" % j, ori.table[:len(ori)]))
                    if self.compact:
                        ds = DescriptorSet(dsc)
                        r["_max"] = ds._max_dev[:1]
                        r["dsc_u8"] = st.fetch("dsc8_%d" % j, ds.u8[:ds.rows])
                        r["_dsc_dev"] = dsc
                    else:
                        r["dsc"] = st.fetch("dsc%d" % j, dsc)
                else:
                    r.update(dsc=dsc, kp=kp.table[:len(kp)], ori=ori.table[:len(ori)])
                out.append((j, r))
            self.streams[w].synchronize()
            for _, r in out:                                    # compact: an entry above 255 does not fit the uint8 table
                if "_max" in r:
                    if int(r.pop("_max").item()) > 255:
                        del r["dsc_u8"]
                        r["dsc"] = r["_dsc_dev"].cpu()
                    del r["_dsc_dev"]
        return out

    def run(self, grids, download=True):
        """``grids``: float32 [x][y][z] maps -- pinned CPU tensors / NumPy arrays are uploaded, CUDA tensors used in place.
        download=True: tables come back as host arrays (views of pinned buffers, valid until the next ``run``)."""
        main = torch.cuda.current_stream()
        for s_ in self.streams:
            s_.wait_stream(main)
        parts = [f.result() for f in [self.pool.submit(self._work, w, grids, download) for w in range(self.nw)]]
        for s_ in self.streams:
            main.wait_stream(s_)
        res = [r for _, r in sorted((x for p in parts for x in p), key=lambda x: x[0])]
        if download:
            self.last_d2h_bytes = int(sum(r[k].numel() * r[k].element_size() for r in res for k in ("dsc", "dsc_u8", "kp", "ori") if k in r))
        return res


def concat_sets(sets):
    """One DescriptorSet holding the rows of several (e.g. all subunits of an assembly) + row offsets,
    so that one matching launch serves them all; pairs come back with global hi rows."""
    offs = np.cumsum([0] + [s.rows for s in sets]).astype(np.int64)
    return DescriptorSet(torch.cat([s.dsc for s in sets], 0)), offs


def match_topk(hi, lo, k=8, lo_index_base=0, impl=None):
    """Per hi row the k best lo rows by (score desc, index asc).  Device tensors (idx, score)."""
    hi, lo = _as_set(hi), _as_set(lo)
    dev = hi.dsc.device
    st = _stream()
    impl, verify = _pick_impl(hi, lo, impl)
    idx = torch.empty((hi.rows, k), dtype=torch.int32, device=dev)
    score = torch.empty((hi.rows, k), dtype=torch.float64, device=dev)
    ws_bytes = _lib.lib.mad_match_topk_workspace_bytes(hi.rows, lo.rows, int(k), impl)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    call("mad_match_topk", C.byref(hi.c), C.byref(lo.c), int(k), int(lo_index_base), _ptr(idx), _ptr(score), _ptr(ws),
         ws_bytes, impl, st)
    if verify:
        _read_counts(torch.zeros(1, dtype=torch.int64, device=dev), hi, lo)
        if _exact_impl(hi, lo) != 0:
            return match_topk(hi, lo, k, lo_index_base)
    return idx, score


def topk_merge(idx_g, score_g):
    """[G, M, k] per-shard lists -> merged [M, k]."""
    g, m, k = idx_g.shape
    dev = idx_g.device
    idx = torch.empty((m, k), dtype=torch.int32, device=dev)
    score = torch.empty((m, k), dtype=torch.float64, device=dev)
    call("mad_topk_merge", _ptr(idx_g.contiguous()), _ptr(score_g.contiguous()), g, m, k, _ptr(idx), _ptr(score), _stream())
    return idx, score


# ---------------------------------------------------------------------------------------------
# next component (SURVEY.md 8f rank 1): MaD._match_dsc including its per-pair repeatability loop
# ---------------------------------------------------------------------------------------------
class FeatureTable(object):
    """Oriented + described features of one structure as device tables: descriptors (DescriptorSet),
    meta int32 [D, 4] = (index, oct_scale, main_bin, sec_bin), sub-voxel map coordinates float64 [D, 3]."""

    def __init__(self, dsc, index, oct_scale, main_bin, sec_bin, subv_map_coords):
        _require_cuda()
        self.set = dsc if isinstance(dsc, DescriptorSet) else DescriptorSet(dsc)
        dev = self.set.dsc.device
        meta = np.stack([np.asarray(index), np.asarray(oct_scale), np.asarray(main_bin), np.asarray(sec_bin)], 1)
        self.meta_host = np.ascontiguousarray(meta, dtype=np.int32)
        self.subv_host = np.ascontiguousarray(subv_map_coords, dtype=np.float64).reshape(-1, 3)
        assert len(self.meta_host) == self.set.rows == len(self.subv_host)
        self.meta = torch.from_numpy(self.meta_host).to(dev)
        self.subv = torch.from_numpy(self.subv_host).to(dev)

    @classmethod
    def from_features(cls, df_list):
        """From a list of DensityFeature (the reference's ``lo_dsc_list`` / ``hi_dsc_list``)."""
        dsc = np.array([df.lin_ar_subeqsp for df in df_list], dtype=np.int16).reshape(-1, DSC_LEN)
        return cls(dsc, [df.index for df in df_list], [df.oct_scale for df in df_list], [df.main_bin for df in df_list],
                   [df.sec_bin for df in df_list], np.array([df.subv_map_coords for df in df_list], dtype=np.float64))


class AnchorCloud(object):
    """np.unique(subv[used], axis=0) built on the device (``mad_anchor_cloud``) and, for the lo side, the uniform grid of
    cell size ``cell`` the repeatability kernel searches (``mad_cloud_grid``): the cell-sorted cloud, cell_start and the
    27-neighbourhood bitmap.  ``org`` float64 [3] / ``dims`` int32 [3] are host copies."""

    def __init__(self, subv, used, cell):
        dev = subv.device
        st = _stream()
        d = int(subv.shape[0])
        self.cell = float(cell)
        self._buf = torch.empty((max(d, 1), 3), dtype=torch.float64, device=dev)
        self.org_dev = torch.empty(3, dtype=torch.float64, device=dev)
        self.info = torch.empty(8, dtype=torch.int64, device=dev)
        ws_bytes = _lib.lib.mad_anchor_cloud_workspace_bytes(d)
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        call("mad_anchor_cloud", _ptr(subv), _ptr(used), d, C.c_double(self.cell), _ptr(self._buf), _ptr(self.org_dev),
             _ptr(self.info), _ptr(ws), ws_bytes, st)
        self.n = None

    def take_info(self, vals):
        """The eight values of ``info`` read back (see ``read_clouds``); refuses a cloud with a non-finite coordinate."""
        n, bad = int(vals[0]), int(vals[1])
        if bad:
            raise _lib.MadError("anchor cloud: %d used feature(s) with a non-finite coordinate" % bad)
        self.n = n
        self.dims64 = np.array(vals[2:5], dtype=np.int64)
        self.org = np.array(vals[5:8], dtype=np.int64).view(np.float64)
        self.dims = self.dims64.astype(np.int32)
        self.cloud = self._buf[:n]
        return self

    def build_grid(self):
        """mad_cloud_grid: lo_sorted, cell_start, near_bits (refused with MadError for a grid of >= 2^31 cells)."""
        dev = self._buf.device
        ncell = int(np.prod([int(v) for v in self.dims64], dtype=object))
        fits = ncell < (1 << 31)
        self.sorted = torch.empty((max(self.n, 1), 3), dtype=torch.float64, device=dev)
        self.cell_start = torch.empty(ncell + 1 if fits else 1, dtype=torch.int32, device=dev)
        self.near_bits = torch.zeros((ncell + 31) // 32 if fits else 1, dtype=torch.int32, device=dev)
        ws_bytes = _lib.lib.mad_cloud_grid_workspace_bytes(self.n)
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        call("mad_cloud_grid", _ptr(self.cloud), self.n, _ptr(self.org_dev), _dptr(self.dims64), C.c_double(self.cell),
             _ptr(self.sorted), _ptr(self.cell_start) if fits else None, _ptr(self.near_bits) if fits else None, _ptr(ws),
             ws_bytes, _stream())
        self.sorted = self.sorted[:self.n]
        return self

    def host(self):
        return self.cloud.cpu().numpy()


def read_clouds(*clouds):
    """One device -> host read of the (n, status, dims, org) of several AnchorClouds."""
    vals = _Readback.read(*[c.info for c in clouds])
    return [c.take_info(vals[8 * i:8 * i + 8]) for i, c in enumerate(clouds)]


def anchor_cloud(subv, used, cell):
    """One AnchorCloud with its grid: ``subv`` float64 [D, 3] and ``used`` uint8 [D] device tensors."""
    c, = read_clouds(AnchorCloud(subv.contiguous(), used.contiguous(), cell))
    return c.build_grid()


class DscMatch(object):
    """What ``match_dsc`` computes before the per-pair loop, and what every rank of ``parallel.match_dsc_sharded`` computes
    alike: the pair list above cc (hi, lo, score device tensors, ``p`` pairs), the hi anchor cloud and the lo anchor cloud
    with its grid (AnchorCloud)."""

    def __init__(self, lo, hi, anchor_dist_thresh=4, cc_threshold=0.65, impl=None, pairs=None):
        """pairs: the (hi, lo, score) list of ``match_threshold(hi.set, lo.set, cc_threshold)`` if already computed."""
        self.lo, self.hi = lo, hi
        self.dist = float(anchor_dist_thresh)
        dev = hi.set.dsc.device
        if pairs is None:
            pairs = match_threshold(hi.set, lo.set, cc_threshold, impl=impl)
        self.ph, self.pl, self.sc = pairs
        self.p = int(self.ph.numel())
        self.hi_cloud = self.lo_cloud = None
        if self.p == 0:
            return
        st = _stream()
        used_hi = torch.zeros(hi.set.rows, dtype=torch.uint8, device=dev)
        used_lo = torch.zeros(lo.set.rows, dtype=torch.uint8, device=dev)
        call("mad_mark_used", _ptr(self.ph), self.p, _ptr(used_hi), st)
        call("mad_mark_used", _ptr(self.pl), self.p, _ptr(used_lo), st)
        self.hi_cloud, self.lo_cloud = read_clouds(AnchorCloud(hi.subv, used_hi, self.dist),       # mad/MaD.py:427
                                                   AnchorCloud(lo.subv, used_lo, self.dist))       # mad/MaD.py:428
        self.lo_cloud.build_grid()
        self.tb = device_tables(dev)

    def _common(self):
        return (_ptr(self.hi.subv), _ptr(self.lo.subv), _ptr(self.hi.meta), _ptr(self.lo.meta), _ptr(self.tb.rf),
                _ptr(self.tb.rf_inv), self.tb.ori_zones)

    def _grid(self):
        g = self.lo_cloud
        return (_ptr(self.hi_cloud.cloud), self.hi_cloud.n, _ptr(g.sorted), _ptr(g.cell_start), _ptr(g.near_bits), _dptr(g.org),
                _dptr(g.dims), C.c_double(self.dist))

    def counts(self, p0, p1):
        """int32 [p1 - p0]: hits of the pairs [p0, p1) (mad_repeat_counts)."""
        out = torch.empty(max(p1 - p0, 1), dtype=torch.int32, device=self.ph.device)
        if p1 > p0:
            call("mad_repeat_counts", _ptr(self.ph), _ptr(self.pl), int(p0), int(p1), *self._common(), *self._grid(), _ptr(out),
                 _stream())
        return out[:p1 - p0]

    def rows(self, counts):
        """float64 [P, 23] result table from the hits of all P pairs (mad_repeat_rows)."""
        if counts.numel() != self.p or counts.dtype != torch.int32 or counts.device != self.ph.device:
            raise _lib.MadError("DscMatch.rows: needs int32 counts of all %d pairs on %s, got %s [%d] on %s"
                                % (self.p, self.ph.device, counts.dtype, counts.numel(), counts.device))
        res = torch.empty((self.p, 23), dtype=torch.float64, device=self.ph.device)
        call("mad_repeat_rows", _ptr(self.ph), _ptr(self.pl), _ptr(self.sc), self.p, *self._common(), _ptr(counts.contiguous()),
             self.hi_cloud.n, _ptr(res), _stream())
        return res

    def table(self):
        """float64 [P, 23] in one call (mad_repeatability: counts + rows without a counts buffer)."""
        res = torch.empty((self.p, 23), dtype=torch.float64, device=self.ph.device)
        call("mad_repeatability", _ptr(self.ph), _ptr(self.pl), _ptr(self.sc), self.p, *self._common(), *self._grid(), _ptr(res),
             _stream())
        return res

    def result(self, table):
        """(table, lo_mapcoords, hi_mapcoords as NumPy arrays): ``match_dsc``'s return value."""
        if self.p == 0:
            return table, np.zeros((0, 3)), np.zeros((0, 3))
        return table, self.lo_cloud.host(), self.hi_cloud.host()

    def empty(self):
        return torch.empty((0, 23), dtype=torch.float64, device=self.ph.device)


def match_dsc(lo, hi, anchor_dist_thresh=4, cc_threshold=0.65, impl=None):
    """``MaD._match_dsc`` (mad/MaD.py:414-453) on the device: cosine matching above ``cc_threshold`` and, per pair, the
    rigid transform R = inv(Rfinal_lo) . Rfinal_hi and the repeatability of the matched hi anchors under it.
    ``lo`` / ``hi``: FeatureTable.  Returns (results float64 [P, 23] device tensor in the reference's row layout,
    lo_mapcoords, hi_mapcoords as NumPy arrays).  The anchor clouds and the lo grid are built on the device (AnchorCloud);
    the host reads one small record between the matching and the per-pair loop.  The clouds equal np.unique's
    (np.array_equal) and are byte for byte the same except that a coordinate equal to zero is always +0.0, where np.unique
    may keep a -0.0 (it treats the two as equal; so does every later use of the clouds)."""
    m = DscMatch(lo, hi, anchor_dist_thresh, cc_threshold, impl)
    return m.result(m.table() if m.p else m.empty())


def match_dsc_lists(lo_dsc_list, hi_dsc_list, anchor_dist_thresh=4, cc_threshold=0.65):
    """Drop-in for ``MaD._match_dsc(lo_dsc_list, hi_dsc_list, anchor_dist_thresh, cc_threshold)``: same arguments
    (lists of DensityFeature), same return value (list of 23-vectors, lo cloud, hi cloud)."""
    res, lo_cloud, hi_cloud = match_dsc(FeatureTable.from_features(lo_dsc_list), FeatureTable.from_features(hi_dsc_list),
                                        anchor_dist_thresh, cc_threshold)
    return list(res.cpu().numpy()), lo_cloud, hi_cloud
