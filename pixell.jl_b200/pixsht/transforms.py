"""map2alm / alm2map with the reference's method table (src/transforms.jl:88-265), on top of the C ABI.

The reference's per-call host work (create_sht_band copies, make_cc_geom_info, the un-flip slice copy) is replaced by
a cached Plan per (geometry, lmax, mmax, dtype): the caller's array goes to the library untouched, flips and padding
are index arithmetic in the FFT kernels.
"""
import ctypes

import numpy as np

from . import _lib
from ._lib import PixshtError, PixshtLib, get_lib, Geom, F64, F32, MAP2ALM, ALM2MAP, HOST, DEVICE  # noqa: F401
from .enmap import Enmap, Alm
from .geometry import sht_band, getlmax


def _ptr_array(ptrs):
    return (ctypes.c_void_p * len(ptrs))(*ptrs)


class Plan:
    """Owner of a pixsht_plan handle (include/pixsht.h)."""

    def __init__(self, band, lmax, mmax=None, dtype=np.float64, device=0, lib=None, devices=None):
        """devices: list of GPU indices -> a multi-GPU plan (pixsht_plan_create_multi: one process drives them all behind the
        same execute call); None -> a single-GPU plan on `device`."""
        self.lib = get_lib() if lib is None else lib
        self.band, self.lmax, self.mmax = band, int(lmax), int(lmax if mmax is None else mmax)
        self.dtype = np.dtype(dtype)
        if self.dtype not in (np.dtype(np.float64), np.dtype(np.float32)):
            raise TypeError("maps must be Float64 or Float32")
        self.cdtype = np.dtype(np.complex128 if self.dtype == np.float64 else np.complex64)
        g = Geom(band.nphi, band.nrings_total, band.ring_first, band.nrings, band.nx, int(band.flipx), int(band.flipy), int(getattr(band, "ring_scheme", 0)),
                 band.phi0)
        h = ctypes.c_void_p()
        dt = F64 if self.dtype == np.float64 else F32
        self.devices = None if devices is None else [int(d) for d in devices]
        if self.devices is None:
            self.lib.check(self.lib.lib.pixsht_plan_create(ctypes.byref(h), ctypes.byref(g), self.lmax, self.mmax, dt, device))
        else:
            arr = (ctypes.c_int * len(self.devices))(*self.devices)
            self.lib.check(self.lib.lib.pixsht_plan_create_multi(ctypes.byref(h), ctypes.byref(g), self.lmax, self.mmax, dt, len(self.devices), arr))
        self.handle = h
        self.nalm = int(self.lib.lib.pixsht_nalm(self.lmax, self.mmax))

    def close(self):
        if getattr(self, "handle", None):
            self.lib.lib.pixsht_plan_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def execute_ptrs(self, direction, alm_ptrs, map_ptrs, location=HOST):
        n = len(alm_ptrs)
        self.lib.check(self.lib.lib.pixsht_execute(self.handle, direction, n, _ptr_array(alm_ptrs), _ptr_array(map_ptrs),
                                                   location))

    def map2alm_iter_ptrs(self, alm_ptrs, map_ptrs, niter, location=HOST):
        """map2alm refined by `niter` Jacobi iterations (pixsht_map2alm_iter); niter = 0 is execute_ptrs(MAP2ALM, ...)."""
        self.lib.check(self.lib.lib.pixsht_map2alm_iter(self.handle, len(alm_ptrs), _ptr_array(alm_ptrs), _ptr_array(map_ptrs),
                                                        int(niter), location))

    def execute_batch_ptrs(self, direction, alm_ptrs, map_ptrs, location=HOST):
        self.lib.check(self.lib.lib.pixsht_execute_batch(self.handle, direction, len(alm_ptrs), _ptr_array(alm_ptrs), _ptr_array(map_ptrs),
                                                         location))

    def alm2map_batch(self, alms):
        """Independent spin-0 syntheses of a list of alm vectors on this plan's geometry (pixsht_execute_batch)."""
        alms = [np.ascontiguousarray(a, dtype=self.cdtype) for a in alms]
        for a in alms:
            if a.shape != (self.nalm,):
                raise ValueError("alm has %d entries, expected %d" % (a.size, self.nalm))
        maps = [np.zeros((self.band.nx, self.band.nrings), dtype=self.dtype, order="F") for _ in alms]
        self.execute_batch_ptrs(ALM2MAP, [a.ctypes.data for a in alms], [m.ctypes.data for m in maps])
        return maps

    def map2alm_batch(self, maps):
        maps = [self._as_map(m) for m in maps]
        alms = [np.zeros(self.nalm, dtype=self.cdtype) for _ in maps]
        self.execute_batch_ptrs(MAP2ALM, [a.ctypes.data for a in alms], [m.ctypes.data for m in maps])
        return alms

    def shards(self):
        """Multi-GPU plan: [(device, first band ring, ring count, m values)] per shard."""
        out = []
        for d in range(len(self.devices or [])):
            info = (ctypes.c_int32 * 4)()
            self.lib.check(self.lib.lib.pixsht_multi_shard(self.handle, d, info, None))
            ml = (ctypes.c_int32 * max(1, info[3]))()
            self.lib.check(self.lib.lib.pixsht_multi_shard(self.handle, d, info, ml))
            out.append((int(info[0]), int(info[1]), int(info[2]), np.array(ml[:info[3]], dtype=np.int32)))
        return out

    def execute_sharded_ptrs(self, direction, ncomp, alm_ptrs, map_ptrs):
        """alm_ptrs / map_ptrs: flat lists [shard][component] of device pointers (pixsht_execute_sharded)."""
        self.lib.check(self.lib.lib.pixsht_execute_sharded(self.handle, direction, ncomp, _ptr_array(alm_ptrs), _ptr_array(map_ptrs)))

    def set_polconv(self, polcconv):
        """Stokes-U sign convention of the maps handed to this plan: "COSMO" (default; the convention the transforms compute in)
        or "IAU" (U negated inside the ring-FFT kernels' row I/O, both directions): pixsht_plan_set_polconv."""
        if polcconv not in ("COSMO", "IAU"):
            raise ValueError("polcconv must be 'COSMO' or 'IAU'")
        self.lib.check(self.lib.lib.pixsht_plan_set_polconv(self.handle, 1 if polcconv == "IAU" else 0))

    def timings(self):
        t = (ctypes.c_double * 8)()
        self.lib.check(self.lib.lib.pixsht_get_timings(self.handle, t))
        return dict(h2d=t[0], legendre=t[1], fft=t[2], d2h=t[3], total=t[4], compute_span=t[5], leg_spin0=t[6], leg_spin2=t[7])

    def work(self, spin):
        """(executed, nominal) (l, m, ring pair) steps of one spin family."""
        w = (ctypes.c_double * 2)()
        self.lib.check(self.lib.lib.pixsht_plan_work(self.handle, spin, w))
        return w[0], w[1]

    def info(self):
        v = (ctypes.c_int32 * 16)()
        self.lib.check(self.lib.lib.pixsht_plan_info(self.handle, v))
        keys = ["nphi", "nrings", "lmax", "mmax", "dtype", "device", "npairs", "sm_count", "nfft", "launches", "R0", "R2", "R0a", "R2a", "ndev"]
        d = dict(zip(keys, list(v)))
        d["fft"] = dict(threads=v[15] & 0xffff, edge_fused=bool(v[15] >> 16 & 1), global_buffers=bool(v[15] >> 17 & 1), super_passes=v[15] >> 20)
        return d

    def weights(self):
        w = np.empty(self.band.nrings)
        th = np.empty(self.band.nrings)
        self.lib.check(self.lib.lib.pixsht_plan_weights(self.handle, w.ctypes.data_as(ctypes.POINTER(ctypes.c_double)),
                                                        th.ctypes.data_as(ctypes.POINTER(ctypes.c_double))))
        return w, th

    # ---- host-array front ends -------------------------------------------------------------------------------
    def map2alm(self, maps, niter=0):
        """maps: list of (nx, ny) Fortran-ordered arrays of the plan dtype (1: T, 2: Q,U, 3: T,Q,U) -> list of alm vectors.
        niter > 0: the analysis refined by niter Jacobi iterations a <- a + A (m - Y a) on the device (pixsht_map2alm_iter)."""
        maps = [self._as_map(m) for m in maps]
        alms = [np.zeros(self.nalm, dtype=self.cdtype) for _ in maps]
        if niter == 0:
            self.execute_ptrs(MAP2ALM, [a.ctypes.data for a in alms], [m.ctypes.data for m in maps])
        else:
            self.map2alm_iter_ptrs([a.ctypes.data for a in alms], [m.ctypes.data for m in maps], niter)
        return alms

    def alm2map(self, alms):
        alms = [np.ascontiguousarray(a, dtype=self.cdtype) for a in alms]
        for a in alms:
            if a.shape != (self.nalm,):
                raise ValueError("alm has %d entries, expected %d" % (a.size, self.nalm))
        maps = [np.zeros((self.band.nx, self.band.nrings), dtype=self.dtype, order="F") for _ in alms]
        self.execute_ptrs(ALM2MAP, [a.ctypes.data for a in alms], [m.ctypes.data for m in maps])
        return maps

    def _as_map(self, m):
        m = np.asarray(m)
        if m.shape != (self.band.nx, self.band.nrings):
            raise ValueError("map has shape %s, expected %s" % (m.shape, (self.band.nx, self.band.nrings)))
        if m.dtype != self.dtype or not m.flags.f_contiguous:
            m = np.asfortranarray(m, dtype=self.dtype)
        return m


_PLANS = {}


def _env_devices():
    """PIXSHT_DEVICES="0,1,2,3" -> [0, 1, 2, 3]; unset or a single index -> None (single-GPU plan on that index is the default 0)."""
    import os
    v = os.environ.get("PIXSHT_DEVICES", "").strip()
    if not v:
        return None
    d = [int(x) for x in v.split(",") if x.strip() != ""]
    return d if len(d) > 1 else None


def _plan_for(shape, wcs, lmax, mmax, dtype, lib=None, devices=None):
    band = sht_band(tuple(shape[:2]), wcs)
    lib = get_lib() if lib is None else lib
    devices = _env_devices() if devices is None else list(devices)
    key = (id(lib), band, lmax, mmax, np.dtype(dtype).str, None if devices is None else tuple(devices))
    p = _PLANS.get(key)
    if p is None:
        if len(_PLANS) >= 8:
            _PLANS.pop(next(iter(_PLANS))).close()
        p = _PLANS[key] = Plan(band, lmax, mmax, dtype=dtype, lib=lib, devices=devices)
    return p


def _compute_dtype(dt, precision=None):
    """Element type of the plan for a map of dtype `dt`.  Default: Float64 whatever the map's type -- the reference promotes every
    map to Float64 before the transform (create_sht_band, src/transforms.jl:71) and so do we (the map is widened on the host,
    like the reference's band copy).  precision="f32" is the explicit opt-in to the Float32-boundary plan for Float32 maps
    (half the PCIe volume, ring FFTs in Float32: rel-RMS ~1e-7 of each ring's dominant mode -- NOT the reference's numerics)."""
    if precision not in (None, "f64", "f32"):
        raise ValueError("precision must be None, 'f64' or 'f32'")
    if precision == "f32" and np.dtype(dt) == np.float32:
        return np.float32
    return np.float64


def pixareamap(shape_or_map, wcs=None, lib=None):
    """pixareamap(shape, wcs) / pixareamap(m::Enmap): an Enmap whose pixel values are the pixel areas in steradians
    (src/projections/car_proj.jl:265-273, src/enmap_ops.jl:124-138).  The per-row areas come from pixsht_ring_pixarea."""
    if isinstance(shape_or_map, Enmap):
        shape, wcs, dtype = shape_or_map.shape, shape_or_map.wcs, shape_or_map.dtype
    else:
        shape, dtype = tuple(shape_or_map), np.float64
    out = Enmap(np.empty(tuple(shape[:2]), dtype=dtype, order="F"), wcs)
    return pixareamap_(out, lib=lib)


def ring_pixarea(shape, wcs, lib=None):
    """Pixel area of each map row (ny values, the map's row order)."""
    lib = get_lib() if lib is None else lib
    band = sht_band(tuple(shape[:2]), wcs)
    g = Geom(band.nphi, band.nrings_total, band.ring_first, band.nrings, band.nx, int(band.flipx), int(band.flipy), int(getattr(band, "ring_scheme", 0)),
             band.phi0)
    area = np.empty(band.nrings)
    lib.check(lib.lib.pixsht_ring_pixarea(ctypes.byref(g), area.ctypes.data_as(ctypes.POINTER(ctypes.c_double))))
    return area


def pixareamap_(pixareas, lib=None):
    """pixareamap!(pixareas::Enmap): in-place (src/enmap_ops.jl:124-138)."""
    area = ring_pixarea(pixareas.shape, pixareas.wcs, lib=lib)
    pixareas.data[...] = area.reshape((1, -1) + (1,) * (pixareas.data.ndim - 2))
    return pixareas


def map2alm(m, lmax=None, mmax=None, lib=None, precision=None, devices=None, polcconv=None, niter=0):
    """map2alm(::Enmap{T,2}) / (::NTuple{2}) / (::NTuple{3}) / (::Enmap{T,3})  (src/transforms.jl:88-165).

    Returns an Alm (spin 0), or a tuple (E, B) / (T, E, B) of Alm -- the reference's return types; the alm are complex128
    whatever the map's element type, as the reference's (ComplexF64).  precision: see _compute_dtype.  devices: list of GPUs
    for a multi-GPU plan (default: the PIXSHT_DEVICES environment variable, else one GPU).  polcconv: "COSMO" | "IAU", the sign
    convention of the U map (default: the Enmap's tag from read_map(..., defer_polcconv=True), else COSMO).  niter: Jacobi
    iterations a <- a + map2alm(m - alm2map(a)) after the plain analysis, as python-pixell's map2alm(niter=...) (single-GPU
    plans only; they help where lmax exceeds (nrings - 1)/2 of the full-sky grid, DESIGN.md section 10)."""
    if isinstance(m, (tuple, list)):
        maps = list(m)
        if len(maps) not in (2, 3) or any(x.ndim != 2 for x in maps):
            raise ValueError("tuples of 2 (Q,U) or 3 (I,Q,U) two-dimensional Enmaps are supported")
        first = maps[0]
        arrays = [x.data for x in maps]
    else:
        first = m
        if m.ndim == 2:
            arrays = [m.data]
        else:
            if m.shape[2] not in (1, 2, 3):
                raise ValueError("SHTs require shape (nx,ny,ncomp) with 1 ≤ ncomp ≤ 3, for I, QU, and IQU.")
            arrays = [m.data[:, :, c] for c in range(m.shape[2])]
    if lmax is None:
        lmax = getlmax(first.wcs)
        mmax = lmax
    mmax = lmax if mmax is None else mmax
    plan = _plan_for(first.shape, first.wcs, lmax, mmax, _compute_dtype(first.dtype, precision), lib, devices)
    # U sign convention of the input: an explicit keyword, else the tag read_map(..., defer_polcconv=True) left on the Enmap
    plan.set_polconv(polcconv if polcconv is not None else getattr(first if not isinstance(m, (tuple, list)) else maps[-1], "polcconv", "COSMO"))
    alms = [Alm(lmax, mmax, np.asarray(a, dtype=np.complex128)) for a in plan.map2alm(arrays, niter=niter)]
    return alms[0] if len(alms) == 1 else tuple(alms)


def alm2map(alm, shape, wcs, dtype=np.float64, lib=None, devices=None, polcconv="COSMO"):
    """alm2map(::Alm, shape, wcs) -> Enmap;  (::NTuple{2,Alm}) -> list of 2 Enmaps;  (::NTuple{3,Alm}) / Vector -> tuple
    (src/transforms.jl:206-265, return-type quirks of SURVEY.md F11 kept)."""
    alms = [alm] if isinstance(alm, Alm) else list(alm)
    if len(alms) not in (1, 2, 3):
        raise ValueError("1, 2 or 3 Alm are supported")
    lmax, mmax = alms[0].lmax, alms[0].mmax
    plan = _plan_for(shape, wcs, lmax, mmax, dtype, lib, devices)
    plan.set_polconv(polcconv)   # "IAU": the U map comes out with the IAU sign (tagged on the Enmap for write_map)
    maps = [Enmap(x, wcs) for x in plan.alm2map([a.alm for a in alms])]
    for x in maps:
        x.polcconv = polcconv
    if len(maps) == 1:
        return maps[0]
    if len(maps) == 2:
        return maps
    return tuple(maps)
