"""ctypes front-end of oracle/sht_oracle.c (TEST INFRASTRUCTURE ONLY, see the C file's header).

Two builds of the same source: "ld" (80-bit long double, the parity checker) and "d" (double + OpenMP, the timed CPU
baseline "port").  Geometry helpers restate src/transforms.jl:33-63 of the reference (ring grid, CC weights x 2pi/nphi).
"""
import atexit
import ctypes
import os
import shutil
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_BUILD = os.path.join(_HERE, "_build")


def build(force=False):
    """(Re)build the oracle shared objects with gcc; no-op when up to date.  When oracle/_build cannot be written (a
    read-only tree), a stale or missing build goes to a fresh temporary directory instead."""
    global _BUILD
    srcs = [os.path.join(_HERE, "sht_oracle.c"), os.path.join(_HERE, "sht_cpu.c")]
    names = ["liborc_ld.so", "liborc_d.so", "libshtcpu.so"]
    libs = [os.path.join(_BUILD, n) for n in names]
    fresh = all(os.path.exists(p) and os.path.getmtime(p) >= max(os.path.getmtime(s) for s in srcs) for p in libs)
    # libshtcpu.so is compiled with -march=native: rebuild it when the snapshot travelled to a machine with another CPU
    tag, tag_file = _cpu_tag(), os.path.join(_BUILD, "libshtcpu.host")
    try:
        same_host = open(tag_file).read() == tag
    except OSError:
        same_host = False
    if (force or not fresh or not same_host) and not os.access(_BUILD if os.path.isdir(_BUILD) else _HERE, os.W_OK):
        _BUILD = tempfile.mkdtemp(prefix="pixsht_oracle_")
        atexit.register(shutil.rmtree, _BUILD, True)
        libs = [os.path.join(_BUILD, n) for n in names]
        tag_file = os.path.join(_BUILD, "libshtcpu.host")
        fresh = False
    if not same_host and os.path.exists(libs[2]):
        os.remove(libs[2])
        fresh = False
    if force or not fresh:
        subprocess.check_call(["make", "-C", _HERE, "-s", "OUT=" + _BUILD] + (["-B"] if force else []))
    if not same_host:
        with open(tag_file, "w") as f:
            f.write(tag)
    return libs


def _cpu_tag():
    try:
        with open("/proc/cpuinfo") as f:
            for line in f:
                if line.startswith("flags"):
                    import hashlib
                    return hashlib.sha1(line.encode()).hexdigest()
    except OSError:
        pass
    return "unknown"


def alm_index(lmax, l, m):
    """0-based index of a_lm in the triangular m-major layout (Healpix.Alm / make_triangular_alm_info(lmax,mmax,1))."""
    return m * (2 * lmax + 1 - m) // 2 + l


def nalm(lmax, mmax=None):
    mmax = lmax if mmax is None else mmax
    return (mmax + 1) * (lmax + 1) - mmax * (mmax + 1) // 2


class Oracle:
    def __init__(self, kind="ld"):
        build()
        self.kind = kind
        self.lib = ctypes.CDLL(os.path.join(_BUILD, "liborc_%s.so" % kind))
        L = self.lib
        dp = ctypes.POINTER(ctypes.c_double)
        pp = ctypes.POINTER(ctypes.c_void_p)
        L.orc_cc_weights.argtypes = [ctypes.c_int, dp]
        L.orc_cc_weights.restype = None
        L.orc_lambda_d.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_double, dp]
        L.orc_lambda_d.restype = None
        L.orc_map2alm.argtypes = [ctypes.c_int, ctypes.c_int, dp, dp, ctypes.c_double, ctypes.c_int, ctypes.c_int,
                                  ctypes.c_int, pp, pp, ctypes.c_int, ctypes.c_int]
        L.orc_map2alm.restype = ctypes.c_int
        L.orc_alm2map.argtypes = [ctypes.c_int, ctypes.c_int, dp, ctypes.c_double, ctypes.c_int, ctypes.c_int,
                                  ctypes.c_int, pp, pp, ctypes.c_int, ctypes.c_int]
        L.orc_alm2map.restype = ctypes.c_int
        L.orc_real_bits.restype = ctypes.c_int
        L.orc_num_threads.restype = ctypes.c_int

    @property
    def threads(self):
        return int(self.lib.orc_num_threads())

    @staticmethod
    def _dp(a):
        return a.ctypes.data_as(ctypes.POINTER(ctypes.c_double))

    @staticmethod
    def _ptrs(arrs):
        return (ctypes.c_void_p * len(arrs))(*[a.ctypes.data for a in arrs])

    def cc_weights(self, n):
        w = np.empty(n, dtype=np.float64)
        self.lib.orc_cc_weights(n, self._dp(w))
        return w

    def lam(self, lmax, m, s, theta):
        out = np.zeros(lmax + 1, dtype=np.float64)
        self.lib.orc_lambda_d(lmax, m, s, float(theta), self._dp(out))
        return out

    def map2alm(self, maps, theta, wgt, phi0, lmax, mmax=None, spin=0, m_stride=1, m_offset=0):
        """maps: (ncomp, nrings, nphi) float64, rings ascending theta, phi ascending from phi0.
        Returns (ncomp, nalm) complex128 (spin 0: T; spin 2: E, B)."""
        mmax = lmax if mmax is None else mmax
        maps = np.ascontiguousarray(maps, dtype=np.float64)
        if maps.ndim == 2:
            maps = maps[None]
        nc, nr, nphi = maps.shape
        assert nc == (1 if spin == 0 else 2)
        theta = np.ascontiguousarray(theta, dtype=np.float64)
        wgt = np.ascontiguousarray(wgt, dtype=np.float64)
        alms = [np.zeros(nalm(lmax, mmax), dtype=np.complex128) for _ in range(nc)]
        mp = [maps[c] for c in range(nc)]
        rc = self.lib.orc_map2alm(spin, nr, self._dp(theta), self._dp(wgt), float(phi0), nphi, lmax, mmax,
                                  self._ptrs(mp), self._ptrs(alms), m_stride, m_offset)
        if rc != 0:
            raise ValueError("orc_map2alm: bad arguments")
        return np.stack(alms)

    def alm2map(self, alms, theta, phi0, nphi, lmax, mmax=None, spin=0, ring_stride=1, ring_offset=0):
        """alms: (ncomp, nalm) complex128.  Returns (ncomp, nrings, nphi) float64 (unselected rings are zero)."""
        mmax = lmax if mmax is None else mmax
        alms = np.ascontiguousarray(alms, dtype=np.complex128)
        if alms.ndim == 1:
            alms = alms[None]
        nc = alms.shape[0]
        assert nc == (1 if spin == 0 else 2) and alms.shape[1] == nalm(lmax, mmax)
        theta = np.ascontiguousarray(theta, dtype=np.float64)
        nr = theta.shape[0]
        maps = [np.zeros((nr, nphi), dtype=np.float64) for _ in range(nc)]
        al = [alms[c] for c in range(nc)]
        rc = self.lib.orc_alm2map(spin, nr, self._dp(theta), float(phi0), nphi, lmax, mmax,
                                  self._ptrs(al), self._ptrs(maps), ring_stride, ring_offset)
        if rc != 0:
            raise ValueError("orc_alm2map: bad arguments")
        return np.stack(maps)


class CpuSht:
    """ctypes front-end of oracle/sht_cpu.c: the libsharp2-style CPU implementation (double, OpenMP, SIMD over rings) that
    bench.py times as the CPU baseline.  Same conventions as Oracle; sampling is by m in both directions."""

    def __init__(self):
        build()
        self.lib = ctypes.CDLL(os.path.join(_BUILD, "libshtcpu.so"))
        L = self.lib
        dp = ctypes.POINTER(ctypes.c_double)
        pp = ctypes.POINTER(ctypes.c_void_p)
        L.cpu_alm2map.argtypes = [ctypes.c_int, ctypes.c_int, dp, ctypes.c_double, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                  pp, pp, ctypes.c_int, ctypes.c_int, dp]
        L.cpu_map2alm.argtypes = [ctypes.c_int, ctypes.c_int, dp, dp, ctypes.c_double, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                  pp, pp, ctypes.c_int, ctypes.c_int, dp]
        L.cpu_num_threads.restype = ctypes.c_int
        L.cpu_fma_peak_gflops.argtypes = [ctypes.c_int, ctypes.c_double]
        L.cpu_fma_peak_gflops.restype = ctypes.c_double
        L.cpu_set_threads.argtypes = [ctypes.c_int]
        L.cpu_set_threads.restype = None
        self.last_times = (0.0, 0.0)

    def use_all_cores(self):
        """All host cores, whatever OMP_NUM_THREADS says (torchrun sets it to 1 for its workers)."""
        try:
            n = len(os.sched_getaffinity(0))
        except AttributeError:
            n = os.cpu_count() or 1
        self.lib.cpu_set_threads(n)
        return n

    @property
    def threads(self):
        return int(self.lib.cpu_num_threads())

    def fma_peak_gflops(self, seconds=0.5):
        """Measured FP64 FMA peak of the host on the threads the port uses (GFLOP/s, 1 FMA = 2 flop)."""
        return float(self.lib.cpu_fma_peak_gflops(self.threads, float(seconds)))

    def alm2map(self, alms, theta, phi0, nphi, lmax, mmax=None, spin=0, m_stride=1, m_offset=0):
        mmax = lmax if mmax is None else mmax
        alms = np.ascontiguousarray(alms, dtype=np.complex128)
        if alms.ndim == 1:
            alms = alms[None]
        nc = alms.shape[0]
        assert nc == (1 if spin == 0 else 2) and alms.shape[1] == nalm(lmax, mmax)
        theta = np.ascontiguousarray(theta, dtype=np.float64)
        maps = [np.zeros((theta.shape[0], nphi), dtype=np.float64) for _ in range(nc)]
        al = [alms[c] for c in range(nc)]
        t = (ctypes.c_double * 2)()
        rc = self.lib.cpu_alm2map(spin, theta.shape[0], Oracle._dp(theta), float(phi0), nphi, lmax, mmax, Oracle._ptrs(al),
                                  Oracle._ptrs(maps), m_stride, m_offset, t)
        if rc != 0:
            raise ValueError("cpu_alm2map: bad arguments")
        self.last_times = (t[0], t[1])
        return np.stack(maps)

    def map2alm(self, maps, theta, wgt, phi0, lmax, mmax=None, spin=0, m_stride=1, m_offset=0):
        mmax = lmax if mmax is None else mmax
        maps = np.ascontiguousarray(maps, dtype=np.float64)
        if maps.ndim == 2:
            maps = maps[None]
        nc, nr, nphi = maps.shape
        assert nc == (1 if spin == 0 else 2)
        theta = np.ascontiguousarray(theta, dtype=np.float64)
        wgt = np.ascontiguousarray(wgt, dtype=np.float64)
        alms = [np.zeros(nalm(lmax, mmax), dtype=np.complex128) for _ in range(nc)]
        mp = [maps[c] for c in range(nc)]
        t = (ctypes.c_double * 2)()
        rc = self.lib.cpu_map2alm(spin, nr, Oracle._dp(theta), Oracle._dp(wgt), float(phi0), nphi, lmax, mmax, Oracle._ptrs(mp),
                                  Oracle._ptrs(alms), m_stride, m_offset, t)
        if rc != 0:
            raise ValueError("cpu_map2alm: bad arguments")
        self.last_times = (t[0], t[1])
        return np.stack(alms)


_CPU = []


def get_cpu_sht():
    if not _CPU:
        _CPU.append(CpuSht())
    return _CPU[0]


_ORACLES = {}


def get_oracle(kind="ld"):
    if kind not in _ORACLES:
        _ORACLES[kind] = Oracle(kind)
    return _ORACLES[kind]


def cc_weights(n):
    return get_oracle("ld").cc_weights(n)


def cc_geometry(nrings_total, nphi, ring_first=0, nrings=None):
    """theta and weights of a (sub-)band of the full-sky Clenshaw-Curtis grid, as src/transforms.jl:44-46 builds them:
    theta_k = pi k/(N-1), w_k = CC_N[k] * 2pi/nphi, for k = ring_first .. ring_first+nrings-1 (0-based)."""
    nrings = nrings_total - ring_first if nrings is None else nrings
    k = np.arange(ring_first, ring_first + nrings)
    theta = np.linspace(0.0, np.pi, nrings_total)[k]
    w = cc_weights(nrings_total)[k] * (2.0 * np.pi / nphi)
    return theta, w
