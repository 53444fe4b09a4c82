"""Host-side mirror of the reference interface (pixell.jl_b200/pixsht/geometry.py, enmap.py) against the reference's own
unit-test expectations (test/test_geometry.jl:5-45,236-269; test/test_transforms.jl:21), and the C-ABI surface: the shared
library loads without a GPU, exports every symbol include/*.h declares, and refuses to compute without a device.  CPU only."""
import ctypes
import math
import os
import re
import subprocess
import sys

import numpy as np
import pytest

import pixsht
from pixsht import (CarClenshawCurtis, fullsky_geometry, geometry, slice_geometry, pix2sky, degree, arcminute, sht_band,
                    fullringsize, fullringnum, getlmax, Enmap, Alm)
from pixsht import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def approx(a, b, tol=1e-12):
    return np.allclose(np.asarray(a, dtype=float), np.asarray(b, dtype=float), rtol=tol, atol=tol)


# ---- test/test_geometry.jl:5-45 ------------------------------------------------------------------------------------
def test_fullsky_geometry_reference_values():
    shape, wcs = fullsky_geometry(math.radians(1 / 60))
    assert shape == (21600, 10801)
    assert approx(wcs.cdelt, [-0.016666666666666666, 0.016666666666666666])
    assert approx(wcs.crpix, [10800.5, 5401.0])
    assert approx(wcs.crval, [0.008333333333333333, 0.0])
    shape, wcs = fullsky_geometry(math.radians(1 / 61))
    assert approx(wcs.cdelt, [-0.01639344262295082, 0.01639344262295082])
    assert approx(wcs.crpix, [10980.5, 5491.0])
    assert approx(wcs.crval, [0.00819672131147541, 0.0])
    shape, wcs = fullsky_geometry(math.radians(5), dims=(3,))
    assert shape == (72, 37, 3)


def test_box_geometry_reference_values():
    shape, wcs = geometry(CarClenshawCurtis, [[10 * degree, -10 * degree], [-5 * degree, 5 * degree]], 0.5 * arcminute)
    assert shape == (2400, 1200)
    assert approx(wcs.cdelt, [-0.008333333333333333, 0.008333333333333333])
    assert approx(wcs.crpix, [1201, 601]) and approx(wcs.crval, [0.0, 0.0])
    shape, wcs = geometry(CarClenshawCurtis, [[11 * degree, -10 * degree], [-6 * degree, 5 * degree]], 0.5 * arcminute)
    assert shape == (2520, 1320)
    assert approx(wcs.crpix, [1261, 721]) and approx(wcs.crval, [0.5, 0.0])
    shape, wcs = geometry(CarClenshawCurtis, [[10 * degree, -4 * degree], [-3 * degree, 5 * degree]], 0.5 * arcminute)
    assert shape == (1680, 960)
    assert approx(wcs.crpix, [841, 361]) and approx(wcs.crval, [3.0, 0.0])


# ---- test/test_geometry.jl:236-269 (1-based Julia ranges a:s:b -> Python slices) ---------------------------------------
def jl(a, s, b):
    """Julia range a:s:b (1-based, inclusive) as a Python slice."""
    if s > 0:
        return slice(a - 1, b, s)
    return slice(a - 1, b - 2 if b >= 2 else None, s)


@pytest.mark.parametrize("sx,sy,eshape,ecdelt,ecrpix", [
    (jl(1, 1, 3), jl(11, -1, 3), (3, 9), [-1.0, -1.0], [180.5, -79.0]),
    (jl(2, 1, 360), jl(6, 1, 11), (359, 6), [-1.0, 1.0], [179.5, 86.0]),
    (jl(2, 2, 359), jl(1, 1, 11), (179, 11), [-2.0, 1.0], [90.0, 91.0]),
    (jl(23, -4, 6), jl(1, 3, 28), (5, 10), [4.0, 3.0], [-38.75, 30.666666666666668]),
    (jl(3, 1, 3), jl(1, 3, 28), (1, 10), [-1.0, 3.0], [178.5, 30.666666666666668]),
])
def test_slice_geometry_reference_values(sx, sy, eshape, ecdelt, ecrpix):
    shape0, wcs0 = fullsky_geometry(math.radians(1))
    shape, wcs = slice_geometry(shape0, wcs0, sx, sy)
    assert tuple(shape) == eshape
    assert approx(wcs.cdelt, ecdelt) and approx(wcs.crpix, ecrpix) and approx(wcs.crval, [0.5, 0.0])


def test_pix2sky_reference_values():
    """test/test_geometry.jl:52-54 (angles wrapped to [0, 2pi) x [0, pi) there)."""
    shape, wcs = fullsky_geometry(math.radians(1))
    for pix, want in (((2.0, 2.0), (3.12413936, -1.55334303)), ((11.0, -12.0), (2.96705973, -1.79768913))):
        a, d = pix2sky(shape, wcs, *pix)
        assert abs(a - want[0]) < 1e-7 and abs(d - want[1]) < 1e-7


# ---- ring bookkeeping of src/transforms.jl:3-30,85 -----------------------------------------------------------------------
def test_ring_bookkeeping_and_bands():
    shape, wcs = fullsky_geometry(10.0 * degree)
    assert fullringsize(wcs) == 36 and fullringnum(wcs) == 19 and getlmax(wcs) == 18
    assert (getlmax(wcs) + 1) * (getlmax(wcs) + 2) // 2 == 190          # test/test_transforms.jl:21
    b = sht_band(shape, wcs)
    assert (b.nphi, b.nrings_total, b.ring_first, b.nrings, b.nx) == (36, 19, 0, 19, 36)
    assert b.flipx and b.flipy                                             # cdelt = (-10, +10): both axes are flipped for libsharp
    m = Enmap(np.zeros(shape, order="F"), wcs)
    sub = m[5:-2, 4:-3]                                                    # test/test_transforms.jl:23 m[6:end-2, 5:end-3]
    bs = sht_band(sub.shape, sub.wcs)
    assert (bs.nx, bs.nrings, bs.nrings_total, bs.nphi) == (29, 12, 19, 36)
    assert bs.ring_first == 3                                              # rows 5..16 of 19, counted from the north after the y flip
    bshape, bwcs = geometry(CarClenshawCurtis, [[10 * degree, -10 * degree], [-5 * degree, 5 * degree]], 1.0 * degree)
    bb = sht_band(bshape, bwcs)
    assert bshape == (20, 10) and (bb.nphi, bb.nrings_total, bb.nx, bb.nrings) == (360, 181, 20, 10)


def test_alm_container_layout():
    a = Alm(4, 4)
    assert a.alm.shape == (15,) and a.alm.dtype == np.complex128
    a2 = Alm(5, 3, np.arange(18, dtype=np.complex128))
    assert a2.lmax == 5 and a2.mmax == 3
    cl = pixsht.alm2cl(Alm(2, 2, np.array([1, 2, 3, 1j, 1 + 1j, 2], dtype=np.complex128)))
    assert approx(cl, [1.0, (4 + 2 * 1) / 3, (9 + 2 * 2 + 2 * 4) / 5])


# ---- C ABI surface -------------------------------------------------------------------------------------------------------
def declared_symbols():
    names = set()
    for h in ("pixsht.h", "pixsht_sharp_shim.h"):
        text = open(os.path.join(ROOT, "include", h)).read()
        text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
        names.update(re.findall(r"\b((?:pixsht|sharp)_[a-z0-9_]+)\s*\(", text))
    return names


def test_library_exports_every_declared_symbol():
    assert os.path.exists(_lib.DEFAULT_LIB), "run `python -c 'import __graft_entry__ as g; g.build()'` first"
    lib = ctypes.CDLL(_lib.DEFAULT_LIB)
    decl = declared_symbols()
    assert len(decl) >= 30
    missing = [s for s in sorted(decl) if not hasattr(lib, s)]
    assert not missing, "libpixsht.so lacks %s" % missing
    assert set(_lib.EXPORTS) == decl                  # the ctypes binding knows exactly the declared surface


_NO_DEVICE_CHECK = """
import pixsht
from pixsht import _lib, fullsky_geometry, sht_band, degree
lib = _lib.PixshtLib(_lib.DEFAULT_LIB)
assert lib.device_count() == 0
shape, wcs = fullsky_geometry(10.0 * degree)
try:
    pixsht.Plan(sht_band(shape, wcs), 18)
except _lib.PixshtError as e:
    assert e.code == _lib.ERR_NODEVICE and "no CPU fallback" in str(e), e
else:
    raise AssertionError("a plan was created without a CUDA device")
"""


def test_library_refuses_to_compute_without_a_device():
    lib = _lib.PixshtLib(_lib.DEFAULT_LIB)
    assert "sm_100a" in lib.version() and "EMULATION" not in lib.version()
    assert int(lib.lib.pixsht_nalm(10800, 10800)) == 58336201
    # in a child process that sees no device, also on a machine that has one
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="", PYTHONPATH=os.pathsep.join([os.path.join(ROOT, "pixell.jl_b200"), ROOT]))
    r = subprocess.run([sys.executable, "-c", _NO_DEVICE_CHECK], env=env, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr


def test_fejer1_geometry_extension():
    """CarFejer1 full-sky grid (extension; the reference has the type but no constructor / SHT path, SURVEY.md F8)."""
    from pixsht import CarFejer1
    shape, wcs = fullsky_geometry(math.radians(1.0), W=CarFejer1)
    assert shape == (360, 180) and isinstance(wcs, CarFejer1)
    assert fullringnum(wcs) == 180 and fullringsize(wcs) == 360
    # ring centres at (k + 1/2) degrees of colatitude, none on the poles
    assert abs(pix2sky(shape, wcs, 1, 1)[1] - math.radians(-89.5)) < 1e-12
    assert abs(pix2sky(shape, wcs, 1, 180)[1] - math.radians(89.5)) < 1e-12
    b = sht_band(shape, wcs)
    assert (b.nrings_total, b.ring_first, b.nrings, b.ring_scheme) == (180, 0, 180, 1)
    sub_shape, sub_wcs = slice_geometry(shape, wcs, slice(0, 360), slice(10, 50))
    bs = sht_band(sub_shape, sub_wcs)
    assert (bs.ring_first, bs.nrings, bs.ring_scheme) == (130, 40, 1)      # rows 10..49 from the south = rings 130..169 from the north
