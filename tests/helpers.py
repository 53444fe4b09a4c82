"""Shared test helpers: reference-style test inputs (test/test_transforms.jl:3-9,40-47) and the host-side band copy
that the reference performs before calling libsharp2 (create_sht_band, src/transforms.jl:66-77)."""
import os
import numpy as np

import pixsht
from oracle import cc_geometry, get_oracle, nalm

GOLDEN = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_alm_golden.npz"))


def golden_alm(name, cols=(0, 1)):
    d = GOLDEN[name]
    return d[:, cols[0]] + 1j * d[:, cols[1]]


def gen_spin0(shape, p=2):
    """m[i,j] = ((j-1)*nx + i)^p, 1-based (test/test_transforms.jl:3-9)."""
    nx, ny = shape[:2]
    i = np.arange(1, nx + 1, dtype=np.float64)[:, None]
    j = np.arange(1, ny + 1, dtype=np.float64)[None, :]
    return np.asfortranarray(((j - 1) * nx + i) ** p)


def gen_spin2(shape):
    """Q = i^2 j, U = i j, 1-based (test/test_transforms.jl:40-47). Returns (nx, ny, 2)."""
    nx, ny = shape[:2]
    i = np.arange(1, nx + 1, dtype=np.float64)[:, None]
    j = np.arange(1, ny + 1, dtype=np.float64)[None, :]
    out = np.zeros((nx, ny, 2), order="F")
    out[:, :, 0] = i ** 2 * j
    out[:, :, 1] = i * j
    return out


def band_copy(m):
    """create_sht_band(m::Enmap) restated: flipped, zero-padded float64 band, returned as (ncomp, nrings, nphi)
    C-ordered (ring-major, phi fastest) -- the flat layout handed to sharp_execute -- plus the ShtBand descriptor."""
    b = pixsht.sht_band(m.shape, m.wcs)
    data = m.data if m.data.ndim == 3 else m.data[:, :, None]
    fx = slice(None, None, -1) if b.flipx else slice(None)
    fy = slice(None, None, -1) if b.flipy else slice(None)
    band = np.zeros((b.nphi, b.nrings, data.shape[2]), dtype=np.float64)
    band[:b.nx] = data[fx, fy, :]
    return np.ascontiguousarray(band.transpose(2, 1, 0)), b


def band_to_map(band, b):
    """Inverse of band_copy for alm2map results: (ncomp, nrings, nphi) -> (nx, ny, ncomp).

    The reference's alm2map (src/transforms.jl:206-225) pads the UNflipped band, so its phi0 is the RA of the virtual
    column `fullringsize` and it reads the last nx band columns back in reverse; here the band follows the map2alm
    convention of ShtBand (phi0 = RA of the flipped map's first column, padding at the end), so map column c is band
    column nx-1-c.  Both address the same (theta, phi) per pixel; for full-sky maps they are the same indices."""
    a = band.transpose(2, 1, 0)  # (nphi, nrings, ncomp)
    xs = slice(b.nx - 1, None, -1) if b.flipx else slice(0, b.nx)
    ys = slice(None, None, -1) if b.flipy else slice(None)
    return np.asfortranarray(a[xs, ys, :])


def oracle_map2alm(m, lmax, mmax=None, spin=0, kind="ld", **kw):
    """Oracle analysis of an Enmap (2-D, or 3-D with the right ncomp for `spin`).  kind: "ld" / "d" = the naive checker in
    long double / double; "cpu" = the libsharp2-style CPU implementation (oracle/sht_cpu.c)."""
    band, b = band_copy(m)
    theta, w = cc_geometry(b.nrings_total, b.nphi, b.ring_first, b.nrings)
    if kind == "cpu":
        from oracle import get_cpu_sht
        return get_cpu_sht().map2alm(band, theta, w, b.phi0, lmax, mmax, spin=spin, **kw)
    return get_oracle(kind).map2alm(band, theta, w, b.phi0, lmax, mmax, spin=spin, **kw)


def oracle_alm2map(alms, shape, wcs, lmax, mmax=None, spin=0, kind="ld", **kw):
    b = pixsht.sht_band(shape, wcs)
    theta, _ = cc_geometry(b.nrings_total, b.nphi, b.ring_first, b.nrings)
    if kind == "cpu":
        from oracle import get_cpu_sht
        return band_to_map(get_cpu_sht().alm2map(alms, theta, b.phi0, b.nphi, lmax, mmax, spin=spin, **kw), b)
    band = get_oracle(kind).alm2map(alms, theta, b.phi0, b.nphi, lmax, mmax, spin=spin, **kw)
    return band_to_map(band, b)


def rel_rms(a, b):
    a = np.asarray(a)
    b = np.asarray(b)
    return float(np.sqrt(np.sum(np.abs(a - b) ** 2) / np.sum(np.abs(b) ** 2)))


def synth_alm(lmax, mmax, seed, spin2=False):
    """Synthetic Gaussian alm of SURVEY.md 8(d): iid N(0,1) re/im, imag(a_l0)=0, l<2 zeroed for E/B."""
    rng = np.random.default_rng(seed)
    n = nalm(lmax, mmax)
    a = rng.standard_normal(n) + 1j * rng.standard_normal(n)
    a[:lmax + 1] = a[:lmax + 1].real
    if spin2:
        for m in range(min(mmax, 1) + 1):
            i0 = m * (2 * lmax + 1 - m) // 2
            a[i0 + m:i0 + 2] = 0  # l = m .. 1
    return a


def fejer1_geometry(nrings_total, nphi, ring_first=0, nrings=None):
    """Colatitudes and ring weights (x 2pi/nphi) of the Fejer-1 grid theta_k = pi (k + 1/2)/N (test-side restatement, independent
    of the device kernel: the weights come from the moment equations sum_k f_k T_j(cos theta_k) = int T_j, solved through the
    orthogonality of the Chebyshev polynomials on these nodes)."""
    N = nrings_total
    k = np.arange(N)
    theta = np.pi * (k + 0.5) / N
    f = np.full(N, 2.0 / N)                                  # j = 0 term: int T_0 = 2
    for j in range(2, N, 2):                                 # int_{-1}^{1} T_j = 2/(1 - j^2) for even j, 0 for odd j
        f += (2.0 / N) * 2.0 / (1.0 - j * j) * np.cos(j * theta)
    w = f * 2.0 * np.pi / nphi
    nrings = N - ring_first if nrings is None else nrings
    return theta[ring_first:ring_first + nrings], w[ring_first:ring_first + nrings]


import contextlib


@contextlib.contextmanager
def plain_fft_kernels():
    """Plans created inside use the plain ring-FFT kernels (fft.cuh) instead of the edge-fused ones (fft_edge.cuh): the
    m-sharded multi-GPU plans run the plain kernels, so a bit-for-bit comparison needs the single-GPU reference on them too."""
    old = os.environ.get("PIXSHT_FFT_EDGE")
    os.environ["PIXSHT_FFT_EDGE"] = "0"
    try:
        yield
    finally:
        if old is None:
            os.environ.pop("PIXSHT_FFT_EDGE", None)
        else:
            os.environ["PIXSHT_FFT_EDGE"] = old
