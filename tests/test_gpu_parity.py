"""Parity tests proper: the nvcc-built sm_100a library, called through the C ABI (ctypes), against the CPU oracle and
the reference's golden alm files.  Need a B200: run with `-m gpu`.

Tolerances (BASELINE.json north_star): relative RMS error <= 1e-10 in Float64 and <= 1e-5 in Float32.
Round trips are compared with the ORACLE's round trip, not with identity (SURVEY.md F6: plain CC weights are not exact
at lmax = nphi/2)."""
import ctypes
import math

import numpy as np
import pytest

import pixsht
from pixsht import Enmap, Alm, CarClenshawCurtis, fullsky_geometry, geometry, degree, arcminute
from pixsht.transforms import Plan, map2alm, alm2map, get_lib, PixshtError
from pixsht import _lib
from helpers import (golden_alm, gen_spin0, gen_spin2, oracle_map2alm, oracle_alm2map, rel_rms, synth_alm, band_copy, plain_fft_kernels)
from oracle import cc_geometry, get_oracle, nalm, alm_index

pytestmark = pytest.mark.gpu
TOL64, TOL32 = 1e-10, 1e-5


def relmax(a, b):
    return float(np.max(np.abs(a - b)) / np.max(np.abs(b)))


def test_library_is_the_cuda_build():
    lib = get_lib()
    assert "sm_100a" in lib.version() and "EMULATION" not in lib.version()
    assert lib.device_count() >= 1


# ---- the reference's own tests (test/test_transforms.jl:11-77) --------------------------------------------------
def test_golden_spin0_fullsky_sliced_box():
    shape, wcs = fullsky_geometry(10.0 * degree)
    m = Enmap(gen_spin0(shape), wcs)
    assert relmax(map2alm(m, lmax=18).alm, golden_alm("simple_analytic_sht")) < 1e-12
    assert len(map2alm(m).alm) == 190
    assert relmax(map2alm(m[5:-2, 4:-3], lmax=18).alm, golden_alm("simple_analytic_sht_sliced")) < 1e-12
    box = [[10 * degree, -10 * degree], [-5 * degree, 5 * degree]]
    bshape, bwcs = geometry(CarClenshawCurtis, box, 1.0 * degree)
    mb = Enmap(gen_spin0(bshape, 2.5), bwcs)
    assert relmax(map2alm(mb, lmax=100).alm, golden_alm("simple_box_analytic_sht")) < 1e-12


def test_golden_spin2_stack_tuple_iqu():
    shape, wcs = fullsky_geometry(10.0 * degree, dims=(2,))
    qu = Enmap(gen_spin2(shape), wcs)
    ref_e, ref_b = golden_alm("simple_pol_analytic_sht", (0, 1)), golden_alm("simple_pol_analytic_sht", (2, 3))
    e, b = map2alm(qu, lmax=3 * 36)
    assert relmax(e.alm, ref_e) < 1e-12 and relmax(b.alm, ref_b) < 1e-12
    e, b = map2alm((Enmap(qu.data[:, :, 0], wcs), Enmap(qu.data[:, :, 1], wcs)), lmax=3 * 36)
    assert relmax(e.alm, ref_e) < 1e-12 and relmax(b.alm, ref_b) < 1e-12
    shape3, wcs3 = fullsky_geometry(10.0 * degree, dims=(3,))
    d = np.zeros(shape3, order="F")
    d[:, :, 0] = gen_spin0(shape3)
    d[:, :, 1:] = gen_spin2(shape3)
    t, e, b = map2alm(Enmap(d, wcs3), lmax=3 * 36)
    assert relmax(t.alm, golden_alm("simple_analytic_sht_fullalm")) < 1e-12
    assert relmax(e.alm, ref_e) < 1e-12 and relmax(b.alm, ref_b) < 1e-12
    t2, e2, b2 = map2alm(tuple(Enmap(d[:, :, c], wcs3) for c in range(3)), lmax=3 * 36)
    assert np.array_equal(t2.alm, t.alm) or relmax(t2.alm, t.alm) < 1e-14


def test_bad_ncomp_is_an_error_not_a_crash():
    shape, wcs = fullsky_geometry(10.0 * degree, dims=(4,))
    with pytest.raises(ValueError):
        map2alm(Enmap(np.zeros(shape, order="F"), wcs), lmax=18)
    lib = get_lib()
    p = Plan(pixsht.sht_band((36, 19), wcs), 18)
    bad = (ctypes.c_void_p * 4)(1, 1, 1, 1)
    rc = lib.lib.pixsht_execute(p.handle, 0, 4, bad, bad, 0)
    assert rc == _lib.ERR_ARG and b"1 <= ncomp <= 3" in lib.lib.pixsht_last_error()
    p.close()


# ---- BASELINE config C1: 360 x 181 Float64 spin-0 round trip, lmax 180 -----------------------------------------
def test_c1_spin0_f64_both_directions_and_roundtrip():
    shape, wcs = fullsky_geometry(1.0 * degree)
    lmax = 180
    alm = synth_alm(lmax, lmax, 1000)
    ref_map = oracle_alm2map(alm[None], shape, wcs, lmax)[:, :, 0]
    got = alm2map(Alm(lmax, lmax, alm), shape, wcs)
    assert rel_rms(got.data, ref_map) < TOL64
    ref_alm = oracle_map2alm(Enmap(ref_map, wcs), lmax)[0]
    got_alm = map2alm(Enmap(ref_map, wcs), lmax=lmax).alm
    assert rel_rms(got_alm, ref_alm) < TOL64
    # round trip vs the oracle's round trip
    rt = map2alm(got, lmax=lmax).alm
    assert rel_rms(rt, ref_alm) < TOL64
    # white-noise (not band-limited) map
    rng = np.random.default_rng(2001)
    noise = Enmap(np.asfortranarray(rng.standard_normal(shape)), wcs)
    assert rel_rms(map2alm(noise, lmax=lmax).alm, oracle_map2alm(noise, lmax)[0]) < TOL64


@pytest.mark.parametrize("res_deg,lmax,mmax", [(0.5, 360, 360), (0.5, 300, 200), (0.25, 720, 720)])
def test_iqu_f64_vs_oracle(res_deg, lmax, mmax):
    shape, wcs = fullsky_geometry(res_deg * degree, dims=(3,))
    alms = [synth_alm(lmax, mmax, 3000 + c, spin2=c > 0) for c in range(3)]
    ref = np.concatenate([oracle_alm2map(alms[0][None], shape, wcs, lmax, mmax),
                          oracle_alm2map(np.stack(alms[1:]), shape, wcs, lmax, mmax, spin=2)], axis=2)
    got = alm2map(tuple(Alm(lmax, mmax, a) for a in alms), shape, wcs)
    assert isinstance(got, tuple) and len(got) == 3
    for c in range(3):
        assert rel_rms(got[c].data, ref[:, :, c]) < TOL64
    m = Enmap(np.asfortranarray(ref), wcs)
    t, e, b = map2alm(m, lmax=lmax, mmax=mmax)
    rt = oracle_map2alm(Enmap(ref[:, :, 0], wcs), lmax, mmax)[0]
    reb = oracle_map2alm(Enmap(ref[:, :, 1:], wcs), lmax, mmax, spin=2)
    assert rel_rms(t.alm, rt) < TOL64 and rel_rms(e.alm, reb[0]) < TOL64 and rel_rms(b.alm, reb[1]) < TOL64


def test_edge_fused_fft_forced_on_small_plans(monkeypatch):
    """The edge-fused ring-FFT kernels (fft_edge.cuh) are the default from 32 KB rings on (C3 / C4 / C5-size tests below run them);
    here they are forced (PIXSHT_FFT_EDGE=2) on small plans of every kind -- IQU, Float32 boundary, band limit below the Nyquist
    mode, a cut-sky flipped band with element-wise row access -- against the oracle and against the plain kernels."""
    shape, wcs = fullsky_geometry(0.5 * degree, dims=(3,))
    band = pixsht.sht_band(shape[:2], wcs)
    for lmax, mmax in ((360, 360), (300, 200)):
        alms = [synth_alm(lmax, mmax, 3100 + c, spin2=c > 0) for c in range(3)]
        ref = np.concatenate([oracle_alm2map(alms[0][None], shape, wcs, lmax, mmax),
                              oracle_alm2map(np.stack(alms[1:]), shape, wcs, lmax, mmax, spin=2)], axis=2)
        rt = oracle_map2alm(Enmap(ref[:, :, 0], wcs), lmax, mmax)[0]
        reb = oracle_map2alm(Enmap(ref[:, :, 1:], wcs), lmax, mmax, spin=2)
        res = {}
        for edge in ("2", "0"):
            monkeypatch.setenv("PIXSHT_FFT_EDGE", edge)
            for dt, tol in ((np.float64, TOL64), (np.float32, TOL32)):
                plan = Plan(band, lmax, mmax, dtype=dt)
                assert plan.info()["fft"]["edge_fused"] == (edge == "2")
                mp = plan.alm2map([a.astype(plan.cdtype) for a in alms])
                assert max(rel_rms(mp[c], ref[:, :, c]) for c in range(3)) < tol
                out = plan.map2alm([np.asfortranarray(ref[:, :, c], dtype=dt) for c in range(3)])
                assert max(rel_rms(out[0], rt), rel_rms(out[1], reb[0]), rel_rms(out[2], reb[1])) < tol
                res[(edge, dt)] = (mp, out)
                plan.close()
        for c in range(3):
            assert rel_rms(res[("2", np.float64)][0][c], res[("0", np.float64)][0][c]) < 1e-14
            assert rel_rms(res[("2", np.float64)][1][c], res[("0", np.float64)][1][c]) < 1e-13
    monkeypatch.setenv("PIXSHT_FFT_EDGE", "2")
    shape, wcs = fullsky_geometry(1.0 * degree)
    full = Enmap(gen_spin0(shape, 1.5), wcs)
    for sub in (full[40:300, 30:120], full[::-1, ::-1][13:341, 5:170]):
        plan = Plan(pixsht.sht_band(sub.data.shape, sub.wcs), 150)
        assert plan.info()["fft"]["edge_fused"]
        assert rel_rms(plan.map2alm([sub.data])[0], oracle_map2alm(sub, 150)[0]) < TOL64
        alm = synth_alm(150, 150, 78)
        assert rel_rms(plan.alm2map([alm])[0], oracle_alm2map(alm[None], sub.data.shape, sub.wcs, 150)[:, :, 0]) < TOL64
        plan.close()


def test_partial_sky_band_and_unflipped_geometry():
    # a cut-sky band sliced out of a full-sky grid, and a geometry with ascending RA / descending DEC (no flips)
    shape, wcs = fullsky_geometry(1.0 * degree)
    full = Enmap(gen_spin0(shape, 1.5), wcs)
    sub = full[40:300, 30:120]
    lmax = 150
    assert rel_rms(map2alm(sub, lmax=lmax).alm, oracle_map2alm(sub, lmax)[0]) < TOL64
    alm = synth_alm(lmax, lmax, 77)
    got = alm2map(Alm(lmax, lmax, alm), sub.shape, sub.wcs)
    assert rel_rms(got.data, oracle_alm2map(alm[None], sub.shape, sub.wcs, lmax)[:, :, 0]) < TOL64
    flipped = full[::-1, ::-1]
    assert rel_rms(map2alm(flipped, lmax=lmax).alm, oracle_map2alm(flipped, lmax)[0]) < TOL64
    got = alm2map(Alm(lmax, lmax, alm), flipped.shape, flipped.wcs)
    assert rel_rms(got.data, oracle_alm2map(alm[None], flipped.shape, flipped.wcs, lmax)[:, :, 0]) < TOL64


def test_float32_maps():
    """Float32 Enmaps: by default promoted to Float64 like the reference (create_sht_band, src/transforms.jl:71; alm are ComplexF64),
    so the result is the Float64 transform of the rounded map; precision="f32" opts in to the Float32-boundary plan (<= 1e-5)."""
    shape, wcs = fullsky_geometry(0.5 * degree)
    lmax = 360
    alm = synth_alm(lmax, lmax, 2000)
    ref = oracle_alm2map(alm[None], shape, wcs, lmax)[:, :, 0]
    got = alm2map(Alm(lmax, lmax, alm), shape, wcs, dtype=np.float32)
    assert got.dtype == np.float32 and rel_rms(got.data, ref) < TOL32
    m32 = np.asfortranarray(ref, dtype=np.float32)
    a_def = map2alm(Enmap(m32, wcs), lmax=lmax)
    assert a_def.alm.dtype == np.complex128
    assert rel_rms(a_def.alm, oracle_map2alm(Enmap(m32.astype(np.float64), wcs), lmax)[0]) < TOL64      # Float64 numerics on the Float32 data
    a32 = map2alm(Enmap(m32, wcs), lmax=lmax, precision="f32")
    assert a32.alm.dtype == np.complex128
    assert rel_rms(a32.alm, oracle_map2alm(Enmap(ref, wcs), lmax)[0]) < TOL32


def test_adjointness_and_linearity_midsize():
    """size-independent properties at a size the full oracle would be slow for: <W Y a, m> = <a, Y^T W m>, linearity."""
    shape, wcs = fullsky_geometry(4.0 * arcminute)   # 5400 x 2701 (geometry of BASELINE config C2)
    lmax = 2700
    band = pixsht.sht_band(shape, wcs)
    plan = Plan(band, lmax)
    w, _ = plan.weights()
    rng = np.random.default_rng(9)
    a1, a2 = synth_alm(lmax, lmax, 91), synth_alm(lmax, lmax, 92)
    m1, m2 = plan.alm2map([a1])[0], plan.alm2map([a2])[0]
    m12 = plan.alm2map([a1 + 0.5 * a2])[0]
    assert rel_rms(m12, m1 + 0.5 * m2) < 1e-12
    x = np.asfortranarray(rng.standard_normal(shape))
    ytx = plan.map2alm([x])[0]
    wrow = w[::-1] if band.flipy else w
    lhs = float(np.sum(m1 * x * wrow[None, :]))
    fac = np.full(a1.shape, 2.0)
    fac[:lmax + 1] = 1.0
    rhs = float(np.sum(fac * (np.conj(a1) * ytx).real))
    assert abs(lhs - rhs) < 1e-10 * abs(lhs)
    # sampled rings / sampled m against the oracle at this size
    ref = oracle_alm2map(a1[None], shape, wcs, lmax, ring_stride=337, ring_offset=5)[:, :, 0]
    rows = np.arange(band.nrings)[5::337]
    rows_map = (band.nrings - 1 - rows) if band.flipy else rows
    assert rel_rms(m1[:, rows_map], ref[:, rows_map]) < TOL64
    ref_alm = oracle_map2alm(Enmap(x, wcs), lmax, m_stride=451, m_offset=7)[0]
    sel = np.concatenate([np.arange(alm_index(lmax, m, m), alm_index(lmax, lmax, m) + 1) for m in range(7, lmax + 1, 451)])
    assert rel_rms(ytx[sel], ref_alm[sel]) < TOL64
    plan.close()


def test_sharp_shim_runs_the_reference_call_sequence():
    """The ccall sequence of src/transforms.jl:33-63,88-108 against the libsharp2-compatible symbols."""
    lib = get_lib()
    L = lib.lib
    shape, wcs = fullsky_geometry(10.0 * degree)
    m = Enmap(gen_spin0(shape), wcs)
    band, b = band_copy(m)
    theta, w = cc_geometry(b.nrings_total, b.nphi, b.ring_first, b.nrings)
    n = b.nrings
    nph = (ctypes.c_int * n)(*([b.nphi] * n))
    ofs = (ctypes.c_ssize_t * n)(*[b.nphi * i for i in range(n)])
    stride = (ctypes.c_int * n)(*([1] * n))
    phi0 = (ctypes.c_double * n)(*([b.phi0] * n))
    th = (ctypes.c_double * n)(*theta)
    wg = (ctypes.c_double * n)(*w)
    geom, ainfo = ctypes.c_void_p(), ctypes.c_void_p()
    L.sharp_make_geom_info(n, nph, ofs, stride, phi0, th, wg, ctypes.byref(geom))
    L.sharp_make_triangular_alm_info(18, 18, 1, ctypes.byref(ainfo))
    assert L.sharp_alm_count(ainfo) == 190 and L.sharp_map_size(geom) == 36 * 19
    alm = np.zeros(190, dtype=np.complex128)
    flat = np.ascontiguousarray(band[0]).ravel()
    SHARP_MAP2ALM, SHARP_ALM2MAP, SHARP_DP = 0, 1, 1 << 4
    L.sharp_execute(SHARP_MAP2ALM, 0, (ctypes.c_void_p * 1)(alm.ctypes.data), (ctypes.c_void_p * 1)(flat.ctypes.data), geom, ainfo,
                    SHARP_DP, None, None)
    assert L.pixsht_shim_status() == 0
    assert relmax(alm, golden_alm("simple_analytic_sht")) < 1e-12
    back = np.zeros_like(flat)
    L.sharp_execute(SHARP_ALM2MAP, 0, (ctypes.c_void_p * 1)(alm.ctypes.data), (ctypes.c_void_p * 1)(back.ctypes.data), geom, ainfo,
                    SHARP_DP, None, None)
    th_full, _ = cc_geometry(b.nrings_total, b.nphi)
    ref = get_oracle("ld").alm2map(alm[None], th_full, b.phi0, b.nphi, 18)[0].ravel()
    assert rel_rms(back, ref) < TOL64
    L.sharp_destroy_alm_info(ainfo)
    L.sharp_destroy_geom_info(geom)


# ---- BASELINE-size checks (C3 / C4 geometries): sampled parity against the oracle + size-independent properties ----------
POLE_TOL64 = 5e-9


def _ring_errors(band, maps, alms, lmax, spin, rings):
    """rel-RMS error per selected band ring of alm2map output against the long-double oracle evaluated on those rings."""
    theta, _ = cc_geometry(band.nrings_total, band.nphi, band.ring_first, band.nrings)
    ref = get_oracle("ld").alm2map(np.stack(alms), theta[rings], band.phi0, band.nphi, lmax, spin=spin)
    num, den = np.zeros(len(rings)), np.zeros(len(rings))
    for i, r in enumerate(rings):
        row = (band.nrings - 1 - r) if band.flipy else r
        for c in range(len(alms)):
            g = maps[c][:, row]
            g = g[::-1] if band.flipx else g
            num[i] += np.sum((g[:band.nx] - ref[c, i, :band.nx]) ** 2)
            den[i] += np.sum(ref[c, i, :band.nx] ** 2)
    return num, den


def _sampled_checks(plan, band, shape, wcs, lmax, alms, spin, ring_stride, ring_offset, m_stride, m_offset, seed):
    """alm2map on sampled rings and map2alm on sampled m against the long-double oracle, plus adjointness of the pair.

    Tolerances: rel-RMS <= 1e-10 (north_star) over the sampled rings / m.  The few rings within ~0.2 deg of a pole are held
    to POLE_TOL64 instead: FP64 three-term recurrences in cos(theta) (this engine and libsharp2 alike) lose ~l^1.5 eps there
    -- measured 1e-9 on the pole ring itself at lmax = 10800 with a white spectrum, 1e-11 from 0.5 deg on (tools/pole_accuracy.py);
    the whole-map rel-RMS stays ~1e-11."""
    nc = len(alms)
    maps = plan.alm2map(alms)
    rings = list(range(ring_offset, band.nrings, ring_stride))
    num, den = _ring_errors(band, maps, alms, lmax, spin, rings)
    assert np.sqrt(num.sum() / den.sum()) < TOL64
    polar = [0, 1, 2, band.nrings - 2, band.nrings - 1]
    num, den = _ring_errors(band, maps, alms, lmax, spin, polar)
    assert np.all(np.sqrt(num / den) < POLE_TOL64)
    rng = np.random.default_rng(seed)
    x = [np.asfortranarray(rng.standard_normal(shape[:2])) for _ in range(nc)]
    ytx = plan.map2alm(x)
    xm = Enmap(x[0], wcs) if nc == 1 else Enmap(np.asfortranarray(np.stack(x, axis=2)), wcs)
    ref_alm = oracle_map2alm(xm, lmax, spin=spin, m_stride=m_stride, m_offset=m_offset)
    sel = np.concatenate([np.arange(alm_index(lmax, m, m), alm_index(lmax, lmax, m) + 1) for m in range(m_offset, lmax + 1, m_stride)])
    for c in range(nc):
        assert rel_rms(ytx[c][sel], ref_alm[c][sel]) < TOL64
    # <W Y a, x> = <a, Y^T W x> over all components
    w, _ = plan.weights()
    wrow = w[::-1] if band.flipy else w
    lhs = sum(float(np.sum(maps[c] * x[c] * wrow[None, :])) for c in range(nc))
    fac = np.full(alms[0].shape, 2.0)
    fac[:lmax + 1] = 1.0
    rhs = sum(float(np.sum(fac * (np.conj(alms[c]) * ytx[c]).real)) for c in range(nc))
    assert abs(lhs - rhs) < 1e-10 * max(abs(lhs), abs(rhs))
    return maps, ytx


def test_c3_size_iqu_sampled_parity_and_adjointness():
    """BASELINE config C3: full-sky CAR 2' (10800 x 5401), lmax 5400, T and (E,B)."""
    shape, wcs = fullsky_geometry(2.0 * arcminute)
    lmax = 5400
    band = pixsht.sht_band(shape, wcs)
    plan = Plan(band, lmax)
    _sampled_checks(plan, band, shape, wcs, lmax, [synth_alm(lmax, lmax, 3000)], 0, 1201, 150, 1777, 5, 31)
    _sampled_checks(plan, band, shape, wcs, lmax, [synth_alm(lmax, lmax, 3001, spin2=True), synth_alm(lmax, lmax, 3002, spin2=True)],
                    2, 1201, 600, 1777, 2, 32)
    plan.close()


def test_c4_size_spin0_and_spin2_sampled_parity():
    """BASELINE config C4 (the headline): full-sky CAR 1' (21600 x 10801), lmax 10800.  Rings next to the pole, mid latitude
    and the equator; low, middle and Nyquist-adjacent m."""
    shape, wcs = fullsky_geometry(1.0 * arcminute)
    lmax = 10800
    band = pixsht.sht_band(shape, wcs)
    plan = Plan(band, lmax)
    _sampled_checks(plan, band, shape, wcs, lmax, [synth_alm(lmax, lmax, 4000)], 0, 1350, 337, 3600, 0, 41)
    _sampled_checks(plan, band, shape, wcs, lmax, [synth_alm(lmax, lmax, 4001, spin2=True), synth_alm(lmax, lmax, 4002, spin2=True)],
                    2, 2700, 1337, 5400, 5399, 42)
    plan.close()


def test_c2_size_float32_sampled_parity():
    """BASELINE config C2: full-sky CAR 4' (5400 x 2701) Float32 T-only, lmax 2700 (also the unit of the 64-map sweep).
    Float32 at the boundary, FP64 inside: rel-RMS <= 1e-5 (north_star's Float32 tolerance) on sampled rings and sampled m.
    PARITY UNPINNED by files: the reference promotes Float32 maps to Float64 (SURVEY.md F7)."""
    shape, wcs = fullsky_geometry(4.0 * arcminute)
    assert shape == (5400, 2701)
    lmax = 2700
    band = pixsht.sht_band(shape, wcs)
    plan = Plan(band, lmax, dtype=np.float32)
    alm = synth_alm(lmax, lmax, 2100).astype(np.complex64)
    maps = plan.alm2map([alm])
    assert maps[0].dtype == np.float32
    rings = list(range(7, band.nrings, 300)) + [0, band.nrings - 1]
    num, den = _ring_errors(band, [maps[0].astype(np.float64)], [alm.astype(np.complex128)], lmax, 0, rings)
    assert np.sqrt(num.sum() / den.sum()) < TOL32
    rng = np.random.default_rng(21)
    x = np.asfortranarray(rng.standard_normal(shape), dtype=np.float32)
    got = plan.map2alm([x])[0]
    assert got.dtype == np.complex64
    m_stride, m_offset = 450, 3
    ref_alm = oracle_map2alm(Enmap(x.astype(np.float64), wcs), lmax, m_stride=m_stride, m_offset=m_offset)[0]
    sel = np.concatenate([np.arange(alm_index(lmax, m, m), alm_index(lmax, lmax, m) + 1) for m in range(m_offset, lmax + 1, m_stride)])
    assert rel_rms(got[sel].astype(np.complex128), ref_alm[sel]) < TOL32
    plan.close()


def test_c5_size_float32_sampled_parity():
    """BASELINE config C5: full-sky CAR 0.5' (43200 x 21601) Float32 T-only, lmax 21600 (the largest config; a 3.7 GB map).
    Sampled rings (pole-adjacent, mid latitude, equator) and sampled m (low, middle, Nyquist-adjacent) against the long-double
    oracle: rel-RMS <= 1e-5 (north_star's Float32 tolerance).  PARITY UNPINNED by files (SURVEY.md F7)."""
    shape, wcs = fullsky_geometry(0.5 * arcminute)
    assert shape == (43200, 21601)
    lmax = 21600
    band = pixsht.sht_band(shape, wcs)
    plan = Plan(band, lmax, dtype=np.float32)
    alm = synth_alm(lmax, lmax, 5000).astype(np.complex64)
    maps = plan.alm2map([alm])
    assert maps[0].dtype == np.float32
    rings = [2, 5400, 10800, 21598]
    num, den = _ring_errors(band, [maps[0].astype(np.float64, copy=False)], [alm.astype(np.complex128)], lmax, 0, rings)
    assert np.sqrt(num.sum() / den.sum()) < TOL32
    assert np.all(np.sqrt(num / den) < 10 * TOL32)       # no single ring (the pole-adjacent ones included) far off
    got = plan.map2alm(maps)[0]                           # analysis of the (band-limited) synthesised map
    assert got.dtype == np.complex64
    theta, w = cc_geometry(band.nrings_total, band.nphi)
    fx = slice(None, None, -1) if band.flipx else slice(None)
    fy = slice(None, None, -1) if band.flipy else slice(None)
    bandmap = np.ascontiguousarray(maps[0].T[fy, fx], dtype=np.float64)[None]
    for m in (3, 10811, 21599):
        ref = get_oracle("ld").map2alm(bandmap, theta, w, band.phi0, lmax, m_stride=lmax + 1, m_offset=m)[0]
        sl = slice(alm_index(lmax, m, m), alm_index(lmax, lmax, m) + 1)
        assert rel_rms(got[sl].astype(np.complex128), ref[sl]) < TOL32
    plan.close()


def test_c3_size_full_map_against_cpu_port():
    """BASELINE config C3, EVERY pixel and EVERY alm (not a sample): the CUDA engine against oracle/sht_cpu.c, the
    libsharp2-style CPU implementation (itself checked against the long-double checker in tests/test_oracle_properties.py).
    Whole-map / whole-alm rel-RMS <= 1e-10."""
    from oracle import get_cpu_sht
    shape, wcs = fullsky_geometry(2.0 * arcminute)
    lmax = 5400
    band = pixsht.sht_band(shape, wcs)
    plan = Plan(band, lmax)
    cpu = get_cpu_sht()
    cpu.use_all_cores()
    theta, w = cc_geometry(band.nrings_total, band.nphi)
    alms = [synth_alm(lmax, lmax, 3100 + c, spin2=c > 0) for c in range(3)]
    maps = plan.alm2map(alms)
    fx = slice(None, None, -1) if band.flipx else slice(None)
    fy = slice(None, None, -1) if band.flipy else slice(None)
    ref_t = cpu.alm2map(alms[0][None], theta, band.phi0, band.nphi, lmax, spin=0)
    ref_qu = cpu.alm2map(np.stack(alms[1:]), theta, band.phi0, band.nphi, lmax, spin=2)
    ref = [ref_t[0], ref_qu[0], ref_qu[1]]
    for c in range(3):
        assert rel_rms(maps[c].T[fy, fx], ref[c]) < TOL64
    rng = np.random.default_rng(33)
    x = [rng.standard_normal((band.nrings, band.nphi)) for _ in range(3)]          # band orientation, not band-limited
    got = plan.map2alm([np.asfortranarray(b[fy, fx].T) for b in x])
    ref_a = [cpu.map2alm(x[0][None], theta, w, band.phi0, lmax, spin=0)[0]] + list(cpu.map2alm(np.stack(x[1:]), theta, w, band.phi0, lmax, spin=2))
    for c in range(3):
        assert rel_rms(got[c], ref_a[c]) < TOL64
    plan.close()


def test_batch_overlapped_staging_equals_serial(monkeypatch):
    """Host-pointer batches: the double-buffered staging on the copy streams (the default) gives the same bits as the serial one,
    on pageable arrays (the plan's stager) and on page-locked ones from pixsht_host_alloc (straight to the copy engines)."""
    shape, wcs = fullsky_geometry(8.0 * arcminute)
    lmax = 1350
    band = pixsht.sht_band(shape, wcs)
    alms = [synth_alm(lmax, lmax, 900 + b).astype(np.complex64) for b in range(11)]      # groups 4 + 4 + 2 + 1
    lib = get_lib()
    for kind in ("pageable", "pinned"):
        res = {}
        for ovl in ("1", "0"):
            monkeypatch.setenv("PIXSHT_BATCH_OVERLAP", ovl)
            plan = Plan(band, lmax, dtype=np.float32)
            if kind == "pageable":
                maps = plan.alm2map_batch(alms)
                back = plan.map2alm_batch(maps)
            else:
                npix = band.nx * band.nrings
                ptrs = []
                def pinned(n, dt):
                    p = ctypes.c_void_p()
                    lib.check(lib.lib.pixsht_host_alloc(ctypes.byref(p), n * np.dtype(dt).itemsize))
                    ptrs.append(p.value)
                    return np.frombuffer((ctypes.c_char * (n * np.dtype(dt).itemsize)).from_address(p.value), dtype=dt)
                h_alm = [pinned(plan.nalm, np.complex64) for _ in alms]
                h_map = [pinned(npix, np.float32) for _ in alms]
                for h, a in zip(h_alm, alms):
                    h[...] = a
                for h in h_map:
                    h[...] = np.nan
                plan.execute_batch_ptrs(_lib.ALM2MAP, [h.ctypes.data for h in h_alm], [h.ctypes.data for h in h_map], _lib.HOST)
                for h in h_alm:
                    h[...] = np.nan
                plan.execute_batch_ptrs(_lib.MAP2ALM, [h.ctypes.data for h in h_alm], [h.ctypes.data for h in h_map], _lib.HOST)
                maps = [h.reshape(band.nrings, band.nx).T.copy() for h in h_map]
                back = [h.copy() for h in h_alm]
                del h_alm, h_map
                for p in ptrs:
                    lib.check(lib.lib.pixsht_host_free(p))
            res[ovl] = (maps, back)
            plan.close()
        for b in range(len(alms)):
            assert np.array_equal(res["1"][0][b], res["0"][0][b])
            assert rel_rms(res["1"][1][b], res["0"][1][b]) < 2e-6
        single = Plan(band, lmax, dtype=np.float32)
        assert rel_rms(res["1"][0][10], single.alm2map([alms[10]])[0]) < 2e-6
        assert rel_rms(res["1"][1][10], single.map2alm([res["1"][0][10]])[0]) < 2e-6
        single.close()


def test_host_and_device_paths_agree_and_iqu_is_t_plus_qu():
    """The pipelined host-pointer path (three streams, split launches) equals the single-stream device path, and the fused
    IQU call equals a T call plus a QU call (the reference runs IQU as two libsharp jobs, src/transforms.jl:143-144)."""
    import torch
    shape, wcs = fullsky_geometry(8.0 * arcminute)
    lmax = 1350
    band = pixsht.sht_band(shape, wcs)
    plan = Plan(band, lmax)
    alms = [synth_alm(lmax, lmax, 70), synth_alm(lmax, lmax, 71, spin2=True), synth_alm(lmax, lmax, 72, spin2=True)]
    host = plan.alm2map(alms)
    t_only = plan.alm2map(alms[:1])
    qu_only = plan.alm2map(alms[1:])
    assert np.array_equal(host[0], t_only[0]) and np.array_equal(host[1], qu_only[0]) and np.array_equal(host[2], qu_only[1])
    dev = torch.device("cuda", 0)
    d_alm = [torch.from_numpy(a).to(dev) for a in alms]
    d_map = [torch.empty(band.nx * band.nrings, dtype=torch.float64, device=dev) for _ in alms]
    plan.execute_ptrs(_lib.ALM2MAP, [a.data_ptr() for a in d_alm], [m.data_ptr() for m in d_map], _lib.DEVICE)
    for c in range(3):
        assert np.array_equal(d_map[c].cpu().numpy().reshape(band.nrings, band.nx).T, host[c])
    back_host = plan.map2alm(host)
    d_out = [torch.empty_like(a) for a in d_alm]
    plan.execute_ptrs(_lib.MAP2ALM, [a.data_ptr() for a in d_out], [m.data_ptr() for m in d_map], _lib.DEVICE)
    for c in range(3):   # atomic accumulation order differs between the split and the single launch: equal to rounding
        assert rel_rms(d_out[c].cpu().numpy(), back_host[c]) < 1e-13
    ex, nom = plan.work(0)
    assert 0.5 < ex / nom < 0.9          # the activation table prunes what never reaches 2^-90
    plan.close()


def _mgpu_worker(rank, world, port, out_dir):
    import os
    import sys
    import torch
    import torch.distributed as dist
    here = os.path.dirname(os.path.abspath(__file__))
    for p in (os.path.dirname(here), os.path.join(os.path.dirname(here), "pixell.jl_b200"), here):
        if p not in sys.path:
            sys.path.insert(0, p)
    import pixsht as px
    from pixsht.distributed import ShardedSHT
    from helpers import synth_alm as sa
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", init_method="tcp://127.0.0.1:%d" % port, rank=rank, world_size=world, device_id=dev)
    shape, wcs = px.fullsky_geometry(8.0 * px.arcminute)
    lmax = 1350
    band = px.sht_band(shape, wcs)
    sht = ShardedSHT(band, lmax, device=dev)
    alms = [torch.from_numpy(sa(lmax, lmax, 70 + c, spin2=c > 0)).to(dev) for c in range(3)]
    a, b = sht.map_rows()
    slabs = [torch.zeros((b - a) * band.nx, dtype=torch.float64, device=dev) for _ in range(3)]
    for _ in range(2):      # twice: the second pass reuses the peer buffers (exercises the stage-ordering barriers)
        sht.alm2map(alms, slabs)
        out = [torch.full((sht.nalm,), 7.0, dtype=torch.complex128, device=dev) for _ in range(3)]
        sht.map2alm(slabs, out)
    torch.cuda.synchronize(dev)
    # host-resident variant (copies overlapped with the stages, one spin family at a time): same numbers
    idx = torch.cat([torch.arange(s, e, device=dev) for (s, e) in sht.alm_columns()])
    h_cols = [x.index_select(0, idx).cpu().pin_memory() for x in alms]
    h_slabs = [torch.zeros(x.numel(), dtype=x.dtype).pin_memory() for x in slabs]
    h_out = [torch.zeros_like(x).pin_memory() for x in h_cols]
    w_alm = [torch.zeros(sht.nalm, dtype=torch.complex128, device=dev) for _ in range(3)]
    w_slab = [torch.zeros_like(x) for x in slabs]
    for _ in range(2):
        sht.alm2map_host(h_cols, h_slabs, w_alm, w_slab)
        sht.map2alm_host(h_slabs, h_out, w_slab, w_alm)
    torch.cuda.synchronize(dev)
    host_ok = all(torch.equal(h.to(dev), x) for h, x in zip(h_slabs, slabs))
    host_ok = host_ok and all(float((h.to(dev) - o.index_select(0, idx)).abs().max()) <= 1e-13 * float(o.abs().max()) for h, o in zip(h_out, out))
    np.save(os.path.join(out_dir, "hostok_%d.npy" % rank), np.array([int(host_ok)]))
    np.save(os.path.join(out_dir, "slab_%d.npy" % rank), np.stack([s.cpu().numpy() for s in slabs]))
    np.save(os.path.join(out_dir, "alm_%d.npy" % rank), np.stack([o.cpu().numpy() for o in out]))
    np.save(os.path.join(out_dir, "rows_%d.npy" % rank), np.array([a, b]))
    sht.close()
    dist.destroy_process_group()


def test_multi_gpu_peer_memory_pipeline_matches_single_gpu(tmp_path):
    """m-sharded Legendre + ring-sharded FFT with the phase rows exchanged through peer memory (no all-to-all pass):
    every rank's slab and alm columns equal the single-GPU transform.  Needs >= 2 GPUs on the box."""
    import os
    import torch
    import torch.multiprocessing as mp
    world = min(torch.cuda.device_count(), 4)
    if world < 2:
        pytest.skip("needs at least 2 GPUs")
    port = 29700 + os.getpid() % 200
    mp.spawn(_mgpu_worker, args=(world, port, str(tmp_path)), nprocs=world, join=True)
    shape, wcs = fullsky_geometry(8.0 * arcminute)
    lmax = 1350
    band = pixsht.sht_band(shape, wcs)
    plan = Plan(band, lmax)
    alms = [synth_alm(lmax, lmax, 70 + c, spin2=c > 0) for c in range(3)]
    maps = plan.alm2map(alms)
    back = plan.map2alm(maps)
    got = np.zeros((3, band.nrings, band.nx))
    for r in range(world):
        a, b = np.load(tmp_path / ("rows_%d.npy" % r))
        got[:, a:b, :] = np.load(tmp_path / ("slab_%d.npy" % r)).reshape(3, b - a, band.nx)
    for c in range(3):
        assert np.array_equal(got[c].T, maps[c])
    alm_sum = sum(np.load(tmp_path / ("alm_%d.npy" % r)) for r in range(world))
    for c in range(3):
        assert rel_rms(alm_sum[c], back[c]) < 1e-13
    assert all(int(np.load(tmp_path / ("hostok_%d.npy" % r))[0]) == 1 for r in range(world))   # alm2map_host / map2alm_host
    plan.close()


# ---- one process, several GPUs behind the C ABI (pixsht_plan_create_multi) ---------------------------------------------------
def _shard_devices(nshard):
    """nshard shards on the GPUs of the box, round-robin (a one-GPU box runs every shard on device 0: same code path --
    partition, per-m address table, slabs, event barriers -- without NVLink)."""
    k = max(1, get_lib().device_count())
    return [i % k for i in range(nshard)]


@pytest.mark.parametrize("nshard", [2, 3, 8])
def test_multi_gpu_plan_equals_single_gpu_plan(nshard, res_arcmin=8.0, lmax=1350, reps=2):
    """The one-process multi-GPU plan against the single-GPU plan on the same inputs: synthesis bit for bit (each (m, ring)
    sum is the same sequence of FMAs wherever it runs; both on the plain ring-FFT kernels, which the m-sharded layout uses),
    analysis to rounding (atomic accumulation order); IQU, T alone, QU alone, Float32, partial-sky / flipped bands, and a batch
    dealt over the shards.  The default single-GPU plan (edge-fused ring FFTs) agrees to rounding."""
    shape, wcs = fullsky_geometry(res_arcmin * arcminute)
    band = pixsht.sht_band(shape, wcs)
    with plain_fft_kernels():
        single = Plan(band, lmax)
    assert not single.info()["fft"]["edge_fused"]
    multi = Plan(band, lmax, devices=_shard_devices(nshard))
    default = Plan(band, lmax)
    assert multi.info()["ndev"] == nshard
    sh = multi.shards()
    assert sorted(np.concatenate([s[3] for s in sh]).tolist()) == list(range(lmax + 1))      # every m exactly once
    assert sum(s[2] for s in sh) == band.nrings and sh[0][1] == 0
    alms = [synth_alm(lmax, lmax, 70 + c, spin2=c > 0) for c in range(3)]
    for comps in ([0, 1, 2], [0], [1, 2]):
        for _ in range(reps):                 # twice: buffers and events are reused
            ref = single.alm2map([alms[c] for c in comps])
            got = multi.alm2map([alms[c] for c in comps])
            for a, b in zip(got, ref):
                assert np.array_equal(a, b)
            back_ref = single.map2alm(ref)
            back = multi.map2alm(got)
            for a, b in zip(back, back_ref):
                assert rel_rms(a, b) < 1e-13
    for a, b in zip(default.alm2map(alms), multi.alm2map(alms)):
        assert rel_rms(a, b) < 1e-14
    single.close(); multi.close(); default.close()
    # Float32 boundary, T only
    with plain_fft_kernels():
        s32 = Plan(band, lmax, dtype=np.float32)
    m32 = Plan(band, lmax, dtype=np.float32, devices=_shard_devices(nshard))
    a32 = alms[0].astype(np.complex64)
    r = s32.alm2map([a32])[0]; g = m32.alm2map([a32])[0]
    assert g.dtype == np.float32 and np.array_equal(g, r)
    assert rel_rms(m32.map2alm([g])[0], s32.map2alm([r])[0]) < 1e-6
    # a batch on a multi-GPU plan: whole transforms dealt to the shards
    nb = nshard + 1
    balm = [synth_alm(lmax, lmax, 500 + b).astype(np.complex64) for b in range(nb)]
    bm = m32.alm2map_batch(balm)
    for b in (0, nb - 1):
        assert rel_rms(bm[b], s32.alm2map([balm[b]])[0]) < 2e-6
    bb = m32.map2alm_batch(bm)
    assert rel_rms(bb[nb - 1], s32.map2alm([bm[nb - 1]])[0]) < 2e-6
    s32.close(); m32.close()


def test_multi_gpu_plan_partial_sky_flips_and_oracle(res_deg=1.0, lmax=150, nshard=3):
    """Cut-sky band (zero-padded rings, ring subset) and an unflipped geometry through the multi-GPU plan, against the oracle."""
    shape, wcs = fullsky_geometry(res_deg * degree)
    full = Enmap(gen_spin0(shape, 1.5), wcs)
    nx, ny = shape
    for sub in (full[nx // 9:nx - nx // 6, ny // 6:ny - ny // 3], full[::-1, ::-1]):
        band = pixsht.sht_band(sub.shape, sub.wcs)
        multi = Plan(band, lmax, devices=_shard_devices(nshard))
        got = multi.map2alm([np.asfortranarray(sub.data)])[0]
        assert rel_rms(got, oracle_map2alm(sub, lmax)[0]) < TOL64
        alm = synth_alm(lmax, lmax, 77)
        mp = multi.alm2map([alm])[0]
        assert rel_rms(mp, oracle_alm2map(alm[None], sub.shape, sub.wcs, lmax)[:, :, 0]) < TOL64
        multi.close()


def test_multi_gpu_plan_sharded_device_buffers(res_arcmin=8.0, lmax=1350, nshard=2):
    """pixsht_execute_sharded: data already distributed (each shard holds its alm columns and its slab of rows on its GPU)."""
    import torch
    shape, wcs = fullsky_geometry(res_arcmin * arcminute)
    band = pixsht.sht_band(shape, wcs)
    devs = _shard_devices(nshard)
    with plain_fft_kernels():       # the kernels of the m-sharded layout: the slabs are compared bit for bit
        single = Plan(band, lmax)
    multi = Plan(band, lmax, devices=devs)
    alms = [synth_alm(lmax, lmax, 70 + c, spin2=c > 0) for c in range(3)]
    ref = single.alm2map(alms)
    back_ref = single.map2alm(ref)
    sh = multi.shards()
    d_alm, d_slab, d_out = [], [], []
    for (dev, r0, nr, ml) in sh:
        td = torch.device("cuda", dev)
        mask = np.zeros(single.nalm, dtype=bool)
        for m in ml:
            mask[alm_index(lmax, int(m), int(m)):alm_index(lmax, lmax, int(m)) + 1] = True
        d_alm.append([torch.from_numpy(np.where(mask, a, 7.0 + 0j)).to(td) for a in alms])      # foreign columns hold junk
        d_slab.append([torch.zeros(nr * band.nx, dtype=torch.float64, device=td) for _ in alms])
        d_out.append([torch.full((single.nalm,), 3.0 + 0j, dtype=torch.complex128, device=td) for _ in alms])
    flat = lambda x: [t.data_ptr() for per in x for t in per]
    multi.execute_sharded_ptrs(_lib.ALM2MAP, 3, flat(d_alm), flat(d_slab))
    for k, (dev, r0, nr, ml) in enumerate(sh):
        a, b = (band.nrings - r0 - nr, band.nrings - r0) if band.flipy else (r0, r0 + nr)
        for c in range(3):
            assert np.array_equal(d_slab[k][c].cpu().numpy().reshape(nr, band.nx).T, ref[c][:, a:b])
    multi.execute_sharded_ptrs(_lib.MAP2ALM, 3, flat(d_out), flat(d_slab))
    for k, (dev, r0, nr, ml) in enumerate(sh):
        for c in range(3):
            o = d_out[k][c].cpu().numpy()
            for m in (int(ml[0]), int(ml[-1])):
                sl = slice(alm_index(lmax, m, m), alm_index(lmax, lmax, m) + 1)
                assert rel_rms(o[sl], back_ref[c][sl]) < 1e-12
    single.close(); multi.close()


def test_c3_size_multi_gpu_plan_sampled_parity():
    """BASELINE config C3 through the one-process multi-GPU plan (every GPU of the box, at least two shards): sampled rings and
    sampled m against the long-double oracle + adjointness, as for the single-GPU plan."""
    shape, wcs = fullsky_geometry(2.0 * arcminute)
    lmax = 5400
    band = pixsht.sht_band(shape, wcs)
    plan = Plan(band, lmax, devices=_shard_devices(max(2, min(8, get_lib().device_count()))))
    _sampled_checks(plan, band, shape, wcs, lmax, [synth_alm(lmax, lmax, 3000)], 0, 1201, 150, 1777, 5, 31)
    _sampled_checks(plan, band, shape, wcs, lmax, [synth_alm(lmax, lmax, 3001, spin2=True), synth_alm(lmax, lmax, 3002, spin2=True)],
                    2, 1201, 600, 1777, 2, 32)
    plan.close()


# ---- edge cases: degenerate band limits, tiny and ragged bands, argument errors --------------------------------------------
@pytest.mark.parametrize("lmax,mmax", [(0, 0), (1, 1), (1, 0), (2, 2), (18, 0), (18, 3), (40, 40)])
def test_edge_band_limits(lmax, mmax):
    """lmax / mmax at the low end (spin 2 has nothing below l = 2), mmax < lmax, and lmax > nphi/2 (aliasing) on a 36 x 19 grid."""
    shape, wcs = fullsky_geometry(10.0 * degree)
    band = pixsht.sht_band(shape, wcs)
    plan = Plan(band, lmax, mmax)
    theta, w = cc_geometry(band.nrings_total, band.nphi)
    orc = get_oracle("ld")
    for spin, nc in ((0, 1), (2, 2)):
        alms = [synth_alm(lmax, mmax, 7 + c, spin2=spin == 2) for c in range(nc)]
        maps = plan.alm2map(alms)
        ref = oracle_alm2map(np.stack(alms), shape, wcs, lmax, mmax, spin=spin)
        scale = max(1.0, float(np.max(np.abs(ref))))
        for c in range(nc):
            assert np.max(np.abs(maps[c] - ref[:, :, c])) < 1e-12 * scale
        rng = np.random.default_rng(5)
        x = [np.asfortranarray(rng.standard_normal(shape)) for _ in range(nc)]
        got = plan.map2alm(x)
        xm = Enmap(x[0], wcs) if nc == 1 else Enmap(np.asfortranarray(np.stack(x, axis=2)), wcs)
        ref_alm = oracle_map2alm(xm, lmax, mmax, spin=spin)
        for c in range(nc):
            assert np.max(np.abs(got[c] - ref_alm[c])) < 1e-12 * max(1.0, float(np.max(np.abs(ref_alm[c]))))
    plan.close()


@pytest.mark.parametrize("nphi,force_global", [(45, 0), (71, 0), (134, 0), (154, 0), (72, 1), (50, 1)])
def test_general_ring_lengths(nphi, force_global, monkeypatch):
    """Ring lengths outside the 2/3/5-smooth even case, which libsharp2 (pocketfft) accepts just the same: odd nphi (complex FFT
    of the real ring, no Nyquist mode), prime factors above the in-register radices (71 odd, 134 = 2 x 67: direct pass), a
    generic small odd radix (154 = 2 x 7 x 11), and -- forced here on small rings -- the global-memory work buffers that rings
    too long for shared memory use.  Checked against the oracle in both directions, spin 0 and spin 2, partial width included."""
    import math
    if force_global:
        monkeypatch.setenv("PIXSHT_FFT_GLOBAL", "1")
    ny = 19
    shape, wcs = fullsky_geometry((2 * math.pi / nphi, math.pi / (ny - 1)))
    assert shape == (nphi, ny)
    band = pixsht.sht_band(shape, wcs)
    lmax = 18 if nphi > 45 else 30          # 30 > 45/2: aliased m on the odd ring as well
    plan = Plan(band, lmax)
    for spin, nc in ((0, 1), (2, 2)):
        alms = [synth_alm(lmax, lmax, 21 + c, spin2=spin == 2) for c in range(nc)]
        maps = plan.alm2map(alms)
        ref = oracle_alm2map(np.stack(alms), shape, wcs, lmax, spin=spin)
        for c in range(nc):
            assert rel_rms(maps[c], ref[:, :, c]) < 1e-12
        rng = np.random.default_rng(nphi)
        x = [np.asfortranarray(rng.standard_normal(shape)) for _ in range(nc)]
        got = plan.map2alm(x)
        xm = Enmap(x[0], wcs) if nc == 1 else Enmap(np.asfortranarray(np.stack(x, axis=2)), wcs)
        ref_alm = oracle_map2alm(xm, lmax, spin=spin)
        for c in range(nc):
            assert rel_rms(got[c], ref_alm[c]) < 1e-12
    plan.close()
    # a band narrower than the ring (zero padding) on the same grid
    m = Enmap(gen_spin0(shape), wcs)
    sub = m[2:-3, 3:-2]
    assert rel_rms(map2alm(sub, lmax=lmax).alm, oracle_map2alm(sub, lmax)[0]) < 1e-12


def test_long_ring_f64_uses_global_work_buffers():
    """A 0.5' Float64 ring (nphi = 43200: 21600 complex samples = 346 KB) does not fit the 227 KB of shared memory; the FFT
    kernels then keep the ring in per-CTA global-memory work buffers.  19 rings (10 degree steps in declination) keep the
    check cheap; IQU, both directions, against the oracle."""
    shape, wcs = fullsky_geometry((0.5 * pixsht.arcminute, 10.0 * degree))
    assert shape == (43200, 19)
    lmax = 18
    band = pixsht.sht_band(shape, wcs)
    plan = Plan(band, lmax)
    for spin, nc in ((0, 1), (2, 2)):
        alms = [synth_alm(lmax, lmax, 31 + c, spin2=spin == 2) for c in range(nc)]
        maps = plan.alm2map(alms)
        ref = oracle_alm2map(np.stack(alms), shape, wcs, lmax, spin=spin, kind="d")
        for c in range(nc):
            assert rel_rms(maps[c], ref[:, :, c]) < 1e-12
        rng = np.random.default_rng(12)
        x = [np.asfortranarray(rng.standard_normal(shape)) for _ in range(nc)]
        got = plan.map2alm(x)
        xm = Enmap(x[0], wcs) if nc == 1 else Enmap(np.asfortranarray(np.stack(x, axis=2)), wcs)
        ref_alm = oracle_map2alm(xm, lmax, spin=spin, kind="d")
        for c in range(nc):
            assert rel_rms(got[c], ref_alm[c]) < 1e-12
    plan.close()


def test_small_plan_does_not_break_a_large_one():
    """A plan whose ring needs the large shared-memory opt-in (nphi = 10800: 106 KB) keeps working after a small plan was
    created and used: the opt-in is a per-kernel attribute of the process, not of the plan."""
    shape_big, wcs_big = fullsky_geometry((2.0 * arcminute, 10.0 * degree))
    assert shape_big == (10800, 19)
    lmax = 18
    big = Plan(pixsht.sht_band(shape_big, wcs_big), lmax)
    alm = synth_alm(lmax, lmax, 77)
    ref = oracle_alm2map(alm[None], shape_big, wcs_big, lmax, kind="d")[:, :, 0]
    assert rel_rms(big.alm2map([alm])[0], ref) < 1e-12
    shape_small, wcs_small = fullsky_geometry(10.0 * degree)
    small = Plan(pixsht.sht_band(shape_small, wcs_small), lmax)
    ref_small = oracle_alm2map(alm[None], shape_small, wcs_small, lmax)[:, :, 0]
    assert rel_rms(small.alm2map([alm])[0], ref_small) < 1e-12
    assert rel_rms(big.alm2map([alm])[0], ref) < 1e-12          # the large plan again, after the small one
    back = big.map2alm([np.asfortranarray(ref)])[0]
    assert rel_rms(back, oracle_map2alm(Enmap(np.asfortranarray(ref), wcs_big), lmax, kind="d")[0]) < 1e-12
    small.close(); big.close()


def test_edge_tiny_and_ragged_bands():
    """One-ring band, a band that contains only southern rings, a band one column wide (everything else of each ring is
    zero padding), and the two pole rings alone."""
    shape0, wcs0 = fullsky_geometry(10.0 * degree)
    full = Enmap(gen_spin0(shape0), wcs0)
    lmax = 18
    for sub in (full[:, 9:10], full[:, 0:4], full[17:18, :], full[3:30, 2:3], full[:, 18:19], full[:, 0:1]):
        got = map2alm(sub, lmax=lmax).alm
        ref = oracle_map2alm(sub, lmax)[0]
        assert np.max(np.abs(got - ref)) < 1e-12 * max(1.0, float(np.max(np.abs(ref))))
        alm = synth_alm(lmax, lmax, 3)
        back = alm2map(Alm(lmax, lmax, alm), sub.shape, sub.wcs)
        refm = oracle_alm2map(alm[None], sub.shape, sub.wcs, lmax)[:, :, 0]
        assert back.data.shape == sub.shape and np.max(np.abs(back.data - refm)) < 1e-12 * max(1.0, float(np.max(np.abs(refm))))


def test_argument_errors_are_reported_not_fatal():
    lib = get_lib()
    L = lib.lib
    h = ctypes.c_void_p()
    g = _lib.Geom(36, 19, 0, 19, 36, 1, 1, 0, 0.0)
    assert L.pixsht_plan_create(ctypes.byref(h), ctypes.byref(g), 10, 11, _lib.F64, 0) == _lib.ERR_ARG          # mmax > lmax
    assert b"mmax" in L.pixsht_last_error()
    assert L.pixsht_plan_create(ctypes.byref(h), ctypes.byref(g), 10, 10, 7, 0) == _lib.ERR_ARG                 # dtype
    bad = _lib.Geom(140000, 70001, 0, 2, 140000, 1, 1, 0, 0.0)
    assert L.pixsht_plan_create(ctypes.byref(h), ctypes.byref(bad), 10, 10, _lib.F64, 0) == _lib.ERR_UNSUPPORTED  # beyond the 16-bit FFT index tables
    assert b"too long" in L.pixsht_last_error()
    bad = _lib.Geom(36, 19, 5, 19, 36, 1, 1, 0, 0.0)
    assert L.pixsht_plan_create(ctypes.byref(h), ctypes.byref(bad), 10, 10, _lib.F64, 0) == _lib.ERR_ARG         # band sticks out of the sphere
    bad = _lib.Geom(36, 19, 0, 19, 40, 1, 1, 0, 0.0)
    assert L.pixsht_plan_create(ctypes.byref(h), ctypes.byref(bad), 10, 10, _lib.F64, 0) == _lib.ERR_ARG         # map wider than a ring
    assert L.pixsht_plan_create(ctypes.byref(h), ctypes.byref(g), 10, 10, _lib.F64, 99) == _lib.ERR_ARG          # device index
    assert L.pixsht_execute(None, 0, 1, None, None, 0) == _lib.ERR_ARG
    p = Plan(pixsht.sht_band((36, 19), fullsky_geometry(10.0 * degree)[1]), 10)
    one = (ctypes.c_void_p * 1)(0)
    assert L.pixsht_execute(p.handle, 0, 1, one, one, 0) == _lib.ERR_ARG                                            # null component pointer
    assert L.pixsht_execute(p.handle, 5, 1, one, one, 0) == _lib.ERR_ARG                                            # direction
    with pytest.raises(ValueError):
        p.alm2map([np.zeros(3, dtype=np.complex128)])                                                              # wrong alm length
    with pytest.raises(ValueError):
        p.map2alm([np.zeros((5, 5))])                                                                              # wrong map shape
    p.close()


def test_alm2cl_on_device_matches_host_mirror():
    """pixsht_alm2cl (SURVEY.md 8f rank 2: the first consumer of the alm) against the numpy mirror of Healpix.alm2cl."""
    lib = get_lib()
    for lmax, mmax in ((0, 0), (7, 7), (40, 25), (300, 300)):
        a = Alm(lmax, mmax, synth_alm(lmax, mmax, 1)); b = Alm(lmax, mmax, synth_alm(lmax, mmax, 2))
        for x, y in ((a, None), (a, b)):
            ref = pixsht.alm2cl(x, y)
            got = pixsht.alm2cl(x, y, lib=lib)
            assert np.max(np.abs(got - ref)) < 1e-13 * max(1.0, float(np.max(np.abs(ref))))


def test_fejer1_rings():
    """Fejer-1 ring grid (named by north_star; the reference declares CarFejer1 but has no SHT path for it, SURVEY.md F8, so
    PARITY IS UNPINNED here: the check is against the oracle run on the same colatitudes and weights, plus the exactness of
    the rule -- a band-limited round trip is the identity while 2 lmax < nrings)."""
    from pixsht import CarFejer1
    from helpers import fejer1_geometry
    shape, wcs = fullsky_geometry(5.0 * degree, W=CarFejer1)
    assert shape == (72, 36)
    band = pixsht.sht_band(shape, wcs)
    assert (band.nphi, band.nrings_total, band.ring_first, band.nrings, band.ring_scheme) == (72, 36, 0, 36, 1)
    lmax = 17                                    # 2 lmax = 34 < 36: exact quadrature
    plan = Plan(band, lmax)
    w_dev, th_dev = plan.weights()
    theta, w = fejer1_geometry(36, 72)
    assert np.max(np.abs(th_dev - theta)) < 1e-15 and np.max(np.abs(w_dev - w) / w) < 1e-13
    assert abs(np.sum(w_dev) * 72 - 4 * np.pi) < 1e-12
    orc = get_oracle("ld")
    for spin, nc in ((0, 1), (2, 2)):
        alms = [synth_alm(lmax, lmax, 60 + c, spin2=spin == 2) for c in range(nc)]
        maps = plan.alm2map(alms)
        ref = orc.alm2map(np.stack(alms), theta, band.phi0, 72, lmax, spin=spin)       # (nc, ring, phi), band orientation
        for c in range(nc):
            got = maps[c][::-1, ::-1].T if (band.flipx and band.flipy) else maps[c].T
            assert rel_rms(got, ref[c]) < 1e-12
        back = plan.map2alm(maps)
        for c in range(nc):
            assert rel_rms(back[c], alms[c]) < 1e-12                                   # exact round trip
    plan.close()
    # a partial band of the Fejer grid through the Enmap front end
    m = Enmap(gen_spin0(shape), wcs)
    sub = m[3:-5, 4:-6]
    bs = pixsht.sht_band(sub.shape, sub.wcs)
    assert bs.ring_scheme == 1 and bs.nrings == 26 and bs.nx == 64
    th_b, w_b = fejer1_geometry(36, 72, bs.ring_first, bs.nrings)
    bandcopy = np.zeros((bs.nrings, 72))
    src = sub.data[::-1, :] if bs.flipx else sub.data
    src = src[:, ::-1] if bs.flipy else src
    bandcopy[:, :bs.nx] = src.T
    ref_alm = orc.map2alm(bandcopy[None], th_b, w_b, bs.phi0, 30, spin=0)[0]
    assert rel_rms(map2alm(sub, lmax=30).alm, ref_alm) < 1e-12


@pytest.mark.parametrize("nbatch,dtype,location", [pytest.param(7, np.float64, "host", id="7-float64"), pytest.param(4, np.float64, "host", id="4-float64"),
                                                   pytest.param(3, np.float32, "host", id="3-float32")] +
                         [pytest.param(n, dt, loc, id="%s-%d-%s" % (loc, n, np.dtype(dt).name)) for loc in ("host", "device")
                          for n, dt in ((1, np.float64), (3, np.float64), (6, np.float32), (9, np.float64))])
def test_batched_spin0_equals_single_transforms(nbatch, dtype, location, res_deg=1.0, lmax=180):
    """pixsht_execute_batch (groups of 4 / 2 / 1 maps on one recurrence) against the single-map path: synthesis bit for bit
    (each ring's sum over l is the same sequence of FMAs), analysis to rounding (the cross-lane reduction is grouped differently).
    Batches of 1, 3, 6 and 9 split into groups 1, 2 + 1, 4 + 2 and 4 + 4 + 1: every group size, alone and after another group.
    location="device": the same batch on device pointers (outputs start as NaN, so a map or alm left unwritten shows)."""
    shape, wcs = fullsky_geometry(res_deg * degree)
    band = pixsht.sht_band(shape, wcs)
    plan = Plan(band, lmax, dtype=dtype)
    alms = [synth_alm(lmax, lmax, 300 + b).astype(plan.cdtype) for b in range(nbatch)]
    rng = np.random.default_rng(8)
    xs = [np.asfortranarray(rng.standard_normal(shape).astype(dtype)) for _ in range(nbatch)]
    if location == "host":
        maps = plan.alm2map_batch(alms)
        back = plan.map2alm_batch(xs)
    else:
        import torch
        d_alm = [torch.from_numpy(a).cuda() for a in alms]
        d_map = [torch.full((band.nx * band.nrings,), float("nan"), dtype=getattr(torch, np.dtype(dtype).name), device="cuda") for _ in alms]
        plan.execute_batch_ptrs(_lib.ALM2MAP, [a.data_ptr() for a in d_alm], [m.data_ptr() for m in d_map], _lib.DEVICE)
        maps = [m.cpu().numpy().reshape(band.nrings, band.nx).T for m in d_map]
        d_x = [torch.from_numpy(np.ravel(x, order="F")).cuda() for x in xs]
        d_out = [torch.full((plan.nalm,), complex("nan+nanj"), dtype=getattr(torch, plan.cdtype.name), device="cuda") for _ in xs]
        plan.execute_batch_ptrs(_lib.MAP2ALM, [a.data_ptr() for a in d_out], [m.data_ptr() for m in d_x], _lib.DEVICE)
        back = [a.cpu().numpy() for a in d_out]
        assert all(np.array_equal(d.cpu().numpy(), np.ravel(x, order="F")) for d, x in zip(d_x, xs))     # inputs untouched
    tol = 1e-13 if dtype == np.float64 else 2e-6
    for b in range(nbatch):
        single = plan.alm2map([alms[b]])[0]
        if dtype == np.float64:
            assert np.array_equal(maps[b], single)
        else:
            assert rel_rms(maps[b], single) < tol
    for b in range(nbatch):
        assert rel_rms(back[b], plan.map2alm([xs[b]])[0]) < tol
    if dtype == np.float64:
        ref = oracle_map2alm(Enmap(xs[-1].astype(np.float64), wcs), lmax)[0]
        assert rel_rms(back[-1], ref) < TOL64
    plan.close()


# ---- SURVEY.md 8(f) rows 3 and 4: the U-sign convention in the kernels, pixel-area ring weights -------------------------------
@pytest.mark.parametrize("nshard", [1, 3])
def test_polconv_iau(nshard, res_deg=1.0, lmax=120):
    """pixsht_plan_set_polconv(IAU): the caller's U has the IAU sign (src/enmap.jl:178-196 flips it on the host at read time; here
    the FFT kernels' row I/O does).  map2alm of (T, Q, -U) under IAU == map2alm of (T, Q, U), bit for bit; alm2map under IAU
    returns -U; host and device pointers, single- and multi-GPU plans, QU alone; batches are untouched by the flag."""
    import torch
    shape, wcs = fullsky_geometry(res_deg * degree)
    band = pixsht.sht_band(shape, wcs)
    plan = Plan(band, lmax) if nshard == 1 else Plan(band, lmax, devices=_shard_devices(nshard))
    alms = [synth_alm(lmax, lmax, 900 + c, spin2=c > 0) for c in range(3)]
    plan.set_polconv("COSMO")
    ref = plan.alm2map(alms)
    back_ref = plan.map2alm(ref)
    plan.set_polconv("IAU")
    got = plan.alm2map(alms)
    assert np.array_equal(got[0], ref[0]) and np.array_equal(got[1], ref[1]) and np.array_equal(got[2], -ref[2])
    back = plan.map2alm(got)
    for a, b in zip(back, back_ref):
        assert rel_rms(a, b) < 1e-13          # the same sums; analysis accumulates atomically, so only to rounding
    qu = plan.alm2map(alms[1:])
    assert np.array_equal(qu[0], ref[1]) and np.array_equal(qu[1], -ref[2])
    t = plan.alm2map(alms[:1])
    assert np.array_equal(t[0], ref[0])       # a single component is never U
    if nshard == 1:
        d_alm = [torch.from_numpy(a).cuda() for a in alms]
        d_map = [torch.empty(band.nx * band.nrings, dtype=torch.float64, device="cuda") for _ in range(3)]
        plan.execute_ptrs(_lib.ALM2MAP, [a.data_ptr() for a in d_alm], [m.data_ptr() for m in d_map], _lib.DEVICE)
        assert np.array_equal(d_map[2].cpu().numpy().reshape(band.nrings, band.nx).T, -ref[2])
        bm = plan.alm2map_batch([alms[0], alms[0]])
        assert np.array_equal(bm[1], ref[0])
    plan.set_polconv("COSMO")
    assert np.array_equal(plan.alm2map(alms)[2], ref[2])
    with pytest.raises(PixshtError):
        get_lib().check(get_lib().lib.pixsht_plan_set_polconv(plan.handle, 7))
    plan.close()
    # the Enmap front end: tag left by read_map(..., defer_polcconv=True), and the explicit keyword
    if nshard == 1:
        m = Enmap(np.asfortranarray(np.dstack([ref[0], ref[1], -ref[2]])), wcs)
        a_kw = map2alm(m, lmax=lmax, polcconv="IAU")
        m.polcconv = "IAU"
        a_tag = map2alm(m, lmax=lmax)
        a_ref = map2alm(Enmap(np.asfortranarray(np.dstack(ref)), wcs), lmax=lmax)
        for x, y, z in zip(a_kw, a_tag, a_ref):
            assert rel_rms(x.alm, z.alm) < 1e-13 and rel_rms(y.alm, z.alm) < 1e-13


def test_pixel_area_weights_as_ring_weights(res_deg=2.0, lmax=60):
    """pixareamap weights (src/projections/car_proj.jl:265-273, src/enmap_ops.jl:124-138) from pixsht_ring_pixarea, used as the ring
    weights of a plan (pixsht_plan_create_rings): the pixel-area-weighted analysis, against the oracle with the same weights."""
    from pixsht.transforms import ring_pixarea, pixareamap
    shape, wcs = fullsky_geometry(res_deg * degree)
    band = pixsht.sht_band(shape, wcs)
    area = ring_pixarea(shape, wcs)                      # map row order
    assert abs(np.sum(area) * shape[0] - 4 * np.pi) < 1e-12
    assert np.array_equal(pixareamap(shape, wcs).data[5, :], area)
    area_band = area[::-1] if band.flipy else area       # ascending colatitude, as the plan wants them
    theta, wcc = cc_geometry(band.nrings_total, band.nphi)
    lib = get_lib()
    h = ctypes.c_void_p()
    dp = ctypes.POINTER(ctypes.c_double)
    th = np.ascontiguousarray(theta); wa = np.ascontiguousarray(area_band)
    lib.check(lib.lib.pixsht_plan_create_rings(ctypes.byref(h), band.nrings, th.ctypes.data_as(dp), wa.ctypes.data_as(dp), band.nphi, band.phi0,
                                               lmax, lmax, _lib.F64, 0))
    rng = np.random.default_rng(17)
    ring_major = np.ascontiguousarray(rng.standard_normal((band.nrings, band.nphi)))     # rings ascending in theta, no flips
    out = np.zeros(nalm(lmax, lmax), dtype=np.complex128)
    lib.check(lib.lib.pixsht_execute(h, _lib.MAP2ALM, 1, (ctypes.c_void_p * 1)(out.ctypes.data), (ctypes.c_void_p * 1)(ring_major.ctypes.data), _lib.HOST))
    lib.lib.pixsht_plan_destroy(h)
    ref = get_oracle("ld").map2alm(ring_major[None], theta, area_band, band.phi0, lmax, spin=0)[0]
    assert rel_rms(out, ref) < TOL64
    # and it is a different (lower-order) quadrature than Clenshaw-Curtis: close, not equal
    ref_cc = get_oracle("ld").map2alm(ring_major[None], theta, wcc, band.phi0, lmax, spin=0)[0]
    assert 1e-6 < rel_rms(out, ref_cc) < 0.2


def test_device_views_at_odd_element_offsets(res_deg=2.0, lmax=60):
    """Device pointers that start at an odd element offset (a torch / CUDA.jl view): the FFT kernels' two-element row accesses need
    pair alignment, so such launches take the element-wise path instead of faulting (ADVICE r01: misaligned-address is sticky)."""
    import torch
    shape, wcs = fullsky_geometry(res_deg * degree)
    band = pixsht.sht_band(shape, wcs)
    for dt, tdt, cdt in ((np.float64, torch.float64, np.complex128), (np.float32, torch.float32, np.complex64)):
        plan = Plan(band, lmax, dtype=dt)
        alm = synth_alm(lmax, lmax, 41).astype(cdt)
        ref = plan.alm2map([alm])[0]
        npix = band.nx * band.nrings
        buf = torch.zeros(npix + 3, dtype=tdt, device="cuda")
        d_alm = torch.from_numpy(alm).cuda()
        for off in (1, 3):
            view = buf[off:off + npix]
            plan.execute_ptrs(_lib.ALM2MAP, [d_alm.data_ptr()], [view.data_ptr()], _lib.DEVICE)
            assert np.array_equal(view.cpu().numpy().reshape(band.nrings, band.nx).T, ref)
            out = torch.zeros_like(d_alm)
            plan.execute_ptrs(_lib.MAP2ALM, [out.data_ptr()], [view.data_ptr()], _lib.DEVICE)
            assert rel_rms(out.cpu().numpy(), plan.map2alm([ref])[0]) < (1e-13 if dt == np.float64 else 1e-6)
        plan.close()
