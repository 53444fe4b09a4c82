"""Kernel-logic tests on the HOST EMULATION build of the CUDA sources (tests/emu/): same .cu/.cuh files compiled
with g++ and tests/emu/cuda_emu.h, one OS thread per CUDA thread.  CPU only.  This checks indexing, parity
bookkeeping, the seek/rescale state machine and the FFT passes before GPU time is spent; the real parity tests
(-m gpu) run the nvcc build on a B200.  The product never loads the emulation library."""
import os
import subprocess

import numpy as np
import pytest

import pixsht
from pixsht import Enmap, CarClenshawCurtis, fullsky_geometry, geometry, degree
from pixsht.transforms import PixshtLib, map2alm, alm2map, Plan
from helpers import (golden_alm, gen_spin0, gen_spin2, oracle_map2alm, oracle_alm2map, rel_rms, synth_alm)
from oracle import cc_geometry

HERE = os.path.dirname(os.path.abspath(__file__))
EMU_SO = os.path.join(HERE, "emu", "_build", "libpixsht_emu.so")


@pytest.fixture(scope="module")
def emu():
    srcs = [os.path.join(HERE, "..", "pixell.jl_b200", "csrc", f) for f in os.listdir(os.path.join(HERE, "..", "pixell.jl_b200", "csrc"))]
    srcs.append(os.path.join(HERE, "emu", "cuda_emu.h"))
    if not os.path.exists(EMU_SO) or any(os.path.getmtime(s) > os.path.getmtime(EMU_SO) for s in srcs):
        subprocess.check_call(["bash", os.path.join(HERE, "emu", "build_emu.sh")])
    lib = PixshtLib(EMU_SO)
    assert "EMULATION" in lib.version()
    return lib


def relmax(a, b):
    return float(np.max(np.abs(a - b)) / np.max(np.abs(b)))


def test_emu_weights_match_oracle(emu):
    shape, wcs = fullsky_geometry(5.0 * degree)
    p = Plan(pixsht.sht_band(shape, wcs), 20, lib=emu)
    w, th = p.weights()
    theta, wref = cc_geometry(37, 72)
    assert np.max(np.abs(w - wref) / wref) < 1e-12
    assert np.max(np.abs(th - theta)) < 1e-15
    p.close()


def test_emu_golden_spin0(emu):
    shape, wcs = fullsky_geometry(10.0 * degree)
    m = Enmap(gen_spin0(shape), wcs)
    alm = map2alm(m, lmax=18, lib=emu)
    assert relmax(alm.alm, golden_alm("simple_analytic_sht")) < 1e-12
    sub = m[5:-2, 4:-3]
    alm = map2alm(sub, lmax=18, lib=emu)
    assert relmax(alm.alm, golden_alm("simple_analytic_sht_sliced")) < 1e-12


def test_emu_golden_spin2_and_iqu(emu):
    shape, wcs = fullsky_geometry(10.0 * degree, dims=(3,))
    d = np.zeros(shape, order="F")
    d[:, :, 0] = gen_spin0(shape)
    d[:, :, 1:] = gen_spin2(shape)
    t, e, b = map2alm(Enmap(d, wcs), lmax=108, lib=emu)
    assert relmax(t.alm, golden_alm("simple_analytic_sht_fullalm")) < 1e-12
    assert relmax(e.alm, golden_alm("simple_pol_analytic_sht", (0, 1))) < 1e-12
    assert relmax(b.alm, golden_alm("simple_pol_analytic_sht", (2, 3))) < 1e-12


@pytest.mark.parametrize("spin", [0, 2])
def test_emu_alm2map_vs_oracle(emu, spin):
    shape, wcs = fullsky_geometry(5.0 * degree)  # 72 x 37
    lmax = 36
    nc = 1 if spin == 0 else 2
    alms = [synth_alm(lmax, lmax, 40 + c, spin2=spin == 2) for c in range(nc)]
    ref = oracle_alm2map(np.stack(alms), shape, wcs, lmax, spin=spin)
    out = alm2map([pixsht.Alm(lmax, lmax, a) for a in alms] if nc > 1 else pixsht.Alm(lmax, lmax, alms[0]), shape, wcs, lib=emu)
    out = [out] if nc == 1 else out
    for c in range(nc):
        assert rel_rms(out[c].data, ref[:, :, c]) < 1e-12


# ---- the small GPU parity cases, replayed on the emulation build (logic check of the test bodies and the kernels) ----
@pytest.fixture()
def emu_default(emu, monkeypatch):
    from pixsht import _lib, transforms
    monkeypatch.setattr(_lib, "_DEFAULT", emu)
    transforms._PLANS.clear()
    yield emu
    transforms._PLANS.clear()


def test_emu_replay_golden_cases(emu_default):
    import test_gpu_parity as g
    g.test_golden_spin0_fullsky_sliced_box()
    g.test_golden_spin2_stack_tuple_iqu()
    g.test_bad_ncomp_is_an_error_not_a_crash()


def test_emu_replay_partial_sky_and_flips(emu_default):
    import test_gpu_parity as g
    g.test_partial_sky_band_and_unflipped_geometry()


def test_emu_replay_sharp_shim(emu_default):
    import test_gpu_parity as g
    g.test_sharp_shim_runs_the_reference_call_sequence()


def test_emu_c1_config(emu_default):
    import test_gpu_parity as g
    g.test_c1_spin0_f64_both_directions_and_roundtrip()


def test_emu_replay_edge_cases(emu_default):
    import test_gpu_parity as g
    for lmax, mmax in ((0, 0), (1, 0), (18, 3)):     # the GPU suite runs the full list
        g.test_edge_band_limits(lmax, mmax)
    g.test_edge_tiny_and_ragged_bands()
    g.test_argument_errors_are_reported_not_fatal()
    g.test_alm2cl_on_device_matches_host_mirror()
    g.test_fejer1_rings()


def test_emu_replay_batched(emu_default):
    import test_gpu_parity as g
    import numpy as np
    g.test_batched_spin0_equals_single_transforms(6, np.float64, "host", res_deg=10.0, lmax=14)      # groups of 4 + 2
    g.test_batched_spin0_equals_single_transforms(3, np.float32, "host", res_deg=10.0, lmax=14)      # groups of 2 + 1


def test_emu_replay_multi_gpu_plan(emu_default, monkeypatch):
    """The one-process multi-GPU plan (pixsht_plan_create_multi) on the emulation build: partition, per-m address table, slabs,
    per-family pipeline and the batch dealing, against the single plan and the oracle."""
    import test_gpu_parity as g
    monkeypatch.setenv("PIXSHT_MULTI_SEGS", "2")
    g.test_multi_gpu_plan_equals_single_gpu_plan(3, res_arcmin=600.0, lmax=18, reps=1)
    g.test_multi_gpu_plan_partial_sky_flips_and_oracle(res_deg=10.0, lmax=14, nshard=2)


@pytest.mark.parametrize("nphi,force_global", [(45, 0), (71, 0), (134, 0), (72, 1)])
def test_emu_replay_general_ring_lengths(emu_default, monkeypatch, nphi, force_global):
    import test_gpu_parity as g
    g.test_general_ring_lengths(nphi, force_global, monkeypatch)


@pytest.mark.parametrize("nc,dt", [(2, np.float64), (3, np.float64), (3, np.float32)])
def test_emu_host_path_two_part_polarisation_analysis(emu_default, monkeypatch, nc, dt):
    """map2alm through host pointers sends the polarisation maps in two parts (equatorial rings, then polar rings) and
    analyses the first part while the second arrives; needs >= 2 ring-pair chunks, hence one pair per lane here."""
    monkeypatch.setenv("PIXSHT_R2A", "1")
    monkeypatch.setenv("PIXSHT_R0A", "1")
    shape, wcs = fullsky_geometry(2.5 * degree, dims=(nc,))     # 144 x 73: 37 ring pairs = 2 chunks of 32
    rng = np.random.default_rng(3)
    m64 = Enmap(np.asfortranarray(rng.standard_normal(shape).astype(dt).astype(np.float64)), wcs)
    m = Enmap(np.asfortranarray(m64.data, dtype=dt), wcs)
    lmax = 40
    got = map2alm(m, lmax=lmax, lib=emu_default)
    m = m64
    if nc == 3:
        ref = np.concatenate([oracle_map2alm(Enmap(np.asfortranarray(m.data[:, :, 0]), wcs), lmax, kind="d"),
                              oracle_map2alm(Enmap(np.asfortranarray(m.data[:, :, 1:]), wcs), lmax, spin=2, kind="d")])
    else:
        ref = oracle_map2alm(m, lmax, spin=2, kind="d")
    for c in range(nc):
        assert rel_rms(got[c].alm, ref[c]) < (1e-12 if dt == np.float64 else 1e-6)


@pytest.mark.parametrize("dt", [np.float64, np.float32])
def test_emu_host_path_single_map_two_phase_pipelines(emu_default, monkeypatch, dt):
    """A single spin-0 map through host pointers on a plan with many ring-pair chunks: alm2map synthesises its last m piece in ring
    ranges whose rows leave one by one, map2alm analyses its last (polar) ring piece in m ranges whose alm columns leave one by one
    (pixsht.cu, execute_host: tonly_rings / tonly_m).  One pair per lane and a lowered threshold make a 0.5 degree grid qualify."""
    monkeypatch.setenv("PIXSHT_R0", "1"); monkeypatch.setenv("PIXSHT_R0A", "1")
    monkeypatch.setenv("PIXSHT_TONLY_MINCHUNKS", "4")
    shape, wcs = fullsky_geometry(0.5 * degree)          # 720 x 361: 181 ring pairs = 6 chunks of 32
    lmax = 100
    tol = 1e-12 if dt == np.float64 else 2e-6
    alm = synth_alm(lmax, lmax, 611)
    plan = Plan(pixsht.sht_band(shape, wcs), lmax, dtype=dt, lib=emu_default)
    mp = plan.alm2map([alm.astype(plan.cdtype)])[0]
    ref = oracle_alm2map(alm[None], shape, wcs, lmax, kind="d")[:, :, 0]
    assert rel_rms(mp, ref) < tol
    x = np.asfortranarray(np.random.default_rng(612).standard_normal(shape).astype(dt))
    got = plan.map2alm([x])[0]
    assert rel_rms(got, oracle_map2alm(Enmap(np.asfortranarray(x, dtype=np.float64), wcs), lmax, kind="d")[0]) < tol
    plan.close()
    if dt == np.float32:
        return
    # a cut-sky band (single rings without a mirror partner in the chunks) and mmax < lmax
    full = Enmap(gen_spin0(shape, 1.5), wcs)
    sub = full[:, 30:290]
    plan = Plan(pixsht.sht_band(sub.data.shape, sub.wcs), 120, 80, dtype=dt, lib=emu_default)
    got = plan.map2alm([np.asfortranarray(sub.data, dtype=dt)])[0]
    assert rel_rms(got, oracle_map2alm(sub, 120, mmax=80)[0]) < tol
    a = synth_alm(120, 80, 613)
    assert rel_rms(plan.alm2map([a.astype(plan.cdtype)])[0], oracle_alm2map(a[None], sub.data.shape, sub.wcs, 120, mmax=80)[:, :, 0]) < tol
    plan.close()


def test_emu_ring_length_sweep(emu):
    """Ring FFT on lengths with every kind of factorisation (two samples, odd primes, squares of generic radices, powers of
    two, a prime above the in-register radices): map2alm / alm2map of a 5-ring grid against the oracle.  The full sweep
    nphi = 2..199 was run once with this body (all within 1e-12)."""
    import math
    for nphi in (2, 3, 5, 6, 9, 14, 49, 121, 128, 130, 169, 194):
        shape, wcs = fullsky_geometry((2 * math.pi / nphi, math.pi / 4))
        band = pixsht.sht_band(shape, wcs)
        lmax = 4
        plan = Plan(band, lmax, lib=emu)
        alm = synth_alm(lmax, lmax, nphi)
        ref = oracle_alm2map(alm[None], shape, wcs, lmax, kind="d")[:, :, 0]
        assert rel_rms(plan.alm2map([alm])[0], ref) < 1e-12, nphi
        x = np.asfortranarray(np.random.default_rng(nphi).standard_normal(shape))
        assert rel_rms(plan.map2alm([x])[0], oracle_map2alm(Enmap(x, wcs), lmax, kind="d")[0]) < 1e-12, nphi
        plan.close()


def test_emu_edge_fused_fft(emu, monkeypatch):
    """The edge-fused ring-FFT kernels (fft_edge.cuh: last pass on butterfly pairs in the phase-row I/O, first super-pass in the
    map-row I/O) on ring lengths with every shape of plan: two super-passes only, single and paired first super-pass, even and
    odd sub-length of the last pass (with / without the self-mirrored butterfly kk = L/2), every last radix 2..5; band limit at,
    just below and far below the Nyquist mode of the ring; against the oracle and against the plain kernels (PIXSHT_FFT_EDGE=0)."""
    import math
    for nphi, lmaxs, both in ((12, (6, 5), True), (16, (8,), False), (20, (10, 9), False), (50, (25,), True), (54, (27,), False),
                              (60, (29,), True), (100, (50,), False), (360, (180,), True)):
        shape, wcs = fullsky_geometry((2 * math.pi / nphi, math.pi / 4))
        band = pixsht.sht_band(shape, wcs)
        for lmax in lmaxs:
            res = {}
            alm = synth_alm(lmax, lmax, nphi)
            x = np.asfortranarray(np.random.default_rng(nphi).standard_normal(shape))
            for edge in (("2", "0") if both else ("2",)):    # 2: also for rings below the 32 KB threshold of the default
                monkeypatch.setenv("PIXSHT_FFT_EDGE", edge)
                plan = Plan(band, lmax, lib=emu)
                assert plan.info()["fft"]["edge_fused"] == (edge == "2"), (nphi, lmax, plan.info())
                res[edge] = (plan.alm2map([alm])[0], plan.map2alm([x])[0])
                plan.close()
            ref = oracle_alm2map(alm[None], shape, wcs, lmax, kind="d")[:, :, 0]
            assert rel_rms(res["2"][0], ref) < 1e-12, (nphi, lmax)
            assert rel_rms(res["2"][1], oracle_map2alm(Enmap(x, wcs), lmax, kind="d")[0]) < 1e-12, (nphi, lmax)
            if both:
                assert rel_rms(res["2"][0], res["0"][0]) < 1e-14 and rel_rms(res["2"][1], res["0"][1]) < 1e-14, (nphi, lmax)
    monkeypatch.setenv("PIXSHT_FFT_EDGE", "1")
    shape, wcs = fullsky_geometry((2 * math.pi / 360, math.pi / 4))
    plan = Plan(pixsht.sht_band(shape, wcs), 100, lib=emu)
    assert not plan.info()["fft"]["edge_fused"]      # default: small rings keep the plain kernels
    plan.close()
    monkeypatch.setenv("PIXSHT_FFT_EDGE", "2")
    # lmax beyond the ring's Nyquist mode (aliasing): stays with the plain kernels
    shape, wcs = fullsky_geometry((2 * math.pi / 24, math.pi / 40))
    plan = Plan(pixsht.sht_band(shape, wcs), 30, lib=emu)
    assert not plan.info()["fft"]["edge_fused"]
    plan.close()
    # Float32 boundary, IQU, a cut-sky flipped band (element-wise row access, zero padding), Fejer-1 rings with a phi0 rotation
    shape, wcs = fullsky_geometry(4.0 * degree, dims=(3,))
    lmax = 40
    alms = [synth_alm(lmax, lmax, 40 + c, spin2=c > 0) for c in range(3)]
    ref = np.concatenate([oracle_alm2map(alms[0][None], shape, wcs, lmax), oracle_alm2map(np.stack(alms[1:]), shape, wcs, lmax, spin=2)], axis=2)
    for dt, tol in ((np.float64, 1e-12), (np.float32, 2e-6)):
        plan = Plan(pixsht.sht_band(shape[:2], wcs), lmax, dtype=dt, lib=emu)
        assert plan.info()["fft"]["edge_fused"]
        mp = plan.alm2map(alms)
        assert max(rel_rms(mp[c], ref[:, :, c]) for c in range(3)) < tol
        out = plan.map2alm([np.asfortranarray(ref[:, :, c], dtype=dt) for c in range(3)])
        rt = oracle_map2alm(Enmap(ref[:, :, 0], wcs), lmax)[0]
        reb = oracle_map2alm(Enmap(ref[:, :, 1:], wcs), lmax, spin=2)
        assert max(rel_rms(out[0], rt), rel_rms(out[1], reb[0]), rel_rms(out[2], reb[1])) < tol
        plan.close()
    full = Enmap(gen_spin0(shape[:2], 1.5), wcs)
    for sub in (full[10:-7, 4:40], full[::-1, ::-1][3:85, 5:40]):
        got = map2alm(sub, lmax=30, lib=emu)
        assert rel_rms(got.alm, oracle_map2alm(sub, 30)[0]) < 1e-12
        back = alm2map(got, sub.data.shape, sub.wcs, lib=emu)
        assert rel_rms(back.data, oracle_alm2map(got.alm[None], sub.data.shape, sub.wcs, 30)[:, :, 0]) < 1e-12


def test_emu_two_step_spin0_kernels(emu, monkeypatch):
    """The two-step spin-0 kernels (legendre_2s.cuh) on the emulation build.  At test sizes every ring pair would fall into the
    chunks that stay with the standard kernels, so the ring tile is shrunk to one pair per lane (32 pairs per chunk): at 1 degree
    (91 pairs) chunk 1 then runs the two-step kernels, chunk 0 (within 3 degrees of the pole) and chunk 2 (|cos theta| < 0.05)
    the standard ones.  Checks: against the oracle, against the same plan with PIXSHT_TWOSTEP=0, an m-limited alm with the other
    parity at the top of the columns, a cut-sky band."""
    monkeypatch.setenv("PIXSHT_R0", "1"); monkeypatch.setenv("PIXSHT_R0A", "1")
    shape, wcs = fullsky_geometry(1.0 * degree)
    band = pixsht.sht_band(shape, wcs)
    lmax = 90
    alm = synth_alm(lmax, lmax, 300)
    res = {}
    for two in ("1", "0"):
        monkeypatch.setenv("PIXSHT_TWOSTEP", two)
        p = Plan(band, lmax, lib=emu)
        ex, nom = p.work(0)
        mp = p.alm2map([alm])[0]
        res[two] = (mp, p.map2alm([mp])[0], ex / nom)
        p.close()
    assert res["1"][2] < 0.97 * res["0"][2]                      # fewer FP64 operations are executed
    assert rel_rms(res["1"][0], oracle_alm2map(alm[None], shape, wcs, lmax)[:, :, 0]) < 1e-12
    assert rel_rms(res["1"][0], res["0"][0]) < 1e-13
    assert rel_rms(res["1"][1], res["0"][1]) < 1e-13
    assert rel_rms(res["1"][1], oracle_map2alm(Enmap(res["0"][0], wcs), lmax)[0]) < 1e-12
    monkeypatch.setenv("PIXSHT_TWOSTEP", "1")
    p = Plan(band, 77, 40, lib=emu)
    a = synth_alm(77, 40, 77)
    mp = p.alm2map([a])[0]
    assert rel_rms(mp, oracle_alm2map(a[None], shape, wcs, 77, mmax=40)[:, :, 0]) < 1e-12
    assert rel_rms(p.map2alm([mp])[0], oracle_map2alm(Enmap(mp, wcs), 77, mmax=40)[0]) < 1e-12
    p.close()
    # a cut-sky, flipped band: single rings without a mirror partner
    full = Enmap(gen_spin0(shape, 1.5), wcs)
    sub = full[40:-25, 12:150]
    got = map2alm(sub, lmax=60, lib=emu)
    assert rel_rms(got.alm, oracle_map2alm(sub, 60)[0]) < 1e-12
