"""The iterative map2alm (pixsht_map2alm_iter: a <- A m, then niter times a <- a + A (m - Y a), with A = map2alm and Y = alm2map,
the whole loop on the device) against what it must equal:

* the same loop built from device-pointer pixsht_execute calls on the same plan, the residual and the sum taken outside the
  library: every m column within a relative RMS of 1e-12 (Float64) or 1e-6 (Float32) -- the loop adds A r into a with the
  analysis kernels' own atomic adds, so only the order of additions differs (and, in Float32, the loop keeps a in Float64);
* the same loop on the CPU oracle, and the convergence the oracle shows on a grid where one analysis is not exact;
* niter = 0: pixsht_execute(MAP2ALM) bit for bit, through device and host pointers.

Every array handed to the library has guard elements on both sides, outputs start as NaN and inputs -- above all the maps, which
the loop must not use as scratch -- must come back unchanged (test_host_pipeline.Buffers).  Each checked call follows a scrub:
the same call on negated maps, which leaves the plan's residual maps, phase rows, staging and Float64 work alm holding wrong
contents.  GPU tests carry the gpu mark; the emulation replays at the end run reduced sets of the same bodies on the
host-emulation build (tests/emu/)."""
import numpy as np
import pytest

import pixsht
from pixsht import Enmap, fullsky_geometry, degree
from pixsht import _lib
from pixsht.transforms import Plan, PixshtError
from helpers import synth_alm, oracle_alm2map, oracle_map2alm
from oracle import cc_geometry
from test_host_pipeline import Buffers, _RingsPlan, _is_torch, _ptr, column_errors, run, A2M, M2A, F64, F32
from test_emu_kernels import emu, emu_default  # noqa: F401  (fixtures of the emulation replays)

COLUMN_TOL = {F64: 1e-12, F32: 1e-6}
ORACLE_TOL = {F64: 1e-10, F32: 1e-5}
COMPONENTS = ((0,), (1, 2), (0, 1, 2))
GPU_KINDS = ("device", "pageable", "pinned", "registered")
# relative error |a_k - a_true| / |a_true| after k iterations at 180 x 91, lmax 80 (DESIGN.md section 10), spin 0 and spin 2
CONVERGENCE = {0: (2.37e-3, 1.71e-4, 1.44e-5, 1.27e-6, 1.13e-7), 2: (3.39e-3, 3.08e-4, 2.93e-5, 2.85e-6, 2.82e-7)}


def run_iter(plan, maps, niter, kind):
    """One pixsht_map2alm_iter call on flat maps held in memory of `kind`.  Returns copies of the alm and the launch count; the
    checks of Buffers (guards, unchanged maps, every alm written) have passed."""
    bufs = Buffers(plan.lib)
    try:
        ins = [bufs.get(kind, x.size, x.dtype, x) for x in maps]
        outs = [bufs.get(kind, plan.nalm, plan.cdtype) for _ in maps]
        plan.map2alm_iter_ptrs([_ptr(a) for a in outs], [_ptr(m) for m in ins], niter, _lib.DEVICE if kind == "device" else _lib.HOST)
        launches = plan.info()["launches"]
        bufs.check()
        return [o.cpu().numpy() if _is_torch(o) else np.array(o) for o in outs], launches
    finally:
        bufs.close()


def scrub(plan, maps, niter):
    neg = [np.negative(x) for x in maps]
    outs = [np.empty(plan.nalm, plan.cdtype) for _ in maps]
    plan.map2alm_iter_ptrs([a.ctypes.data for a in outs], [m.ctypes.data for m in neg], niter, _lib.HOST)


def loop_from_parts(plan, maps, niter):
    """a_0 .. a_niter of the loop built from device-pointer pixsht_execute calls on `plan`, with r = m - s and a + A r taken in
    the plan's element types outside the library; and the launch counts of one map2alm and one alm2map call."""
    a, l_m2a = run(plan, M2A, maps, "device")
    out, l_a2m = [a], 0
    for _ in range(niter):
        s, l_a2m = run(plan, A2M, a, "device")
        d, _ = run(plan, M2A, [m - x for m, x in zip(maps, s)], "device")
        a = [x + y for x, y in zip(a, d)]
        out.append(a)
    return out, l_m2a, l_a2m


def random_maps(n, count, seed):
    """Maps of n pixels rounded through Float32, so that Float32 plans see exactly the Float64 values."""
    rng = np.random.default_rng(seed)
    return [rng.standard_normal(n).astype(np.float32).astype(np.float64) for _ in range(count)]


# ---- 1. the loop equals its parts --------------------------------------------------------------------------------------------
GEOMETRIES = ["flipped", "unflipped", "cut_sky", "mmax_below_lmax", "iau", "rings"]


def make_plans(case, res, lmax, dtypes):
    shape, wcs = fullsky_geometry(res)
    nx, ny = shape
    if case == "rings":       # pixsht_plan_create_rings: rings of the full-sky CC grid, nx = nphi, no flips (Float64 only)
        theta, w = cc_geometry(ny, nx)
        return [_RingsPlan(theta, w, nx, lmax)]
    full = Enmap(np.zeros(shape, order="F"), wcs)
    sub = {"unflipped": full[::-1, ::-1], "cut_sky": full[:, ny // 2 - (2 * ny) // 5:ny // 2 + ny // 10]}.get(case, full)
    band = pixsht.sht_band(sub.shape[:2], sub.wcs)
    assert band.flipy == (case != "unflipped")
    plans = []
    for dt in dtypes:
        plan = Plan(band, lmax, lmax // 2 if case == "mmax_below_lmax" else lmax, dtype=dt)
        if case == "iau":
            plan.set_polconv("IAU")
        plans.append(plan)
    return plans


def parts_case(case, res=1.0 * degree, lmax=150, dtypes=(F64, F32), components=None, niter=3, kinds=None):
    """For each plan and component set: the loop from its parts up to `niter`, then pixsht_map2alm_iter for niter = 1 .. `niter`
    in every memory kind, each after a scrub: every m column equals the parts, and the launch count is one map2alm, plus k times
    one alm2map and one map2alm, plus k residual launches, less the 2 k ncomp Float32 conversions the separate calls make and the
    loop does not (it converts once, at the end, like one map2alm)."""
    components = components or (((1, 2), (0, 1, 2)) if case == "iau" else COMPONENTS)
    for plan in make_plans(case, res, lmax, dtypes):
        kinds_ = kinds or (GPU_KINDS if case == "flipped" else ("device", "pageable"))
        npix = plan.band.nx * plan.band.nrings
        allmaps = random_maps(npix, 3, 9100)
        for comps in components:
            maps = [allmaps[c].astype(plan.dtype) for c in comps]
            ncomp = len(comps)
            scrub(plan, maps, niter)
            ref, l_m2a, l_a2m = loop_from_parts(plan, maps, niter)
            for k in range(1, niter + 1):
                expect = l_m2a + k * (l_a2m + l_m2a) + k - (2 * k * ncomp if plan.dtype == F32 else 0)
                for kind in kinds_:
                    scrub(plan, maps, k)
                    got, n = run_iter(plan, maps, k, kind)
                    assert n == expect, (case, plan.dtype, comps, k, kind, n, expect)
                    for c in range(ncomp):
                        err = column_errors(plan.lmax, plan.mmax, got[c], ref[k][c])
                        assert err.max() <= COLUMN_TOL[plan.dtype], \
                            "%s %s %s niter %d %s component %d: column m = %d off by %.2e" % (case, plan.dtype, comps, k, kind, c, int(err.argmax()), err.max())
        plan.close()


@pytest.mark.gpu
@pytest.mark.parametrize("case", GEOMETRIES)
def test_loop_equals_its_parts(case):
    parts_case(case)


# ---- 2. against the oracle ---------------------------------------------------------------------------------------------------
def oracle_loop(maps, shape, wcs, lmax, spin, niter):
    """The loop on the CPU oracle (double): maps is (nx, ny) for spin 0, (nx, ny, 2) for spin 2."""
    m = np.asfortranarray(maps)
    a = oracle_map2alm(Enmap(m, wcs), lmax, spin=spin, kind="d")
    for _ in range(niter):
        s = oracle_alm2map(a, shape, wcs, lmax, spin=spin, kind="d")
        a = a + oracle_map2alm(Enmap(np.asfortranarray(m - (s[:, :, 0] if spin == 0 else s)), wcs), lmax, spin=spin, kind="d")
    return a


def oracle_case(res=2.0 * degree, lmax=80, niter=3, dtypes=(F64, F32), components=COMPONENTS, kind="device"):
    shape, wcs = fullsky_geometry(res)
    allmaps = [x.reshape(shape, order="F") for x in random_maps(shape[0] * shape[1], 3, 9200)]
    ref = [oracle_loop(allmaps[0], shape, wcs, lmax, 0, niter)[0]] + list(oracle_loop(np.stack(allmaps[1:], axis=2), shape, wcs, lmax, 2, niter))
    for dt in dtypes:
        plan = Plan(pixsht.sht_band(shape, wcs), lmax, dtype=dt)
        for comps in components:
            maps = [np.ravel(allmaps[c], order="F").astype(dt) for c in comps]
            scrub(plan, maps, niter)
            got, _ = run_iter(plan, maps, niter, kind)
            for c, g in zip(comps, got):
                err = column_errors(lmax, lmax, g, ref[c])
                assert err.max() <= ORACLE_TOL[dt], (dt, comps, c, int(err.argmax()), err.max())
        plan.close()


@pytest.mark.gpu
def test_loop_against_the_oracle():
    oracle_case()


# ---- 3. convergence ----------------------------------------------------------------------------------------------------------
def convergence_case(spin, kind="device"):
    """Truth alm -> alm2map -> pixsht_map2alm_iter at 180 x 91 with lmax 80 > (nrings - 1)/2: the error after k iterations stays
    within twice the oracle's, for k = 0 .. 4."""
    shape, wcs = fullsky_geometry(2.0 * degree)
    lmax = 80
    plan = Plan(pixsht.sht_band(shape, wcs), lmax)
    truth = [synth_alm(lmax, lmax, 1 + c, spin2=spin == 2) for c in range(1 if spin == 0 else 2)]
    maps = [np.ravel(m, order="F") for m in plan.alm2map(truth)]
    for k, bound in enumerate(CONVERGENCE[spin]):
        scrub(plan, maps, k)
        got, _ = run_iter(plan, maps, k, kind)
        err = np.sqrt(sum(np.sum(np.abs(g - t) ** 2) for g, t in zip(got, truth)) / sum(np.sum(np.abs(t) ** 2) for t in truth))
        assert err < 2 * bound, (spin, k, err, bound)
    plan.close()


@pytest.mark.gpu
@pytest.mark.parametrize("spin", [0, 2])
def test_convergence(spin):
    convergence_case(spin)


# ---- 4. niter = 0 is pixsht_execute(MAP2ALM) ---------------------------------------------------------------------------------
def niter_zero_case(kinds, res=2.0 * degree, lmax=80):
    """Bit for bit, on a grid of one ring-pair chunk per Legendre launch (each alm element receives one atomic add, so the
    result does not depend on the order of the adds)."""
    shape, wcs = fullsky_geometry(res)
    for dt in (F64, F32):
        plan = Plan(pixsht.sht_band(shape, wcs), lmax, dtype=dt)
        allmaps = random_maps(shape[0] * shape[1], 3, 9300)
        for comps in COMPONENTS:
            maps = [allmaps[c].astype(dt) for c in comps]
            for kind in kinds:
                scrub(plan, maps, 0)
                got, n_iter = run_iter(plan, maps, 0, kind)
                ref, n_exec = run(plan, M2A, maps, kind)
                assert n_iter == n_exec
                for g, r in zip(got, ref):
                    assert np.array_equal(g, r), (dt, comps, kind)
        plan.close()


@pytest.mark.gpu
def test_niter_zero_is_plain_map2alm():
    niter_zero_case(("device", "pageable", "pinned"))


# ---- 5. errors ---------------------------------------------------------------------------------------------------------------
def errors_case(res=5.0 * degree, lmax=30):
    shape, wcs = fullsky_geometry(res)
    band = pixsht.sht_band(shape, wcs)
    maps = [x.reshape(shape, order="F") for x in random_maps(shape[0] * shape[1], 3, 9400)]
    plan = Plan(band, lmax)
    with pytest.raises(PixshtError) as e:
        plan.map2alm_iter_ptrs([np.empty(plan.nalm, plan.cdtype).ctypes.data], [maps[0].ctypes.data], -1)
    assert e.value.code == _lib.ERR_ARG
    ref = plan.map2alm(maps, niter=2)            # the plan still works
    assert all(np.all(np.isfinite(a)) for a in ref)
    multi = Plan(band, lmax, devices=[0, 0])
    with pytest.raises(PixshtError) as e:
        multi.map2alm(maps, niter=1)
    assert e.value.code == _lib.ERR_UNSUPPORTED and "multi-GPU" in str(e.value)
    got = multi.map2alm(maps)                    # niter = 0 on the same plan: the ordinary multi-GPU analysis
    single = plan.map2alm(maps)
    for g, r in zip(got, single):
        assert column_errors(lmax, lmax, g, r).max() <= COLUMN_TOL[F64]
    multi.close()
    plan.close()


@pytest.mark.gpu
def test_errors():
    errors_case()


@pytest.mark.gpu
def test_python_front_end_takes_niter():
    """pixsht.map2alm(..., niter=k) equals Plan.map2alm(..., niter=k); niter = 0 is today's call."""
    from pixsht.transforms import map2alm
    shape, wcs = fullsky_geometry(2.0 * degree, dims=(3,))
    m = Enmap(np.asfortranarray(np.random.default_rng(9500).standard_normal(shape)), wcs)
    plan = Plan(pixsht.sht_band(shape[:2], wcs), 80)
    planes = [np.asfortranarray(m.data[:, :, c]) for c in range(3)]
    for k in (0, 2):
        got = map2alm(m, lmax=80, niter=k)
        ref = plan.map2alm(planes, niter=k)
        for g, r in zip(got, ref):
            assert column_errors(80, 80, g.alm, r).max() <= COLUMN_TOL[F64]
    plan.close()


# ---- emulation replays: reduced sets on a 5 degree grid (72 x 37) with lmax 30 > 18; the streams of the emulation build run
# one after another and its memory kinds are all ordinary host memory ------------------------------------------------------------
EMU = dict(res=5.0 * degree, lmax=30)


def test_emu_replay_loop_equals_its_parts(emu_default):
    parts_case("flipped", dtypes=(F64, F32), components=((0,), (0, 1, 2)), niter=2, kinds=("device", "pageable"), **EMU)
    parts_case("cut_sky", dtypes=(F64,), components=((1, 2),), niter=1, kinds=("pageable",), **EMU)
    parts_case("rings", components=((0,),), niter=1, kinds=("device",), **EMU)


def test_emu_replay_oracle_and_convergence(emu_default):
    oracle_case(res=5.0 * degree, lmax=30, niter=2, components=((0, 1, 2),))
    convergence_case(0)


def test_emu_replay_niter_zero_and_errors(emu_default):
    niter_zero_case(("device", "pageable"), **EMU)
    errors_case()
