"""The pipelined host-pointer path of a single-GPU plan (pixsht.cu, execute_host: three streams, pieces of graded size, the
single-map schedule of large plans, the pageable-array stager of host_stage.inl) against the device-pointer path of the same
plan, which runs every stage as one launch on one stream.  Any difference between the two is a fault in the scheduling or in
the copies:

* alm2map: host == device bit for bit (chunks reach the two-step kernels by absolute index, so splitting a launch changes no sum);
* map2alm: the two paths differ only in the order of the atomic adds: the relative RMS of EVERY m column is <= 1e-12 (Float64)
  or <= 1e-6 (Float32) -- a whole-vector figure would hide a small column that was dropped or counted twice;
* every array handed to the library has guard elements on both sides that must come back unchanged, inputs must come back
  unchanged, and outputs start as NaN, so that a piece which is never written shows.

The schedule depends on switches read when a plan is created (PIXSHT_R0 / R0A / R2 / R2A: ring pairs per lane, hence the number
of 32-lane chunks; PIXSHT_SPLITS: the number of pieces), on every call (PIXSHT_TONLY_MINCHUNKS: the single-map schedule of
large plans) and once per process (PIXSHT_PIECE_SHAPE, PIXSHT_STAGE: run in a child process).  Each case proves by launch
counts that the single-map schedule ran exactly where it is expected to: a T-only call's count is compared with the same call
with that schedule forced off.  GPU tests carry the gpu mark; the emulation replays at the
end run the same bodies on the host-emulation build (tests/emu/), whose streams run one after another."""
import ctypes
import functools
import os
import subprocess
import sys

import numpy as np
import pytest

import pixsht
from pixsht import Enmap, fullsky_geometry, degree, arcminute
from pixsht import _lib
from pixsht.transforms import Plan, get_lib
from helpers import synth_alm, rel_rms, oracle_alm2map, oracle_map2alm
from oracle import alm_index, cc_geometry
from test_emu_kernels import emu, emu_default  # noqa: F401  (fixtures of the emulation replays)

HERE = os.path.dirname(os.path.abspath(__file__))
A2M, M2A = _lib.ALM2MAP, _lib.MAP2ALM
F64, F32 = np.dtype(np.float64), np.dtype(np.float32)
GUARD = 64                          # elements on either side of every array (a multiple of 16 bytes: alignment is kept)
GUARD_VALUE = -1.5 * 2.0 ** 100     # exact in Float32 and Float64
COLUMN_TOL = {F64: 1e-12, F32: 1e-6}
ORACLE_TOL = {F64: 1e-10, F32: 1e-5}
NEVER = "1000000"                   # a PIXSHT_TONLY_MINCHUNKS no plan reaches: the single-map schedule off
PIECE_SHAPE = os.environ.get("PIXSHT_PIECE_SHAPE", "1") != "0"     # the library reads it once per process


def _is_torch(x):
    return type(x).__module__.startswith("torch")


def _ptr(x):
    return x.data_ptr() if _is_torch(x) else x.ctypes.data


class Buffers:
    """The arrays of one call.  Host kinds: "pageable" (numpy), "pinned" (pixsht_host_alloc), "registered" (numpy, page-locked
    with pixsht_host_register); "device": a torch CUDA tensor -- on the emulation build, whose device pointers are host
    pointers, a numpy array.  Every array has GUARD elements on both sides; outputs start as NaN."""

    def __init__(self, lib):
        self.lib = lib
        self.emu = "EMULATION" in lib.version()
        self.arrays = []                      # (whole buffer, region handed to the library, input copy or None)
        self.pinned, self.registered = [], []

    def get(self, kind, n, dtype, data=None):
        dtype = np.dtype(dtype)
        total = n + 2 * GUARD
        if kind == "device" and not self.emu:
            import torch
            tdt = {F64: torch.float64, F32: torch.float32, np.dtype(np.complex128): torch.complex128, np.dtype(np.complex64): torch.complex64}[dtype]
            whole = torch.empty(total, dtype=tdt, device="cuda")
            real = torch.view_as_real(whole) if whole.is_complex() else whole
            real.fill_(GUARD_VALUE)
            if whole.is_complex():
                real[:, 1] = 0.0
            region = whole[GUARD:GUARD + n]
            if data is None:
                (torch.view_as_real(region) if region.is_complex() else region).fill_(float("nan"))
            else:
                region.copy_(torch.from_numpy(np.ascontiguousarray(data)))
        else:
            if kind == "pinned":
                p = ctypes.c_void_p()
                self.lib.check(self.lib.lib.pixsht_host_alloc(ctypes.byref(p), total * dtype.itemsize))
                self.pinned.append(p.value)
                whole = np.frombuffer((ctypes.c_char * (total * dtype.itemsize)).from_address(p.value), dtype=dtype)
            elif kind in ("pageable", "registered", "device"):
                whole = np.empty(total, dtype=dtype)
                if kind == "registered":
                    self.lib.check(self.lib.lib.pixsht_host_register(whole.ctypes.data, whole.nbytes))
                    self.registered.append(whole.ctypes.data)
            else:
                raise ValueError(kind)
            whole[:GUARD] = GUARD_VALUE
            whole[-GUARD:] = GUARD_VALUE
            region = whole[GUARD:GUARD + n]
            if data is None:
                region.view(np.float32 if dtype.itemsize // (2 if dtype.kind == "c" else 1) == 4 else np.float64)[...] = np.nan
            else:
                region[...] = data
        self.arrays.append((whole, region, None if data is None else data))
        return region

    def check(self):
        """Guards unchanged, inputs unchanged, no output element left unwritten."""
        for i, (whole, region, data) in enumerate(self.arrays):
            if _is_torch(whole):
                import torch
                guards = torch.cat([whole[:GUARD], whole[-GUARD:]]).cpu().numpy()
                assert np.all(guards == guards.dtype.type(GUARD_VALUE)), "array %d: guard overwritten" % i
                if data is None:
                    assert not bool(torch.isnan(region).any()), "array %d: output element never written" % i
                else:
                    assert torch.equal(region, torch.from_numpy(np.ascontiguousarray(data)).to(region.device)), "array %d: input changed" % i
            else:
                assert np.all(whole[:GUARD] == whole.dtype.type(GUARD_VALUE)) and np.all(whole[-GUARD:] == whole.dtype.type(GUARD_VALUE)), \
                    "array %d: guard overwritten" % i
                if data is None:
                    bad = np.flatnonzero(np.isnan(region))
                    assert bad.size == 0, "array %d: %d output elements never written, first at %d" % (i, bad.size, bad[0])
                else:
                    assert np.array_equal(region, data), "array %d: input changed" % i

    def close(self):
        self.arrays = []
        for p in self.registered:
            self.lib.check(self.lib.lib.pixsht_host_unregister(p))
        for p in self.pinned:
            self.lib.check(self.lib.lib.pixsht_host_free(p))
        self.registered, self.pinned = [], []


def run(plan, direction, inputs, kind, batch=False):
    """One call of `plan` on flat `inputs` (alm vectors, or maps raveled in Fortran order) held in memory of `kind` (one kind,
    or one per component).  Returns copies of the outputs and the plan's launch count; the checks of Buffers have passed."""
    kinds = list(kind) if isinstance(kind, (list, tuple)) else [kind] * len(inputs)
    a2m = direction == A2M
    nout, dout = (plan.band.nx * plan.band.nrings, plan.dtype) if a2m else (plan.nalm, plan.cdtype)
    bufs = Buffers(plan.lib)
    try:
        ins = [bufs.get(k, x.size, x.dtype, x) for k, x in zip(kinds, inputs)]
        outs = [bufs.get(k, nout, dout) for k in kinds]
        alms, maps = (ins, outs) if a2m else (outs, ins)
        loc = _lib.DEVICE if kinds[0] == "device" else _lib.HOST
        ex = plan.execute_batch_ptrs if batch else plan.execute_ptrs
        ex(direction, [_ptr(a) for a in alms], [_ptr(m) for m in maps], loc)
        launches = plan.info()["launches"]
        bufs.check()
        return [o.cpu().numpy() if _is_torch(o) else np.array(o) for o in outs], launches
    finally:
        bufs.close()


def column_errors(lmax, mmax, a, b):
    """Relative RMS error of every m column of alm vector `a` against `b`."""
    starts = np.array([alm_index(lmax, m, m) for m in range(mmax + 1)])
    num = np.add.reduceat(np.abs(a - b) ** 2, starts, dtype=np.float64)
    den = np.add.reduceat(np.abs(b) ** 2, starts, dtype=np.float64)
    assert np.all(den > 0)
    return np.sqrt(num / den)


def assert_same(plan, direction, got, ref, what=""):
    for c, (g, r) in enumerate(zip(got, ref)):
        if direction == A2M:
            bad = np.flatnonzero(g != r)
            assert bad.size == 0, "%s component %d: %d pixels differ, first at ring %d" % (what, c, bad.size, bad[0] // plan.band.nx)
        else:
            err = column_errors(plan.lmax, plan.mmax, g, r)
            assert err.max() <= COLUMN_TOL[plan.dtype], "%s component %d: column m = %d off by %.2e" % (what, c, int(err.argmax()), err.max())


def scrub(plan, direction, inputs, batch=False):
    """The same call on negated inputs: afterwards every buffer of the plan (phase rows, staged maps and alm, the Float64 alm of
    a Float32 plan) holds wrong contents for the next call on `inputs`."""
    nout, dout = (plan.band.nx * plan.band.nrings, plan.dtype) if direction == A2M else (plan.nalm, plan.cdtype)
    neg = [np.negative(x) for x in inputs]
    outs = [np.empty(nout, dout) for _ in inputs]
    alms, maps = (neg, outs) if direction == A2M else (outs, neg)
    ex = plan.execute_batch_ptrs if batch else plan.execute_ptrs
    ex(direction, [a.ctypes.data for a in alms], [m.ctypes.data for m in maps], _lib.HOST)


def host_vs_device(plan, direction, inputs, kinds=("pageable",), batch=False):
    """A host call per memory kind (one kind, or a list of one kind per component), then the device call; each host result
    equals the device result.  Returns (device result, host launches, device launches).  Each host call follows a scrub: an
    earlier call on the same inputs would leave every plan buffer holding exactly what a copy, FFT or Legendre launch that runs
    before its event wait should have waited for, and hide the fault."""
    hosts, lh = [], None
    for k in kinds:
        scrub(plan, direction, inputs, batch)
        host, n = run(plan, direction, inputs, k, batch)
        assert lh is None or n == lh, "the memory kind changed the schedule"
        hosts.append(host)
        lh = n
    dev, ld = run(plan, direction, inputs, "device", batch)
    for k, host in zip(kinds, hosts):
        assert_same(plan, direction, host, dev, "%s %s" % ("alm2map" if direction == A2M else "map2alm", k))
    return dev, lh, ld


def single_map_launches_off(plan, direction, inputs, monkeypatch):
    """Host launch count of the same call with the single-map schedule forced off (PIXSHT_TONLY_MINCHUNKS is read per call)."""
    prev = os.environ.get("PIXSHT_TONLY_MINCHUNKS")
    monkeypatch.setenv("PIXSHT_TONLY_MINCHUNKS", NEVER)
    try:
        return host_vs_device(plan, direction, inputs)[1]
    finally:
        if prev is None:
            monkeypatch.delenv("PIXSHT_TONLY_MINCHUNKS")
        else:
            monkeypatch.setenv("PIXSHT_TONLY_MINCHUNKS", prev)


def expect_single_map(plan, minchunks, nsplit=8):
    """Whether a T-only call takes the single-map schedule (alm2map, map2alm), from the plan's chunk counts: alm2map needs
    >= minchunks chunks of 32 R0 pairs, 5 pieces and mmax + 1 >= 64; map2alm >= minchunks chunks of 32 R0A pairs and the
    equator-first order (>= 4 chunks, >= 4 pieces).  Both need the graded pieces (PIXSHT_PIECE_SHAPE)."""
    info = plan.info()
    nch0 = -(-info["npairs"] // (32 * info["R0"]))
    nch0a = -(-info["npairs"] // (32 * info["R0a"]))
    return (PIECE_SHAPE and nsplit >= 5 and plan.mmax + 1 >= 64 and nch0 >= minchunks,
            PIECE_SHAPE and nsplit >= 4 and nch0a >= max(4, minchunks))


def _emulated():
    return "EMULATION" in get_lib().version()


def _flat(x):
    return np.ravel(x, order="F")


def _set_env(monkeypatch, env):
    for k, v in env.items():
        monkeypatch.setenv(k, v)


# ---- 2. schedule sweep at 8' ------------------------------------------------------------------------------------------------
TILES1 = {"PIXSHT_R0": "1", "PIXSHT_R0A": "1", "PIXSHT_R2": "1", "PIXSHT_R2A": "1"}     # 32 ring pairs per chunk (22 chunks at 8')
# name: (switches, single-map schedule expected on a T-only (alm2map, map2alm) call).  What the launch counts prove: the
# single-map schedule runs exactly where expected (against the same call with it forced off), and a host call with more than one
# piece runs more launches than the device call.  The comments name the other branches each set is configured to reach (by the
# conditions of execute_host: >= 4 chunks and >= 4 pieces for equator-first rows, >= 2 chunks for the two-part analysis); their
# piece shape and order are not visible in a launch count and are not proven separately.
SWEEP = {
    "defaults": ({}, (False, False)),                                              # 6 / 11 chunks: graded pieces, two-part QU analysis
    "tiles1": (TILES1, (True, True)),                                              # 22 chunks: tonly_rings / tonly_m
    "tiles1_off": (dict(TILES1, PIXSHT_TONLY_MINCHUNKS=NEVER), (False, False)),    # same chunks, single-map schedule off
    "tiles1_splits5": (dict(TILES1, PIXSHT_SPLITS="5"), (True, True)),             # the fewest pieces tonly_rings runs with
    "tiles1_splits4": (dict(TILES1, PIXSHT_SPLITS="4"), (False, True)),            # no tonly_rings; equator-first rows (tonly_m) on
    "tiles1_splits3": (dict(TILES1, PIXSHT_SPLITS="3"), (False, False)),           # too few pieces for equator-first rows
    "tiles1_splits1": (dict(TILES1, PIXSHT_SPLITS="1"), (False, False)),           # one piece
    "odd_tiles": ({"PIXSHT_R0": "3", "PIXSHT_R0A": "6", "PIXSHT_R2": "3", "PIXSHT_R2A": "6"}, (False, False)),   # other chunk boundaries
}
COMPONENTS = ((0,), (1, 2), (0, 1, 2))


@functools.lru_cache(maxsize=2)
def sweep_inputs(res, lmax):
    """T, E, B alm and T, Q, U maps, rounded through Float32 so that the Float32 plans see exactly the Float64 inputs."""
    shape, wcs = fullsky_geometry(res)
    alms = [synth_alm(lmax, lmax, 8100 + c, spin2=c > 0).astype(np.complex64).astype(np.complex128) for c in range(3)]
    rng = np.random.default_rng(8200)
    maps = [np.asfortranarray(rng.standard_normal(shape).astype(np.float32).astype(np.float64)) for _ in range(3)]
    return shape, wcs, alms, maps


@functools.lru_cache(maxsize=2)
def sweep_oracle(res, lmax):
    """Every pixel and every alm of the sweep inputs from the CPU port (oracle/sht_cpu.c)."""
    from oracle import get_cpu_sht
    get_cpu_sht().use_all_cores()
    shape, wcs, alms, maps = sweep_inputs(res, lmax)
    t = oracle_alm2map(alms[0][None], shape, wcs, lmax, kind="cpu")[:, :, 0]
    qu = oracle_alm2map(np.stack(alms[1:]), shape, wcs, lmax, spin=2, kind="cpu")
    ta = oracle_map2alm(Enmap(maps[0], wcs), lmax, kind="cpu")[0]
    eb = oracle_map2alm(Enmap(np.asfortranarray(np.stack(maps[1:], axis=2)), wcs), lmax, spin=2, kind="cpu")
    return [t, qu[:, :, 0], qu[:, :, 1]], [ta, eb[0], eb[1]]


def sweep_case(name, monkeypatch, res=8.0 * arcminute, lmax=1350, minchunks=16, dtypes=(F64, F32), components=COMPONENTS):
    env, (on_a2m, on_m2a) = SWEEP[name]
    _set_env(monkeypatch, env)
    if "PIXSHT_TONLY_MINCHUNKS" not in env:
        monkeypatch.setenv("PIXSHT_TONLY_MINCHUNKS", str(minchunks))
    kinds = ("pageable", "pinned", "registered") if name in ("defaults", "tiles1") and not _emulated() else ("pageable",)
    shape, wcs, alms, maps = sweep_inputs(res, lmax)
    band = pixsht.sht_band(shape, wcs)
    for dt in dtypes:
        plan = Plan(band, lmax, dtype=dt)
        nsplit = int(env.get("PIXSHT_SPLITS", 8))
        assert expect_single_map(plan, int(env.get("PIXSHT_TONLY_MINCHUNKS", minchunks)), nsplit) == (on_a2m and PIECE_SHAPE, on_m2a and PIECE_SHAPE), \
            "the sweep set no longer reaches its branch: %s" % plan.info()
        for comps in components:
            for direction, inputs in ((A2M, [alms[c].astype(plan.cdtype) for c in comps]), (M2A, [_flat(maps[c]).astype(dt) for c in comps])):
                dev, lh, ld = host_vs_device(plan, direction, inputs, kinds)
                if nsplit > 1:
                    assert lh > ld, "the host call ran no pieces"
                if comps == (0,):
                    on = on_a2m if direction == A2M else on_m2a
                    off = single_map_launches_off(plan, direction, inputs, monkeypatch)
                    assert (lh != off) == (on and PIECE_SHAPE), (name, dt, direction, lh, off)
                if name == "defaults":       # the device result, every pixel and alm, against the CPU port
                    ref_maps, ref_alms = sweep_oracle(res, lmax)
                    for c, d in zip(comps, dev):
                        if direction == A2M:
                            err = rel_rms(d.reshape(shape, order="F"), ref_maps[c])
                        else:
                            err = rel_rms(d, ref_alms[c])
                        assert err <= ORACLE_TOL[F64 if dt == F64 else F32], (comps, c, direction, dt, err)
        plan.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(SWEEP))
def test_host_path_schedule_sweep(name, monkeypatch):
    sweep_case(name, monkeypatch)


# ---- 3. geometries, on 32-pair chunks --------------------------------------------------------------------------------------
GEOMETRIES = ["unflipped", "north_only", "straddles_equator", "narrower_than_ring", "mmax_half", "mmax_below_64", "iau"]


def geometry_case(case, monkeypatch, res=8.0 * arcminute, lmax=1350, minchunks=16, components=None):
    _set_env(monkeypatch, TILES1)
    monkeypatch.setenv("PIXSHT_TONLY_MINCHUNKS", str(minchunks))
    shape, wcs = fullsky_geometry(res)
    nx, ny = shape
    full = Enmap(np.zeros(shape, order="F"), wcs)
    mmax = {"mmax_half": lmax // 2, "mmax_below_64": 40}.get(case, lmax)
    sub = {"unflipped": full[::-1, ::-1],                                # flipy = False: ring_rows maps rings to rows directly
           "north_only": full[:, ny // 2 + ny // 20:],                   # ring pairs of one member
           "straddles_equator": full[:, ny // 2 - (2 * ny) // 5:ny // 2 + ny // 10],
           "narrower_than_ring": full[nx // 20:nx - nx // 3, ny // 10:]}.get(case, full)
    band = pixsht.sht_band(sub.shape[:2], sub.wcs)
    if case == "unflipped":
        assert not band.flipy
    plan = Plan(band, lmax, mmax)
    if case == "iau":
        plan.set_polconv("IAU")
    expect = expect_single_map(plan, minchunks)
    assert expect[1], "the case does not reach the single-map schedule: %s" % plan.info()
    assert expect[0] == (case != "mmax_below_64")
    rng = np.random.default_rng(8300)
    alms = [synth_alm(lmax, mmax, 8310 + c, spin2=c > 0) for c in range(3)]
    maps = [rng.standard_normal(band.nx * band.nrings) for _ in range(3)]
    for comps in components or (((1, 2), (0, 1, 2)) if case == "iau" else COMPONENTS):
        for direction, inputs in ((A2M, [alms[c] for c in comps]), (M2A, [maps[c] for c in comps])):
            dev, lh, ld = host_vs_device(plan, direction, inputs)
            if comps == (0,):
                off = single_map_launches_off(plan, direction, inputs, monkeypatch)
                assert (lh != off) == expect[0 if direction == A2M else 1], (case, direction, lh, off)
    plan.close()


@pytest.mark.gpu
@pytest.mark.parametrize("case", GEOMETRIES)
def test_host_path_geometries(case, monkeypatch):
    geometry_case(case, monkeypatch)


class _RingsPlan(Plan):
    """A plan on an explicit ring set (pixsht_plan_create_rings): rings in the caller's order, nx = nphi, no flips."""

    def __init__(self, theta, weight, nphi, lmax):
        from types import SimpleNamespace
        self.lib = get_lib()
        self.band = SimpleNamespace(nx=nphi, nrings=len(theta))
        self.lmax = self.mmax = lmax
        self.dtype, self.cdtype, self.devices = F64, np.dtype(np.complex128), None
        h = ctypes.c_void_p()
        dp = ctypes.POINTER(ctypes.c_double)
        th, w = np.ascontiguousarray(theta, dtype=np.float64), np.ascontiguousarray(weight, dtype=np.float64)
        self.lib.check(self.lib.lib.pixsht_plan_create_rings(ctypes.byref(h), len(th), th.ctypes.data_as(dp), w.ctypes.data_as(dp), nphi, 0.0,
                                                             lmax, lmax, _lib.F64, 0))
        self.handle = h
        self.nalm = int(self.lib.lib.pixsht_nalm(lmax, lmax))


def unordered_rings_case(monkeypatch, nphi=2700, nrings=1351, lmax=1350, minchunks=16):
    """Rings handed over in no order of colatitude (even ring numbers first, then odd ones): a piece's ring pairs no longer
    map to one contiguous ring range per hemisphere (pair_range_rings fails), and every pipeline falls back to whole-component
    copies and FFTs.  Host == device on that plan, its results equal the sorted plan's with rows permuted, and each of its host
    calls runs fewer launches than the same call on the sorted plan (which takes the ring-range pieces)."""
    _set_env(monkeypatch, TILES1)
    monkeypatch.setenv("PIXSHT_TONLY_MINCHUNKS", str(minchunks))
    nr = nrings
    theta, w = cc_geometry(nr, nphi)
    order = np.concatenate([np.arange(0, nr, 2), np.arange(1, nr, 2)])
    srt, prm = _RingsPlan(theta, w, nphi, lmax), _RingsPlan(theta[order], w[order], nphi, lmax)
    rng = np.random.default_rng(8400)
    alms = [synth_alm(lmax, lmax, 8410 + c, spin2=c > 0) for c in range(3)]
    maps = [rng.standard_normal((nphi, nr)) for _ in range(3)]
    for comps in COMPONENTS:
        d_srt, l_srt, _ = host_vs_device(srt, A2M, [alms[c] for c in comps])
        d_prm, l_prm, _ = host_vs_device(prm, A2M, [alms[c] for c in comps])
        assert l_prm < l_srt, (comps, l_prm, l_srt)
        for a, b in zip(d_prm, d_srt):
            assert rel_rms(a.reshape(nphi, nr, order="F"), b.reshape(nphi, nr, order="F")[:, order]) < 1e-13
        d_srt, l_srt, _ = host_vs_device(srt, M2A, [_flat(maps[c]) for c in comps])
        d_prm, l_prm, _ = host_vs_device(prm, M2A, [_flat(maps[c][:, order]) for c in comps])
        assert l_prm < l_srt, (comps, l_prm, l_srt)
        for a, b in zip(d_prm, d_srt):
            assert column_errors(lmax, lmax, a, b).max() < 1e-12
    srt.close()
    prm.close()


@pytest.mark.gpu
def test_host_path_unordered_rings_fall_back_to_whole_components(monkeypatch):
    unordered_rings_case(monkeypatch)


# ---- 4. large single maps, default settings (the product case) --------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("config", ["c4_f64", "c5_f32"])
def test_large_single_map_host_path_equals_device_path(config, monkeypatch):
    """C4 (1', lmax 10800) T-only Float64 and C5 (0.5', lmax 21600) T-only Float32: host calls on pageable and page-locked
    arrays against the device call, every pixel and every alm, both directions; both take the single-map schedule."""
    res, lmax, dt = {"c4_f64": (1.0, 10800, F64), "c5_f32": (0.5, 21600, F32)}[config]
    shape, wcs = fullsky_geometry(res * arcminute)
    plan = Plan(pixsht.sht_band(shape, wcs), lmax, dtype=dt)
    assert expect_single_map(plan, 16) == (PIECE_SHAPE, PIECE_SHAPE)
    alm = [synth_alm(lmax, lmax, 9000).astype(plan.cdtype)]
    dev_map, lh, ld = host_vs_device(plan, A2M, alm, ("pageable", "pinned"))
    assert (single_map_launches_off(plan, A2M, alm, monkeypatch) != lh) == PIECE_SHAPE
    del alm
    _, lh, ld = host_vs_device(plan, M2A, dev_map, ("pageable", "pinned"))      # the band-limited synthesised map
    assert (single_map_launches_off(plan, M2A, dev_map, monkeypatch) != lh) == PIECE_SHAPE
    plan.close()


# ---- 5. the stager with small slots, and calls that follow each other --------------------------------------------------------
def stager_case(monkeypatch, res=8.0 * arcminute, lmax=1350):
    """A fresh plan whose stager has two 1 MB slots (read when the plan first stages a pageable copy; copies of >= 4 MB are
    staged, so an 8' Float64 map crosses the two slots about 15 times): a mixed sequence of calls, each equal to the device
    call, so that slot generations and the dependency events carry over from call to call; then calls whose components mix
    pageable and page-locked arrays."""
    monkeypatch.setenv("PIXSHT_STAGE_CHUNK_MB", "1")
    monkeypatch.setenv("PIXSHT_STAGE_SLOTS", "2")
    shape, wcs, alms, maps = sweep_inputs(res, lmax)
    plan = Plan(pixsht.sht_band(shape, wcs), lmax)
    fm = [_flat(m) for m in maps]
    host_vs_device(plan, A2M, alms[:1])
    host_vs_device(plan, M2A, fm)
    host_vs_device(plan, A2M, alms[1:])
    host_vs_device(plan, M2A, fm[:1])
    host_vs_device(plan, A2M, alms, batch=True)
    host_vs_device(plan, M2A, fm, batch=True)
    mixed = ["pageable", "pinned", "registered"]
    host_vs_device(plan, M2A, fm, (mixed,))
    host_vs_device(plan, A2M, alms, (mixed[::-1],))
    plan.close()


@pytest.mark.gpu
def test_stager_small_slots_and_call_sequence(monkeypatch):
    stager_case(monkeypatch)


# ---- 7. switches read once per process: the sweep subset in a child process ---------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("switch", ["PIXSHT_PIECE_SHAPE=0", "PIXSHT_STAGE=0"])
def test_process_wide_switches_in_a_child_process(switch):
    """PIXSHT_PIECE_SHAPE=0: equal pieces, pole first, no single-map schedule (the sweep's expectations follow it);
    PIXSHT_STAGE=0: pageable arrays go to the driver instead of the stager."""
    key, val = switch.split("=")
    env = dict(os.environ, **{key: val})
    ids = ["%s::test_host_path_schedule_sweep[%s]" % (os.path.join(HERE, "test_host_pipeline.py"), n) for n in ("tiles1", "tiles1_splits4", "odd_tiles")]
    cmd = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + ["-m", "pytest", "-q", "-p", "no:cacheprovider", "-m", "gpu"] + ids
    r = subprocess.run(cmd, env=env, cwd=os.path.dirname(HERE), capture_output=True, text=True, timeout=900)
    assert r.returncode == 0 and "3 passed" in r.stdout, r.stdout[-4000:] + r.stderr[-2000:]


# ---- emulation replays: the bodies above on the host-emulation build, on a 2 x 0.5 degree grid (180 x 361: 181 ring pairs, 6
# chunks of 32) with lmax 80 and the single-map schedule lowered to 4 chunks.  Its streams run one after another and its stager
# is compiled out: these rehearse the schedules' arithmetic and the checks, not the ordering. -----------------------------------
EMU_RES, EMU_LMAX = (2.0 * degree, 0.5 * degree), 80


@pytest.mark.parametrize("name", ["defaults", "tiles1", "tiles1_splits4"])
def test_emu_replay_schedule_sweep(emu_default, monkeypatch, name):
    sweep_case(name, monkeypatch, EMU_RES, EMU_LMAX, minchunks=4, dtypes=(F64, F32) if name == "tiles1" else (F64,),
               components=((0,), (0, 1, 2)) if name == "tiles1" else ((0,),))


def test_emu_replay_geometry_and_unordered_rings(emu_default, monkeypatch):
    geometry_case("straddles_equator", monkeypatch, EMU_RES, EMU_LMAX, minchunks=4, components=((0,),))
    unordered_rings_case(monkeypatch, nphi=180, nrings=361, lmax=EMU_LMAX, minchunks=4)


def test_emu_replay_call_sequence(emu_default, monkeypatch):
    stager_case(monkeypatch, EMU_RES, EMU_LMAX)
