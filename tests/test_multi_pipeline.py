"""The pipelined host-pointer path of a multi-GPU plan (multi.inl: execute_multi, multi_alm2map, multi_map2alm -- m-sharded
Legendre stages, cross-shard event barriers, ring-range pieces, alm columns copied in runs of consecutive m) against a single-GPU
plan on the plain ring-FFT kernels called with device pointers.  The m-sharded layout runs the plain kernels too, so:

* alm2map: multi == single bit for bit;
* map2alm: the relative RMS of EVERY m column is <= 1e-12 (Float64) or <= 1e-6 (Float32) (atomic accumulation order);
* guards, unchanged inputs and NaN-filled outputs are checked as in test_host_pipeline.py, and every multi call follows a scrub
  (the same call on negated inputs), so that a copy or launch which runs before its event wait finds wrong values.

The switches are read when a plan is created.  Every set runs on 32-pair chunks (TILES1), so that each family has several
chunks: the defaults; no pieces at all (the m-piece Legendre branch); three analysis ring pieces (equal-count bounds instead of
the equatorial third); one m segment per shard.  A call whose last family runs in several ring pieces must run more launches
than the same call with no pieces: the pieced branches ran.  GPU tests carry the gpu mark; the emulation replay at the end
runs a reduced set on the host-emulation build (tests/emu/), whose streams run one after another: it checks the pieces'
arithmetic and the copies, not their ordering."""
import numpy as np
import pytest

import pixsht
from pixsht import Enmap, fullsky_geometry, arcminute
from pixsht.transforms import Plan
from helpers import synth_alm, plain_fft_kernels
from test_gpu_parity import _shard_devices
from test_host_pipeline import A2M, M2A, F64, F32, TILES1, EMU_RES, run, scrub, assert_same
from test_emu_kernels import emu, emu_default  # noqa: F401  (fixtures of the emulation replay)

NO_PIECES = dict(TILES1, PIXSHT_MULTI_PIECES="1", PIXSHT_MULTI_RING_PIECES="1", PIXSHT_MULTI_RING_PIECES_M2A="1",
                 PIXSHT_MULTI_RING_PIECES_T="1")
SWITCHES = {
    "defaults": TILES1,
    "no_pieces": NO_PIECES,
    "m2a3": dict(TILES1, PIXSHT_MULTI_RING_PIECES_M2A="3"),
    "segs1": dict(TILES1, PIXSHT_MULTI_SEGS="1"),
}
SWITCH_KEYS = sorted({k for env in SWITCHES.values() for k in env})
COMPONENTS = ((0,), (1, 2), (0, 1, 2))


def _band(res, geometry):
    shape, wcs = fullsky_geometry(res)
    nx, ny = shape
    full = Enmap(np.zeros(shape, order="F"), wcs)
    sub = {"full": full,
           "unflipped": full[::-1, ::-1],
           "cut": full[nx // 9:nx - nx // 6, ny // 6:ny - ny // 3]}[geometry]
    band = pixsht.sht_band(sub.shape[:2], sub.wcs)
    if geometry == "unflipped":
        assert not band.flipy
    return band


def _use_switches(monkeypatch, name):
    for k in SWITCH_KEYS:
        monkeypatch.delenv(k, raising=False)
    for k, v in SWITCHES[name].items():
        monkeypatch.setenv(k, v)


def multi_case(monkeypatch, nshard, sets, res=8.0 * arcminute, lmax=1350, geometry="full", dtypes=(F64, F32),
               components=COMPONENTS, pinned=()):
    """Every call of `components` x both directions through a multi plan of `nshard` shards under each switch set of `sets`
    (pageable arrays; also page-locked ones for the sets in `pinned`), against the single-GPU reference; then the launch counts
    of the pieced sets against the no-pieces set, when it ran."""
    band = _band(res, geometry)
    rng = np.random.default_rng(8500)
    alms = [synth_alm(lmax, lmax, 8510 + c, spin2=c > 0).astype(np.complex64).astype(np.complex128) for c in range(3)]
    maps = [rng.standard_normal(band.nx * band.nrings).astype(np.float32).astype(np.float64) for _ in range(3)]
    devices = _shard_devices(nshard)
    for dt in dtypes:
        _use_switches(monkeypatch, "defaults")
        with plain_fft_kernels():
            single = Plan(band, lmax, dtype=dt)
        refs, launches = {}, {}
        for name in sets:
            _use_switches(monkeypatch, name)
            multi = Plan(band, lmax, dtype=dt, devices=devices)
            assert multi.info()["ndev"] == nshard
            for comps in components:
                for direction, inputs in ((A2M, [alms[c].astype(multi.cdtype) for c in comps]), (M2A, [maps[c].astype(dt) for c in comps])):
                    if (comps, direction) not in refs:
                        refs[comps, direction] = run(single, direction, inputs, "device")[0]
                    for kind in ("pageable", "pinned") if name in pinned else ("pageable",):
                        scrub(multi, direction, inputs)
                        got, n = run(multi, direction, inputs, kind)
                        what = "%s %s shards=%d %s comps=%s %s" % (geometry, name, nshard, dt.name, comps, "alm2map" if direction == A2M else "map2alm")
                        assert_same(multi, direction, got, refs[comps, direction], what)
                    launches[name, comps, direction] = n
            multi.close()
        single.close()
        for (name, comps, direction), n in launches.items():
            if name != "no_pieces" and ("no_pieces", comps, direction) in launches:
                assert n > launches["no_pieces", comps, direction], (name, nshard, dt, comps, direction, n)


@pytest.mark.gpu
@pytest.mark.parametrize("nshard", [1, 2, 3])
def test_multi_host_path_switch_sets(nshard, monkeypatch):
    multi_case(monkeypatch, nshard, list(SWITCHES), pinned=("defaults",))


@pytest.mark.gpu
@pytest.mark.parametrize("nshard", [2, 3])
@pytest.mark.parametrize("geometry", ["cut", "unflipped"])
def test_multi_host_path_geometries(geometry, nshard, monkeypatch):
    multi_case(monkeypatch, nshard, ["defaults"], geometry=geometry)


# ---- emulation replay: the same body on the host-emulation build, on the 2 x 0.5 degree grid of test_host_pipeline.py (180 x
# 361: 181 ring pairs, 6 chunks of 32) with lmax 40: T and IQU, the defaults and no pieces, Float32 once ---------------------
@pytest.mark.parametrize("nshard", [2, 3])
def test_emu_replay_multi_host_path(emu_default, monkeypatch, nshard):
    multi_case(monkeypatch, nshard, ["defaults", "no_pieces"], EMU_RES, 40, dtypes=(F64,), components=((0,), (0, 1, 2)))
    if nshard == 2:
        multi_case(monkeypatch, nshard, ["defaults"], EMU_RES, 40, dtypes=(F32,), components=((0, 1, 2),))
