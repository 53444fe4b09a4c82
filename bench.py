#!/usr/bin/env python
"""bench.py -- alm2map + map2alm wall time on the BASELINE.json configs (default: C4, full-sky CAR 1' IQU, lmax 10800, F64).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--workload C1|C2|C3|C4] [--impl b200|reference] [--dump-outputs DIR]

A step = one alm2map followed by one map2alm of the whole IQU (or T) set.  One JSON line is printed by rank 0:
  value   : ms per step, inputs and outputs resident in HBM (device pointers through the C ABI / stage API)
  e2e     : ms per step through the host-pointer C ABI call (pinned host buffers, H2D + D2H inside the timed region)
  roofline: Legendre kernels (the dominant ones) against the measured FP64 FMA peak; roofline_fft against measured HBM
  cpu_baseline: oracle/sht_cpu.c, a libsharp2-style CPU implementation ("port", not libsharp2) on a bounded sample of m
N > 1: launched by torchrun, one rank per GPU, m-sharded Legendre + NCCL all-to-all + ring-sharded FFT (strong scaling).
--impl reference: times that CPU implementation of the reference path (all host threads); the real
Pixell.jl/libsharp2 cannot run here (no Julia, no libsharp2: DESIGN.md).
--dump-outputs DIR (one process): after the timed steps, writes what the last one returned -- DIR/map.npy (alm2map
output, one row per component or batch member) and DIR/alm.npy (map2alm output as (re, im) pairs) -- in the workload's
float type.  Outputs larger than 32 MB are sampled at positions drawn with a fixed seed from their length alone, so two
builds run with the same arguments (same seeded inputs) can be compared value for value.
"""
import argparse
import ctypes
import json
import math
import os
import subprocess
import sys
import threading

ROOT = os.path.dirname(os.path.abspath(__file__))
for _p in (ROOT, os.path.join(ROOT, "pixell.jl_b200"), os.path.join(ROOT, "tests")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import numpy as np  # noqa: E402

WORKLOADS = {
    "C1": dict(res_arcmin=60.0, lmax=180, ncomp=1, dtype="f64", desc="full-sky CAR 1deg (360x181) Float64 spin-0, lmax=180"),
    "C2": dict(res_arcmin=4.0, lmax=2700, ncomp=1, dtype="f32", desc="full-sky CAR 4' (5400x2701) Float32 T-only, lmax=2700"),
    "C3": dict(res_arcmin=2.0, lmax=5400, ncomp=3, dtype="f64", desc="full-sky CAR 2' (10800x5401) Float64 IQU, lmax=5400"),
    "C4": dict(res_arcmin=1.0, lmax=10800, ncomp=3, dtype="f64", desc="full-sky CAR 1' (21600x10801) Float64 IQU, lmax=10800"),
    "C5": dict(res_arcmin=0.5, lmax=21600, ncomp=1, dtype="f32", desc="full-sky CAR 0.5' (43200x21601) Float32 T-only, lmax=21600"),
    "C2x64": dict(res_arcmin=4.0, lmax=2700, ncomp=1, dtype="f32", batch=64,
                  desc="64-sim batched sweep: full-sky CAR 4' (5400x2701) Float32 T-only, lmax=2700 (configs[4], second part)"),
}
METRIC = "alm2map+map2alm wall time"


def algorithmic_flops(nalm, nrings, ncomp):
    """SURVEY.md 8(d): per (l, m, ring pair) 4 FMA (spin 0), 12 (spin 2), 16 (IQU); 1 FMA = 2 flop; per direction."""
    fma = {1: 4, 2: 12, 3: 16}[ncomp]
    return 2.0 * fma * nalm * math.ceil(nrings / 2)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index=0):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            pass
        sm, mx, reasons, pw = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1])); pw.append(float(f[2]))
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------------------------------
# CPU baseline (oracle "d" build; test infrastructure used here ONLY as the timed baseline, never as the product)
# ------------------------------------------------------------------------------------------------------------------
_CPU_INPUTS = {}


def cpu_baseline(wl, target_s=12.0, maps=None, alms=None):
    """Times oracle/sht_cpu.c -- a CPU implementation with libsharp2's algorithm (ring-pair folding, scaled-exponent seek,
    pruning, OpenMP over m, SIMD over rings; "port", not libsharp2 itself) -- on all host threads, on a bounded sample: every
    `stride`-th m in both directions.  The ring FFTs run in full; the Legendre time is extrapolated linearly in the number of
    m (uniform stride => representative mix of long and short m columns)."""
    import pixsht
    from oracle import get_cpu_sht, cc_geometry, nalm as nalm_of
    cpu = get_cpu_sht()
    cpu.use_all_cores()
    res = wl["res_arcmin"] * pixsht.arcminute
    shape, wcs = pixsht.fullsky_geometry(res)
    band = pixsht.sht_band(shape, wcs)
    lmax, nc = wl["lmax"], wl["ncomp"]
    theta, w = cc_geometry(band.nrings_total, band.nphi)
    n = nalm_of(lmax)
    if alms is None or maps is None:
        key = (wl["res_arcmin"], lmax, nc)
        if key not in _CPU_INPUTS:      # generated once per process (the reference arm calls this every step)
            rng = np.random.default_rng(4242)
            _CPU_INPUTS.clear()
            _CPU_INPUTS[key] = ([rng.standard_normal(2 * n).view(np.complex128) for _ in range(nc)],
                                [rng.standard_normal((band.nrings, band.nphi)) for _ in range(nc)])
        alms, maps = _CPU_INPUTS[key] if alms is None else alms, _CPU_INPUTS[key][1] if maps is None else maps
        if isinstance(alms, tuple):
            alms = alms[0]
    jobs = [(0, [0])] if nc == 1 else ([(2, [0, 1])] if nc == 2 else [(0, [0]), (2, [1, 2])])
    nm = lmax + 1

    def run(stride):
        """-> (Legendre seconds, FFT seconds, number of m) summed over both directions and all jobs"""
        leg = fft = 0.0
        nsel = len(range(stride // 2, nm, stride))
        for spin, idx in jobs:
            cpu.alm2map(np.stack([alms[i] for i in idx]), theta, band.phi0, band.nphi, lmax, spin=spin, m_stride=stride, m_offset=stride // 2)
            leg += cpu.last_times[0]; fft += cpu.last_times[1]
            cpu.map2alm(np.stack([maps[i] for i in idx]), theta, w, band.phi0, lmax, spin=spin, m_stride=stride, m_offset=stride // 2)
            leg += cpu.last_times[0]; fft += cpu.last_times[1]
        return leg, fft, nsel

    thr = cpu.threads
    stride = max(1, nm // (2 * thr))                # calibration: two m per thread
    leg, fft, nsel = run(stride)
    per_m = leg / nsel
    want = max(2 * thr, int(max(0.0, target_s - 2.0 * fft) / max(per_m, 1e-9)))
    if want >= nm or stride == 1:
        stride2 = 1
    else:
        stride2 = max(1, nm // want)
    if stride2 < stride:
        leg, fft, nsel = run(stride2); stride = stride2
    full_ms = 1e3 * (leg * nm / nsel + fft)
    out = {"value": full_ms, "unit": "ms", "cores": thr, "kind": "port",
           "sample": "oracle/sht_cpu.c (libsharp2-style CPU implementation: ring-pair folding, scaled seek, pruning, OpenMP over m, "
                     "SIMD over rings; not libsharp2 itself): alm2map + map2alm on every %d-th m (%d of %d m, Legendre %.1f s, "
                     "extrapolated linearly in m) + all ring FFTs (%.1f s)" % (stride, nsel, nm, leg, fft)}
    # how good a stand-in for libsharp2 is it?  Its Legendre rate (un-pruned SURVEY 8(d) flop count, as for the GPU roofline)
    # against the host's measured FP64 FMA peak on the same threads.  libsharp2's hand-vectorised kernels reach ~50-60 % of peak
    # on the executed (pruned, ~2/3 of nominal) work, i.e. ~0.8-0.9 of peak in these nominal units.
    try:
        peak = cpu.fma_peak_gflops(0.4)
        nom = 2.0 * algorithmic_flops(n, band.nrings, nc)
        rate = nom / max(leg * nm / nsel, 1e-9) * 1e-9
        out.update({"host_fma_peak_gflops": peak, "legendre_gflops_nominal": rate, "frac_of_host_peak": rate / peak})
    except Exception as ex:
        out["host_fma_peak_error"] = repr(ex)[:100]
    return out


def cpu_calibration(target="C3"):
    """The sampling of cpu_baseline checked against a FULL run (every m) of the same code on a config where that is affordable:
    ratio = full / extrapolated."""
    import pixsht
    from oracle import get_cpu_sht, cc_geometry, nalm as nalm_of
    wl = WORKLOADS[target]
    est = cpu_baseline(wl, target_s=3.0)
    cpu = get_cpu_sht()
    res = wl["res_arcmin"] * pixsht.arcminute
    shape, wcs = pixsht.fullsky_geometry(res)
    band = pixsht.sht_band(shape, wcs)
    lmax, nc = wl["lmax"], wl["ncomp"]
    theta, w = cc_geometry(band.nrings_total, band.nphi)
    alms, maps = _CPU_INPUTS[(wl["res_arcmin"], lmax, nc)]
    jobs = [(0, [0])] if nc == 1 else ([(2, [0, 1])] if nc == 2 else [(0, [0]), (2, [1, 2])])
    t = 0.0
    for spin, idx in jobs:
        cpu.alm2map(np.stack([alms[i] for i in idx]), theta, band.phi0, band.nphi, lmax, spin=spin)
        t += sum(cpu.last_times)
        cpu.map2alm(np.stack([maps[i] for i in idx]), theta, w, band.phi0, lmax, spin=spin)
        t += sum(cpu.last_times)
    _CPU_INPUTS.clear()
    return {"workload": target, "full_run_ms": 1e3 * t, "sampled_estimate_ms": est["value"], "full_over_estimate": 1e3 * t / est["value"],
            "cores": est["cores"]}


# ------------------------------------------------------------------------------------------------------------------
# parity of the timed path's own outputs against the long-double oracle (the checker; after the timed region)
# ------------------------------------------------------------------------------------------------------------------
def parity_sampled(band, lmax, nc, alms, maps, outs, f64=True, nrings_sample=3, m_sample=2):
    """alms[c]: the step's input alm (host, complex); maps[c]: its alm2map output as (nrings, nx) arrays in the caller's row
    order; outs[c]: the map2alm output of those maps.  Checks alm2map on sampled rings and map2alm on sampled m against
    oracle/sht_oracle.c (80-bit long double, naive sums).  Returns rel-RMS errors over the samples."""
    from oracle import get_oracle, cc_geometry, alm_index
    orc = get_oracle("ld")
    theta, w = cc_geometry(band.nrings_total, band.nphi, band.ring_first, band.nrings)
    nr = band.nrings
    rings = sorted(set(int(round(x)) for x in np.linspace(nr * 0.07, nr * 0.5, nrings_sample)))
    msel = sorted(set(int(round(x)) for x in np.linspace(lmax * 0.11, lmax * 0.83, m_sample)))
    jobs = [(0, [0])] if nc == 1 else ([(2, [0, 1])] if nc == 2 else [(0, [0]), (2, [1, 2])])
    num = den = 0.0
    anum = aden = 0.0
    fy = slice(None, None, -1) if band.flipy else slice(None)
    fx = slice(None, None, -1) if band.flipx else slice(None)
    for spin, idx in jobs:
        a = np.stack([np.asarray(alms[c]).astype(np.complex128) for c in idx])
        ref = orc.alm2map(a, theta[rings], band.phi0, band.nphi, lmax, spin=spin)
        for k, c in enumerate(idx):
            for i, r in enumerate(rings):
                row = (nr - 1 - r) if band.flipy else r
                g = np.asarray(maps[c][row], dtype=np.float64)[fx]
                num += float(np.sum((g - ref[k, i, :band.nx]) ** 2)); den += float(np.sum(ref[k, i, :band.nx] ** 2))
        bandmaps = np.zeros((len(idx), nr, band.nphi))
        for k, c in enumerate(idx):
            bandmaps[k, :, :band.nx] = np.asarray(maps[c], dtype=np.float64)[fy, fx]
        for m in msel:
            # every (lmax+1)-th m starting at m: exactly this m
            refa = orc.map2alm(bandmaps, theta, w, band.phi0, lmax, spin=spin, m_stride=lmax + 1, m_offset=m)
            sl = slice(alm_index(lmax, m, m), alm_index(lmax, lmax, m) + 1)
            for k, c in enumerate(idx):
                got = np.asarray(outs[c][sl]).astype(np.complex128)
                anum += float(np.sum(np.abs(got - refa[k][sl]) ** 2)); aden += float(np.sum(np.abs(refa[k][sl]) ** 2))
    tol = 1e-10 if f64 else 1e-5
    e1, e2 = math.sqrt(num / den), math.sqrt(anum / aden)
    return {"alm2map_rel_rms": e1, "map2alm_rel_rms": e2, "tolerance": tol, "ok": bool(e1 <= tol and e2 <= tol),
            "checker": "oracle/sht_oracle.c (long double)", "rings": rings, "m": msel}


# ------------------------------------------------------------------------------------------------------------------
def synth_alm_device(torch, nalm, lmax, seed, spin2, device, cdtype):
    g = torch.Generator(device=device)
    g.manual_seed(seed)
    a = torch.randn(nalm, 2, generator=g, device=device, dtype=torch.float64)
    a[:lmax + 1, 1] = 0          # a_l0 real
    if spin2:
        a[0:2] = 0               # m = 0: l = 0, 1
        a[lmax + 1:lmax + 2] = 0  # m = 1: l = 1
    a = torch.view_as_complex(a)
    return a.to(cdtype).contiguous()


DUMP_BYTES = 32 * 10 ** 6     # per dumped file: map.npy + alm.npy stay under 64 MB


def dump_outputs(torch, out_dir, name, tensors):
    """Writes out_dir/<name>.npy: one row per tensor (all of one length), complex values as (re, im) pairs.  When the rows
    together exceed DUMP_BYTES, each keeps the same positions: a sample drawn with a fixed seed, so it depends on the length alone."""
    flat = [torch.view_as_real(t).reshape(-1, 2) if t.is_complex() else t.reshape(-1, 1) for t in tensors]
    n, width = flat[0].shape
    keep = DUMP_BYTES // (len(flat) * width * flat[0].element_size())
    if n > keep:
        idx = torch.from_numpy(np.unique(np.random.default_rng(12345).integers(0, n, keep))).to(flat[0].device)
        flat = [f.index_select(0, idx) for f in flat]
    arr = np.stack([f.cpu().numpy() for f in flat])
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, name + ".npy"), arr[:, :, 0] if width == 1 else arr)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--workload", default="C4", choices=sorted(WORKLOADS))
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-pageable", action="store_true")
    ap.add_argument("--no-calibration", action="store_true")
    ap.add_argument("--no-extras", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs as DIR/map.npy and DIR/alm.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    wl = WORKLOADS[args.workload]
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.dump_outputs and (args.impl != "b200" or world > 1):
        ap.error("--dump-outputs needs the one-process GPU path (--impl b200, one rank)")
    config = {"workload": "%s: %s" % (args.workload, wl["desc"]), "ncomp": wl["ncomp"], "lmax": wl["lmax"],
              "step": "one alm2map + one map2alm", "l2": "inputs larger than L2 (map+alm+phase >> 126 MB)" if args.workload in ("C3", "C4", "C5") else
              "inputs smaller than L2; 256 MB scratch written between timed steps"}

    if args.impl == "reference":
        if rank != 0:
            return
        vals = []
        base = None
        per_step = max(1.0, min(8.0, 150.0 / max(1, args.warmup + args.steps)))   # the whole run stays within a few minutes
        for i in range(args.warmup + args.steps):
            base = cpu_baseline(wl, target_s=per_step)
            if i >= args.warmup:
                vals.append(base["value"])
        v = float(np.mean(vals))
        base["value"] = v
        print(json.dumps({"impl": "reference", "metric": METRIC, "value": v, "unit": "ms", "n_gpus": args.gpus, "steps": args.steps,
                          "warmup": args.warmup, "ms_per_step": v, "higher_is_better": False, "scaling": "strong", "vs_baseline": None,
                          "dtype": "f64", "data": "synthetic", "config": config, "cpu_baseline": base,
                          "e2e": {"value": v, "unit": "ms", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                          "note": "CPU implementation of the Pixell.jl/libsharp2 path with libsharp2's algorithm (oracle/sht_cpu.c); Julia and "
                                  "libsharp2 are not available in this image, so the unmodified reference cannot be run"}))
        return

    import torch
    import pixsht
    from pixsht.transforms import Plan, get_lib, MAP2ALM, ALM2MAP, HOST, DEVICE
    from pixsht.distributed import ShardedSHT

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=device)
    lib = get_lib()
    res = wl["res_arcmin"] * pixsht.arcminute
    shape, wcs = pixsht.fullsky_geometry(res)
    band = pixsht.sht_band(shape, wcs)
    lmax, nc = wl["lmax"], wl["ncomp"]
    f64 = wl["dtype"] == "f64"
    rdt, cdt = (torch.float64, torch.complex128) if f64 else (torch.float32, torch.complex64)
    npdt = np.float64 if f64 else np.float32
    esz = 8 if f64 else 4
    seed0 = 1000 * int(args.workload[1])
    stream = torch.cuda.current_stream(device)
    if "batch" in wl:
        return bench_batch(args, wl, config, torch, pixsht, Plan, lib, band, lmax, device, stream, rdt, cdt, npdt, local_rank,
                           MAP2ALM, ALM2MAP, DEVICE)
    l2_scratch = None if args.workload in ("C3", "C4", "C5") else torch.empty(64 * 1024 * 1024, dtype=torch.float32, device=device)

    def flush_l2():
        if l2_scratch is not None:
            l2_scratch.zero_()

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize(device)

    def timed(fn, nwarm, nsteps):
        for _ in range(nwarm):
            fn(); flush_l2()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(nsteps):
            fn(); flush_l2()
        e1.record(stream)
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=device, dtype=torch.float64)
        if dist is not None:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()) / nsteps

    launches = 0
    stage = {}
    parity = None
    e2e_pageable = None
    one_process = None
    if world == 1:
        plan = Plan(band, lmax, dtype=npdt)
        lib.check(lib.lib.pixsht_plan_set_stream(plan.handle, ctypes.c_void_p(stream.cuda_stream), 1))
        nalm = plan.nalm
        d_alm = [synth_alm_device(torch, nalm, lmax, seed0 + c, c > 0, device, cdt) for c in range(nc)]
        d_out = [torch.empty_like(a) for a in d_alm]
        d_map = [torch.empty(band.nx * band.nrings, dtype=rdt, device=device) for _ in range(nc)]
        acc = {"leg": 0.0, "fft": 0.0, "n": 0, "launches": 0, "synth0": 0.0, "synth2": 0.0, "anal0": 0.0, "anal2": 0.0,
               "fft_a2m": 0.0, "fft_m2a": 0.0}

        def step_dev():
            plan.execute_ptrs(ALM2MAP, [a.data_ptr() for a in d_alm], [m.data_ptr() for m in d_map], DEVICE)
            t1 = plan.timings(); l1 = plan.info()["launches"]
            plan.execute_ptrs(MAP2ALM, [a.data_ptr() for a in d_out], [m.data_ptr() for m in d_map], DEVICE)
            t2 = plan.timings(); l2 = plan.info()["launches"]
            acc["leg"] += t1["legendre"] + t2["legendre"]; acc["fft"] += t1["fft"] + t2["fft"]; acc["n"] += 1
            acc["synth0"] += t1["leg_spin0"]; acc["synth2"] += t1["leg_spin2"]; acc["anal0"] += t2["leg_spin0"]; acc["anal2"] += t2["leg_spin2"]
            acc["fft_a2m"] += t1["fft"]; acc["fft_m2a"] += t2["fft"]
            acc["launches"] = l1 + l2

        clk = ClockSampler(local_rank); clk.start()
        for _ in range(args.warmup):
            step_dev(); flush_l2()
        for k in list(acc):
            acc[k] = 0 if k in ("n", "launches") else 0.0
        ms_dev = timed(step_dev, 0, args.steps)
        clocks = clk.stop()
        if args.dump_outputs:
            dump_outputs(torch, args.dump_outputs, "map", d_map)
            dump_outputs(torch, args.dump_outputs, "alm", d_out)
        leg_ms, fft_ms = acc["leg"] / acc["n"], acc["fft"] / acc["n"]
        launches = acc["launches"] * args.steps
        stage = {"legendre_ms": leg_ms, "fft_ms": fft_ms}
        kern_ms = {k: acc[k] / acc["n"] for k in ("synth0", "synth2", "anal0", "anal2", "fft_a2m", "fft_m2a")}
        work = {}
        if nc != 2:
            work[0] = plan.work(0)
        if nc >= 2:
            work[2] = plan.work(2)
        h2d = d2h = 0
        e2e = None
        host_maps = host_alms = None
        if not args.no_e2e:
            h_alm = [torch.empty(nalm, dtype=cdt).pin_memory() for _ in range(nc)]
            h_out = [torch.empty(nalm, dtype=cdt).pin_memory() for _ in range(nc)]
            h_map = [torch.empty(band.nx * band.nrings, dtype=rdt).pin_memory() for _ in range(nc)]
            for h, d in zip(h_alm, d_alm):
                h.copy_(d)
            torch.cuda.synchronize(device)

            def step_host():
                plan.execute_ptrs(ALM2MAP, [a.data_ptr() for a in h_alm], [m.data_ptr() for m in h_map], HOST)
                plan.execute_ptrs(MAP2ALM, [a.data_ptr() for a in h_out], [m.data_ptr() for m in h_map], HOST)

            ms_e2e = timed(step_host, min(args.warmup, 3), args.steps)
            h2d = sum(a.numel() * a.element_size() for a in h_alm) + sum(m.numel() * m.element_size() for m in h_map)
            d2h = sum(m.numel() * m.element_size() for m in h_map) + sum(a.numel() * a.element_size() for a in h_out)
            e2e = {"value": ms_e2e, "unit": "ms", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                   "api": "pixsht_execute(..., PIXSHT_HOST) on pinned host buffers"}
            # the two directions on their own (same buffers): shows where the copies are not hidden
            e2e["alm2map_ms"] = timed(lambda: plan.execute_ptrs(ALM2MAP, [a.data_ptr() for a in h_alm], [m.data_ptr() for m in h_map], HOST), 1, max(1, min(args.steps, 3)))
            e2e["map2alm_ms"] = timed(lambda: plan.execute_ptrs(MAP2ALM, [a.data_ptr() for a in h_out], [m.data_ptr() for m in h_map], HOST), 1, max(1, min(args.steps, 3)))
            # sanity: device-resident and host paths agree
            chk = float((h_out[0].to(device) - d_out[0]).abs().max().item())
            e2e["host_vs_device_maxabs"] = chk
            host_maps = [m.numpy().reshape(band.nrings, band.nx).astype(np.float64, copy=False) for m in h_map]
            host_alms = [a.numpy().astype(np.complex128, copy=False) for a in h_alm]
            # the same call on ordinary (pageable) host arrays -- what a caller who did not allocate through pixsht_host_alloc /
            # pixsht_host_register gets
            if not args.no_pageable:
                p_alm = [np.array(a.numpy()) for a in h_alm]
                p_out = [np.empty_like(a) for a in p_alm]
                p_map = [np.empty(band.nx * band.nrings, dtype=npdt) for _ in range(nc)]

                def step_pageable():
                    plan.execute_ptrs(ALM2MAP, [a.ctypes.data for a in p_alm], [m.ctypes.data for m in p_map], HOST)
                    plan.execute_ptrs(MAP2ALM, [a.ctypes.data for a in p_out], [m.ctypes.data for m in p_map], HOST)

                ms_pg = timed(step_pageable, 1, max(1, min(args.steps, 3)))
                e2e_pageable = {"value": ms_pg, "unit": "ms", "ratio_to_pinned": ms_pg / ms_e2e,
                                "api": "pixsht_execute(..., PIXSHT_HOST) on pageable numpy arrays (staged through the library's pinned "
                                       "bounce buffers by its copy threads)",
                                "maxabs_vs_pinned": float(np.max(np.abs(p_out[0] - h_out[0].numpy())))}
                del p_alm, p_out, p_map
            # parity of the timed path's own output (the host-pointer call) against the long-double oracle
            if not args.no_parity:
                parity = parity_sampled(band, lmax, nc, [a.numpy() for a in h_alm], [m.numpy().reshape(band.nrings, band.nx) for m in h_map],
                                        [a.numpy() for a in h_out], f64=f64)
        nrings = band.nrings
        plan_info = plan.info()
    else:
        sht = ShardedSHT(band, lmax, device=device, dtype=rdt)
        nalm = sht.nalm
        a, b = sht.map_rows()
        d_alm = [synth_alm_device(torch, nalm, lmax, seed0 + c, c > 0, device, cdt) for c in range(nc)]
        d_out = [torch.empty_like(x) for x in d_alm]
        d_slab = [torch.empty((b - a) * band.nx, dtype=rdt, device=device) for _ in range(nc)]
        acc = {"a2m": None, "m2a": None}

        def step_dev():
            sht.alm2map(d_alm, d_slab)
            sht.map2alm(d_slab, d_out)

        clk = ClockSampler(local_rank); clk.start()
        ms_dev = timed(step_dev, args.warmup, args.steps)
        clocks = clk.stop()
        s1, s2 = sht.stage_ms("alm2map"), sht.stage_ms("map2alm")
        leg_ms, fft_ms, a2a_ms = s1[0] + s2[2], s1[2] + s2[0], s1[1] + s2[1]
        t = torch.tensor([leg_ms, fft_ms, a2a_ms], device=device, dtype=torch.float64)
        per_rank = [torch.zeros_like(t) for _ in range(world)]
        dist.all_gather(per_rank, t)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        leg_ms, fft_ms, a2a_ms = [float(x) for x in t.tolist()]
        stage = {"legendre_ms": leg_ms, "fft_ms": fft_ms, "exchange_ms": a2a_ms,
                 "per_rank": {"legendre_ms": [round(float(x[0]), 3) for x in per_rank], "fft_ms": [round(float(x[1]), 3) for x in per_rank],
                              "barrier_ms": [round(float(x[2]), 3) for x in per_rank], "m_per_rank": None},
                 "exchange": "fused: the FFT kernels' row loads/stores fetch/put every m in the phase buffer of the GPU that owns it "
                             "(peer memory over NVLink, 256-byte runs); exchange_ms is the stage-ordering barrier (includes waiting "
                             "for the slowest rank)"}
        nfam = 2 if nc == 3 else 1   # spin families: each costs a prep + a synthesis launch one way and an analysis launch back
        # per rank and step, counted from the stage calls: per spin family a record preparation + its synthesis launch(es) one way and
        # its analysis launch(es) back (T: up to three each -- two-step kernels plus the polar and equatorial chunks on the standard
        # ones -- and a second preparation), one FFT launch per direction
        nT = 3 if nc != 2 else 0
        launches = ((2 + 2 * nT if nT else 0) + (3 if nc >= 2 else 0) + 2) * args.steps
        # ---- the ONE-PROCESS path (include/pixsht.h: pixsht_plan_create_multi): rank 0 alone drives all N GPUs through the
        # blocking C-ABI call on whole host arrays -- what a Julia caller gets.  The other ranks idle at a host-side (gloo)
        # barrier meanwhile, so that nothing of theirs runs on the GPUs.
        gloo = dist.new_group(backend="gloo")
        shm = "/dev/shm/pixsht_bench_%d_" % int(os.environ.get("MASTER_PORT", "0"))
        e2e = None
        nrings = band.nrings
        torch.cuda.synchronize(device)
        dist.barrier(group=gloo)
        if rank == 0 and not args.no_e2e:
            import time
            mplan = Plan(band, lmax, dtype=npdt, devices=list(range(world)))
            # page-locked host arrays from the library's own allocator (pixsht_host_alloc: what the Julia binding hands out;
            # NUMA-interleaved on a multi-socket host because every GPU pulls its own columns / rows)
            host_ptrs = []

            def host_array(n, np_dtype):
                ptr = ctypes.c_void_p()
                lib.check(lib.lib.pixsht_host_alloc(ctypes.byref(ptr), int(n) * np.dtype(np_dtype).itemsize))
                host_ptrs.append(ptr)
                arr = np.ctypeslib.as_array(ctypes.cast(ptr, ctypes.POINTER(ctypes.c_uint8)), shape=(int(n) * np.dtype(np_dtype).itemsize,)).view(np_dtype)
                return torch.from_numpy(arr)

            npc = np.complex128 if f64 else np.complex64
            h_alm = [host_array(nalm, npc) for _ in range(nc)]
            h_out = [host_array(nalm, npc) for _ in range(nc)]
            h_map = [host_array(band.nx * band.nrings, npdt) for _ in range(nc)]
            for h, d in zip(h_alm, d_alm):
                h.copy_(d)
            torch.cuda.synchronize(device)
            pa, po, pm = [a.data_ptr() for a in h_alm], [a.data_ptr() for a in h_out], [m.data_ptr() for m in h_map]

            def step_host():
                mplan.execute_ptrs(ALM2MAP, pa, pm, HOST)
                t1 = mplan.timings()["compute_span"]
                mplan.execute_ptrs(MAP2ALM, po, pm, HOST)
                return t1 + mplan.timings()["compute_span"]

            for _ in range(min(args.warmup, 3)):
                step_host()
            t0 = time.perf_counter()
            span = 0.0
            for _ in range(args.steps):
                span += step_host()
            ms_e2e = 1e3 * (time.perf_counter() - t0) / args.steps
            nbytes = sum(x.numel() * x.element_size() for x in h_alm) + sum(x.numel() * x.element_size() for x in h_map)
            e2e = {"value": ms_e2e, "unit": "ms", "h2d_bytes_per_step": nbytes, "d2h_bytes_per_step": nbytes,
                   "device_span_ms": span / args.steps,
                   "timing": "host wall clock around the blocking calls (they return when the caller's arrays are complete); "
                             "device_span_ms = max over the GPUs of the CUDA-event span of each call",
                   "api": "pixsht_execute on a pixsht_plan_create_multi plan: one process, %d GPUs, whole page-locked host arrays from "
                          "pixsht_host_alloc (each GPU copies its alm columns / map rows itself); no torch, no NCCL on this path" % world,
                   "host_numa": os.environ.get("PIXSHT_HOST_NUMA", "interleave")}
            # the same plan with the data already distributed over the GPUs (nothing copied): pixsht_execute_sharded
            try:
                sh = mplan.shards()
                sa, sm, so = [], [], []
                for (dv, r0, nr, ml) in sh:
                    td = torch.device("cuda", dv)
                    sa.append([a.to(td) for a in d_alm])
                    sm.append([torch.empty(nr * band.nx, dtype=rdt, device=td) for _ in range(nc)])
                    so.append([torch.empty(nalm, dtype=cdt, device=td) for _ in range(nc)])
                flat = lambda x: [t.data_ptr() for per in x for t in per]
                fa, fm, fo = flat(sa), flat(sm), flat(so)

                def step_sharded():
                    mplan.execute_sharded_ptrs(ALM2MAP, nc, fa, fm)
                    t1 = mplan.timings()["compute_span"]
                    mplan.execute_sharded_ptrs(MAP2ALM, nc, fo, fm)
                    return t1 + mplan.timings()["compute_span"]

                for _ in range(2):
                    step_sharded()
                t0 = time.perf_counter(); span = 0.0
                for _ in range(args.steps):
                    span += step_sharded()
                one_process = {"device_resident_ms": 1e3 * (time.perf_counter() - t0) / args.steps, "device_span_ms": span / args.steps,
                               "api": "pixsht_execute_sharded: shards of alm / map resident on their GPUs, one process"}
                del sa, sm, so
            except Exception as ex:
                one_process = {"error": repr(ex)[:200]}
            # parity of the one-process path's own output against the long-double oracle
            if not args.no_parity:
                parity = parity_sampled(band, lmax, nc, [a.numpy() for a in h_alm], [m.numpy().reshape(band.nrings, band.nx) for m in h_map],
                                        [a.numpy() for a in h_out], f64=f64)
            for c in range(nc):
                np.save(shm + "map%d.npy" % c, h_map[c].numpy())
                np.save(shm + "alm%d.npy" % c, h_out[c].numpy())
            mplan.close()
            del h_alm, h_out, h_map
            for ptr in host_ptrs:
                lib.lib.pixsht_host_free(ptr)
        dist.barrier(group=gloo)
        # ---- every rank: its device-resident slab / alm columns (the torchrun pipeline timed as `value`) against the one-process
        # result: the same (m, ring) sums wherever they run -> maps bit for bit, alm to rounding (atomic accumulation order)
        cross = torch.zeros(2, dtype=torch.float64, device=device)
        if not args.no_e2e and os.path.exists(shm + "map0.npy"):
            for c in range(nc):
                ref = np.load(shm + "map%d.npy" % c, mmap_mode="r")[a * band.nx:b * band.nx]
                got = d_slab[c].cpu().numpy()
                cross[0] = max(float(cross[0]), float(np.max(np.abs(got - ref))) / max(float(np.max(np.abs(ref))), 1e-300))
                refa = np.load(shm + "alm%d.npy" % c, mmap_mode="r")
                o = d_out[c].cpu().numpy()
                for (s0, s1) in sht.alm_columns()[::max(1, sht.nm // 16)]:
                    den = max(float(np.sqrt(np.sum(np.abs(refa[s0:s1]) ** 2))), 1e-300)
                    cross[1] = max(float(cross[1]), float(np.sqrt(np.sum(np.abs(o[s0:s1] - refa[s0:s1]) ** 2))) / den)
        dist.all_reduce(cross, op=dist.ReduceOp.MAX)
        dist.barrier(group=gloo)
        if rank == 0:
            for c in range(nc):
                for nm_ in ("map%d.npy" % c, "alm%d.npy" % c):
                    try:
                        os.remove(shm + nm_)
                    except OSError:
                        pass
            if parity is not None:
                parity["ranks_vs_one_process"] = {"map_maxabs_rel": float(cross[0]), "alm_rel_rms_max": float(cross[1]),
                                                  "note": "each torchrun rank's slab and sampled alm columns (the pipeline timed as `value`) "
                                                          "against the one-process result that the oracle check above covers"}
                tol = parity["tolerance"]
                parity["ok"] = bool(parity["ok"] and float(cross[0]) <= tol and float(cross[1]) <= tol)
        plan_info = {"npairs": math.ceil(nrings / 2), "sm_count": None}
        host_maps = host_alms = None
        kern_ms, work = None, None
        sht.close()

    if rank != 0:
        if dist is not None:
            dist.barrier(); dist.destroy_process_group()
        return

    # ---- rooflines -----------------------------------------------------------------------------------------------
    peaks = {}
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            peaks = json.load(f)
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    hbm_src = "MEASURED_PEAKS.json (of measured)" if "hbm_gbs" in peaks else "fallback 6650 GB/s (of fallback)"
    fp64_peak, fp32_peak = lib.measure_fma_peak(local_rank)
    peak_src = ("pixsht_measure_fma_peak: FP64 FMA probe (16 independent accumulators per thread, one warp-uniform operand) "
                "measured on this GPU in this run; datasheet FP64 vector peak 37.2 TFLOP/s at 1965 MHz; MEASURED_PEAKS.json has no FP64 figure")
    flops = 2.0 * algorithmic_flops(nalm, nrings, nc)            # both directions, all ranks together
    leg_tf = flops / world / (leg_ms * 1e-3) / 1e12             # per GPU
    stage_roof = {"kernel": "leg_synth<0|2> + leg_anal<0|2> (Legendre stage, both directions)", "achieved": leg_tf, "peak": fp64_peak,
                  "unit": "TFLOP/s", "frac": leg_tf / fp64_peak, "algorithmic_flop_per_step": flops,
                  "note": "un-pruned, north/south-folded count of SURVEY.md 8(d); per GPU"}
    traffic = {}
    try:
        with open(os.path.join(ROOT, "profiles", "r02", "ncu_dram_traffic.json")) as f:   # ncu capture of the kernels as they are now
            traffic = json.load(f).get(args.workload, {})
    except Exception:
        pass
    if kern_ms is not None:
        # per kernel: algorithmic flop = 2 * (4 | 12) * nominal (l, m, ring pair) steps (SURVEY.md 8(d)); "executed" is the share
        # of those steps the activation table lets the kernel run, so achieved * executed / peak is the FP64 pipe utilisation
        kernels = []
        for name, spin, key in (("leg_synth_2s<%d> + leg_synth<0,%d>" % (plan_info["R0"], plan_info["R0"]), 0, "synth0"), ("leg_synth<2,%d>" % plan_info["R2"], 2, "synth2"),
                                ("leg_anal_2s<%d> + leg_anal<0,%d>" % (plan_info["R0a"], plan_info["R0a"]), 0, "anal0"), ("leg_anal<2,%d>" % plan_info["R2a"], 2, "anal2")):
            if spin not in work:
                continue
            ex, nom = work[spin]
            fl = 2.0 * (4 if spin == 0 else 12) * nom
            tf = fl / (kern_ms[key] * 1e-3) / 1e12
            kernels.append({"kernel": name, "ms": kern_ms[key], "algorithmic_flop": fl, "achieved": tf, "frac": tf / fp64_peak,
                            "executed_share": ex / nom, "fp64_pipe_utilisation": tf * ex / nom / fp64_peak,
                            "traffic": traffic.get(name.split(" + ")[-1].split(",")[0] + ">")})
        dom = max(kernels, key=lambda k: k["ms"])
        roofline = {"bound": "fp64_fma", "kernel": dom["kernel"], "achieved": dom["achieved"], "peak": fp64_peak, "unit": "TFLOP/s",
                    "frac": dom["frac"], "traffic": dom["traffic"], "peak_source": peak_src,
                    "algorithmic_flop_per_launch": dom["algorithmic_flop"], "executed_share": dom["executed_share"],
                    "fp64_pipe_utilisation": dom["fp64_pipe_utilisation"], "launch_ms": dom["ms"],
                    "note": "dominant kernel; algorithmic = un-pruned, north/south-folded count of SURVEY.md 8(d) (12 FP64 FMA-class ops per "
                            "(l, m, ring pair) for spin 2); timed with CUDA events around the launch inside pixsht_execute",
                    "traffic_note": "dram bytes per launch from ncu (profiles/r02/ncu_c4_metrics_final.csv). The kernel is FP64 bound; in the default "
                                    "chunk-major grid order every chunk of ring pairs re-reads the (alpha, delta, gamma) column of its m and re-touches "
                                    "the alm lines it adds to (about 56 B per (l, m, chunk): 154 GB = 0.7 TB/s at C4, 11 % of the HBM rate), against 9 GB "
                                    "in m-major order (PIXSHT_LEG_ORDER=0), which runs 3 % slower (DESIGN.md 4.1)",
                    "kernels": kernels, "legendre_stage": stage_roof}
    else:
        roofline = dict(stage_roof, bound="fp64_fma", traffic=None, peak_source=peak_src)
    fft_bytes = 2.0 * (nc * band.nx * nrings * esz + nc * (lmax + 1) * nrings * 16)
    roofline_fft = {"bound": "hbm", "kernel": "fft_phase2map_edge + fft_map2phase_edge" if plan_info.get("fft", {}).get("edge_fused") else "fft_phase2map + fft_map2phase", "achieved": fft_bytes / world / (fft_ms * 1e-3) / 1e9,
                    "peak": hbm_peak, "unit": "GB/s", "traffic": traffic.get("fft"), "peak_source": hbm_src,
                    "algorithmic_bytes_per_step": fft_bytes}
    roofline_fft["frac"] = roofline_fft["achieved"] / hbm_peak

    line = {"metric": METRIC, "value": ms_dev, "unit": "ms", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_dev, "higher_is_better": False, "scaling": "strong", "vs_baseline": None,
            "dtype": wl["dtype"], "data": "synthetic", "config": config, "clocks": clocks, "gpu_launches": launches,
            "stages": stage, "roofline": roofline, "roofline_fft": roofline_fft, "fp32_fma_peak_tflops": fp32_peak,
            "transforms_per_s": 2.0 * 1e3 / ms_dev, "plan": {k: plan_info.get(k) for k in ("npairs", "sm_count", "R0", "R2", "R0a", "R2a")}}
    if e2e is not None:
        line["e2e"] = e2e
    if e2e_pageable is not None:
        line["e2e_pageable"] = e2e_pageable
    if parity is not None:
        line["parity"] = parity
    if one_process is not None:
        line["one_process"] = one_process
    if world == 1 and not args.no_cpu_baseline:
        try:
            line["cpu_baseline"] = cpu_baseline(wl, maps=host_maps, alms=host_alms)
            if args.workload in ("C4", "C5") and not args.no_calibration:
                del host_maps, host_alms
                line["cpu_baseline"]["calibration"] = cpu_calibration("C3")
        except Exception as ex:  # never lose the GPU numbers to a baseline problem
            line["cpu_baseline"] = dict(line.get("cpu_baseline") or {}, error=repr(ex))
    if world == 1 and args.workload == "C4" and not args.no_extras:
        line["extra"] = run_extras(args)
    print(json.dumps(line))
    if dist is not None:
        dist.barrier(); dist.destroy_process_group()
    if parity is not None and not parity["ok"]:
        raise SystemExit("bench.py: PARITY FAILURE against the oracle: %s" % json.dumps(parity))


def run_extras(args):
    """The other single-GPU BASELINE configs, measured in the same driver run (each in a fresh process, after this process has
    released the GPU's memory is not required: they are small): C3 (2' IQU F64), C2 (4' T F32) and the 64-map sweep C2x64.
    Returns {workload: trimmed bench line}."""
    out = {}
    for name in ("C3", "C2", "C2x64"):
        cmd = [sys.executable, os.path.abspath(__file__), "--workload", name, "--steps", "3", "--warmup", "3", "--no-cpu-baseline",
               "--no-pageable", "--no-extras"]
        try:
            r = subprocess.run(cmd, capture_output=True, text=True, timeout=300)
            d = json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("{")][-1])
            keep = {k: d.get(k) for k in ("value", "unit", "ms_per_step", "dtype", "clocks", "gpu_launches", "stages", "e2e", "parity",
                                          "sims_per_s", "one_by_one_ms", "batch_speedup", "transforms_per_s")}
            keep["config"] = d.get("config", {}).get("workload")
            rf = d.get("roofline") or {}
            keep["roofline"] = {k: rf.get(k) for k in ("bound", "kernel", "achieved", "peak", "unit", "frac", "fp64_pipe_utilisation")}
            if d.get("roofline_fft"):
                keep["roofline_fft"] = {k: d["roofline_fft"].get(k) for k in ("achieved", "peak", "unit", "frac")}
            out[name] = keep
        except Exception as ex:
            out[name] = {"error": repr(ex)[:200]}
    return out


def bench_batch(args, wl, config, torch, pixsht, Plan, lib, band, lmax, device, stream, rdt, cdt, npdt, local_rank, MAP2ALM, ALM2MAP, DEVICE):
    """Simulation sweep: B independent T transforms on one geometry, batched (pixsht_execute_batch: four maps per recurrence)
    against the same B transforms issued one by one.  Device-resident, one GPU."""
    B = wl["batch"]
    plan = Plan(band, lmax, dtype=npdt)
    lib.check(lib.lib.pixsht_plan_set_stream(plan.handle, ctypes.c_void_p(stream.cuda_stream), 1))
    nalm = plan.nalm
    alm = [synth_alm_device(torch, nalm, lmax, 5000 + i, False, device, cdt) for i in range(B)]
    out = [torch.empty_like(a) for a in alm]
    mp = [torch.empty(band.nx * band.nrings, dtype=rdt, device=device) for _ in range(B)]

    def run(fn):
        for _ in range(args.warmup):
            fn()
        torch.cuda.synchronize(device)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(args.steps):
            fn()
        e1.record(stream)
        torch.cuda.synchronize(device)
        return e0.elapsed_time(e1) / args.steps

    def batched():
        plan.execute_batch_ptrs(ALM2MAP, [a.data_ptr() for a in alm], [m.data_ptr() for m in mp], DEVICE)
        plan.execute_batch_ptrs(MAP2ALM, [a.data_ptr() for a in out], [m.data_ptr() for m in mp], DEVICE)

    def one_by_one():
        for i in range(B):
            plan.execute_ptrs(ALM2MAP, [alm[i].data_ptr()], [mp[i].data_ptr()], DEVICE)
            plan.execute_ptrs(MAP2ALM, [out[i].data_ptr()], [mp[i].data_ptr()], DEVICE)

    clk = ClockSampler(local_rank); clk.start()
    ms_b = run(batched)
    clocks = clk.stop()
    if args.dump_outputs:      # before one_by_one() overwrites the buffers
        dump_outputs(torch, args.dump_outputs, "map", mp)
        dump_outputs(torch, args.dump_outputs, "alm", out)
    ms_s = run(one_by_one)
    fp64_peak, _ = lib.measure_fma_peak(local_rank)
    # end to end: the same sweep through the host-pointer call on pinned buffers (H2D + D2H inside the timed region)
    e2e = None
    if not args.no_e2e:
        from pixsht._lib import HOST
        try:
            h_alm = [torch.empty(nalm, dtype=cdt).pin_memory() for _ in range(B)]
            h_out = [torch.empty(nalm, dtype=cdt).pin_memory() for _ in range(B)]
            h_map = [torch.empty(band.nx * band.nrings, dtype=rdt).pin_memory() for _ in range(B)]
            for h, d in zip(h_alm, alm):
                h.copy_(d)
            torch.cuda.synchronize(device)

            def batched_host():
                plan.execute_batch_ptrs(ALM2MAP, [a.data_ptr() for a in h_alm], [m.data_ptr() for m in h_map], HOST)
                plan.execute_batch_ptrs(MAP2ALM, [a.data_ptr() for a in h_out], [m.data_ptr() for m in h_map], HOST)

            ms_h = run(batched_host)
            nbytes = sum(x.numel() * x.element_size() for x in h_alm) + sum(x.numel() * x.element_size() for x in h_map)
            e2e = {"value": ms_h, "unit": "ms", "h2d_bytes_per_step": nbytes, "d2h_bytes_per_step": nbytes,
                   "api": "pixsht_execute_batch(..., PIXSHT_HOST) on pinned host buffers",
                   "overlap": bool(int(os.environ.get("PIXSHT_BATCH_OVERLAP", "0") or 0)),
                   "host_vs_device_maxabs": float((h_out[0].to(device) - out[0]).abs().max().item())}
        except Exception as ex:   # the device-resident numbers above stand on their own
            e2e = {"unavailable": str(ex)[:200]}
    nom = 2.0 * 2.0 * 4 * nalm * math.ceil(band.nrings / 2) * B      # flop the B single transforms would take, both directions
    print(json.dumps({"metric": METRIC, "value": ms_b, "unit": "ms", "n_gpus": 1, "steps": args.steps, "warmup": args.warmup,
                      "ms_per_step": ms_b, "higher_is_better": False, "scaling": "strong", "vs_baseline": None, "dtype": wl["dtype"],
                      "data": "synthetic", "config": dict(config, batch=B, step="alm2map + map2alm of all %d maps" % B), "clocks": clocks,
                      "sims_per_s": 1e3 * B / ms_b, "one_by_one_ms": ms_s, "one_by_one_sims_per_s": 1e3 * B / ms_s,
                      "batch_speedup": ms_s / ms_b, "e2e": e2e,
                      "roofline": {"bound": "fp64_fma", "kernel": "leg_synth_b + leg_anal_b (+ ring FFTs) of the whole sweep",
                                   "achieved": nom / (ms_b * 1e-3) / 1e12, "peak": fp64_peak, "unit": "TFLOP/s",
                                   "frac": nom / (ms_b * 1e-3) / 1e12 / fp64_peak, "traffic": None,
                                   "note": "algorithmic = 4 FP64 ops per (l, m, ring pair) and map, as for single transforms; the batched "
                                           "kernels execute 2 + 2 NB per NB maps, so frac can exceed 1"}}))


if __name__ == "__main__":
    main()
