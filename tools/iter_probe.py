#!/usr/bin/env python
"""Cost of the iterative map2alm (pixsht_map2alm_iter) at C3 and C4 (full-sky CAR 2' / 1', IQU, Float64), one GPU.

For niter = 0, 1, 2, 3, with device pointers and with page-locked host pointers: the time per call (host clock around the call,
which synchronises; median of --reps after one warm-up), its ratio to niter * (alm2map + map2alm) + map2alm with each of those
timed alone in the same run and the same memory kind, and the kernels launched.  A ratio below 1 is what the loop saves over
separate calls: with host pointers, the copies of every intermediate map and alm; with device pointers, nothing but launch
gaps (the loop runs the same kernels plus one residual pass per iteration).  The card's name and power limit are printed with
the numbers.  Usage: iter_probe.py [--workloads C3 C4] [--reps 3] [--out FILE.json]"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "pixell.jl_b200")]
import torch  # noqa: E402
import pixsht  # noqa: E402
from pixsht import _lib  # noqa: E402
from pixsht.transforms import Plan  # noqa: E402

WORKLOADS = {"C3": (2.0, 5400), "C4": (1.0, 10800)}
NITERS = (0, 1, 2, 3)


def card():
    name = torch.cuda.get_device_name(0)
    try:
        power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                               capture_output=True, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        power = "unknown"
    return name, power or "unknown"


def timed(fn, reps):
    fn()                                   # warm-up
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        ts.append((time.perf_counter() - t0) * 1e3)
    return statistics.median(ts)


def probe(wl, reps):
    res, lmax = WORKLOADS[wl]
    shape, wcs = pixsht.fullsky_geometry(res * pixsht.arcminute)
    band = pixsht.sht_band(shape, wcs)
    plan = Plan(band, lmax)
    npix = band.nx * band.nrings
    g = torch.Generator(device="cuda").manual_seed(1)
    d_alm = [torch.randn(plan.nalm, dtype=torch.complex128, device="cuda", generator=g) for _ in range(3)]
    d_map = [torch.empty(npix, dtype=torch.float64, device="cuda") for _ in range(3)]
    d_out = [torch.empty(plan.nalm, dtype=torch.complex128, device="cuda") for _ in range(3)]
    P = lambda ts: [t.data_ptr() for t in ts]    # noqa: E731
    plan.execute_ptrs(_lib.ALM2MAP, P(d_alm), P(d_map), _lib.DEVICE)        # band-limited input maps
    h_map = [m.cpu().pin_memory() for m in d_map]
    h_alm = [a.cpu().pin_memory() for a in d_alm]
    h_out = [torch.empty(plan.nalm, dtype=torch.complex128).pin_memory() for _ in range(3)]
    rows = []
    for where, loc, alms, maps, outs in (("device", _lib.DEVICE, d_alm, d_map, d_out), ("pinned host", _lib.HOST, h_alm, h_map, h_out)):
        t_a2m = timed(lambda: plan.execute_ptrs(_lib.ALM2MAP, P(alms), P(maps), loc), reps)
        n_a2m = plan.info()["launches"]
        t_m2a = timed(lambda: plan.execute_ptrs(_lib.MAP2ALM, P(outs), P(maps), loc), reps)
        n_m2a = plan.info()["launches"]
        for k in NITERS:
            t = timed(lambda: plan.map2alm_iter_ptrs(P(outs), P(maps), k, loc), reps)
            tm = plan.timings()
            row = dict(workload=wl, memory=where, niter=k, ms=round(t, 1), compute_span_ms=round(tm["compute_span"], 1),
                       separate_ms=round(k * (t_a2m + t_m2a) + t_m2a, 1), alm2map_ms=round(t_a2m, 1), map2alm_ms=round(t_m2a, 1),
                       launches=plan.info()["launches"], separate_launches=k * (n_a2m + n_m2a) + n_m2a)
            row["ratio"] = round(row["ms"] / row["separate_ms"], 3)
            rows.append(row)
            print("%s %-11s niter %d: %8.1f ms per call (compute span %8.1f)  separate calls %8.1f ms  ratio %.3f  launches %d (separate %d)"
                  % (wl, where, k, row["ms"], row["compute_span_ms"], row["separate_ms"], row["ratio"], row["launches"], row["separate_launches"]),
                  flush=True)
    plan.close()
    del d_alm, d_map, d_out, h_map, h_alm, h_out
    torch.cuda.empty_cache()
    return rows


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--workloads", nargs="+", default=["C3", "C4"], choices=sorted(WORKLOADS))
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None, help="write the rows as JSON here")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("iter_probe.py needs a CUDA device")
    name, power = card()
    print("card: %s, power limit %s; IQU Float64, median of %d calls after one warm-up" % (name, power, args.reps), flush=True)
    rows = [r for wl in args.workloads for r in probe(wl, args.reps)]
    if args.out:
        with open(args.out, "w") as f:
            json.dump(dict(card=name, power_limit=power, reps=args.reps, rows=rows), f, indent=1)


if __name__ == "__main__":
    main()
