#!/usr/bin/env python
"""bench_over.py -- gen.phiOver on the device against the dense gen.phi it replaces, on a benchmark proband list.

    python bench_over.py --config C3 --thresholds 0.0625,0.015625,0.00390625 --steps 3 --warmup 1 [--scale S] [--devices 0,1]

A phiOver step is one genlib_phi_over call per threshold: host rank arrays in, the gen.phi plan and layers, then the
selection on the devices (a count pass, the host's offsets, a select pass) and the copy of the pairs into NumPy.  A
dense step is one genlib_phi / genlib_phi_multi call on the same list and devices into a page-locked n x n Float32
matrix, the way bench.py times gen.phi end to end.  The two alternate within every step, in one process.

Per threshold: `n_pairs`, and medians over the timed steps of `e2e_ms` (host clock around the call), `ms_kernels` (the
layers, CUDA events), `ms_fetch` (selection and copy back) and `d2h_bytes` (per-row counts plus pairs).  The same for the
dense call.  Where the dense matrix fits in half the host's available memory, `identical` tells whether GENLIB's host
phiOver on that matrix gives the device's pairs bit for bit.  A last call per threshold runs under torch.profiler
(CUDA activity, summed over the devices) to split the fetch into the two selection kernels and the device-to-host
copies (`profile`).  Prints one JSON line; writes nothing.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from bench_gc import gpu_card  # noqa: E402


def workload(gen, name: str, scale: float):
    if name == "genea140":
        ped = gen.genealogy(gen.genea140)
        return ped, gen.pro(ped)
    s = gen.synth.config(name, scale)
    return gen.genealogy(s.as_columns()), s.probands


def host_bytes_available() -> int:
    try:
        with open("/proc/meminfo") as fh:
            for line in fh:
                if line.startswith("MemAvailable:"):
                    return int(line.split()[1]) * 1024
    except OSError:
        pass
    return 0


def profile_once(gen, ped, ranks, t, devices):
    """Device time of the selection kernels and of the device-to-host copies in one genlib_phi_over call."""
    try:
        import torch
        from torch.profiler import ProfilerActivity, profile
        torch.cuda.init()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            gen.phi_over_arrays(ped.father, ped.mother, ranks, t, devices=devices)
        out = {"count_ms": 0.0, "select_ms": 0.0, "d2h_ms": 0.0, "layer_ms": 0.0, "other_ms": 0.0}
        for e in prof.events():
            if e.device_type != torch.autograd.DeviceType.CUDA:
                continue
            ms = e.device_time / 1e3 if hasattr(e, "device_time") else e.cuda_time / 1e3
            name = e.name
            key = ("count" if "phi_over_count_kernel" in name else "select" if "phi_over_select_kernel" in name else
                   "d2h" if "DtoH" in name or "Device -> Pageable" in name or "Device -> Pinned" in name else
                   "layer" if "layer_kernel" in name else "other")
            out[f"{key}_ms"] += ms
        return out
    except Exception as e:  # noqa: BLE001 -- reported, not fatal
        return {"error": repr(e)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", default="C3", choices=["genea140", "C3", "C4"])
    ap.add_argument("--scale", type=float, default=1.0)
    ap.add_argument("--devices", default="0", help="comma-separated device list")
    ap.add_argument("--thresholds", default="0.0625,0.015625,0.00390625")
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--numerics", default="reference", choices=["reference", "fp64"])
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    thresholds = [float(t) for t in args.thresholds.split(",")]
    if any(np.isnan(t) for t in thresholds):
        ap.error("a threshold is NaN")
    devices = [int(d) for d in args.devices.split(",")]
    import genlib_b200 as gen
    name, power = gpu_card()
    ped, pro = workload(gen, args.config, args.scale)
    ranks = ped.rank_of(pro)
    n = len(np.unique(ranks))
    dense_bytes = n * n * 4
    dense_fits = dense_bytes <= host_bytes_available() // 2

    over = {t: {"e2e_ms": [], "ms_kernels": [], "ms_fetch": [], "d2h_bytes": [], "n_pairs": None} for t in thresholds}
    dense = {"e2e_ms": [], "ms_kernels": [], "ms_fetch": [], "d2h_bytes": []}
    results = {}
    pinned = gen.PinnedMatrix(n, np.float32) if dense_fits else None
    dev_kw = {"devices": devices} if len(devices) > 1 else {"device": devices[0]}
    for step in range(args.warmup + args.steps):
        timed = step >= args.warmup
        for t in thresholds:
            t0 = time.perf_counter()
            line, column, kin, st = gen.phi_over_arrays(ped.father, ped.mother, ranks, t, numerics=args.numerics,
                                                        devices=devices)
            t1 = time.perf_counter()
            results[t] = (line, column, kin)
            rec = over[t]
            rec["n_pairs"] = int(len(line))
            if timed:
                rec["e2e_ms"].append((t1 - t0) * 1e3)
                for k in ("ms_kernels", "ms_fetch", "d2h_bytes"):
                    rec[k].append(st[k])
        if pinned is not None:
            t0 = time.perf_counter()
            _, st = gen.phi_arrays(ped.father, ped.mother, ranks, numerics=args.numerics, out=pinned.array, **dev_kw)
            t1 = time.perf_counter()
            if timed:
                dense["e2e_ms"].append((t1 - t0) * 1e3)
                for k in ("ms_kernels", "ms_fetch", "d2h_bytes"):
                    dense[k].append(st[k])

    def med(rec):
        return {k: (float(np.median(v)) if isinstance(v, list) else v) for k, v in rec.items()} | \
               {"e2e_ms_all": rec["e2e_ms"]}

    out = {"metric": "gen.phiOver e2e", "config": args.config, "scale": args.scale, "n_unique": n,
           "numerics": args.numerics, "n_dev": len(devices), "devices": devices, "gpu": name, "power_limit": power,
           "steps": args.steps, "warmup": args.warmup,
           "over": {repr(t): med(over[t]) for t in thresholds}}
    if pinned is not None:
        out["dense"] = med(dense)
        ids = np.arange(n, dtype=np.int64)
        for t in thresholds:
            want = gen.phiOver(pinned.array, t, ids)
            line, column, kin = results[t]
            out["over"][repr(t)]["identical"] = bool(np.array_equal(want.line, line) and np.array_equal(want.column, column)
                                                     and want.kinship.tobytes() == kin.tobytes())
        pinned.free()
    else:
        out["dense"] = {"skipped": f"the {dense_bytes / 1e9:.1f} GB matrix does not fit half the host's available memory"}
    for t in thresholds:
        out["over"][repr(t)]["profile"] = profile_once(gen, ped, ranks, t, devices)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
