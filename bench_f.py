#!/usr/bin/env python
"""bench_f.py -- gen.f (inbreeding coefficients) of many individuals on a benchmark pedigree.

    python bench_f.py --config C3 --ids all --steps 3 --warmup 1 [--scale S] [--devices 0]

A step is one genlib_f call: host rank arrays in, planning (on a worker thread, beside the device), upload, every
layer with the read of Psi[father, mother] of each couple just before its layer, one D2H copy of the per-couple
values and the host's mapping to the list.  `--ids all` lists every individual, `pro` the benchmark's probands,
K a seeded sample of K individuals.  With `--ids pro` the same run also times the method gen.f used before, the
Float64 phi matrix of the probands' parents through the public API (gen.phi(ped, parents, numerics="fp64")), and
checks that both give the same bits.

`e2e_ms` (host clock around the call), `ms_plan` and `ms_kernels` (CUDA events from the first launch to the last,
the gathers included) are medians over the timed steps.  One more call, after them, runs under torch.profiler to
split the device time into the layer kernels and the gather launches (`profile`).  `alg_bytes` is the traffic the
layers cannot avoid, 8 (4 n L + 3 n^2) per layer plus 8 bytes per couple with both parents; `frac_of_peak` divides
it by ms_kernels and the HBM peak.  The C3 frontier (tens of GB) is far larger than the 126 MB L2.
Prints one JSON line; writes nothing.
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from bench import measured_peaks  # noqa: E402
from bench_gc import gpu_card  # noqa: E402


def workload(gen, name: str, scale: float, ids: str, seed: int):
    if name == "genea140":
        ped = gen.genealogy(gen.genea140)
        pro = gen.pro(ped)
    else:
        s = gen.synth.config(name, scale)
        ped = gen.genealogy(s.as_columns())
        pro = s.probands
    if ids == "all":
        chosen = ped.ids
    elif ids == "pro":
        chosen = np.asarray(pro, np.int64)
    else:
        chosen = np.sort(np.random.default_rng(seed).choice(ped.ids, int(ids), replace=False))
    return ped, ped.rank_of(chosen)


def profile_once(gen, ped, ranks, devices):
    """Device time of the layer kernels and of the gather launches in one call (torch.profiler, CUDA activity)."""
    try:
        import torch
        from torch.profiler import ProfilerActivity, profile
        torch.cuda.init()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            gen.f_arrays(ped.father, ped.mother, ranks, dtype=np.float64, devices=devices)
        out = {"layer_ms": 0.0, "layer_launches": 0, "gather_ms": 0.0, "gather_launches": 0, "other_ms": 0.0}
        for e in prof.events():
            if e.device_type != torch.autograd.DeviceType.CUDA:
                continue
            ms = e.device_time / 1e3 if hasattr(e, "device_time") else e.cuda_time / 1e3
            key = "gather" if "couple_kinship_kernel" in e.name else "layer" if "layer_kernel" in e.name else None
            if key is None:
                out["other_ms"] += ms
            else:
                out[f"{key}_ms"] += ms
                out[f"{key}_launches"] += 1
        return out
    except Exception as e:  # noqa: BLE001 -- reported, not fatal
        return {"error": repr(e)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", default="C3", choices=["genea140", "C3", "C5"])
    ap.add_argument("--scale", type=float, default=1.0)
    ap.add_argument("--ids", default="all", help="all, pro or a sample size K")
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--seed", type=int, default=1)
    ap.add_argument("--devices", default="0", help="comma-separated device list")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.ids not in ("all", "pro") and not args.ids.isdigit():
        ap.error("--ids must be all, pro or a number")
    import genlib_b200 as gen
    devices = [int(d) for d in args.devices.split(",")]
    ped, ranks = workload(gen, args.config, args.scale, args.ids, args.seed)

    e2e, ms_plan, ms_kernels, res, st = [], [], [], None, None
    for step in range(args.warmup + args.steps):
        t0 = time.perf_counter()
        res, st = gen.f_arrays(ped.father, ped.mother, ranks, dtype=np.float64, devices=devices)
        t1 = time.perf_counter()
        if step >= args.warmup:
            e2e.append((t1 - t0) * 1e3)
            ms_plan.append(st["ms_plan"])
            ms_kernels.append(st["ms_kernels"])
    peak, peak_src = measured_peaks()
    mk = float(np.median(ms_kernels))
    name, power = gpu_card()
    out = {"metric": "gen.f required bytes / kernel time", "config": args.config, "scale": args.scale,
           "ids": args.ids, "n_ids": int(len(ranks)), "n_unique": st["n_unique"], "n_dev": len(devices),
           "e2e_ms": float(np.median(e2e)), "e2e_ms_all": e2e, "ms_plan": float(np.median(ms_plan)),
           "ms_kernels": mk, "ms_kernels_all": ms_kernels, "ms_fetch": st["ms_fetch"], "n_layers": st["n_layers"],
           "row_updates": st["row_updates"], "capacity": st["capacity"], "device_bytes": st["device_bytes"],
           "alg_bytes": st["alg_bytes"], "achieved_gbs": st["alg_bytes"] / mk / 1e6 if mk > 0 else None,
           "frac_of_peak": st["alg_bytes"] / mk / 1e6 / peak if mk > 0 else None, "peak_gbs": peak,
           "peak_source": peak_src, "h2d_bytes": st["h2d_bytes"], "d2h_bytes": st["d2h_bytes"],
           "kernel_launches": st["kernel_launches"],
           "output_sha256": hashlib.sha256(res.tobytes()).hexdigest()}
    out["profile"] = profile_once(gen, ped, ranks, devices)
    if args.ids == "pro":                        # the replaced method: the Float64 phi matrix of the parents
        fa, mo = ped.father[ranks], ped.mother[ranks]
        both = (fa >= 0) & (mo >= 0)
        parents = np.unique(np.concatenate([fa[both], mo[both]]))
        t0 = time.perf_counter()
        k, ost = gen.phi(ped, ped.ids[parents], numerics="fp64", dtype=np.float64, return_stats=True)
        t1 = time.perf_counter()
        old = np.zeros(len(ranks))
        old[both] = k[np.searchsorted(parents, fa[both]), np.searchsorted(parents, mo[both])]
        out["parents_matrix"] = {"n_parents": int(len(parents)), "e2e_ms": (t1 - t0) * 1e3,
                                 "ms_kernels": ost["ms_kernels"], "ms_plan": ost["ms_plan"],
                                 "device_bytes": ost["device_bytes"], "d2h_bytes": ost["d2h_bytes"],
                                 "bitwise_equal": bool(np.array_equal(old, res))}
    out.update({"gpu": name, "power_limit": power, "steps": args.steps, "warmup": args.warmup})
    print(json.dumps(out))


if __name__ == "__main__":
    main()
