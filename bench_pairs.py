#!/usr/bin/env python
"""bench_pairs.py -- gen.phi_pairs (the kinship of each pair of a list) on a benchmark pedigree.

    python bench_pairs.py --config C3 --pairs couples --steps 3 --warmup 1 [--scale S] [--devices 0]

A step is one genlib_phi_pairs call: host rank arrays in, planning (on a worker thread, beside the device), upload,
every layer with the reads of its pairs just before it, one D2H copy of the per-read values and the host's scatter to
list order.  The lists a user would run:
  couples         every distinct (father, mother) pair of the pedigree
  same-depth:K    K seeded pairs of individuals of one depth below the founders, over all depths
  pro:K           all K*K ordered pairs of K seeded probands; the run also times the method this replaces, the Float64
                  phi matrix of those probands through the public API (gen.phi(ped, named, numerics="fp64")), and checks
                  that both give the same bits

`e2e_ms` (host clock around the call), `ms_plan` and `ms_kernels` (CUDA events from the first launch to the last) are
medians over the timed steps.  One more call, after them, runs under torch.profiler to split the device time into the
layer kernels and the pair reads (`profile`).  `capacity` is the frontier width W the engine was sized with, which
pairs across generations widen.  Prints one JSON line; writes nothing.
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

from bench_gc import gpu_card  # noqa: E402


def depths(father, mother):
    d = np.zeros(len(father), np.int64)
    for x in range(len(father)):                                     # parents precede children
        f, m = father[x], mother[x]
        d[x] = max(d[f] + 1 if f >= 0 else 0, d[m] + 1 if m >= 0 else 0)
    return d


def workload(gen, name: str, scale: float, pairs: str, seed: int):
    """(pedigree, a, b, named proband IDs or None)."""
    if name == "genea140":
        ped = gen.genealogy(gen.genea140)
        pro = gen.pro(ped)
    else:
        s = gen.synth.config(name, scale)
        ped = gen.genealogy(s.as_columns())
        pro = s.probands
    rng = np.random.default_rng(seed)
    if pairs == "couples":
        both = (ped.father >= 0) & (ped.mother >= 0)
        key = np.unique(ped.father[both].astype(np.int64) * len(ped.ids) + ped.mother[both])
        return ped, (key // len(ped.ids)).astype(np.int32), (key % len(ped.ids)).astype(np.int32), None
    kind, k = pairs.split(":")
    k = int(k)
    if kind == "same-depth":
        d = depths(ped.father, ped.mother)
        order = np.argsort(d, kind="stable")
        start = np.searchsorted(d[order], np.arange(d.max() + 2))
        which = rng.integers(0, d.max() + 1, k)                     # a depth per pair, then two of its individuals
        size = start[which + 1] - start[which]
        while (size == 0).any():
            which[size == 0] = rng.integers(0, d.max() + 1, int((size == 0).sum()))
            size = start[which + 1] - start[which]
        a = order[start[which] + rng.integers(0, size)]
        b = order[start[which] + rng.integers(0, size)]
        return ped, a.astype(np.int32), b.astype(np.int32), None
    named = rng.choice(np.asarray(pro, np.int64), k, replace=False)
    r = ped.rank_of(named)
    i, j = np.meshgrid(np.arange(k), np.arange(k), indexing="ij")
    return ped, r[i.ravel()], r[j.ravel()], named


def profile_once(gen, ped, a, b, devices):
    """Device time of the layer kernels and of the pair reads in one call (torch.profiler, CUDA activity)."""
    try:
        import torch
        from torch.profiler import ProfilerActivity, profile
        torch.cuda.init()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            gen.phi_pairs_arrays(ped.father, ped.mother, a, b, devices=devices)
        out = {"layer_ms": 0.0, "layer_launches": 0, "reads_ms": 0.0, "reads_launches": 0, "other_ms": 0.0}
        for e in prof.events():
            if e.device_type != torch.autograd.DeviceType.CUDA:
                continue
            ms = e.device_time / 1e3 if hasattr(e, "device_time") else e.cuda_time / 1e3
            key = "reads" if "pair_kinship_kernel" in e.name else "layer" if "layer_kernel" in e.name else None
            if key is None:
                out["other_ms"] += ms
            else:
                out[f"{key}_ms"] += ms
                out[f"{key}_launches"] += 1
        total = out["layer_ms"] + out["reads_ms"] + out["other_ms"]
        out["reads_share"] = out["reads_ms"] / total if total > 0 else None
        return out
    except Exception as e:  # noqa: BLE001 -- reported, not fatal
        return {"error": repr(e)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", default="C3", choices=["genea140", "C3", "C5"])
    ap.add_argument("--scale", type=float, default=1.0)
    ap.add_argument("--pairs", default="couples", help="couples, same-depth:K or pro:K")
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--seed", type=int, default=1)
    ap.add_argument("--devices", default="0", help="comma-separated device list")
    ap.add_argument("--plan-only", action="store_true", help="plan on the host and report the frontier; no device")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    kind, _, k = args.pairs.partition(":")
    if not (args.pairs == "couples" or (kind in ("same-depth", "pro") and k.isdigit())):
        ap.error("--pairs must be couples, same-depth:K or pro:K")
    import genlib_b200 as gen
    devices = [int(d) for d in args.devices.split(",")]
    ped, a, b, named = workload(gen, args.config, args.scale, args.pairs, args.seed)
    out = {"metric": "gen.phi_pairs plan, host only" if args.plan_only else "gen.phi_pairs e2e", "config": args.config,
           "scale": args.scale, "pairs": args.pairs, "n_pairs": int(len(a)), "n_dev": len(devices)}
    if args.plan_only:
        t0 = time.perf_counter()
        plan = gen.Plan.pairs(ped.father, ped.mother, a, b, world=len(devices))
        out.update({"plan_ms": (time.perf_counter() - t0) * 1e3, "n_unique": plan.n_unique, "n_layers": plan.n_layers,
                    "capacity": plan.capacity, "device_bytes_rank0": plan.device_bytes("fp64", 0)})
        print(json.dumps(out))
        return

    e2e, ms_plan, ms_kernels, res, st = [], [], [], None, None
    for step in range(args.warmup + args.steps):
        t0 = time.perf_counter()
        res, st = gen.phi_pairs_arrays(ped.father, ped.mother, a, b, devices=devices)
        t1 = time.perf_counter()
        if step >= args.warmup:
            e2e.append((t1 - t0) * 1e3)
            ms_plan.append(st["ms_plan"])
            ms_kernels.append(st["ms_kernels"])
    name, power = gpu_card()
    out.update({"n_unique": st["n_unique"], "e2e_ms": float(np.median(e2e)), "e2e_ms_all": e2e,
                "ms_plan": float(np.median(ms_plan)), "ms_kernels": float(np.median(ms_kernels)),
                "ms_kernels_all": ms_kernels, "ms_fetch": st["ms_fetch"], "n_layers": st["n_layers"],
                "row_updates": st["row_updates"], "capacity": st["capacity"], "device_bytes": st["device_bytes"],
                "h2d_bytes": st["h2d_bytes"], "d2h_bytes": st["d2h_bytes"], "kernel_launches": st["kernel_launches"],
                "output_sha256": hashlib.sha256(res.tobytes()).hexdigest()})
    out["profile"] = profile_once(gen, ped, a, b, devices)
    if named is not None:                        # the replaced method: the Float64 phi matrix of the named probands
        t0 = time.perf_counter()
        m, ost = gen.phi(ped, named, numerics="fp64", dtype=np.float64, return_stats=True)
        t1 = time.perf_counter()
        out["phi_matrix"] = {"n_named": int(len(named)), "e2e_ms": (t1 - t0) * 1e3, "ms_kernels": ost["ms_kernels"],
                             "ms_plan": ost["ms_plan"], "capacity": ost["capacity"], "device_bytes": ost["device_bytes"],
                             "d2h_bytes": ost["d2h_bytes"], "bitwise_equal": bool(np.array_equal(m.ravel(), res))}
    out.update({"gpu": name, "power_limit": power, "steps": args.steps, "warmup": args.warmup})
    print(json.dumps(out))


if __name__ == "__main__":
    main()
