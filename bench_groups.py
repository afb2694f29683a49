#!/usr/bin/env python
"""bench_groups.py -- gen.phiMeanGroups on the device against the dense gen.phi plus a host reduction it replaces.

    python bench_groups.py --config C3 --steps 3 --warmup 1 [--scale S] [--devices 0,1]
    python bench_groups.py --config C4 --scale 0.5 --groups 20

The probands of C3 are grouped by their deme (20 demes, migration 0.02); C4 has one deme, so its probands get
`position % --groups` as labels.  A groups step is one genlib_phi_groups call: host rank arrays in, the gen.phi plan and
layers, the reduction of the proband rows on the devices, P x G doubles copied back and the host's T and divisions.  A
dense step is one genlib_phi / genlib_phi_multi call on the same list and devices into a page-locked P x P Float32
matrix, then the same means on the host from indicator products in float64 (row blocks of the widened matrix, its
diagonal zeroed, times the P x G one-hot matrix).  The two alternate within every step, in one process.

Reported: medians over the timed steps of `e2e_ms` (host clock around everything), `ms_kernels` (the layers, CUDA events),
`ms_fetch` (groups: the reduction, the copies and the host's part; dense: the matrix copy), `host_ms` (dense: the host
reduction), `d2h_bytes`, the host bytes each result needs, and `max_rel_diff`, the largest relative difference between
the two paths' means.  A last call under torch.profiler (CUDA activity, summed over the devices) gives the time of
phi_groups_kernel, and, as the yardstick on the same rows, rowsum_kernel's (Engine.row_sums, one device).  Prints one
JSON line; writes nothing.
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
from bench_over import host_bytes_available  # noqa: E402


def workload(gen, name: str, scale: float, n_groups: int):
    """(pedigree, proband IDs in list order, group index per proband, number of groups)."""
    s = gen.synth.config(name, scale)
    pro = s.probands
    if name == "C3":
        labels = s.deme[pro - 1]                                   # IDs are 1..N in file order
    else:
        labels = np.arange(len(pro)) % n_groups
    levels, index = np.unique(labels, return_inverse=True)
    return gen.genealogy(s.as_columns()), pro, index.astype(np.int32), len(levels)


def dense_means(m, index, G):
    """proband_mean and group_mean of the P x P matrix m by indicator products in float64, in row blocks."""
    P = m.shape[0]
    E = np.zeros((P, G))
    E[np.arange(P), index] = 1.0
    S = np.empty((P, G))
    step = max(1, (1 << 25) // P)                                  # the float64 block stays at 256 MB
    for r0 in range(0, P, step):
        b = m[r0:r0 + step].astype(np.float64)
        k = np.arange(len(b))
        b[k, r0 + k] = 0.0
        S[r0:r0 + step] = b @ E
    size = np.bincount(index, minlength=G).astype(np.float64)
    T = E.T @ S
    pairs = np.outer(size, size) - np.diag(size)
    own = E.astype(bool)
    with np.errstate(invalid="ignore", divide="ignore"):
        pm = S / (size[None, :] - own)
        up = np.triu(T)
        gm = (up + np.triu(up, 1).T) / pairs
    return pm, gm


def max_rel_diff(a, b):
    ok = np.isfinite(a) & np.isfinite(b)
    if not np.array_equal(np.isnan(a), np.isnan(b)):
        return float("inf")
    d = np.abs(a[ok] - b[ok]) / np.maximum(np.abs(b[ok]), np.finfo(np.float64).tiny)
    return float(d.max()) if d.size else 0.0


def profile_once(gen, ped, ranks, index, G, devices):
    """Device time of phi_groups_kernel and its copies in one call; rowsum_kernel on the same rows (one device)."""
    try:
        import torch
        from torch.profiler import ProfilerActivity, profile
        torch.cuda.init()
        out = {"groups_kernel_ms": 0.0, "d2h_ms": 0.0, "layer_ms": 0.0, "other_ms": 0.0, "rowsum_kernel_ms": 0.0}

        def add(prof, rowsum):
            for e in prof.events():
                if e.device_type != torch.autograd.DeviceType.CUDA:
                    continue
                ms = e.device_time / 1e3 if hasattr(e, "device_time") else e.cuda_time / 1e3
                name = e.name
                if rowsum:
                    if "rowsum_kernel" in name:
                        out["rowsum_kernel_ms"] += ms
                    continue
                key = ("groups_kernel" if "phi_groups_kernel" in name else
                       "d2h" if "DtoH" in name or "Device -> Pageable" in name or "Device -> Pinned" in name else
                       "layer" if "layer_kernel" in name else "other")
                out[f"{key}_ms"] += ms

        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            gen.phi_groups_arrays(ped.father, ped.mother, ranks, index, G, devices=devices)
        add(prof, False)
        eng = gen.Engine(gen.Plan(ped.father, ped.mother, ranks), device=devices[0])
        try:
            eng.run()
            eng.row_sums()                                          # (warm)
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                eng.row_sums()
            add(prof, True)
        finally:
            eng.close()
        return out
    except Exception as e:  # noqa: BLE001 -- reported, not fatal
        return {"error": repr(e)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", default="C3", choices=["C3", "C4", "C5"])
    ap.add_argument("--scale", type=float, default=1.0)
    ap.add_argument("--groups", type=int, default=20, help="labels position %% groups (configs without demes)")
    ap.add_argument("--devices", default="0", help="comma-separated device list")
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--numerics", default="reference", choices=["reference", "fp64"])
    args = ap.parse_args()
    if args.steps < 1 or args.groups < 1:
        ap.error("--steps and --groups must be at least 1")
    devices = [int(d) for d in args.devices.split(",")]
    import genlib_b200 as gen
    name, power = gpu_card()
    ped, pro, index, G = workload(gen, args.config, args.scale, args.groups)
    ranks = ped.rank_of(pro)
    P = len(ranks)
    dense_bytes = P * P * 4
    dense_fits = dense_bytes <= host_bytes_available() // 2
    keys = ("ms_kernels", "ms_fetch", "d2h_bytes")
    grp = {"e2e_ms": [], **{k: [] for k in keys}}
    dense = {"e2e_ms": [], "host_ms": [], **{k: [] for k in keys}}
    pinned = gen.PinnedMatrix(P, np.float32) if dense_fits else None
    dev_kw = {"devices": devices} if len(devices) > 1 else {"device": devices[0]}
    got = want = None
    for step in range(args.warmup + args.steps):
        timed = step >= args.warmup
        t0 = time.perf_counter()
        pm, gm, st = gen.phi_groups_arrays(ped.father, ped.mother, ranks, index, G, numerics=args.numerics, devices=devices)
        t1 = time.perf_counter()
        got = (pm, gm)
        if timed:
            grp["e2e_ms"].append((t1 - t0) * 1e3)
            for k in keys:
                grp[k].append(st[k])
        if pinned is not None:
            t0 = time.perf_counter()
            _, st = gen.phi_arrays(ped.father, ped.mother, ranks, numerics=args.numerics, out=pinned.array, **dev_kw)
            t1 = time.perf_counter()
            want = dense_means(pinned.array, index, G)
            t2 = time.perf_counter()
            if timed:
                dense["e2e_ms"].append((t2 - t0) * 1e3)
                dense["host_ms"].append((t2 - t1) * 1e3)
                for k in keys:
                    dense[k].append(st[k])

    def med(rec):
        return {k: float(np.median(v)) for k, v in rec.items()} | {"e2e_ms_all": rec["e2e_ms"]}

    out = {"metric": "gen.phiMeanGroups e2e", "config": args.config, "scale": args.scale, "n_unique": P, "n_groups": G,
           "numerics": args.numerics, "n_dev": len(devices), "devices": devices, "gpu": name, "power_limit": power,
           "steps": args.steps, "warmup": args.warmup,
           "groups": med(grp) | {"host_bytes": P * G * 8 + G * G * 8}}
    if pinned is not None:
        out["dense"] = med(dense) | {"host_bytes": dense_bytes}
        out["max_rel_diff"] = {"proband": max_rel_diff(got[0], want[0]), "mean": max_rel_diff(got[1], want[1])}
        pinned.free()
    else:
        out["dense"] = {"skipped": f"the {dense_bytes / 1e9:.1f} GB matrix does not fit half the host's available memory"}
    out["profile"] = profile_once(gen, ped, ranks, index, G, devices)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
