#!/usr/bin/env python
"""bench_product.py -- gen.phiProduct on the device against the dense gen.phi plus a host product it replaces.

    python bench_product.py --config C3 --ks 1,8,64 --steps 3 --warmup 1
    python bench_product.py --config C4 --scale 0.5 --ks 1,8,64 --steps 2 --warmup 1

X is P x k standard normal (seeded).  A product step is one genlib_phi_product call: host rank arrays and X in, the
gen.phi plan and layers, the products of the proband rows on the devices, P x k doubles copied back.  A dense step is
one genlib_phi / genlib_phi_multi call on the same list and devices into a page-locked P x P Float32 matrix, then M X on
the host in float64 (row blocks of the widened matrix).  The two alternate within every step, in one process.

Reported per k: medians over the timed steps of `e2e_ms` (host clock around everything), `ms_kernels` (the layers, CUDA
events), `ms_fetch` (product: the kernel, the copies and the host's part; dense: the matrix copy), `host_ms` (dense: the
host product) and `d2h_bytes`; `max_err_over_bound`, the largest |Y_product - Y_dense| over the bound 2 P 2^-53 (M |X|)
that two reordered float64 sums of the same terms stay within (<= 1: the two paths agree).  A separate pass on one live
engine (one device) times phi_product_kernel under torch.profiler (CUDA activity records, summed over the call's
launches), and rowsum_kernel (Engine.row_sums) on the same rows as the yardstick: the median of five calls each,
alternated, with their range.  With it: the bytes the kernel must
move (own rows x P x element size + 4 P of slots + 8 P k of X read + 8 P k of Y written) and the flops (2 P^2 k), the
achieved GB/s and GFLOP/s, and the share of the 7.7 TB/s HBM bound at k = 1 only, where bytes bound the kernel.  Prints
one JSON line per k; writes nothing.
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

HBM_BYTES_PER_S = 7.7e12          # HGX B200 data sheet, one GPU


def dense_product(m, X):
    """M X on the host in float64, in row blocks of the widened Float32 matrix (256 MB each)."""
    P = m.shape[0]
    Y = np.empty((P, X.shape[1]))
    step = max(1, (1 << 25) // P)
    for r0 in range(0, P, step):
        Y[r0:r0 + step] = m[r0:r0 + step].astype(np.float64) @ X
    return Y


def err_over_bound(got, want, m, X):
    bound = 2 * m.shape[0] * 2.0 ** -53 * dense_product(m, np.abs(X))      # (M >= 0: |M| = M)
    with np.errstate(invalid="ignore", divide="ignore"):
        r = np.abs(got - want) / bound
    r[(got == want)] = 0.0
    return float(np.nanmax(r))


def kernel_times(gen, ped, ranks, Xs, numerics, device, repeats=5):
    """Per k: phi_product_kernel's device time on a live engine; rowsum_kernel's on the same rows.  Each is the median
    of `repeats` profiled calls, alternated, and the spread (min, max) comes with it."""
    try:
        import torch
        from torch.profiler import ProfilerActivity, profile
        torch.cuda.init()

        def device_ms(prof, name):
            t = 0.0
            for e in prof.events():
                if e.device_type == torch.autograd.DeviceType.CUDA and name in e.name:
                    t += (e.device_time if hasattr(e, "device_time") else e.cuda_time) / 1e3
            return t

        def timed(fn, name):
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                fn()
            return device_ms(prof, name)

        eng = gen.Engine(gen.Plan(ped.father, ped.mother, ranks), numerics=numerics, device=device)
        try:
            eng.run()
            own = len(eng.own_probands())
            eng.row_sums()                                              # (warm)
            for X in Xs.values():
                eng.phi_product(X)
            rowsum, product = [], {k: [] for k in Xs}
            for _ in range(repeats):
                rowsum.append(timed(eng.row_sums, "rowsum_kernel"))
                for k, X in Xs.items():
                    product[k].append(timed(lambda: eng.phi_product(X), "phi_product_kernel"))
            return {"own_rows": own, "repeats": repeats, "rowsum_kernel_ms": float(np.median(rowsum)),
                    "rowsum_kernel_ms_range": [min(rowsum), max(rowsum)],
                    "product_kernel_ms": {k: float(np.median(v)) for k, v in product.items()},
                    "product_kernel_ms_range": {k: [min(v), max(v)] for k, v in product.items()}}
        finally:
            eng.close()
    except Exception as e:  # noqa: BLE001 -- reported, not fatal
        return {"error": repr(e)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", default="C3", choices=["C3", "C4", "C5"])
    ap.add_argument("--scale", type=float, default=1.0)
    ap.add_argument("--ks", default="1,8,64", help="comma-separated column counts")
    ap.add_argument("--devices", default="0", help="comma-separated device list")
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--numerics", default="reference", choices=["reference", "fp64"])
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    devices = [int(d) for d in args.devices.split(",")]
    ks = [int(k) for k in args.ks.split(",")]
    import genlib_b200 as gen
    name, power = gpu_card()
    s = gen.synth.config(args.config, args.scale)
    ped = gen.genealogy(s.as_columns())
    ranks = ped.rank_of(s.probands)
    P = len(ranks)
    es = 4 if args.numerics == "reference" else 8
    rng = np.random.default_rng(20261022)
    Xs = {k: rng.standard_normal((P, k)) for k in ks}
    dense_bytes = P * P * 4
    dense_fits = dense_bytes <= host_bytes_available() // 3
    pinned = gen.PinnedMatrix(P, np.float32) if dense_fits else None
    dev_kw = {"devices": devices} if len(devices) > 1 else {"device": devices[0]}
    times = kernel_times(gen, ped, ranks, Xs, args.numerics, devices[0])
    keys = ("ms_kernels", "ms_fetch", "d2h_bytes")
    for k in ks:
        X = Xs[k]
        prod = {"e2e_ms": [], **{key: [] for key in keys}}
        dense = {"e2e_ms": [], "host_ms": [], **{key: [] for key in keys}}
        got = want = None
        for step in range(args.warmup + args.steps):
            timed = step >= args.warmup
            t0 = time.perf_counter()
            got, _, st = gen.phi_product_arrays(ped.father, ped.mother, ranks, X, numerics=args.numerics, devices=devices)
            t1 = time.perf_counter()
            if timed:
                prod["e2e_ms"].append((t1 - t0) * 1e3)
                for key in keys:
                    prod[key].append(st[key])
            if pinned is not None:
                t0 = time.perf_counter()
                _, st = gen.phi_arrays(ped.father, ped.mother, ranks, numerics=args.numerics, out=pinned.array, **dev_kw)
                t1 = time.perf_counter()
                want = dense_product(pinned.array, X)
                t2 = time.perf_counter()
                if timed:
                    dense["e2e_ms"].append((t2 - t0) * 1e3)
                    dense["host_ms"].append((t2 - t1) * 1e3)
                    for key in keys:
                        dense[key].append(st[key])

        def med(rec):
            return {key: float(np.median(v)) for key, v in rec.items()} | {"e2e_ms_all": rec["e2e_ms"]}

        out = {"metric": "gen.phiProduct e2e", "config": args.config, "scale": args.scale, "n_unique": P, "k": k,
               "numerics": args.numerics, "n_dev": len(devices), "devices": devices, "gpu": name,
               "power_limit": power, "steps": args.steps, "warmup": args.warmup,
               "product": med(prod) | {"host_bytes": P * k * 8}}
        if pinned is not None:
            out["dense"] = med(dense) | {"host_bytes": dense_bytes}
            out["max_err_over_bound"] = err_over_bound(got, want, pinned.array, X)
        else:
            out["dense"] = {"skipped": f"the {dense_bytes / 1e9:.1f} GB matrix does not fit a third of the host's available memory"}
        if "error" in times:
            out["kernel"] = times
        else:
            own = times["own_rows"]
            kb = own * P * es + 4 * P + 16 * P * k                  # the bytes the kernel must move
            fl = 2 * own * P * k
            ms = times["product_kernel_ms"][k]
            kern = {"product_kernel_ms": ms, "product_kernel_ms_range": times["product_kernel_ms_range"][k],
                    "rowsum_kernel_ms": times["rowsum_kernel_ms"], "rowsum_kernel_ms_range": times["rowsum_kernel_ms_range"],
                    "ratio_to_rowsum": ms / times["rowsum_kernel_ms"] if times["rowsum_kernel_ms"] else None,
                    "bytes": kb, "flops": fl}
            if ms > 0:
                kern["achieved_GBps"] = kb / ms / 1e6
                kern["achieved_GFLOPps"] = fl / ms / 1e6
                if k == 1:
                    kern["share_of_hbm_bound"] = kb / HBM_BYTES_PER_S / (ms / 1e3)
            out["kernel"] = kern
        print(json.dumps(out), flush=True)
    if pinned is not None:
        pinned.free()


if __name__ == "__main__":
    main()
