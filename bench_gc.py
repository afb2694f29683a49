#!/usr/bin/env python
"""bench_gc.py -- gen.gc (proband x ancestor genetic contributions), gen.occ, gen.rec and gen.findMRCA on a
benchmark pedigree.

    python bench_gc.py --config C3 --steps 5 --warmup 1 [--direction descend|ascend] [--ancestors K]
                       [--function gc|occ|occ_total|rec|meioses|mrca]

A step is one genlib_gc call: host rank arrays in, planning, upload, every layer, gather and D2H of the
whole len(pro) x len(ancestors) Float64 matrix into pinned host memory.  `--function occ` is one genlib_occ
call that returns the len(ancestors) x len(pro) Int64 path counts the same way; `occ_total` (its row sums)
and `rec` (descendant counts) reduce on the device and fetch len(ancestors) Int64 values.  `meioses` is one
genlib_meioses call: the len(pro) x len(ancestors) Int64 minimum meioses, 2 bytes per column on the device.
`mrca` is one findMRCA of the probands: the genlib_mrca pass (a gen.rec over the probands' ancestors-or-self)
and the genlib_meioses pass to the MRCAs, each reported with its own kernel time and bytes; `--ids K` takes a
seeded sample of K probands instead (the whole proband list of C3 or genea140 has no common ancestor, so
its distance pass is empty).  `ms_kernels` (CUDA events
around the layer kernels, slowest device) and `e2e_ms` (host clock around the call) are medians over
the timed steps.  `alg_bytes` is the traffic the layers cannot avoid (input rows read, frontier and
output rows written, 8 bytes per column -- gen.rec: per 64-column word -- plus one read of the output block
for a reduction); `frac_of_peak` divides it by ms_kernels and the measured HBM peak.
The C3 working set (frontier and output block, GBs) is far larger than the 126 MB L2; genea140's is
not.  Prints one JSON line; writes nothing.
"""
from __future__ import annotations

import argparse
import ctypes as C
import hashlib
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from bench import measured_peaks  # noqa: E402


def gpu_card():
    """Name and power limit of GPU 0 (read-only query)."""
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        name, power = (x.strip() for x in out[0].split(",", 1))
        return name, power
    except Exception as e:  # noqa: BLE001 -- reported, not fatal
        return f"unknown ({e})", "unknown"


def workload(gen, name: str, scale: float, n_anc: int | None, seed: int):
    if name == "genea140":
        ped = gen.genealogy(gen.genea140)
        pro = gen.pro(ped)
    else:
        s = gen.synth.config(name, scale)
        ped = gen.genealogy(s.as_columns())
        pro = s.probands
    anc = gen.founder(ped)
    if n_anc is not None and n_anc < len(anc):          # a seeded sample of the founders, in ID order
        anc = np.sort(np.random.default_rng(seed).choice(anc, n_anc, replace=False))
    return ped, ped.rank_of(pro), ped.rank_of(anc), n_anc is None


METRIC_NAME = {"gc": "gc", "occ": "occ", "occ_total": "occ(TOTAL)", "rec": "rec", "meioses": "meioses"}


def bench_mrca(gen, ped, pro, devices, args):
    """findMRCA of the whole proband list: the common-ancestor pass and the distance pass, timed apart."""
    if args.ids is not None and args.ids < len(pro):
        pro = np.random.default_rng(args.seed).choice(pro, args.ids, replace=False)
    ids = ped.ids[pro]
    passes = {"mrca": [], "meioses": []}
    e2e, res, stats = [], None, None
    for step in range(args.warmup + args.steps):
        t0 = time.perf_counter()
        res, stats = gen.findMRCA(ped, ids, devices=devices, return_stats=True)
        t1 = time.perf_counter()
        if step >= args.warmup:
            e2e.append((t1 - t0) * 1e3)
            for k in passes:
                passes[k].append(stats[k])
    name, power = gpu_card()
    out = {"metric": "gen.findMRCA required bytes / kernel time, per pass", "config": args.config,
           "scale": args.scale, "n_ids": len(ids), "ids": "probands" if args.ids is None else f"{len(ids)} sampled probands, seed {args.seed}",
           "n_mrca": len(res.ancestors), "n_dev": len(devices),
           "e2e_ms": float(np.median(e2e)), "e2e_ms_all": e2e,
           "output_sha256": hashlib.sha256(res.ancestors.tobytes() + res.meioses.tobytes()).hexdigest()}
    for k, runs in passes.items():
        ms_k = [s["ms_kernels"] for s in runs]
        ms = float(np.median(ms_k))
        last = runs[-1]
        out[k] = {"direction": last["direction"], "n_pro": last["n_pro"], "n_anc": last["n_anc"],
                  "width": last["width"], "n_layers": last["n_layers"], "rows": last["rows"],
                  "ms_kernels": ms, "ms_kernels_all": ms_k, "ms_plan": last["ms_plan"], "ms_fetch": last["ms_fetch"],
                  "alg_bytes": last["alg_bytes"], "achieved_gbs": last["alg_bytes"] / ms / 1e6 if ms > 0 else None,
                  "device_bytes": last["device_bytes"], "d2h_bytes": last["d2h_bytes"],
                  "kernel_launches": last["kernel_launches"]}
    out.update({"gpu": name, "power_limit": power, "steps": args.steps, "warmup": args.warmup})
    print(json.dumps(out))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", default="C3", help="genea140, C3, C4 or C5")
    ap.add_argument("--scale", type=float, default=1.0)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--direction", choices=["auto", "descend", "ascend"], default="auto")
    ap.add_argument("--ancestors", type=int, default=None, help="a seeded sample of this many founders")
    ap.add_argument("--seed", type=int, default=1)
    ap.add_argument("--ids", type=int, default=None, help="mrca: a seeded sample of this many probands")
    ap.add_argument("--devices", default="0", help="comma-separated device list")
    ap.add_argument("--function", choices=["gc", "occ", "occ_total", "rec", "meioses", "mrca"], default="gc")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.direction == "auto":
        os.environ.pop("GENLIB_GC_DIRECTION", None)
    else:
        os.environ["GENLIB_GC_DIRECTION"] = args.direction
    import genlib_b200 as gen
    if gen.lib().genlib_device_count() < 1:
        raise SystemExit("no CUDA device: gen.gc has no CPU fallback")
    devices = [int(d) for d in args.devices.split(",")]
    ped, pro, anc, all_founders = workload(gen, args.config, args.scale, args.ancestors, args.seed)
    if args.function == "mrca":
        return bench_mrca(gen, ped, pro, devices, args)
    shape = {"gc": (len(pro), len(anc)), "occ": (len(anc), len(pro)), "occ_total": (len(anc), 1),
             "rec": (len(anc),), "meioses": (len(pro), len(anc))}[args.function]
    dtype = np.float64 if args.function == "gc" else np.int64
    nbytes = max(1, int(np.prod(shape)) * 8)
    p = C.c_void_p()
    gen._lib.check(gen.lib().genlib_pinned_alloc(nbytes, C.byref(p)))
    try:
        out = np.frombuffer((C.c_char * nbytes).from_address(p.value), dtype, count=int(np.prod(shape))).reshape(shape)
        call = {
            "gc": lambda: gen.gc_arrays(ped.father, ped.mother, pro, anc, out=out, devices=devices),
            "occ": lambda: gen.occ_arrays(ped.father, ped.mother, pro, anc, out=out, devices=devices),
            "occ_total": lambda: gen.occ_arrays(ped.father, ped.mother, pro, anc, typeOcc="TOTAL", out=out,
                                                devices=devices),
            "rec": lambda: gen.rec_arrays(ped.father, ped.mother, pro, anc, out=out, devices=devices),
            "meioses": lambda: gen.meioses_arrays(ped.father, ped.mother, pro, anc, out=out, devices=devices),
        }[args.function]
        ms_k, e2e, stats = [], [], None
        for step in range(args.warmup + args.steps):
            t0 = time.perf_counter()
            _, stats = call()
            t1 = time.perf_counter()
            if step >= args.warmup:
                ms_k.append(stats["ms_kernels"]); e2e.append((t1 - t0) * 1e3)
        sums = out.sum(axis=1) if args.function == "gc" else None
        digest = hashlib.sha256(out.tobytes()).hexdigest()
    finally:
        gen.lib().genlib_pinned_free(p)
    peak_gbs, peak_src = measured_peaks()
    ms = float(np.median(ms_k))
    name, power = gpu_card()
    res = {
        "metric": f"gen.{METRIC_NAME[args.function]} required bytes / kernel time", "config": args.config,
        "scale": args.scale,
        "shape": list(shape), "ancestors": "founders" if all_founders else f"{len(anc)} sampled founders",
        "direction": stats["direction"], "width": stats["width"], "capacity": stats["capacity"],
        "n_layers": stats["n_layers"], "rows": stats["rows"], "inputs": stats["inputs"],
        "device_bytes": stats["device_bytes"], "n_dev": stats["n_dev"],
        "ms_kernels": ms, "ms_kernels_all": ms_k, "e2e_ms": float(np.median(e2e)), "e2e_ms_all": e2e,
        "ms_plan": stats["ms_plan"], "ms_fetch": stats["ms_fetch"], "d2h_bytes": stats["d2h_bytes"],
        "kernel_launches": stats["kernel_launches"],
        "alg_bytes": stats["alg_bytes"], "achieved_gbs": stats["alg_bytes"] / ms / 1e6 if ms > 0 else None,
        "hbm_peak_gbs": peak_gbs, "hbm_peak_source": peak_src,
        "frac_of_peak": stats["alg_bytes"] / ms / 1e6 / peak_gbs if ms > 0 else None,
        "output_sha256": digest,
        "rows_summing_to_one": int((sums == 1.0).sum()) if args.function == "gc" else None, "n_pro": len(pro),
        "gpu": name, "power_limit": power, "steps": args.steps, "warmup": args.warmup,
    }
    print(json.dumps(res))


if __name__ == "__main__":
    main()
