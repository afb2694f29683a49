#!/usr/bin/env python
"""bench_gc_groups.py -- gen.gcGroups on the device against the dense gen.gc plus the host group sums it replaces.

    python bench_gc_groups.py --steps 3 --warmup 1 [--workload c3_pro,c3_both,c4_pro]

Workloads (the defaults of each configuration):
  c3_pro   C3, probands grouped by deme (20 groups) x all 50 000 founders
  c3_both  C3, founders by deme x probands by deme: a 20 x 20 table
  c4_pro   C4 at full size, 100 000 probands in 20 seeded hashed groups (C4 has one deme) x all founders, one device
A groups step is one genlib_gc_groups call: host rank arrays in, planning, upload, the layers over one column per
group, the sums over the target side's groups when it is grouped, and R x C doubles copied back.  A dense step is one
genlib_gc call on the same lists into a page-locked P x A float64 matrix, then the group sums on the host (indicator
products in float64).  On C3 the two alternate within every step, in one process; C4's dense matrix (133 GB) is not
formed, which the output says.  Reported: medians over the timed steps of `e2e_ms` (host clock around the call),
`ms_kernels` (CUDA events, slowest device), `ms_plan` (host planning), and for the dense arm `host_ms` (its group
sums); `d2h_bytes`, `alg_bytes` (the plan's byte model) and `max_abs_diff` between the two arms' results.  Prints one
JSON line per workload; writes nothing.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import math
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from bench_gc import gpu_card  # noqa: E402


def _index(labels):
    levels, index = np.unique(labels, return_inverse=True)
    return index.astype(np.int32), len(levels)


def workload(gen, name: str):
    """(pedigree, proband ranks, proband groups or None, n_pro_groups, founder ranks, founder groups or None,
    n_anc_groups, description)."""
    cfg = "C3" if name.startswith("c3") else "C4"
    s = gen.synth.config(cfg, 1.0)
    ped = gen.genealogy(s.as_columns())
    pro, anc = ped.rank_of(s.probands), ped.rank_of(gen.founder(ped))
    if cfg == "C3":
        pg, npg = _index(s.deme[ped.ids[pro] - 1])                 # IDs are 1..N in file order
    else:
        h = (np.arange(len(pro), dtype=np.int64) * 0x9E3779B1 + 20261022) & 0xFFFFFFFF
        pg, npg = _index(h % 20)
    ag, nag = _index(s.deme[ped.ids[anc] - 1]) if name == "c3_both" else (None, 0)
    what = {"c3_pro": "C3 defaults: probands by deme x all founders",
            "c3_both": "C3 defaults: probands by deme x founders by deme",
            "c4_pro": "C4 defaults: probands in 20 seeded hashed groups x all founders"}[name]
    return ped, pro, pg, npg, anc, ag, nag, what


def group_sums(G, pg, npg, ag, nag):
    """The dense arm's host reduction: indicator products in float64 (exact here: every partial sum is a float64)."""
    E = np.zeros((npg, G.shape[0]))
    E[pg, np.arange(G.shape[0])] = 1.0
    T = E @ G
    if ag is not None:
        F = np.zeros((G.shape[1], nag))
        F[np.arange(G.shape[1]), ag] = 1.0
        T = T @ F
    return T


def run(gen, name, args):
    ped, pro, pg, npg, anc, ag, nag, what = workload(gen, name)
    devices = [0]
    dense = name != "c4_pro"
    groups_call = lambda: gen.gc_groups_arrays(ped.father, ped.mother, pro, anc, pro_group=pg, n_pro_groups=npg,
                                               anc_group=ag, n_anc_groups=nag, devices=devices)
    runs = {"groups": {"e2e_ms": [], "ms_kernels": [], "ms_plan": []},
            "dense": {"e2e_ms": [], "ms_kernels": [], "ms_plan": [], "host_ms": []}}
    p = C.c_void_p()
    nbytes = len(pro) * len(anc) * 8
    if dense:
        gen._lib.check(gen.lib().genlib_pinned_alloc(nbytes, C.byref(p)))
    try:
        out = np.frombuffer((C.c_char * nbytes).from_address(p.value), np.float64).reshape(len(pro), len(anc)) \
            if dense else None
        res = want = st_g = st_d = None
        for step in range(args.warmup + args.steps):
            t0 = time.perf_counter()
            res, st_g = groups_call()
            t1 = time.perf_counter()
            if step >= args.warmup:
                r = runs["groups"]
                r["e2e_ms"].append((t1 - t0) * 1e3); r["ms_kernels"].append(st_g["ms_kernels"])
                r["ms_plan"].append(st_g["ms_plan"])
            if dense:
                t0 = time.perf_counter()
                _, st_d = gen.gc_arrays(ped.father, ped.mother, pro, anc, out=out, devices=devices)
                t1 = time.perf_counter()
                want = group_sums(out, pg, npg, ag, nag)
                t2 = time.perf_counter()
                if step >= args.warmup:
                    r = runs["dense"]
                    r["e2e_ms"].append((t2 - t0) * 1e3); r["ms_kernels"].append(st_d["ms_kernels"])
                    r["ms_plan"].append(st_d["ms_plan"]); r["host_ms"].append((t2 - t1) * 1e3)
    finally:
        if dense:
            gen.lib().genlib_pinned_free(p)
    name_gpu, power = gpu_card()
    med = lambda v: float(np.median(v)) if v else None
    size = np.bincount(pg, minlength=npg)
    line = {
        "metric": "gen.gcGroups against dense gen.gc + host group sums", "workload": name, "what": what,
        "n_pro": len(pro), "n_anc": len(anc), "shape": list(res.shape), "direction": st_g["direction"],
        "width": st_g["width"], "n_layers": st_g["n_layers"], "rows": st_g["rows"], "capacity": st_g["capacity"],
        "device_bytes": st_g["device_bytes"], "d2h_bytes": st_g["d2h_bytes"], "alg_bytes": st_g["alg_bytes"],
        "kernel_launches": st_g["kernel_launches"],
        "groups": {k: med(v) for k, v in runs["groups"].items()} | {"e2e_ms_all": runs["groups"]["e2e_ms"]},
        "group_totals_equal_sizes": all(math.fsum(res[g]) == size[g] for g in range(npg)) if ag is None else None,
    }
    if dense:
        line["dense"] = {k: med(v) for k, v in runs["dense"].items()} | {
            "e2e_ms_all": runs["dense"]["e2e_ms"], "d2h_bytes": st_d["d2h_bytes"], "alg_bytes": st_d["alg_bytes"],
            "direction": st_d["direction"], "width": st_d["width"]}
        line["max_abs_diff"] = float(np.abs(res - want).max())
    else:
        line["dense"] = (f"not run: the {len(pro)} x {len(anc)} float64 matrix needs {nbytes / 1e9:.0f} GB of host "
                         "memory and more device memory than one B200 has")
    line.update({"gpu": name_gpu, "power_limit": power, "steps": args.steps, "warmup": args.warmup})
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="c3_pro,c3_both,c4_pro")
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    names = args.workload.split(",")
    for n in names:
        if n not in ("c3_pro", "c3_both", "c4_pro"):
            ap.error(f"unknown workload {n}")
    os.environ.pop("GENLIB_GC_DIRECTION", None)
    import genlib_b200 as gen
    if gen.lib().genlib_device_count() < 1:
        raise SystemExit("no CUDA device: gen.gcGroups has no CPU fallback")
    for n in names:
        run(gen, n, args)


if __name__ == "__main__":
    main()
