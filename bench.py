#!/usr/bin/env python
"""bench.py -- gen.phi on the named synthetic pedigree: kinship row-updates/s.

    python bench.py --gpus N --steps K --warmup W            (N = 1: this process;
    N > 1: one rank per GPU under torchrun, RANK/LOCAL_RANK/WORLD_SIZE from the env)
    python bench.py --impl reference ...                     (CPU restatement of the
    reference algorithm on the host cores, same metric and config)

A "step" is one complete pass of the hot path -- every generation layer of
gen.phi(ped, probands) -- over one synthetic pedigree.  `value` counts the pass
with the schedule already resident in HBM (CUDA events on the engine's
stream); `e2e` is the public call with HOST buffers: planning, H2D of the
schedule, all layers, proband gather and D2H into pinned host memory.
Both arms print the sha256 of the proband matrix they produced
(`output_sha256`) next to the committed golden one (tests/golden/, made by the
oracle alone).  Prints ONE JSON line (rank 0).  `--dump-outputs DIR` (one GPU,
or a full pass of the reference arm) also writes that matrix, or a seeded
sample of its rows, to DIR as .npy for output-by-output comparison of builds.
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "gen.phi kinship row-updates/s"
UNIT = "row-updates/s"


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as fh:
            return float(json.load(fh)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md: 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks/throttle reasons DURING the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "50", "-i", str(self.index)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def __exit__(self, *a):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self):
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
                for name, v in zip(names, r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                "samples": len(sm)}


# ---- what both arms agree on -------------------------------------------------------------------
def workload_desc(name: str, scale: float) -> str:
    if name == "genea140":
        return "genea140 (41523 individuals, 140 probands)"
    sys.path.insert(0, os.path.join(ROOT, "genlib.jl_b200"))
    from oracle.binding import _synth
    p = dict(_synth().CONFIGS[name])
    if scale != 1.0:
        p["n_individuals"] = max(p["generations"] * 4, int(round(p["n_individuals"] * scale)))
        p["n_probands"] = max(2, int(round(p["n_probands"] * scale)))
    return (f"{name} synthetic: {p['n_individuals']} individuals, {p['generations']} generations, "
            f"{p['n_probands']} probands, alpha={p['alpha']}, demes={p['demes']}, migration={p['migration']}, "
            f"overlap={p['overlap']}, seed={p['seed']}" + (f", scale={scale}" if scale != 1 else ""))


def shared_config(args, row_updates: int) -> dict:
    """The `config` object: identical in both arms for the same command line."""
    return {"workload": workload_desc(args.workload, args.scale), "numerics": args.numerics,
            "row_updates_per_step": int(row_updates), "output": "n_probands x n_probands Float32, host memory",
            "l2": "working set >> L2 (no flush needed)"}


def golden_record(args):
    name = f"{args.workload.lower()}_full.sha256" if args.scale == 1.0 else f"{args.workload.lower()}_x{args.scale:g}.sha256"
    try:
        with open(os.path.join(ROOT, "tests", "golden", name)) as fh:
            return json.load(fh)
    except Exception:
        return None


DUMP_BYTES = 60 << 20                # the whole dump, .npy header included, stays below 64 MB


def dump_outputs(out_dir: str, phi: np.ndarray):
    """Write the proband kinship matrix of the last timed step to `out_dir`, so that two builds can be
    compared output for output: phi.npy when it fits DUMP_BYTES, else phi_row_sample.npy, the rows
    sorted(default_rng(0).choice(n, k, replace=False)) with k as large as fits (the same rows for the
    same command line)."""
    os.makedirs(out_dir, exist_ok=True)
    n = phi.shape[0]
    k = DUMP_BYTES // max(1, n * phi.itemsize)
    if k >= n:
        np.save(os.path.join(out_dir, "phi.npy"), phi)
    else:
        rows = np.sort(np.random.default_rng(0).choice(n, k, replace=False))
        np.save(os.path.join(out_dir, "phi_row_sample.npy"), phi[rows])


def rows_digest(rows: np.ndarray) -> bytes:
    """Concatenated sha256 digests of the rows (32 bytes each): ranks hash their own rows, the
    digest of the concatenation in proband order is independent of how the rows were sharded."""
    return b"".join(hashlib.sha256(np.ascontiguousarray(r).tobytes()).digest() for r in rows)


def parity_fields(args, full_sha, rows_sha):
    g = golden_record(args) if args.numerics == "reference" else None
    out = {"output_sha256": full_sha, "output_rows_sha256": rows_sha,
           "golden_sha256": g["sha256"] if g else None, "golden_rows_sha256": g.get("rows_sha256") if g else None}
    if g and full_sha is not None:
        out["matches_golden"] = full_sha == g["sha256"]
    elif g and g.get("rows_sha256") and rows_sha is not None:
        out["matches_golden"] = rows_sha == g["rows_sha256"]
    else:
        out["matches_golden"] = None
    return out


def build_workload(args):
    """The product's own loader (C++), for the GPU arm."""
    import genlib_b200 as gen
    if args.workload == "genea140":
        ped = gen.genealogy(gen.genea140)
        pro = gen.pro(ped)
    else:
        s = gen.synth.config(args.workload, args.scale)
        ped = gen.genealogy(s.as_columns())
        pro = s.probands
    return gen, ped, ped.rank_of(pro)


# ---- the reference arm: the oracle on the host cores, no product library in the process -----------
def cpu_sample(father, mother, ranks, seconds):
    """Bounded sample: the first generation steps of the workload until `seconds` have elapsed."""
    from oracle import binding as ob
    cores = ob.num_threads()
    t0 = time.time()
    steps = ob.bounded_steps(father, mother, ranks, seconds, nthreads=cores)
    wall = time.time() - t0
    secs = float(steps[:, 5].sum()) if len(steps) else 0.0
    rows = float(steps[:, 4].sum()) if len(steps) else 0.0
    pairs = float(steps[:, 3].sum()) if len(steps) else 0.0
    return {"value": rows / secs if secs > 0 else 0.0, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": (f"first {len(steps)} generation steps ({int(rows)} row-updates, {pairs:.3g} pair "
                       f"evaluations) of the same pedigree, {secs:.1f} s in the pair loops, {wall:.1f} s wall; "
                       "C restatement of the reference algorithm (Julia is not installable here)"),
            "seconds": secs}


def cpu_baseline(ped, ranks, seconds):
    return cpu_sample(ped.father, ped.mother, ranks, seconds)


def run_reference(args, rank, world):
    """ONE complete pass of the whole workload through the oracle (all host threads): an unsampled
    CPU figure and the sha256 of its matrix.  C4 does not fit a host (2 x 71 GB step matrices):
    there, and with --ref-mode sample, K bounded samples of the first steps are timed instead."""
    if rank != 0:
        return
    from oracle import binding as ob
    father, mother, ranks, _ = ob.workload(args.workload, args.scale)
    cores = ob.num_threads()
    full = args.ref_mode == "full" or (args.ref_mode == "auto" and not (args.workload == "C4" and args.scale > 0.25))
    if args.dump_outputs and not full:
        raise SystemExit("bench.py: --dump-outputs with --impl reference needs a full pass (--ref-mode full)")
    for _ in range(min(args.warmup, 1)):
        cpu_sample(father, mother, ranks, 2.0)                      # pages the pedigree in, spins the cores up
    if full:
        t0 = time.time()
        phi, steps = ob.phi_ranks(father, mother, ranks, nthreads=cores)
        wall = time.time() - t0
        rows = int(steps[:, 4].sum())
        value, ms, k = rows / wall, wall * 1e3, 1
        base = {"value": value, "unit": UNIT, "cores": cores, "kind": "port",
                "sample": (f"the WHOLE workload, once: {len(steps)} generation steps, {rows} row-updates, "
                           f"{steps[:, 3].sum():.3g} pair evaluations, {wall:.1f} s wall (loops {steps[:, 5].sum():.1f} s); "
                           "C restatement of the reference algorithm (Julia is not installable here)"),
                "seconds": wall}
        par = parity_fields(args, ob.matrix_sha256(phi), hashlib.sha256(rows_digest(phi)).hexdigest())
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, phi)
    else:
        per = max(1.0, args.cpu_seconds / max(1, args.steps))
        vals, base = [], None
        t0 = time.time()
        for _ in range(args.steps):
            base = cpu_sample(father, mother, ranks, per)
            vals.append(base["value"])
        ms, k = (time.time() - t0) * 1e3 / max(1, args.steps), args.steps
        value = float(np.mean(vals))
        base["value"] = value
        rows = 0
        par = parity_fields(args, None, None)
    if not rows:                                                    # row-updates of a full pass, for `config`
        rows = ob.row_updates(father, mother, ranks)
    cfg = shared_config(args, rows)
    emit({"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
          "steps": k, "steps_requested": args.steps, "warmup": min(args.warmup, 1), "ms_per_step": ms,
          "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": data_tag(args),
          "config": cfg, "cpu_baseline": base, "parity": par,
          "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
          "gpu_launches": 0})


def data_tag(args):
    return "synthetic" if args.workload != "genea140" else "genea140.csv"


_REAL_STDOUT = None


def quiet_stdout():
    """Libraries (NCCL, torchrun banners) print to fd 1; the contract is ONE JSON line on stdout.
    Everything written to fd 1 from here on goes to stderr; emit() writes the line to the real one."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def emit(line: dict):
    out = _REAL_STDOUT if _REAL_STDOUT is not None else sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


# ---- roofline of the layer kernel ------------------------------------------------------------------
def roofline_record(infos, layer_ms, K, esize, peak, peak_src, world, args):
    """infos: per-layer dicts of this rank (summed over ranks by the caller for N > 1: dram/l2/nvlink
    bytes); layer_ms: (K, n_layers) device time of the layer kernel (slowest rank)."""
    dram = np.array([i["dram_read_bytes"] + i["dram_write_bytes"] for i in infos])
    l2 = np.array([i["l2_bytes"] for i in infos])
    nvl = np.array([i["nvlink_bytes"] for i in infos])
    alg = np.array([esize * i["alg_elems"] for i in infos])
    launched = np.array([i["n_new"] > 0 for i in infos])
    t = float(layer_ms[:, launched].sum()) * 1e-3
    achieved = float(dram[launched].sum()) * K / t / 1e9 if t > 0 else 0.0
    rec = {"bound": "hbm", "kernel": "layer_kernel", "achieved": achieved, "peak": peak * world, "unit": "GB/s",
           "frac": achieved / (peak * world),
           "bytes": "required DRAM bytes of the step from the plan: parent rows of the couples over the live columns "
                    "read once + new rows (and their mirror columns in carried rows) written once; the transposed "
                    "strip scratch stays in L2 and is not counted",
           "peak_source": (f"{world} x " if world > 1 else "") + peak_src,
           "launches": int(launched.sum()) * K,
           "avg_launch_ms": float(layer_ms[:, launched].mean()) if launched.any() else 0.0,
           "required_bytes_per_launch": float(dram[launched].mean()) if launched.any() else 0.0,
           "l2_scratch_bytes_per_launch": float(l2[launched].mean()) if launched.any() else 0.0,
           "nvlink_bytes_per_step": float(nvl.sum()),
           "share_of_step": 1.0,
           "survey_model": {"bytes": "s*(4nL+3n^2) per layer (SURVEY.md 8d): counts a row per individual and three passes "
                                     "over the intra-layer block; the engine moves less (one row per couple, one pass)",
                            "achieved": float(alg.sum()) * K / t / 1e9 if t > 0 else 0.0,
                            "frac": (float(alg.sum()) * K / t / 1e9 / (peak * world)) if t > 0 else 0.0}}
    # measured DRAM bytes of one launch, from a committed `ncu --set full` capture of this exact workload
    rec["traffic"], rec["traffic_source"] = None, "no ncu capture of this workload / GPU count under profiles/"
    try:
        with open(os.path.join(ROOT, "profiles", "r02", "ncu_traffic.json")) as fh:
            cap = json.load(fh)
        key = f"{args.workload}:{args.scale:g}:{args.numerics}:{world}"
        if key in cap:
            c = cap[key]
            rec["traffic"] = c["dram_bytes"]
            rec["traffic_source"] = c["source"]
            rec["traffic_layer"] = c["layer"]
            rec["traffic_required_bytes_same_launch"] = float(dram[c["layer"]])
    except Exception:
        pass
    return rec


def main():
    quiet_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="C3", choices=["C3", "C4", "C5", "genea140"])
    ap.add_argument("--scale", type=float, default=1.0)
    ap.add_argument("--numerics", default="reference", choices=["reference", "fp64"])
    ap.add_argument("--cpu-seconds", type=float, default=20.0, help="CPU baseline budget of the GPU arm (0 = skip)")
    ap.add_argument("--ref-mode", default="auto", choices=["auto", "full", "sample"],
                    help="reference arm: one full pass (sha256, unsampled) or bounded samples")
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--layers-json", default="", help="write per-layer timings here")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="write the proband matrix of the last timed step to DIR as .npy (a seeded sample of its rows above 60 MiB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.dump_outputs and world > 1:
        ap.error("--dump-outputs runs on one GPU only")
    if args.impl == "reference":
        return run_reference(args, rank, world)
    if world > 1:
        from bench_dist import main_dist          # sharded path (one rank per GPU)
        return main_dist(args, rank, world, local, sys.modules[__name__])

    gen, ped, ranks = build_workload(args)
    if gen.lib().genlib_device_count() < 1:
        raise SystemExit("bench.py: no CUDA device; the engine has no CPU fallback")
    esize = 4 if args.numerics == "reference" else 8
    t0 = time.time()
    plan = gen.Plan(ped.father, ped.mother, ranks)
    eng = gen.Engine(plan, numerics=args.numerics, device=local)
    setup_s = time.time() - t0
    rows = plan.metric_row_updates
    W = max(args.warmup, 3)
    for _ in range(W):
        eng.run()
    K = args.steps
    layer_ms, step_ms = [], []
    with ClockSampler(local) as clocks:
        time.sleep(0.6)                      # let nvidia-smi start sampling
        n0 = len(clocks.rows)
        while len(clocks.rows) == n0 and clocks.proc and time.time() < t0 + 60:
            eng.run()                        # keep the GPU under load until the first sample lands
        clocks.rows.clear()
        t0 = time.time()
        for _ in range(K):
            step_ms.append(eng.run(time_layers=True))
            layer_ms.append([eng.layer_info(t)["ms_layer"] for t in range(plan.n_layers)])
        wall_ms = (time.time() - t0) * 1e3
    stats = eng.stats()
    infos = [eng.layer_info(t) for t in range(plan.n_layers)]
    total_ms = float(np.sum(step_ms))
    value = rows * K / (total_ms * 1e-3)
    layer_ms = np.array(layer_ms)
    peak, peak_src = measured_peaks()
    roofline = roofline_record(infos, layer_ms, K, esize, peak, peak_src, 1, args)
    roofline["share_of_step"] = float(layer_ms.sum() / total_ms)
    if args.layers_json:
        with open(args.layers_json, "w") as fh:
            json.dump([{**i, "ms_layer": float(layer_ms[:, t].mean())} for t, i in enumerate(infos)], fh, indent=1)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, eng.fetch(dtype=np.float32 if esize == 4 else np.float64))
    eng.close()

    # ---- end to end: the public call with host buffers, pinned output ----
    n = plan.n_unique
    pinned = gen.PinnedMatrix(n, np.float32)
    e2e_t, h2d, d2h, st = [], 0, 0, None
    for it in range(args.e2e_steps + 1):
        t0 = time.time()
        _, st = gen.phi_arrays(ped.father, ped.mother, ranks, numerics=args.numerics, device=local,
                               out=pinned.array)
        dt = time.time() - t0
        if it > 0 or args.e2e_steps == 0:
            e2e_t.append(dt)
        h2d = st["h2d_bytes"] + ped.father.nbytes + ped.mother.nbytes + ranks.nbytes
        d2h = st["d2h_bytes"]
    e2e = {"value": rows / float(np.mean(e2e_t)), "unit": UNIT, "h2d_bytes_per_step": int(h2d),
           "d2h_bytes_per_step": int(d2h), "ms_per_call": float(np.mean(e2e_t)) * 1e3,
           "breakdown_ms": {k: st[k] for k in ("ms_plan", "ms_upload", "ms_kernels", "ms_fetch")}}
    parity = parity_fields(args, hashlib.sha256(pinned.array.tobytes()).hexdigest(),
                           hashlib.sha256(rows_digest(pinned.array)).hexdigest())
    checksum = float(pinned.array.astype(np.float64).sum())
    pinned.free()

    base = cpu_baseline(ped, ranks, args.cpu_seconds) if args.cpu_seconds > 0 else None
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": 1, "steps": K, "warmup": W,
            "ms_per_step": total_ms / K, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f64", "data": data_tag(args), "config": shared_config(args, rows),
            "engine": {"storage_bytes": esize, "layers": plan.n_layers, "capacity_slots": int(plan.capacity),
                       "device_bytes": int(stats["device_bytes"]), "alg_bytes_per_step": float(stats["alg_bytes"]),
                       "setup_s": setup_s, "host_wall_ms_per_step": wall_ms / K, "output_checksum": checksum},
            "roofline": roofline, "cpu_baseline": base, "e2e": e2e, "parity": parity,
            "gpu_launches": int(stats["kernel_launches"]) * K, "clocks": clocks.summary()}
    emit(line)


if __name__ == "__main__":
    main()
