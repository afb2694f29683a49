"""Plan / Engine handles over the C ABI and the `gen.phi` front end.

`phi` keeps the reference's signature and behaviour (src/compute.jl:233-304):
    phi(pedigree, probandIDs = pro(pedigree); verbose = false, compute = true)
returns a symmetric Float32 matrix in probandIDs order (duplicates collapsed),
`None` when compute is false, raises KeyError for an unknown ID.
"""
from __future__ import annotations

import ctypes as C
from collections.abc import Mapping
from typing import Optional

import numpy as np

from . import _lib
from . import pedigree as _pedigree
from ._lib import GcStats, LaunchShape, LayerInfo, PlanBoundsExceeded, Stats, check, lib, ptr
from .pedigree import Individual, Pedigree, pro


class Plan:
    """Host schedule (levels, Kirkpatrick frontier, slots). Needs no GPU."""

    def __init__(self, father, mother, proband_ranks, world: int = 1, schedule: str = "phi", ids=None,
                 stream: bool = False):
        """stream=True: the plan is made on a worker thread (genlib_plan_create_async); an Engine created on
        it runs every layer as soon as it is planned.  Any query but n_unique / world waits for the whole plan."""
        self.father = np.ascontiguousarray(father, np.int32)
        self.mother = np.ascontiguousarray(mother, np.int32)
        self.probands = np.ascontiguousarray(proband_ranks, np.int32)
        if len(self.father) != len(self.mother):
            raise ValueError("father and mother must have the same length")
        # sparse_phi's queue starts with the founders sorted by ID (identify.jl:15-19)
        self.ids = None if ids is None else np.ascontiguousarray(ids, np.int64)
        if self.ids is not None and len(self.ids) != len(self.father):
            raise ValueError("ids must have one entry per individual")
        h = C.c_void_p()
        create = lib().genlib_plan_create_async if stream else lib().genlib_plan_create_ex
        check(create(len(self.father), ptr(self.father), ptr(self.mother), ptr(self.ids),
                     len(self.probands), ptr(self.probands), world, _lib.SCHEDULES[schedule], C.byref(h)))
        self._h = h
        self.world = world
        self.schedule = schedule

    @classmethod
    def pairs(cls, father, mother, a, b, world: int = 1, stream: bool = False) -> "Plan":
        """The plan of gen.phi_pairs (genlib_plan_create_pairs): the pairs (a[k], b[k]) of ranks, read by the layers
        (`pair_reads`); stream=True makes it on a worker thread like Plan(..., stream=True)."""
        self = cls.__new__(cls)
        self.father = np.ascontiguousarray(father, np.int32)
        self.mother = np.ascontiguousarray(mother, np.int32)
        self.a, self.b = np.ascontiguousarray(a, np.int32), np.ascontiguousarray(b, np.int32)
        if len(self.father) != len(self.mother) or len(self.a) != len(self.b):
            raise ValueError("father and mother, and the two sides of the pairs, must have the same length")
        self.probands, self.ids = np.zeros(0, np.int32), None
        h = C.c_void_p()
        check(lib().genlib_plan_create_pairs(len(self.father), ptr(self.father), ptr(self.mother), len(self.a),
                                             ptr(self.a), ptr(self.b), world, int(stream), C.byref(h)))
        self._h, self.world, self.schedule = h, world, "pairs"
        return self

    def pair_reads(self, layer: int) -> dict:
        """The reads of a pairs plan just before `layer` (layer == n_layers: after the last one), in list order:
        list position, row slot (the higher-ranked member), column slot, the row's owner and local row."""
        n = lib().genlib_plan_pair_reads(self._h, layer, None, None, None, None, None)
        if n < 0:
            check(_lib.EINVAL)
        out = {"pos": np.zeros(n, np.int64)}
        out.update({k: np.zeros(n, np.int32) for k in ("row_slot", "col_slot", "owner", "lrow")})
        lib().genlib_plan_pair_reads(self._h, layer, *(ptr(out[k]) for k in ("pos", "row_slot", "col_slot", "owner", "lrow")))
        return out

    def __del__(self):
        h, self._h = getattr(self, "_h", None), None
        if h:
            lib().genlib_plan_destroy(h)

    n_unique = property(lambda s: lib().genlib_plan_n_unique(s._h))
    n_layers = property(lambda s: lib().genlib_plan_n_layers(s._h))
    capacity = property(lambda s: lib().genlib_plan_capacity(s._h))
    row_updates = property(lambda s: lib().genlib_plan_row_updates(s._h))     # rows the engine writes (every layer)

    @property
    def metric_row_updates(self) -> int:
        """The benchmark's unit (SURVEY.md 8d): proband-ancestors born AFTER the top level -- what the
        reference's steps compute (compute.jl:276-302); the top level is only the initial 1/2 I."""
        return int(self.row_updates - (self.layer_info(0)["n_new"] if self.n_layers > 0 else 0))

    def device_bytes(self, numerics="reference", rank: int = 0) -> int:
        return lib().genlib_plan_device_bytes(self._h, _lib.NUMERICS[numerics], rank)

    def layer_info(self, layer: int) -> dict:
        info = LayerInfo()
        check(lib().genlib_plan_layer_info(self._h, layer, C.byref(info)))
        return info.as_dict()

    def launch_shape(self, layer: int, numerics="reference", rank: int = 0, sm_count: int = 148) -> dict:
        """How an engine of `rank` would launch the layer kernel of `layer` on a device with `sm_count` SMs
        (genlib_plan_launch_shape: the GENLIB_* tuning variables of the environment apply); all zero when the
        rank has no couple in the layer."""
        shape = LaunchShape()
        check(lib().genlib_plan_launch_shape(self._h, layer, _lib.NUMERICS[numerics], rank, sm_count, C.byref(shape)))
        return shape.as_dict()

    def layers(self):
        return [self.layer_info(t) for t in range(self.n_layers)]

    def layer_arrays(self, layer: int) -> dict:
        info = self.layer_info(layer)
        n, nf = info["n_new"], info["n_fam"]
        out = {k: np.zeros(n, np.int32) for k in ("member_ind", "member_slot", "member_fam", "member_owner")}
        out.update({k: np.zeros(nf, np.int32) for k in ("fam_father_slot", "fam_mother_slot")})
        check(lib().genlib_plan_layer_arrays(self._h, layer, ptr(out["member_ind"]), ptr(out["member_slot"]),
                                             ptr(out["member_fam"]), ptr(out["fam_father_slot"]),
                                             ptr(out["fam_mother_slot"]), ptr(out["member_owner"])))
        flags = np.zeros(max(self.capacity, 1), np.uint8)
        check(lib().genlib_plan_layer_flags(self._h, layer, ptr(flags)))
        out["live_flags"] = flags
        out["member_rank"] = np.zeros(n, np.int32)
        if n:
            check(lib().genlib_plan_layer_ranks(self._h, layer, ptr(out["member_rank"])))
        return out

    def layer_shard(self, layer: int) -> dict:
        """Row sharding of a layer: own couple/member ranges per rank, local rows, parents' homes."""
        info = self.layer_info(layer)
        n, nf, w = info["n_new"], info["n_fam"], self.world
        out = {"fam_base": np.zeros(w + 1, np.int32), "mem_base": np.zeros(w + 1, np.int32),
               "member_lrow": np.zeros(n, np.int32)}
        out.update({k: np.zeros(nf, np.int32) for k in ("fam_father_owner", "fam_father_lrow",
                                                        "fam_mother_owner", "fam_mother_lrow")})
        check(lib().genlib_plan_layer_shard(self._h, layer, ptr(out["fam_base"]), ptr(out["mem_base"]),
                                            ptr(out["member_lrow"]), ptr(out["fam_father_owner"]),
                                            ptr(out["fam_father_lrow"]), ptr(out["fam_mother_owner"]),
                                            ptr(out["fam_mother_lrow"])))
        cap = max(self.capacity, 1)
        out["live_owner"], out["live_lrow"] = np.zeros(cap, np.int32), np.zeros(cap, np.int32)
        check(lib().genlib_plan_layer_live_rows(self._h, layer, ptr(out["live_owner"]), ptr(out["live_lrow"])))
        return out

    def rank_rows(self, rank: int) -> int:
        return lib().genlib_plan_rank_rows(self._h, rank)

    def proband_rows(self):
        n = self.n_unique
        owner, lrow = np.zeros(n, np.int32), np.zeros(n, np.int32)
        if n:
            check(lib().genlib_plan_proband_rows(self._h, ptr(owner), ptr(lrow)))
        return owner, lrow

    def proband_slots(self) -> np.ndarray:
        s = np.zeros(self.n_unique, np.int32)
        if self.n_unique:
            check(lib().genlib_plan_proband_slots(self._h, ptr(s)))
        return s

    def verbose_lines(self, running: bool = False):
        """The reference's per-step lines (src/compute.jl:257-260 and :281-284)."""
        infos = self.layers()[1:]
        S1 = len(infos)
        for k, i in enumerate(infos, 1):
            counts = (f"{i['ref_founders']} founders, {i['ref_probands']} probands, {i['ref_both']} both")
            yield (f"Running step {k} of {S1} ({counts})." if running else f"Step {k} of {S1}: {counts}.")


class Engine:
    """Device state of one rank: frontier rows, scratch, uploaded schedule.

    rank=None: the whole problem on one GPU.  With a plan built for world > 1, pass this
    process's rank; exchange `ipc_handle()` with the peers and `attach()` them before `run()`
    (see `phi_distributed`)."""

    def __init__(self, plan: Plan, numerics="reference", device: int = -1, rank: Optional[int] = None):
        self.plan = plan
        self.numerics = _lib.NUMERICS[numerics]
        self.rank = 0 if rank is None else rank
        h = C.c_void_p()
        if rank is None:
            check(lib().genlib_engine_create(plan._h, self.numerics, device, C.byref(h)))
        else:
            check(lib().genlib_engine_create_dist(plan._h, self.numerics, device, rank, C.byref(h)))
        self._h = h

    def ipc_handle(self) -> bytes:
        buf = C.create_string_buffer(64)
        check(lib().genlib_engine_ipc_export(self._h, buf))
        return buf.raw

    def attach(self, handles):
        """handles: one 64-byte CUDA-IPC handle per rank, rank-major (this rank's own is ignored)."""
        blob = b"".join(handles)
        assert len(blob) == 64 * self.plan.world
        check(lib().genlib_engine_ipc_attach(self._h, blob, 64))

    def own_probands(self) -> np.ndarray:
        n = lib().genlib_engine_own_probands(self._h, None)
        idx = np.zeros(n, np.int32)
        if n:
            lib().genlib_engine_own_probands(self._h, ptr(idx))
        return idx

    def close(self):
        h, self._h = getattr(self, "_h", None), None
        if h:
            lib().genlib_engine_destroy(h)

    __del__ = close

    def run(self, time_layers: bool = False, layer_limit: int = -1) -> float:
        """All generation steps on the device; returns CUDA-event milliseconds."""
        check(lib().genlib_engine_set_layer_limit(self._h, layer_limit))
        check(lib().genlib_engine_run(self._h, int(time_layers)))
        return self.stats()["ms_kernels"]

    def stats(self) -> dict:
        s = Stats()
        check(lib().genlib_engine_stats(self._h, C.byref(s)))
        return s.as_dict()

    def layer_info(self, layer: int) -> dict:
        info = LayerInfo()
        check(lib().genlib_engine_layer_info(self._h, layer, C.byref(info)))
        return info.as_dict()

    def fetch(self, out: Optional[np.ndarray] = None, dtype=np.float32) -> np.ndarray:
        """Rows of this rank's probands (all of them on one GPU) x all probands."""
        n = self.plan.n_unique
        rows = n if self.plan.world == 1 else lib().genlib_engine_own_probands(self._h, None)
        if out is None:
            out = np.empty((rows, n), dtype)
        if out.shape != (rows, n) or not out.flags.c_contiguous or out.dtype not in _lib.DTYPES:
            raise ValueError("out must be a C-contiguous (own rows, n_unique) float32/float64 array")
        check(lib().genlib_engine_fetch(self._h, ptr(out), _lib.DTYPES[out.dtype]))
        return out

    def phi_mean(self) -> float:
        v = C.c_double(0)
        check(lib().genlib_engine_phi_mean(self._h, C.byref(v)))
        return v.value

    def row_sums(self) -> np.ndarray:
        """(n_own, 2): per own proband row, the sum over all proband columns and the diagonal entry
        (binary64, fixed order).  Ranks' rows added in proband order give a rank-count-independent mean."""
        n = lib().genlib_engine_own_probands(self._h, None)
        out = np.zeros((n, 2), np.float64)
        if n:
            check(lib().genlib_engine_row_sums(self._h, ptr(out)))
        return out

    def phi_product(self, X, return_diagonal: bool = False):
        """Y = M X for this rank's proband rows (genlib_engine_phi_product), M the proband block of the run: X has
        plan.n_unique rows in the plan's proband order, the result one row per own proband (own_probands() order; one
        rank: list order).  A 1-D X gives a 1-D result.  The bits are gen.phiProduct's; the layers are not run again,
        so an iterative method can call this as often as it needs.  return_diagonal=True also returns M[i, i]."""
        X = np.asarray(X, np.float64)
        one = X.ndim == 1
        X2 = np.ascontiguousarray(X[:, None] if one else X)
        if X2.ndim != 2 or X2.shape[0] != self.plan.n_unique:
            raise ValueError(f"phi_product: X needs {self.plan.n_unique} rows, one per proband; it has shape {X.shape}")
        n = lib().genlib_engine_own_probands(self._h, None)
        Y = np.empty((n, X2.shape[1]), np.float64)
        d = np.empty(n, np.float64) if return_diagonal else None
        check(lib().genlib_engine_phi_product(self._h, X2.shape[1], ptr(X2), ptr(Y), ptr(d)))
        Y = Y[:, 0] if one else Y
        return (Y, d) if return_diagonal else Y

    def read_block(self, slots) -> np.ndarray:
        slots = np.ascontiguousarray(slots, np.int32)
        out = np.zeros((len(slots), len(slots)), np.float64)
        check(lib().genlib_engine_read_block(self._h, len(slots), ptr(slots), ptr(out)))
        return out


class PinnedMatrix:
    """A page-locked (n, n) host matrix for `out=` (genlib_pinned_alloc)."""

    def __init__(self, n: int, dtype=np.float32):
        self.dtype = np.dtype(dtype)
        nbytes = max(1, n * n * self.dtype.itemsize)
        p = C.c_void_p()
        check(lib().genlib_pinned_alloc(nbytes, C.byref(p)))
        self._p = p
        buf = (C.c_char * nbytes).from_address(p.value)
        self.array = np.frombuffer(buf, dtype=self.dtype, count=n * n).reshape(n, n)

    def free(self):
        p, self._p = getattr(self, "_p", None), None
        if p:
            self.array = None
            lib().genlib_pinned_free(p)

    __del__ = free


def phi(pedigree: Pedigree, probandIDs=None, *, verbose: bool = False, compute: bool = True,
        numerics="reference", dtype=np.float32, device: int = -1, out: Optional[np.ndarray] = None,
        return_stats: bool = False, devices=None):
    """gen.phi(pedigree, probandIDs; verbose, compute) on the B200 engine.  `devices=[0, 1, ...]` shards
    the frontier over several GPUs of the box from this one process (genlib_phi_multi).

    gen.phi(ind1, ind2) with two Individuals of one pedigree is the reference's scalar method
    (src/compute.jl:66-95): their kinship as a Python float, through `phi_pairs` with one pair."""
    if isinstance(pedigree, Individual):
        ind1, ind2 = pedigree, probandIDs
        if not isinstance(ind2, Individual) or ind2._ped is not ind1._ped:
            raise ValueError("gen.phi(ind1, ind2): two Individuals of one pedigree")
        ped = ind1._ped
        res, _ = phi_pairs_arrays(ped.father, ped.mother, [ind1._r], [ind2._r], device=device, devices=devices)
        return float(res[0])
    IDs = pro(pedigree) if probandIDs is None else np.asarray(probandIDs, np.int64)
    ranks = pedigree.rank_of(IDs)                       # KeyError, like pedigree[ID]
    plan = Plan(pedigree.father, pedigree.mother, ranks, stream=compute and not verbose and devices is None)
    if verbose or not compute:
        for line in plan.verbose_lines():
            print(line)
    if not compute:
        return None
    n = plan.n_unique
    if n == 0:
        res = np.zeros((0, 0), dtype)
        return (res, {}) if return_stats else res
    if verbose:
        for line in plan.verbose_lines(running=True):
            print(line)
    if devices is not None and len(devices) > 1:
        if out is None:
            out = np.empty((n, n), dtype)
        res, stats = phi_arrays(pedigree.father, pedigree.mother, ranks, numerics=numerics, out=out, devices=devices)
        return (res, stats) if return_stats else res
    if devices is not None and len(devices) == 1:
        device = int(devices[0])
    eng = Engine(plan, numerics=numerics, device=device)
    try:
        try:
            eng.run()
        except PlanBoundsExceeded:                      # a bound of the streamed plan did not hold: the plan is finished now
            eng.close()
            eng = Engine(plan, numerics=numerics, device=device)
            eng.run()
        res = eng.fetch(out=out, dtype=dtype)
        stats = eng.stats()
    finally:
        eng.close()
    return (res, stats) if return_stats else res


def run_distributed(plan: Plan, numerics="reference", device: int = 0, rank: int = 0) -> Engine:
    """This rank's engine of a `torch.distributed` job, attached to its peers and run once.  Collective.
    With a streamed plan (Plan(..., stream=True)) the layers run while the later ones are planned; if a size
    bound of that plan does not hold, every rank finds out (same plan, same bounds) and all start over.
    The ranks agree on the outcome before anybody goes on to fetch or gather: a failure of one rank (an
    inter-GPU barrier that timed out also marks every peer) raises on all of them instead of leaving the
    others waiting in the next collective."""
    import torch.distributed as dist
    for attempt in (0, 1):
        eng = Engine(plan, numerics=numerics, device=device, rank=rank)
        outcome, error = "ok", None
        try:
            handles = [None] * plan.world
            dist.all_gather_object(handles, eng.ipc_handle())
            eng.attach(handles)
            dist.barrier()
            try:
                eng.run()
            except PlanBoundsExceeded:
                outcome = "restart"
            except Exception as e:                                  # noqa: BLE001 -- reported to every rank below
                outcome, error = "failed", e
            outcomes = [None] * plan.world
            dist.all_gather_object(outcomes, outcome)              # (also: nobody unmaps while a peer may still read)
        except BaseException:
            eng.close()
            raise
        if all(o == "ok" for o in outcomes):
            return eng
        eng.close()
        if "failed" in outcomes:
            if error is not None:
                raise error
            raise RuntimeError(f"gen.phi: rank(s) {[g for g, o in enumerate(outcomes) if o == 'failed']} failed")
        if attempt:
            raise PlanBoundsExceeded(7, "the plan's bounds did not hold on the finished plan")
    raise AssertionError("unreachable")


def phi_distributed(pedigree: Pedigree, probandIDs=None, *, numerics="reference", dtype=np.float32,
                    device: Optional[int] = None, gather: bool = True, return_stats: bool = False,
                    schedule: str = "phi"):
    """gen.phi on all ranks of a `torch.distributed` job (one process per GPU of one box).

    Every rank builds the same plan, owns a share of the frontier rows, reads parent rows and
    pushes couple-matrix rows through NVLink peer mappings.  Collective: call on every rank.
    gather=True returns the full matrix on rank 0 (None elsewhere); gather=False returns
    (own_proband_indices, own_rows) on every rank.  schedule="sparse_phi" gives the values of
    gen.sparse_phi instead (dense, in proband order)."""
    import torch.distributed as dist
    rank, world = dist.get_rank(), dist.get_world_size()
    IDs = pro(pedigree) if probandIDs is None else np.asarray(probandIDs, np.int64)
    ranks = pedigree.rank_of(IDs)
    plan = Plan(pedigree.father, pedigree.mother, ranks, world=world, schedule=schedule,
                ids=pedigree.ids if schedule != "phi" else None, stream=True)
    n = plan.n_unique
    if n == 0:
        res = np.zeros((0, 0), dtype)
        return (res, {}) if return_stats else res
    if device is None:
        import os
        device = int(os.environ.get("LOCAL_RANK", rank))
    eng = run_distributed(plan, numerics=numerics, device=device, rank=rank)
    try:
        own, rows = eng.own_probands(), eng.fetch(dtype=dtype)
        stats = eng.stats()
        dist.barrier()                      # nobody unmaps while a peer may still read
    finally:
        eng.close()
    if not gather:
        return ((own, rows), stats) if return_stats else (own, rows)
    parts = [None] * world if rank == 0 else None
    dist.gather_object((own, rows), parts, dst=0)
    res = None
    if rank == 0:
        res = np.empty((n, n), dtype)
        for idx, blk in parts:
            res[idx] = blk
    return (res, stats) if return_stats else res


def phi_arrays(father, mother, proband_ranks, *, numerics="reference", dtype=np.float32,
               device: int = -1, out: Optional[np.ndarray] = None, devices=None):
    """One-shot C-ABI call `genlib_phi` on flat arrays (what the Julia shim ccalls); with
    `devices=[...]` the same through `genlib_phi_multi` (one process, several GPUs)."""
    father = np.ascontiguousarray(father, np.int32)
    mother = np.ascontiguousarray(mother, np.int32)
    pr = np.ascontiguousarray(proband_ranks, np.int32)
    n_unique = len(np.unique(pr)) if ((pr >= 0) & (pr < len(father))).all() else len(pr)
    if out is None:
        out = np.empty((n_unique, n_unique), dtype)
    st = Stats()
    if devices is not None:
        dv = np.ascontiguousarray(devices, np.int32)
        check(lib().genlib_phi_multi(len(father), ptr(father), ptr(mother), len(pr), ptr(pr), ptr(out),
                                     _lib.DTYPES[np.dtype(out.dtype)], _lib.NUMERICS[numerics], len(dv), ptr(dv),
                                     C.byref(st)))
    else:
        check(lib().genlib_phi(len(father), ptr(father), ptr(mother), len(pr), ptr(pr), ptr(out),
                               _lib.DTYPES[np.dtype(out.dtype)], _lib.NUMERICS[numerics], device, C.byref(st)))
    return out, st.as_dict()


class PhiOver:
    """What gen.phiOver returns, GENLIB's data frame `line, column, pro1, pro2, kinship`: one entry per proband pair whose
    kinship reaches the threshold, ordered by line, then column.  `line` < `column` are 0-based positions in the
    deduplicated proband list (the rows and columns of gen.phi's matrix), `pro1` / `pro2` the IDs at those positions,
    `kinship` the matrix entry, bit for bit (float32, or float64)."""

    def __init__(self, line, column, pro1, pro2, kinship, threshold: float):
        self.line, self.column = np.asarray(line, np.int64), np.asarray(column, np.int64)
        self.pro1, self.pro2 = np.asarray(pro1, np.int64), np.asarray(pro2, np.int64)
        self.kinship = np.asarray(kinship)
        self.threshold = threshold

    def __len__(self) -> int:
        return len(self.line)

    def __repr__(self) -> str:
        return f"PhiOver({len(self)} pairs with kinship >= {self.threshold!r}, {self.kinship.dtype})"


def _first_occurrences(ids) -> np.ndarray:
    """The IDs with duplicates collapsed onto their first occurrence (the rows of gen.phi's matrix)."""
    _, first = np.unique(ids, return_index=True)
    return ids[np.sort(first)]


def _phi_over_host(phi_matrix, threshold: float, probandIDs) -> PhiOver:
    """GENLIB's phiOver(phiMatrix, threshold) on a matrix in host memory: the pairs (i, j), i < j, with
    M[i, j] >= threshold, M[i, j] compared as a float64."""
    m = np.asarray(phi_matrix)
    if m.ndim != 2 or m.shape[0] != m.shape[1]:
        raise ValueError(f"gen.phiOver: a Pedigree or a square kinship matrix, not an array of shape {m.shape}")
    n = m.shape[0]
    ids = np.arange(n, dtype=np.int64) if probandIDs is None else \
        _first_occurrences(np.asarray(probandIDs, np.int64).reshape(-1))
    if len(ids) != n:
        raise ValueError(f"gen.phiOver: {len(ids)} distinct proband IDs for a {n} x {n} matrix")
    lines, cols = [np.zeros(0, np.int64)], [np.zeros(0, np.int64)]
    step = max(1, (1 << 24) // max(n, 1))                  # rows per block: the float64 copy stays at 128 MB
    for r0 in range(0, n, step):
        i, j = np.nonzero(m[r0:r0 + step].astype(np.float64) >= threshold)
        i += r0
        keep = j > i
        lines.append(i[keep])
        cols.append(j[keep])
    line, column = np.concatenate(lines), np.concatenate(cols)
    return PhiOver(line, column, ids[line], ids[column], m[line, column], threshold)


def phiOver(pedigree, threshold, probandIDs=None, *, numerics="reference", dtype=np.float32, max_pairs=None,
            device: int = -1, devices=None, return_stats: bool = False):
    """GENLIB's phiOver: the proband pairs whose kinship is at least `threshold`, as a `PhiOver` record.

    gen.phiOver(pedigree, threshold, probandIDs = pro(pedigree)) runs gen.phi's plan and layers on the device and
    selects there, from the proband rows each device holds (genlib_phi_over): only the pairs (and 8 bytes per row)
    leave the device, never the matrix.  The result is `np.nonzero(np.triu(M >= threshold, 1))` of the matrix M that
    gen.phi(pedigree, probandIDs, numerics=numerics, dtype=dtype) returns, with M at those positions, the same bits
    for any number of devices: the diagonal is never selected, M[i, j] is compared as a float64 (a float32 entry is
    widened exactly), threshold <= 0 selects every pair, +inf none.  More than `max_pairs` pairs raise
    GenlibOverflowError (an OverflowError) naming their number and the threshold; fewer than two distinct probands
    give an empty result without a device.  ValueError on a NaN threshold, KeyError on an unknown ID.

    gen.phiOver(phi_matrix, threshold, probandIDs=None), with a square array first, is the same selection on a matrix
    already in host memory; `probandIDs` (duplicates collapse, as in gen.phi) names its rows, else pro1 / pro2 are the
    positions."""
    threshold = float(threshold)
    if np.isnan(threshold):
        raise ValueError("gen.phiOver: the threshold is NaN")
    if not isinstance(pedigree, Pedigree):
        res, stats = _phi_over_host(pedigree, threshold, probandIDs), {}
        return (res, stats) if return_stats else res
    IDs = pro(pedigree) if probandIDs is None else np.asarray(probandIDs, np.int64).reshape(-1)
    ranks = pedigree.rank_of(IDs)                       # KeyError, like pedigree[ID]
    ids = _first_occurrences(IDs)
    line, column, kinship, stats = phi_over_arrays(pedigree.father, pedigree.mother, ranks, threshold, numerics=numerics,
                                                   dtype=dtype, max_pairs=max_pairs, device=device, devices=devices)
    res = PhiOver(line, column, ids[line], ids[column], kinship, threshold)
    return (res, stats) if return_stats else res


def phi_over_arrays(father, mother, proband_ranks, threshold, *, numerics="reference", dtype=np.float32,
                    max_pairs=None, device: int = -1, devices=None):
    """One-shot C-ABI call `genlib_phi_over` on flat rank arrays (what the Julia shim ccalls).  Returns
    (line, column, kinship, stats): 0-based positions in the deduplicated proband list, line < column, in (line,
    column) order, and the matrix entries as float32 or float64.  The library's arrays are copied and freed."""
    father = np.ascontiguousarray(father, np.int32)
    mother = np.ascontiguousarray(mother, np.int32)
    pr = np.ascontiguousarray(proband_ranks, np.int32)
    dt = np.dtype(dtype)
    if dt not in _lib.DTYPES:
        raise ValueError("dtype must be float32 or float64")
    dv = np.ascontiguousarray([device] if devices is None else devices, np.int32)
    res, st = _lib.KinshipPairs(), Stats()
    rc = lib().genlib_phi_over(len(father), ptr(father), ptr(mother), len(pr), ptr(pr), float(threshold),
                               -1 if max_pairs is None else int(max_pairs), _lib.DTYPES[dt], _lib.NUMERICS[numerics],
                               len(dv), ptr(dv), C.byref(res), C.byref(st))
    try:
        check(rc)
        n = res.n

        def take(p, t):
            t = np.dtype(t)
            return np.frombuffer((C.c_char * (n * t.itemsize)).from_address(p), t, n).copy() if n else np.zeros(0, t)

        line, column, kinship = take(res.row, np.int32), take(res.col, np.int32), take(res.value, dt)
    finally:
        lib().genlib_kinship_pairs_free(C.byref(res))
    return line.astype(np.int64), column.astype(np.int64), kinship, st.as_dict()


class GroupKinship:
    """What gen.phiMeanGroups returns.  `ids`: the probands, sorted; `groups`: the group labels, sorted; `size`: the
    probands per group (int64); `mean[h, g]`: the mean kinship between groups h and g, pairs of distinct probands
    (G x G, symmetric, float64); `proband[i, g]`: the mean kinship of proband ids[i] with the other members of group g
    (P x G, float64).  A proband alone in its group has NaN in its own column; a one-member group NaN on the diagonal."""

    def __init__(self, ids, groups, size, mean, proband):
        self.ids, self.groups, self.size = ids, groups, size
        self.mean, self.proband = mean, proband

    def __repr__(self) -> str:
        return f"GroupKinship({len(self.ids)} probands in {len(self.groups)} groups)"


def _group_mapping(pedigree: Pedigree, groups):
    """A {ID: label} mapping read as (IDs sorted, labels sorted, each ID's label index, members per label (int64),
    the IDs' ranks).  TypeError on labels that do not compare, KeyError on an unknown ID."""
    ids = np.array(sorted(int(i) for i in groups), np.int64)
    labels = np.empty(len(ids), object)
    labels[:] = [groups[int(i)] for i in ids]
    levels, index = np.unique(labels, return_inverse=True)          # (TypeError on labels that do not compare)
    levels = np.array(levels.tolist())
    size = np.bincount(index, minlength=len(levels)).astype(np.int64)
    return ids, levels, index, size, pedigree.rank_of(ids)          # KeyError, like pedigree[ID]


def phiMeanGroups(pedigree: Pedigree, groups, *, numerics="reference", device: int = -1, devices=None,
                  return_stats: bool = False) -> GroupKinship:
    """Mean kinship within and between groups of probands, and of each proband with each group, as a `GroupKinship`.

    `groups` maps proband IDs to labels (`{ID: population}`, what GenLib's `_pop` reads from pop140.csv).  The probands
    are its IDs sorted ascending, the groups its distinct labels sorted (TypeError when labels do not compare, e.g. str
    and int).  M is the matrix gen.phi(pedigree, ids, numerics=numerics) returns, widened exactly to float64; the means
    are over pairs of distinct probands (the diagonal is skipped).  gen.phi's plan and layers run on the device and
    every device reduces the proband rows it holds (genlib_phi_groups): only P x G doubles leave the device, never the
    matrix.  The order of every sum is fixed by the list and the groups, so the result is the same bits on any number
    of devices; where every partial sum is a float64 number each mean is the exact rational rounded once.  An empty
    mapping gives an empty record without a device; KeyError on an unknown ID."""
    ids, levels, index, size, ranks = _group_mapping(pedigree, groups)
    if len(ids) == 0:
        res, stats = GroupKinship(ids, levels, size, np.zeros((0, 0)), np.zeros((0, 0))), {}
    else:
        pm, gm, stats = phi_groups_arrays(pedigree.father, pedigree.mother, ranks, index, len(levels), numerics=numerics,
                                          device=device, devices=devices)
        res = GroupKinship(ids, levels, size, gm, pm)
    return (res, stats) if return_stats else res


def phi_groups_arrays(father, mother, proband_ranks, group_index, n_groups, *, numerics="reference", device: int = -1,
                      devices=None):
    """One-shot C-ABI call `genlib_phi_groups` on flat rank arrays (what the Julia shim ccalls): distinct proband ranks
    in list order, each one's group in [0, n_groups).  Returns (proband_mean (P x G), group_mean (G x G), stats)."""
    father = np.ascontiguousarray(father, np.int32)
    mother = np.ascontiguousarray(mother, np.int32)
    pr = np.ascontiguousarray(proband_ranks, np.int32).reshape(-1)
    gi = np.ascontiguousarray(group_index, np.int32).reshape(-1)
    if len(gi) != len(pr):
        raise ValueError(f"phi_groups_arrays: {len(gi)} group indices for {len(pr)} probands")
    n_groups = int(n_groups)
    pm = np.empty((len(pr), max(n_groups, 0)), np.float64)
    gm = np.empty((max(n_groups, 0), max(n_groups, 0)), np.float64)
    dv = np.ascontiguousarray([device] if devices is None else devices, np.int32)
    st = Stats()
    check(lib().genlib_phi_groups(len(father), ptr(father), ptr(mother), len(pr), ptr(pr), ptr(gi), n_groups,
                                  _lib.NUMERICS[numerics], len(dv), ptr(dv), ptr(pm), ptr(gm), C.byref(st)))
    return pm, gm, st.as_dict()


def phiProduct(pedigree: Pedigree, X, probandIDs=None, *, numerics="reference", device: int = -1, devices=None,
               return_diagonal: bool = False, return_stats: bool = False):
    """The proband kinship matrix times a block of vectors, Y = M X, formed on the device (genlib_phi_product).

    M is the matrix gen.phi(pedigree, probandIDs, numerics=numerics) returns, widened exactly to float64; probandIDs
    defaults to pro(pedigree) and must not repeat an ID.  X has one row per proband in probandIDs order (P x k, or a
    vector of P for a 1-D result); Y[i, c] = sum over all j of M[i, j] X[j, c], the diagonal included.  With
    return_diagonal=True the result is (Y, diag), diag[i] = M[i, i], so that the sum over relatives j != i is
    Y - diag[:, None] * X.  gen.phi's plan and layers run on the device and every device multiplies the proband rows
    it holds: only P x k doubles leave the device, never the matrix.  Each entry is summed in a fixed order that
    depends only on P, so a column of X gives the same bits alone or in a block, on any number of devices and through
    Engine.phi_product; where every product and partial sum is a float64 number (integer X on geneaJi or genea140) Y
    is exact.  ValueError on a repeated ID or a row count that is not P, KeyError on an unknown ID, both before any
    device work."""
    IDs = pro(pedigree) if probandIDs is None else np.asarray(probandIDs, np.int64).reshape(-1)
    if len(np.unique(IDs)) != len(IDs):
        raise ValueError("phiProduct: duplicate proband IDs")
    X = np.asarray(X, np.float64)
    if X.ndim not in (1, 2) or X.shape[0] != len(IDs):
        raise ValueError(f"phiProduct: X needs {len(IDs)} rows, one per proband; it has shape {X.shape}")
    ranks = pedigree.rank_of(IDs)                       # KeyError, like pedigree[ID]
    Y, d, stats = phi_product_arrays(pedigree.father, pedigree.mother, ranks, X[:, None] if X.ndim == 1 else X,
                                     numerics=numerics, device=device, devices=devices, diagonal=return_diagonal)
    Y = Y[:, 0] if X.ndim == 1 else Y
    res = (Y, d) if return_diagonal else Y
    return (res, stats) if return_stats else res


def phi_product_arrays(father, mother, proband_ranks, X, *, numerics="reference", device: int = -1, devices=None,
                       diagonal: bool = False):
    """One-shot C-ABI call `genlib_phi_product` on flat arrays (what the Julia shim ccalls): distinct proband ranks in
    list order and X (P x k, its rows in that order).  Returns (Y (P x k), diag (P) or None, stats)."""
    father = np.ascontiguousarray(father, np.int32)
    mother = np.ascontiguousarray(mother, np.int32)
    pr = np.ascontiguousarray(proband_ranks, np.int32).reshape(-1)
    X = np.ascontiguousarray(X, np.float64)
    if X.ndim != 2 or X.shape[0] != len(pr):
        raise ValueError(f"phi_product_arrays: X of shape {X.shape} for {len(pr)} probands")
    k = X.shape[1]
    Y = np.empty((len(pr), k), np.float64)
    d = np.empty(len(pr), np.float64) if diagonal else None
    dv = np.ascontiguousarray([device] if devices is None else devices, np.int32)
    st = Stats()
    check(lib().genlib_phi_product(len(father), ptr(father), ptr(mother), len(pr), ptr(pr), k, ptr(X),
                                   _lib.NUMERICS[numerics], len(dv), ptr(dv), ptr(Y), ptr(d), C.byref(st)))
    return Y, d, st.as_dict()


class GcPlan:
    """The schedule of gen.gc (genlib_gc_plan_*): direction, layers, frontier slots.  Needs no GPU."""

    def __init__(self, father, mother, proband_ranks, ancestor_ranks, *, pro_group=None, n_pro_groups: int = 0,
                 anc_group=None, n_anc_groups: int = 0):
        """With `pro_group` and/or `anc_group` (a group index per rank), gen.gcGroups' schedule
        (genlib_gc_groups_plan_create)."""
        self.father = np.ascontiguousarray(father, np.int32)
        self.mother = np.ascontiguousarray(mother, np.int32)
        self.probands = np.ascontiguousarray(proband_ranks, np.int32)
        self.ancestors = np.ascontiguousarray(ancestor_ranks, np.int32)
        if len(self.father) != len(self.mother):
            raise ValueError("father and mother must have the same length")
        h = C.c_void_p()
        if pro_group is None and anc_group is None:
            check(lib().genlib_gc_plan_create(len(self.father), ptr(self.father), ptr(self.mother), len(self.probands),
                                              ptr(self.probands), len(self.ancestors), ptr(self.ancestors), C.byref(h)))
        else:
            pg, ag = _group_array(pro_group, self.probands), _group_array(anc_group, self.ancestors)
            check(lib().genlib_gc_groups_plan_create(len(self.father), ptr(self.father), ptr(self.mother),
                                                     len(self.probands), ptr(self.probands), ptr(pg), int(n_pro_groups),
                                                     len(self.ancestors), ptr(self.ancestors), ptr(ag),
                                                     int(n_anc_groups), C.byref(h)))
        self._h = h

    def __del__(self):
        h, self._h = getattr(self, "_h", None), None
        if h:
            lib().genlib_gc_plan_destroy(h)

    def info(self) -> dict:
        """genlib_gc_stats without timings; `direction` is "descend" or "ascend"."""
        s = GcStats()
        check(lib().genlib_gc_plan_info(self._h, C.byref(s)))
        d = s.as_dict()
        d["direction"] = _lib.GC_DIRECTIONS[d["direction"]]
        return d

    def layer_arrays(self, layer: int) -> dict:
        n_rows, n_in = C.c_int32(), C.c_int64()
        check(lib().genlib_gc_plan_layer(self._h, layer, C.byref(n_rows), C.byref(n_in)))
        out = {k: np.zeros(n_rows.value, np.int32) for k in ("row_ind", "row_slot", "row_seed", "row_out")}
        out["in_ptr"] = np.zeros(n_rows.value + 1, np.int64)
        out["in_slot"] = np.zeros(n_in.value, np.int32)
        check(lib().genlib_gc_plan_layer_arrays(self._h, layer, *(ptr(out[k]) for k in (
            "row_ind", "row_slot", "row_seed", "row_out", "in_ptr", "in_slot"))))
        return out

    def layers(self):
        return [self.layer_arrays(t) for t in range(self.info()["n_layers"])]


def gc(pedigree: Pedigree, pro=None, ancestors=None, *, dtype=np.float64, device: int = -1, devices=None,
       out: Optional[np.ndarray] = None, return_stats: bool = False):
    """gen.gc(pedigree; pro = pro(pedigree), ancestors = founder(pedigree)) on the B200 engine
    (src/compute.jl:518-595): the genetic contribution of every ancestor to every proband,
    G[p, a] = sum over descent paths a -> p of (1/2)^length, a len(pro) x len(ancestors) Float64 matrix
    in list order, duplicates kept.  KeyError on an unknown ID.  `devices=[0, 1, ...]` splits the
    columns over several GPUs of the box (genlib_gc)."""
    pro_ids = _pedigree.pro(pedigree) if pro is None else np.asarray(pro, np.int64)
    anc_ids = _pedigree.founder(pedigree) if ancestors is None else np.asarray(ancestors, np.int64)
    res, stats = gc_arrays(pedigree.father, pedigree.mother, pedigree.rank_of(pro_ids), pedigree.rank_of(anc_ids),
                           dtype=dtype, device=device, devices=devices, out=out)
    return (res, stats) if return_stats else res


def gc_arrays(father, mother, proband_ranks, ancestor_ranks, *, dtype=np.float64, device: int = -1, devices=None,
              out: Optional[np.ndarray] = None, col_major: bool = False):
    """One-shot C-ABI call `genlib_gc` on flat rank arrays (what the Julia shim ccalls).  Returns
    (matrix, stats); col_major=True fills a Fortran-ordered matrix (a Julia Matrix) without a transpose."""
    father = np.ascontiguousarray(father, np.int32)
    mother = np.ascontiguousarray(mother, np.int32)
    pr = np.ascontiguousarray(proband_ranks, np.int32)
    an = np.ascontiguousarray(ancestor_ranks, np.int32)
    shape = (len(pr), len(an))
    if out is None:
        out = np.empty(shape, dtype, order="F" if col_major else "C")
    contiguous = out.flags.f_contiguous if col_major else out.flags.c_contiguous
    if out.shape != shape or not contiguous or out.dtype not in _lib.DTYPES:
        raise ValueError(f"out must be a {'Fortran' if col_major else 'C'}-contiguous {shape} float32/float64 array")
    dv = np.ascontiguousarray([device] if devices is None else devices, np.int32)
    st = GcStats()
    check(lib().genlib_gc(len(father), ptr(father), ptr(mother), len(pr), ptr(pr), len(an), ptr(an), ptr(out),
                          _lib.DTYPES[np.dtype(out.dtype)], int(col_major), len(dv), ptr(dv), C.byref(st)))
    stats = st.as_dict()
    stats["direction"] = _lib.GC_DIRECTIONS[stats["direction"]]
    return out, stats


class GroupContribution:
    """What gen.gcGroups returns.  `rows` / `cols`: the output positions of the proband / ancestor side -- a grouped
    side's labels, sorted, or a list's IDs in list order; `row_size` / `col_size`: the individuals in each (int64, 1 for
    a list entry); `total[r, c]`: the sum of G[p, a] over the probands p of row r and the ancestors a of column c
    (float64); `mean = total / row_size[:, None]`: the mean contribution of column c to one proband of row r."""

    def __init__(self, rows, cols, row_size, col_size, total):
        self.rows, self.cols, self.row_size, self.col_size = rows, cols, row_size, col_size
        self.total = total
        self.mean = total / row_size[:, None]

    def __repr__(self) -> str:
        return f"GroupContribution({len(self.rows)} x {len(self.cols)})"


def gcGroups(pedigree: Pedigree, pro=None, ancestors=None, *, device: int = -1, devices=None,
             return_stats: bool = False) -> GroupContribution:
    """gen.gc summed over groups, as a `GroupContribution`: total[r, c] = the sum of G[p, a] over p in row r and a in
    column c, where G is what gen.gc returns for the same lists.

    Each of `pro` and `ancestors` is None (gen.pro / gen.founder, as in gen.gc), a list of IDs (one row / column per
    entry, duplicates kept) or a {ID: label} mapping (one row / column per label; IDs sorted, labels sorted, TypeError
    when labels do not compare).  At least one side must be a mapping (ValueError otherwise: that is gen.gc).  G is
    linear, so the engine propagates one column per group and sums the other side's rows per group on the device
    (genlib_gc_groups): only the R x C result leaves it, never the proband x ancestor matrix.  Where every partial
    sum is a float64 number (founders as ancestors, any realistic group size) the result is the exact sum.  KeyError
    on an unknown ID."""
    sides = []
    for arg, default in ((pro, _pedigree.pro), (ancestors, _pedigree.founder)):
        if isinstance(arg, Mapping):
            _, levels, index, size, ranks = _group_mapping(pedigree, arg)
            sides.append((levels, size, ranks, index, len(levels)))
        else:
            ids = default(pedigree) if arg is None else np.asarray(arg, np.int64)
            sides.append((ids, np.ones(len(ids), np.int64), pedigree.rank_of(ids), None, 0))
    (rows, row_size, pr, pg, npg), (cols, col_size, an, ag, nag) = sides
    if pg is None and ag is None:
        raise ValueError("gen.gcGroups needs a {ID: group} mapping for pro or ancestors; for two lists use gen.gc")
    total, stats = gc_groups_arrays(pedigree.father, pedigree.mother, pr, an, pro_group=pg, n_pro_groups=npg,
                                    anc_group=ag, n_anc_groups=nag, device=device, devices=devices)
    res = GroupContribution(rows, cols, row_size, col_size, total)
    return (res, stats) if return_stats else res


def _group_array(group, ranks):
    if group is None:
        return None
    g = np.ascontiguousarray(group, np.int32).reshape(-1)
    if len(g) != len(ranks):
        raise ValueError(f"{len(g)} group indices for {len(ranks)} ranks")
    return g


def gc_groups_arrays(father, mother, proband_ranks, ancestor_ranks, *, pro_group=None, n_pro_groups: int = 0,
                     anc_group=None, n_anc_groups: int = 0, device: int = -1, devices=None, col_major: bool = False):
    """One-shot C-ABI call `genlib_gc_groups` on flat rank arrays (what the Julia shim ccalls).  A side with a group
    array (distinct ranks, each one's group in [0, n_groups)) is grouped, a side without one is a list as in
    gc_arrays.  Returns (total, stats): R x C float64, R = n_pro_groups or len(proband_ranks), C likewise."""
    father = np.ascontiguousarray(father, np.int32)
    mother = np.ascontiguousarray(mother, np.int32)
    pr = np.ascontiguousarray(proband_ranks, np.int32).reshape(-1)
    an = np.ascontiguousarray(ancestor_ranks, np.int32).reshape(-1)
    pg, ag = _group_array(pro_group, pr), _group_array(anc_group, an)
    shape = (len(pr) if pg is None else max(int(n_pro_groups), 0), len(an) if ag is None else max(int(n_anc_groups), 0))
    out = np.empty(shape, np.float64, order="F" if col_major else "C")
    dv = np.ascontiguousarray([device] if devices is None else devices, np.int32)
    st = GcStats()
    check(lib().genlib_gc_groups(len(father), ptr(father), ptr(mother), len(pr), ptr(pr), ptr(pg), int(n_pro_groups),
                                 len(an), ptr(an), ptr(ag), int(n_anc_groups), ptr(out), int(col_major), len(dv),
                                 ptr(dv), C.byref(st)))
    stats = st.as_dict()
    stats["direction"] = _lib.GC_DIRECTIONS[stats["direction"]]
    return out, stats


OCC_TYPES = {"IND": 0, "TOTAL": 1}


def _occ_type(typeOcc) -> int:
    if typeOcc not in OCC_TYPES:
        raise ValueError(f"typeOcc must be \"IND\" or \"TOTAL\", not {typeOcc!r}")
    return OCC_TYPES[typeOcc]


def _named_overflow(pedigree: Pedigree, pro_ids, anc_ids, e):
    """The library's overflow error with the pair it names given as IDs."""
    i, j = e.ancestor_index, e.proband_index
    if i is None or j is None or j < 0:
        return e
    err = _lib.GenlibOverflowError(e.status, f"gen.occ: the number of descent paths from ancestor {int(anc_ids[i])} "
                                   f"to proband {int(pro_ids[j])} does not fit an Int64 ({e})")
    err.ancestor_index, err.proband_index = i, j
    return err


def occ(pedigree: Pedigree, pro=None, ancestors=None, typeOcc: str = "IND", *, device: int = -1, devices=None,
        return_stats: bool = False):
    """gen.occ(pedigree; pro = pro(pedigree), ancestors = founder(pedigree), typeOcc = "IND") on the B200
    engine: O[a, p] = the number of descent paths from ancestor a to proband p (1 for a == p itself), a
    len(ancestors) x len(pro) Int64 matrix in list order, duplicates kept -- ROWS ARE ANCESTORS.
    typeOcc = "TOTAL" returns the len(ancestors) x 1 row sums, reduced on the device.  ValueError on another
    typeOcc, KeyError on an unknown ID, an OverflowError (also a GenlibError) naming the first
    (ancestor, proband) pair whose count or row sum does not fit an Int64."""
    _occ_type(typeOcc)
    pro_ids = _pedigree.pro(pedigree) if pro is None else np.asarray(pro, np.int64)
    anc_ids = _pedigree.founder(pedigree) if ancestors is None else np.asarray(ancestors, np.int64)
    pr, an = pedigree.rank_of(pro_ids), pedigree.rank_of(anc_ids)
    try:
        res, stats = occ_arrays(pedigree.father, pedigree.mother, pr, an, typeOcc=typeOcc, device=device,
                                devices=devices)
    except _lib.GenlibOverflowError as e:
        raise _named_overflow(pedigree, pro_ids, anc_ids, e) from None
    return (res, stats) if return_stats else res


def occ_arrays(father, mother, proband_ranks, ancestor_ranks, *, typeOcc: str = "IND", device: int = -1,
               devices=None, out: Optional[np.ndarray] = None, col_major: bool = False):
    """One-shot C-ABI call `genlib_occ` on flat rank arrays.  Returns (result, stats): typeOcc = "IND" gives
    the len(ancestors) x len(pro) int64 matrix (col_major=True: Fortran order, a Julia Matrix), "TOTAL" the
    len(ancestors) x 1 int64 row sums."""
    kind = _occ_type(typeOcc)
    father = np.ascontiguousarray(father, np.int32)
    mother = np.ascontiguousarray(mother, np.int32)
    pr = np.ascontiguousarray(proband_ranks, np.int32)
    an = np.ascontiguousarray(ancestor_ranks, np.int32)
    ind = kind == OCC_TYPES["IND"]
    shape = (len(an), len(pr)) if ind else (len(an), 1)
    if out is None:
        out = np.empty(shape, np.int64, order="F" if ind and col_major else "C")
    contiguous = out.flags.f_contiguous if ind and col_major else out.flags.c_contiguous
    if out.shape != shape or not contiguous or out.dtype != np.int64:
        raise ValueError(f"out must be a {'Fortran' if ind and col_major else 'C'}-contiguous {shape} int64 array")
    dv = np.ascontiguousarray([device] if devices is None else devices, np.int32)
    st = GcStats()
    check(lib().genlib_occ(len(father), ptr(father), ptr(mother), len(pr), ptr(pr), len(an), ptr(an), ptr(out),
                           kind, int(col_major), len(dv), ptr(dv), C.byref(st)))
    stats = st.as_dict()
    stats["direction"] = _lib.GC_DIRECTIONS[stats["direction"]]
    return out, stats


def rec(pedigree: Pedigree, pro=None, ancestors=None, *, device: int = -1, devices=None, return_stats: bool = False):
    """gen.rec(pedigree; pro = pro(pedigree), ancestors = founder(pedigree)) on the B200 engine: for every
    ancestor, the number of entries of `pro` that descend from it, the ancestor itself included (duplicates
    counted) -- an Int64 vector in ancestor-list order, reduced on the device."""
    pro_ids = _pedigree.pro(pedigree) if pro is None else np.asarray(pro, np.int64)
    anc_ids = _pedigree.founder(pedigree) if ancestors is None else np.asarray(ancestors, np.int64)
    res, stats = rec_arrays(pedigree.father, pedigree.mother, pedigree.rank_of(pro_ids), pedigree.rank_of(anc_ids),
                            device=device, devices=devices)
    return (res, stats) if return_stats else res


def rec_arrays(father, mother, proband_ranks, ancestor_ranks, *, device: int = -1, devices=None,
               out: Optional[np.ndarray] = None):
    """One-shot C-ABI call `genlib_rec` on flat rank arrays.  Returns (counts, stats)."""
    father = np.ascontiguousarray(father, np.int32)
    mother = np.ascontiguousarray(mother, np.int32)
    pr = np.ascontiguousarray(proband_ranks, np.int32)
    an = np.ascontiguousarray(ancestor_ranks, np.int32)
    if out is None:
        out = np.empty(len(an), np.int64)
    if out.shape != (len(an),) or not out.flags.c_contiguous or out.dtype != np.int64:
        raise ValueError(f"out must be a contiguous ({len(an)},) int64 array")
    dv = np.ascontiguousarray([device] if devices is None else devices, np.int32)
    st = GcStats()
    check(lib().genlib_rec(len(father), ptr(father), ptr(mother), len(pr), ptr(pr), len(an), ptr(an), ptr(out),
                           len(dv), ptr(dv), C.byref(st)))
    stats = st.as_dict()
    stats["direction"] = _lib.GC_DIRECTIONS[stats["direction"]]
    return out, stats


class GenMatrix:
    """gen.GenMatrix (src/identify.jl:129-133), what `findMRCA` returns: `individuals` (the IDs as given),
    `ancestors` (the MRCAs, sorted by ID) and `meioses[i, j]`, the number of meioses on the shortest descent
    path from ancestors[j] down to individuals[i] (Int64)."""

    def __init__(self, individuals, ancestors, meioses):
        self.individuals = np.asarray(individuals, np.int64)
        self.ancestors = np.asarray(ancestors, np.int64)
        self.meioses = np.asarray(meioses, np.int64)
        if self.meioses.shape != (len(self.individuals), len(self.ancestors)):
            raise ValueError("meioses must be len(individuals) x len(ancestors)")

    def __repr__(self) -> str:
        return (f"GenMatrix({len(self.individuals)} individuals x {len(self.ancestors)} ancestors: "
                f"{self.ancestors.tolist()})")


def meioses_arrays(father, mother, proband_ranks, ancestor_ranks, *, device: int = -1, devices=None,
                   out: Optional[np.ndarray] = None, col_major: bool = False):
    """One-shot C-ABI call `genlib_meioses` on flat rank arrays.  Returns (matrix, stats): the
    len(pro) x len(ancestors) int64 minimum meioses from each ancestor down to each proband, -1 where the
    proband does not descend from the ancestor (0 on the diagonal a == p); col_major=True: Fortran order."""
    father = np.ascontiguousarray(father, np.int32)
    mother = np.ascontiguousarray(mother, np.int32)
    pr = np.ascontiguousarray(proband_ranks, np.int32)
    an = np.ascontiguousarray(ancestor_ranks, np.int32)
    shape = (len(pr), len(an))
    if out is None:
        out = np.empty(shape, np.int64, order="F" if col_major else "C")
    contiguous = out.flags.f_contiguous if col_major else out.flags.c_contiguous
    if out.shape != shape or not contiguous or out.dtype != np.int64:
        raise ValueError(f"out must be a {'Fortran' if col_major else 'C'}-contiguous {shape} int64 array")
    dv = np.ascontiguousarray([device] if devices is None else devices, np.int32)
    st = GcStats()
    check(lib().genlib_meioses(len(father), ptr(father), ptr(mother), len(pr), ptr(pr), len(an), ptr(an), ptr(out),
                               int(col_major), len(dv), ptr(dv), C.byref(st)))
    stats = st.as_dict()
    stats["direction"] = _lib.GC_DIRECTIONS[stats["direction"]]
    return out, stats


def mrca_arrays(father, mother, ranks, *, device: int = -1, devices=None):
    """One-shot C-ABI call `genlib_mrca` on flat rank arrays.  Returns (MRCA ranks ascending, stats of the
    device pass that decides who is a common ancestor)."""
    father = np.ascontiguousarray(father, np.int32)
    mother = np.ascontiguousarray(mother, np.int32)
    r = np.ascontiguousarray(ranks, np.int32)
    out = np.empty(max(len(father), 1), np.int32)
    m = C.c_int32(0)
    dv = np.ascontiguousarray([device] if devices is None else devices, np.int32)
    st = GcStats()
    check(lib().genlib_mrca(len(father), ptr(father), ptr(mother), len(r), ptr(r), ptr(out), C.byref(m), len(dv),
                            ptr(dv), C.byref(st)))
    stats = st.as_dict()
    stats["direction"] = _lib.GC_DIRECTIONS[stats["direction"]]
    return out[:m.value].copy(), stats


def findMRCA(pedigree: Pedigree, IDs, *, device: int = -1, devices=None, return_stats: bool = False):
    """gen.findMRCA(pedigree, IDs) (src/identify.jl:153-161) on the B200 engine: the most recent common
    ancestors of IDs and the minimum meioses from each of them to each ID, as a `GenMatrix`.  A common ancestor
    is a proper ancestor of every ID (an individual is not its own ancestor); an MRCA is a common ancestor
    none of whose descendants is common.  `ancestors` are sorted by ID; no common ancestor gives a
    len(IDs) x 0 matrix.  KeyError on an unknown ID.  return_stats: also {"mrca": the common-ancestor pass,
    "meioses": the distance pass}."""
    ids = np.asarray(IDs, np.int64).reshape(-1)
    ranks = pedigree.rank_of(ids)                       # KeyError, like pedigree[ID]
    stats = {}
    if len(ids) == 0:
        res = GenMatrix(ids, np.zeros(0, np.int64), np.zeros((0, 0), np.int64))
        return (res, stats) if return_stats else res
    anc, stats["mrca"] = mrca_arrays(pedigree.father, pedigree.mother, ranks, device=device, devices=devices)
    anc_ids = np.sort(pedigree.ids[anc])
    d, stats["meioses"] = meioses_arrays(pedigree.father, pedigree.mother, ranks, pedigree.rank_of(anc_ids),
                                         device=device, devices=devices)
    res = GenMatrix(ids, anc_ids, d)
    return (res, stats) if return_stats else res


def findDistance(pedigree: Pedigree, IDs, ancestorID, *, device: int = -1) -> int:
    """gen.findDistance(pedigree, IDs, ancestorID) (src/describe.jl:296-300) on the B200 engine: the sum over
    IDs of the minimum meioses from ancestorID down to each of them (for two individuals, the meioses that
    separate them through that ancestor).  An ID equal to ancestorID adds 0.  ValueError naming the first ID
    that does not descend from ancestorID; KeyError on an unknown ID."""
    ids = np.asarray(IDs, np.int64).reshape(-1)
    ranks = pedigree.rank_of(ids)
    anc = pedigree.rank_of([ancestorID])
    if len(ids) == 0:
        return 0
    d, _ = meioses_arrays(pedigree.father, pedigree.mother, ranks, anc, device=device)
    bad = np.flatnonzero(d[:, 0] < 0)
    if len(bad):
        raise ValueError(f"gen.findDistance: {int(ids[bad[0]])} does not descend from {int(ancestorID)}")
    return int(d[:, 0].sum())


def f(pedigree: Pedigree, IDs, *, device: int = -1, devices=None, return_stats: bool = False):
    """gen.f(pedigree, IDs): inbreeding coefficients, Float32 in list order (src/compute.jl:500-511).

    F of an individual is the kinship of its parents, 0 when a parent is missing.  The reference runs the
    exponential pairwise recursion in Float64 per ID and rounds once; here ONE sweep of the engine with Float64
    storage over the IDs' ancestors-or-self, layered by depth below the founders, reads Psi[father, mother] of
    every couple on the device just before the couple's layer (genlib_f), so the cost grows with the pedigree,
    not with the square of the number of IDs: the inbreeding of a whole population is one call.  Exact while
    kinships fit 53 bits (about 26 generations, e.g. genea140); in deeper pedigrees the last Float64 bits follow
    this schedule's order of the sums and may differ from the reference's before the rounding to Float32.
    Duplicates are kept; KeyError on an unknown ID.  `devices=[0, 1, ...]` shards the frontier over several
    GPUs of the box, with the same result.  SURVEY.md 8(f) N3."""
    IDs = np.asarray(IDs, np.int64).reshape(-1)
    ranks = pedigree.rank_of(IDs)                       # KeyError, like pedigree[ID]
    res, stats = f_arrays(pedigree.father, pedigree.mother, ranks, device=device, devices=devices)
    return (res, stats) if return_stats else res


def f_arrays(father, mother, ranks, *, dtype=np.float32, device: int = -1, devices=None,
             out: Optional[np.ndarray] = None):
    """One-shot C-ABI call `genlib_f` on flat rank arrays (what the Julia shim ccalls).  Returns
    (coefficients in list order as float32 or float64, stats)."""
    father = np.ascontiguousarray(father, np.int32)
    mother = np.ascontiguousarray(mother, np.int32)
    r = np.ascontiguousarray(ranks, np.int32)
    if out is None:
        out = np.empty(len(r), dtype)
    if out.shape != (len(r),) or not out.flags.c_contiguous or out.dtype not in _lib.DTYPES:
        raise ValueError(f"out must be a contiguous ({len(r)},) float32/float64 array")
    dv = np.ascontiguousarray([device] if devices is None else devices, np.int32)
    st = Stats()
    check(lib().genlib_f(len(father), ptr(father), ptr(mother), len(r), ptr(r), ptr(out),
                         _lib.DTYPES[np.dtype(out.dtype)], len(dv), ptr(dv), C.byref(st)))
    return out, st.as_dict()


def phi_pairs(pedigree: Pedigree, IDs1, IDs2, *, dtype=np.float64, device: int = -1, devices=None,
              return_stats: bool = False):
    """The kinship of each pair (IDs1[k], IDs2[k]), in list order (duplicates and reversed pairs kept): what the
    reference's scalar phi(ind1, ind2) (src/compute.jl:66-95) gives one pair at a time, for a whole list.

    ONE sweep of the engine with Float64 storage over the ancestors-or-self of everybody named, layered by depth
    below the founders, reads each pair on the device in the layer after its later-born member's (genlib_phi_pairs);
    no matrix is formed.  phi(a, b) == phi(b, a) bitwise, phi(a, a) = 1/2 + 1/2 F_a, unrelated pairs give 0.  Exact
    while kinships fit 53 bits; deeper pedigrees follow this schedule's order of the sums, like gen.f.  Both rows of
    a pair stay on the device until it is read: pairs of members born many generations apart widen the frontier
    (MemoryError when it does not fit).  ValueError on lists of unequal length, KeyError on an unknown ID.
    `devices=[0, 1, ...]` shards the frontier over several GPUs of the box, with the same result."""
    a = np.asarray(IDs1, np.int64).reshape(-1)
    b = np.asarray(IDs2, np.int64).reshape(-1)
    if len(a) != len(b):
        raise ValueError(f"gen.phi_pairs: {len(a)} IDs against {len(b)}")
    ra, rb = pedigree.rank_of(a), pedigree.rank_of(b)   # KeyError, like pedigree[ID]
    res, stats = phi_pairs_arrays(pedigree.father, pedigree.mother, ra, rb, dtype=dtype, device=device, devices=devices)
    return (res, stats) if return_stats else res


def phi_pairs_arrays(father, mother, a, b, *, dtype=np.float64, device: int = -1, devices=None,
                     out: Optional[np.ndarray] = None):
    """One-shot C-ABI call `genlib_phi_pairs` on flat rank arrays (what the Julia shim ccalls).  Returns
    (kinships in list order as float64 or float32, stats)."""
    father = np.ascontiguousarray(father, np.int32)
    mother = np.ascontiguousarray(mother, np.int32)
    a, b = np.ascontiguousarray(a, np.int32).reshape(-1), np.ascontiguousarray(b, np.int32).reshape(-1)
    if len(a) != len(b):
        raise ValueError(f"phi_pairs_arrays: {len(a)} ranks against {len(b)}")
    if out is None:
        out = np.empty(len(a), dtype)
    if out.shape != (len(a),) or not out.flags.c_contiguous or out.dtype not in _lib.DTYPES:
        raise ValueError(f"out must be a contiguous ({len(a)},) float32/float64 array")
    dv = np.ascontiguousarray([device] if devices is None else devices, np.int32)
    st = Stats()
    check(lib().genlib_phi_pairs(len(father), ptr(father), ptr(mother), len(a), ptr(a), ptr(b), ptr(out),
                                 _lib.DTYPES[np.dtype(out.dtype)], len(dv), ptr(dv), C.byref(st)))
    return out, st.as_dict()


class KinshipMatrix:
    """gen.KinshipMatrix (src/compute.jl:31-46): what `sparse_phi` returns, indexed by ID.

    `k[ID1, ID2]` is the reference's getindex (:36-40): the entry filed under phi[lower rank][higher
    rank], 0 when there is none.  The reference files a kinship under phi[earlier processed][later
    processed] (:393); where sparse_phi's queue order inverts the rank order of two individuals of one
    depth the value is never found again, reads as 0 here as there, and is missing from everything
    computed from it.  `stored` counts the entries a look-up can find (the diagonal and the non-zero
    lower->higher pairs); the reference's `show` line (:42-46) also counts misfiled and orphaned keys,
    which no look-up ever reads -- they coincide when the queue order follows the ranks (e.g. the
    reference's own test, test/runtests.jl:56)."""

    def __init__(self, ids: np.ndarray, ranks: np.ndarray, dense: np.ndarray):
        """`dense`: the symmetric matrix in the order of `ids`.  Kept are the entries the reference's Dict of Dicts
        holds where a look-up finds them (:391-394, zeros are never stored): per individual, in rank order, the
        diagonal and the non-zero kinships with higher-ranked individuals -- compressed sparse rows."""
        order = np.argsort(ranks, kind="stable")
        self._ids = np.asarray(ids)[order]
        self._pos = {int(i): k for k, i in enumerate(self._ids)}
        dense = np.asarray(dense, np.float32)
        n = len(order)
        indptr = np.zeros(n + 1, np.int64)
        cols, vals = [], []
        for k in range(n):
            row = dense[order[k]][order[k:]]                 # (k, j) for j >= k, in rank order
            nz = np.flatnonzero(row != 0)
            if len(nz) == 0 or nz[0] != 0:
                nz = np.concatenate(([0], nz))               # the diagonal is always there (:398)
            cols.append(nz + k)
            vals.append(row[nz])
            indptr[k + 1] = indptr[k] + len(nz)
        self._indptr = indptr
        self._indices = np.concatenate(cols).astype(np.int64) if n else np.zeros(0, np.int64)
        self._data = np.concatenate(vals).astype(np.float32) if n else np.zeros(0, np.float32)

    def _row(self, k: int):
        a, b = self._indptr[k], self._indptr[k + 1]
        return self._indices[a:b], self._data[a:b]

    def __getitem__(self, key) -> np.float32:
        a, b = key
        ka, kb = self._pos[int(a)], self._pos[int(b)]        # KeyError on an unknown ID, like the Dict
        lo, hi = (ka, kb) if ka < kb else (kb, ka)           # phi[lower rank][higher rank] (:36-40)
        cols, vals = self._row(lo)
        p = int(np.searchsorted(cols, hi))
        return vals[p] if p < len(cols) and cols[p] == hi else np.float32(0)

    @property
    def stored(self) -> int:
        return len(self._data)

    def to_dense(self) -> np.ndarray:
        """The symmetric Float32 matrix in rank order (zeros where nothing is stored)."""
        n = len(self._ids)
        d = np.zeros((n, n), np.float32)
        rows = np.repeat(np.arange(n), np.diff(self._indptr))
        d[rows, self._indices] = self._data
        d[self._indices, rows] = self._data
        return d

    _dense = property(to_dense)

    def to_dict(self) -> dict:
        """{lower-ranked ID: {higher-ranked ID: kinship}}: the entries of `KinshipMatrix.dict` a look-up finds."""
        out = {}
        for k, i in enumerate(self._ids):
            cols, vals = self._row(k)
            out[int(i)] = {int(self._ids[j]): v for j, v in zip(cols, vals)}
        return out

    def __len__(self) -> int:
        return len(self._ids)

    def __repr__(self) -> str:                                            # src/compute.jl:42-46
        return f"{len(self)}\u00d7{len(self)} KinshipMatrix with {self.stored} stored entries."


def sparse_phi(pedigree: Pedigree, probandIDs=None, *, device: int = -1, symmetric: bool = False) -> KinshipMatrix:
    """gen.sparse_phi(pedigree, probandIDs = pro(pedigree)) (src/compute.jl:321-447) on the GPU.

    Same engine, planned for sparse_phi's own floating-point schedule: founders in ID order
    (identify.jl:15-19), then its queue; the later-processed individual of a pair is climbed; every
    stored kinship is a Float32 and is halved in Float32; kinships the reference misfiles (see
    KinshipMatrix) read as 0.  Look-ups are bit-identical to the reference's KinshipMatrix.
    symmetric=True keeps the misfiled kinships instead (the consistent variant of the schedule).
    SURVEY.md 8(f) N2."""
    ids = pro(pedigree) if probandIDs is None else np.asarray(probandIDs, np.int64)
    ranks = pedigree.rank_of(ids)                                         # KeyError on an unknown ID
    _, first = np.unique(ranks, return_index=True)                        # duplicates collapse (Dict keys)
    first.sort()
    plan = Plan(pedigree.father, pedigree.mother, ranks, ids=pedigree.ids,
                schedule="sparse_phi_symmetric" if symmetric else "sparse_phi")
    n = plan.n_unique
    if n == 0:
        return KinshipMatrix(np.zeros(0, np.int64), np.zeros(0, np.int32), np.zeros((0, 0), np.float32))
    eng = Engine(plan, "reference", device)
    try:
        eng.run()
        dense = eng.fetch()
    finally:
        eng.close()
    return KinshipMatrix(np.asarray(ids)[first], ranks[first], dense)


def _julia_sum_f32(a: np.ndarray) -> np.float32:
    """Base.sum of a Float32 array as Julia's mapreduce does it: pairwise halving down to blocks of
    1024 elements (Base.pairwise_blocksize), the block summed left to right.  (Julia's block loop is
    `@simd`, so the reference's last bits depend on the machine's vector width; this is the scalar order.)"""
    a = np.ascontiguousarray(a, np.float32).ravel()

    def rec(lo: int, hi: int) -> np.float32:
        if hi - lo <= 1024:
            acc = np.float32(0) if hi == lo else a[lo]
            for x in a[lo + 1:hi]:
                acc = np.float32(acc + x)
            return acc
        mid = (lo + hi) >> 1
        return np.float32(rec(lo, mid) + rec(mid, hi))

    return rec(0, len(a))


def phiMean(phi_matrix) -> np.float32:
    """gen.phiMean(::Matrix{Float32}) (src/compute.jl:454-459) and gen.phiMean(::KinshipMatrix)
    (:466-472), host side.  Matrix: `sum(phi)` (Float32, Julia's pairwise order over the column-major
    buffer -- the matrix is symmetric, so that is this buffer), minus the diagonal summed left to right,
    divided by n^2 - n in Float32.  KinshipMatrix: the reference adds the stored entries in Dict
    iteration order; here the entries a look-up can find are added in rank order -- the same number
    whenever the Float32 sum is exact, e.g. the reference's own test, test/runtests.jl:55."""
    if isinstance(phi_matrix, KinshipMatrix):
        k, n = phi_matrix, len(phi_matrix)
        total, diag = np.float32(0), np.float32(0)
        for r in range(n):                                   # sum(values(kinships)) per individual (:467), then their sum
            vals = k._row(r)[1]
            total = np.float32(total + vals.sum(dtype=np.float32))
            diag = np.float32(diag + vals[0])                # the diagonal leads its row
        total = np.float32(total - diag)
        return np.float32(total / (n * (n - 1) / 2))
    m = np.asarray(phi_matrix, np.float32)
    big = m.size > (1 << 22)                                        # the scalar emulation is slow: NumPy's pairwise sum
    total = m.sum(dtype=np.float32) if big else _julia_sum_f32(m)
    diag = np.float32(0)
    for x in np.diag(m):
        diag = np.float32(diag + x)
    total = np.float32(total - diag)
    return np.float32(total / np.float32(m.size - m.shape[0]))
