"""Plan / Engine handles over the C ABI and the `gen.phi` front end.

`phi` keeps the reference's signature and behaviour (src/compute.jl:233-304):
    phi(pedigree, probandIDs = pro(pedigree); verbose = false, compute = true)
returns a symmetric Float32 matrix in probandIDs order (duplicates collapsed),
`None` when compute is false, raises KeyError for an unknown ID.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional

import numpy as np

from . import _lib
from . import pedigree as _pedigree
from ._lib import GcStats, LayerInfo, PlanBoundsExceeded, Stats, check, lib, ptr
from .pedigree import Pedigree, pro


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
    the frontier over several GPUs of the box from this one process (genlib_phi_multi)."""
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


class GcPlan:
    """The schedule of gen.gc (genlib_gc_plan_*): direction, layers, frontier slots.  Needs no GPU."""

    def __init__(self, father, mother, proband_ranks, ancestor_ranks):
        self.father = np.ascontiguousarray(father, np.int32)
        self.mother = np.ascontiguousarray(mother, np.int32)
        self.probands = np.ascontiguousarray(proband_ranks, np.int32)
        self.ancestors = np.ascontiguousarray(ancestor_ranks, np.int32)
        if len(self.father) != len(self.mother):
            raise ValueError("father and mother must have the same length")
        h = C.c_void_p()
        check(lib().genlib_gc_plan_create(len(self.father), ptr(self.father), ptr(self.mother), len(self.probands),
                                          ptr(self.probands), len(self.ancestors), ptr(self.ancestors), C.byref(h)))
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


def f(pedigree: Pedigree, IDs, *, device: int = -1) -> np.ndarray:
    """gen.f(pedigree, IDs): inbreeding coefficients, Float32 (src/compute.jl:500-511).

    The reference evaluates phi(father, mother) by the exponential pairwise recursion in Float64
    and rounds once; here the parents of all requested individuals go through ONE sweep of the
    engine with Float64 storage (exact while kinships fit 53 bits, i.e. up to ~26 generations)
    and the result is rounded to Float32.  SURVEY.md 8(f) N3."""
    IDs = np.asarray(IDs, np.int64)
    ranks = pedigree.rank_of(IDs)
    fa, mo = pedigree.father[ranks], pedigree.mother[ranks]
    both = (fa >= 0) & (mo >= 0)
    out = np.zeros(len(IDs), np.float32)
    if both.any():
        parents = np.unique(np.concatenate([fa[both], mo[both]]))
        k = phi(pedigree, pedigree.ids[parents], numerics="fp64", dtype=np.float64, device=device)
        pos = {int(r): i for i, r in enumerate(parents)}
        idx = np.nonzero(both)[0]
        out[idx] = [np.float32(k[pos[int(fa[i])], pos[int(mo[i])]]) for i in idx]
    return out


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
