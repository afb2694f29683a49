"""genlib.jl_b200 -- B200-native kinship engine behind GenLib.jl's `gen.phi` (and `gen.gc`, `gen.occ`, `gen.rec`, `gen.findMRCA`).

Usage mirrors the reference (`import GenLib as gen`):
    import genlib_b200 as gen
    ped = gen.genealogy(gen.genea140)
    phi = gen.phi(ped)                     # float32, probands in gen.pro(ped) order
    g = gen.gc(ped)                        # float64, gen.pro(ped) x gen.founder(ped)
    o = gen.occ(ped)                       # int64 path counts, gen.founder(ped) x gen.pro(ped)
    r = gen.rec(ped)                       # int64, probands descending from each founder
    m = gen.findMRCA(ped, [1, 2])          # GenMatrix: MRCAs sorted by ID, int64 meioses
    F = gen.f(ped, ped.ids)                # float32 inbreeding of everyone, one device sweep
    k = gen.phi_pairs(ped, [1, 2], [29, 2])  # float64 kinship of each pair, list order, no matrix formed
    o = gen.phiOver(ped, 1 / 64)           # proband pairs at or above 1/64, selected on the device
    g = gen.phiMeanGroups(ped, {1: "a", 2: "a", 29: "b"})  # mean kinship within / between groups, and per proband
    c = gen.gcGroups(ped, {1: "a", 2: "a", 29: "b"})       # gen.gc summed over proband groups, no matrix formed
    y = gen.phiProduct(ped, x)             # the proband kinship matrix times x (P, or P x k), no matrix fetched
"""
import os as _os

from .pedigree import Individual, Pedigree, founder, genealogy, pro  # noqa: F401
from .engine import (Engine, GcPlan, GenMatrix, GroupKinship, KinshipMatrix, PinnedMatrix, Plan, f, f_arrays,  # noqa: F401
                     findDistance, findMRCA, gc, gc_arrays, gc_groups_arrays, gcGroups, GroupContribution, meioses_arrays, mrca_arrays, occ, occ_arrays, phi, phi_arrays,
                     phi_distributed, phi_groups_arrays, phi_over_arrays, phi_pairs, phi_pairs_arrays, phiMean,
                     phiMeanGroups, phiOver, phi_product_arrays, phiProduct, PhiOver, rec, rec_arrays, run_distributed,
                     sparse_phi)
from . import synth  # noqa: F401
from ._lib import GenlibError, GenlibOverflowError, LIB_PATH, PlanBoundsExceeded, lib  # noqa: F401

_DATA = _os.path.join(_os.path.dirname(_os.path.dirname(_os.path.abspath(__file__))), "tests", "data")
genea140 = _os.path.join(_DATA, "genea140.csv")   # src/GenLib.jl:27
geneaJi = _os.path.join(_DATA, "geneaJi.csv")     # src/GenLib.jl:43
