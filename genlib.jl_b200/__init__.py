"""genlib.jl_b200 -- B200-native kinship engine behind GenLib.jl's `gen.phi` (and `gen.gc`, `gen.occ`, `gen.rec`).

Usage mirrors the reference (`import GenLib as gen`):
    import genlib_b200 as gen
    ped = gen.genealogy(gen.genea140)
    phi = gen.phi(ped)                     # float32, probands in gen.pro(ped) order
    g = gen.gc(ped)                        # float64, gen.pro(ped) x gen.founder(ped)
    o = gen.occ(ped)                       # int64 path counts, gen.founder(ped) x gen.pro(ped)
    r = gen.rec(ped)                       # int64, probands descending from each founder
"""
import os as _os

from .pedigree import Individual, Pedigree, founder, genealogy, pro  # noqa: F401
from .engine import (Engine, GcPlan, KinshipMatrix, PinnedMatrix, Plan, f, gc, gc_arrays, occ, occ_arrays,  # noqa: F401
                     phi, phi_arrays, phi_distributed, phiMean, rec, rec_arrays, run_distributed, sparse_phi)
from . import synth  # noqa: F401
from ._lib import GenlibError, GenlibOverflowError, LIB_PATH, PlanBoundsExceeded, lib  # noqa: F401

_DATA = _os.path.join(_os.path.dirname(_os.path.dirname(_os.path.abspath(__file__))), "tests", "data")
genea140 = _os.path.join(_DATA, "genea140.csv")   # src/GenLib.jl:27
geneaJi = _os.path.join(_DATA, "geneaJi.csv")     # src/GenLib.jl:43
