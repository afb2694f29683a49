"""genlib.jl_b200 -- B200-native kinship engine behind GenLib.jl's `gen.phi` (and `gen.gc`).

Usage mirrors the reference (`import GenLib as gen`):
    import genlib_b200 as gen
    ped = gen.genealogy(gen.genea140)
    phi = gen.phi(ped)                     # float32, probands in gen.pro(ped) order
    g = gen.gc(ped)                        # float64, gen.pro(ped) x gen.founder(ped)
"""
import os as _os

from .pedigree import Individual, Pedigree, founder, genealogy, pro  # noqa: F401
from .engine import (Engine, GcPlan, KinshipMatrix, PinnedMatrix, Plan, f, gc, gc_arrays, phi, phi_arrays,  # noqa: F401
                     phi_distributed, phiMean, run_distributed, sparse_phi)
from . import synth  # noqa: F401
from ._lib import GenlibError, LIB_PATH, PlanBoundsExceeded, lib  # noqa: F401

_DATA = _os.path.join(_os.path.dirname(_os.path.dirname(_os.path.abspath(__file__))), "tests", "data")
genea140 = _os.path.join(_DATA, "genea140.csv")   # src/GenLib.jl:27
geneaJi = _os.path.join(_DATA, "geneaJi.csv")     # src/GenLib.jl:43
