"""Deterministic synthetic pedigrees of the shapes BASELINE.json names (SURVEY.md 8d).

The generator is workload infrastructure (benchmarks, parity tests); it is not
part of the reference.  It emits the reference's own file format
(`ind<TAB>father<TAB>mother<TAB>sex` with a header, src/create.jl:161-189), so
the same pedigrees can be fed to GenLib.jl elsewhere.

Model: IDs 1..N generation-major, generation 0 = founders, sex alternates with
the ID (odd = 1 male, even = 2 female).  For every later generation the
parental pool is the previous `overlap` generations; inside each deme males and
females are shuffled and paired without replacement (monogamous couples); with
probability `alpha` a family that has both a son and a daughter in the pool
contributes a full-sib couple first (controlled inbreeding).  Every child picks
a couple uniformly, inherits the couple's deme, and migrates to a random deme
with probability `migration`.  Probands are `n_probands` individuals of the last
generation sampled without replacement, sorted by ID.  All randomness comes
from one splitmix64 counter stream, so the output is a pure function of the
arguments.
"""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np

_GOLDEN = np.uint64(0x9E3779B97F4A7C15)


class SplitMix64:
    def __init__(self, seed: int):
        self.state = np.uint64(seed & 0xFFFFFFFFFFFFFFFF)

    def next(self, n: int) -> np.ndarray:
        with np.errstate(over="ignore"):
            z = self.state + (np.arange(1, n + 1, dtype=np.uint64) * _GOLDEN)
            self.state = self.state + np.uint64(n) * _GOLDEN
            z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
            z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
            return z ^ (z >> np.uint64(31))

    def uniform(self, n: int) -> np.ndarray:
        return (self.next(n) >> np.uint64(11)).astype(np.float64) * (1.0 / 9007199254740992.0)

    def below(self, n: int, m: int) -> np.ndarray:
        return np.minimum((self.uniform(n) * m).astype(np.int64), m - 1)

    def permutation(self, n: int) -> np.ndarray:
        return np.argsort(self.next(n), kind="stable")


@dataclass
class SyntheticPedigree:
    ind: np.ndarray
    father: np.ndarray      # IDs, 0 = unknown
    mother: np.ndarray
    sex: np.ndarray
    probands: np.ndarray    # IDs, sorted
    generation: np.ndarray
    params: dict
    deme: np.ndarray        # per individual, in [0, demes): a natural grouping for gen.phiMeanGroups

    def to_csv(self, path: str):
        with open(path, "w") as fh:
            fh.write("ind\tfather\tmother\tsex\n")
            np.savetxt(fh, np.stack([self.ind, self.father, self.mother, self.sex], 1), fmt="%d", delimiter="\t")

    def as_columns(self) -> dict:
        return {"ind": self.ind, "father": self.father, "mother": self.mother, "sex": self.sex}


def generate(n_individuals: int, generations: int, n_probands: int, alpha: float = 0.0,
             demes: int = 1, migration: float = 0.0, overlap: int = 1, seed: int = 20261018
             ) -> SyntheticPedigree:
    N, G = int(n_individuals), int(generations)
    assert G >= 1 and N >= G
    rng = SplitMix64(seed)
    sizes = np.full(G, N // G, np.int64)
    sizes[: N % G] += 1
    starts = np.concatenate([[0], np.cumsum(sizes)])
    ind = np.arange(1, N + 1, dtype=np.int64)
    sex = np.where(ind % 2 == 1, 1, 2).astype(np.int32)
    father = np.zeros(N, np.int64)
    mother = np.zeros(N, np.int64)
    gen = np.repeat(np.arange(G), sizes).astype(np.int32)
    deme = np.zeros(N, np.int64)
    deme[: sizes[0]] = (np.arange(sizes[0]) // 2) % demes   # pairs (male, female) share a deme
    family = np.full(N, -1, np.int64)      # id of the parental couple (for sib matings)
    next_family = 0
    for g in range(1, G):
        lo, hi = starts[max(0, g - overlap)], starts[g]
        pool = np.arange(lo, hi)
        pool = pool[rng.permutation(len(pool))]
        used = np.zeros(N, bool)
        hus, wif = [], []
        if alpha > 0:
            # full-sib couples: families with a son and a daughter in the pool
            fam = family[pool]
            ok = fam >= 0
            pm, pf = pool[ok & (sex[pool] == 1)], pool[ok & (sex[pool] == 2)]
            um, im = np.unique(family[pm], return_index=True)
            uf, i_f = np.unique(family[pf], return_index=True)
            common, am, af = np.intersect1d(um, uf, return_indices=True)
            pick = rng.uniform(len(common)) < alpha
            h, w = pm[im[am[pick]]], pf[i_f[af[pick]]]
            same = deme[h] == deme[w]
            h, w = h[same], w[same]
            used[h] = True
            used[w] = True
            hus.append(h)
            wif.append(w)
        rest = pool[~used[pool]]
        for d in range(demes):
            sel = rest[deme[rest] == d] if demes > 1 else rest
            m_, f_ = sel[sex[sel] == 1], sel[sex[sel] == 2]
            k = min(len(m_), len(f_))
            hus.append(m_[:k])
            wif.append(f_[:k])
        hus, wif = np.concatenate(hus), np.concatenate(wif)
        if len(hus) == 0:
            raise ValueError(f"generation {g}: no couple could be formed")
        n = int(sizes[g])
        c = rng.below(n, len(hus))
        kids = np.arange(starts[g], starts[g + 1])
        father[kids] = ind[hus[c]]
        mother[kids] = ind[wif[c]]
        family[kids] = next_family + c
        next_family += len(hus)
        deme[kids] = deme[hus[c]]
        if demes > 1 and migration > 0:
            mig = rng.uniform(n) < migration
            dest = rng.below(n, demes)
            deme[kids] = np.where(mig, dest, deme[kids])
    last = np.arange(starts[G - 1], starts[G])
    P = min(int(n_probands), len(last))
    probands = np.sort(ind[last[rng.permutation(len(last))[:P]]])
    params = dict(n_individuals=N, generations=G, n_probands=P, alpha=alpha, demes=demes,
                  migration=migration, overlap=overlap, seed=seed)
    return SyntheticPedigree(ind, father, mother, sex, probands, gen, params, deme)


# The shapes BASELINE.json's configs name (SURVEY.md 8d table).
CONFIGS = {
    "C3": dict(n_individuals=1_000_000, generations=20, n_probands=10_000, alpha=0.01, demes=20,
               migration=0.02, overlap=1, seed=20261018),
    "C4": dict(n_individuals=5_000_000, generations=30, n_probands=100_000, alpha=0.001, demes=1,
               migration=0.0, overlap=1, seed=20261018),
    "C5": dict(n_individuals=1_000_000, generations=200, n_probands=5_000, alpha=0.10, demes=1,
               migration=0.0, overlap=3, seed=20261018),
}


def config(name: str, scale: float = 1.0) -> SyntheticPedigree:
    """A named configuration; `scale` < 1 shrinks individuals and probands alike
    (generations, rates and structure are kept)."""
    p = dict(CONFIGS[name])
    if scale != 1.0:
        p["n_individuals"] = max(p["generations"] * 4, int(round(p["n_individuals"] * scale)))
        p["n_probands"] = max(2, int(round(p["n_probands"] * scale)))
    return generate(**p)
