"""gen.f for whole pedigrees: the GENLIB_SCHEDULE_F plan (members = the IDs' ancestors-or-self, layers by depth
below the founders, no row kept to the end) and the device read of Psi[father, mother] in each couple's layer."""
from fractions import Fraction

import numpy as np
import pytest

from plan_replay import replay
from util import exact_kinship, ladder_pedigree, random_pedigree


def _sibship():
    n = 3002 + 1000                                  # a 1000-child sibship and 3000 unrelated founders
    father = np.full(n, -1, np.int32)
    mother = np.full(n, -1, np.int32)
    father[3002:] = 0
    mother[3002:] = 1
    return father, mother, np.arange(n, dtype=np.int32)


def make_case(gen, name):
    """(father, mother, listed ranks): every individual, unless the name says otherwise."""
    if name in ("geneaJi", "genea140"):
        ped = gen.genealogy(getattr(gen, name))
    elif name.startswith("random"):                 # single parents, overlapping generations, permuted IDs
        seed = int(name[6:])
        rng = np.random.default_rng(seed)
        ped = gen.genealogy(random_pedigree(rng, (600, 1200, 900)[seed % 3], (20, 40, 8)[seed % 3], p_single=0.15,
                                            p_none=0.03, window=(0, 40, 120)[seed % 3]))
    elif name == "ladder":
        cols, _ = ladder_pedigree(80)
        ped = gen.genealogy(cols)
    elif name == "sibship":
        return _sibship()
    elif name.startswith(("C3x", "C5x")):
        ped = gen.genealogy(gen.synth.config(name[:2], float(name[3:])).as_columns())
    else:
        raise KeyError(name)
    return ped.father, ped.mother, np.arange(len(ped.father), dtype=np.int32)


def members_and_depth(father, mother, ranks):
    """The ancestors-or-self of the listed individuals with both parents, and every individual's depth below the
    founders of that set."""
    n = len(father)
    member = np.zeros(n, bool)
    r = np.asarray(ranks)
    member[r[(father[r] >= 0) & (mother[r] >= 0)]] = True
    for x in range(n - 1, -1, -1):
        if member[x]:
            for p in (father[x], mother[x]):
                if p >= 0:
                    member[p] = True
    depth = np.zeros(n, np.int64)
    for x in np.nonzero(member)[0]:
        d = [depth[p] + 1 for p in (father[x], mother[x]) if p >= 0]
        depth[x] = max(d) if d else 0
    return member, depth


def f_plan(gen, father, mother, ranks, world=1, stream=False):
    return gen.Plan(father, mother, ranks, world=world, schedule="f", stream=stream)


class _NoProbandMatrix:
    """A gen.f plan as the replay sees it: it keeps no proband to the end, so there is no matrix to extract."""

    def __init__(self, plan):
        self._plan = plan

    def __getattr__(self, name):
        return getattr(self._plan, name)

    def proband_slots(self):
        return np.zeros(0, np.int32)


def replay_f(plan, father, mother, ranks):
    """F of every listed rank from the Float64 replay of the plan: Psi[father slot, mother slot] per couple."""
    got = {}

    def on_layer(t, A, live):
        a = plan.layer_arrays(t)
        pf, pm = a["fam_father_slot"][a["member_fam"]], a["fam_mother_slot"][a["member_fam"]]
        both = (pf >= 0) & (pm >= 0)
        for x, v in zip(a["member_ind"][both], A[pf[both], pm[both]]):
            got[int(x)] = v

    replay(_NoProbandMatrix(plan), "fp64", on_layer=on_layer)
    return np.array([got[int(r)] if father[r] >= 0 and mother[r] >= 0 else 0.0 for r in ranks], np.float64)


def assert_exact(got, father, mother, ranks):
    """Exact rationals; equal wherever the value fits 53 bits, within 2^-50 relative elsewhere."""
    phi = exact_kinship(father, mother)
    for v, r in zip(got, ranks):
        want = phi(int(father[r]), int(mother[r])) if father[r] >= 0 and mother[r] >= 0 else Fraction(0)
        if Fraction(float(want)) == want:
            assert Fraction(float(v)) == want, (r, v, want)
        else:
            assert abs(Fraction(float(v)) - want) <= want * Fraction(1, 2 ** 50), (r, v, want)


# ---- the plan, on the CPU -------------------------------------------------------------------------------------

SHAPE_CASES = ["geneaJi", "genea140", "random0", "random1", "random2", "sibship", "ladder"]


@pytest.mark.parametrize("case", SHAPE_CASES)
def test_plan_shape(gen, case, monkeypatch):
    """Every member is born in the layer of its depth below the founders; a couple's parents are both live in its
    layer; a row is live exactly from the layer after its birth to the layer of its last child (a childless row is
    never live again); nothing is live after the last layer; the plan passes the planner's own checks."""
    monkeypatch.setenv("GENLIB_PLAN_VERIFY", "1")
    father, mother, ranks = make_case(gen, case)
    if case == "geneaJi":                            # also: duplicates and individuals with a missing parent
        ranks = np.concatenate([ranks, ranks[::3]])
    member, depth = members_and_depth(father, mother, ranks)
    plan = f_plan(gen, father, mother, ranks)
    listed = np.unique(ranks[(father[ranks] >= 0) & (mother[ranks] >= 0)])
    assert plan.n_unique == len(listed) and plan.n_layers == depth[member].max() + 1
    assert plan.row_updates == member.sum()
    last_child = np.full(len(father), -1)
    for x in np.nonzero(member)[0]:
        for p in (father[x], mother[x]):
            if p >= 0:
                last_child[p] = max(last_child[p], depth[x])
    born = np.zeros(len(father), bool)
    occupant = {}
    for t in range(plan.n_layers):
        a, info = plan.layer_arrays(t), plan.layer_info(t)
        ind = a["member_ind"]
        assert np.array_equal(a["member_rank"], ind)                     # phi's arithmetic: mem_ind is the rank
        assert (depth[ind] == t).all() and member[ind].all() and not born[ind].any()
        live = np.nonzero(a["live_flags"] & 1)[0]
        who = np.array(sorted(occupant[s] for s in live), np.int64)
        want = np.nonzero(born & (last_child >= t))[0]
        assert np.array_equal(who, want), f"layer {t}: live rows"
        carried = np.array(sorted(occupant[s] for s in np.nonzero(a["live_flags"] & 2)[0]), np.int64)
        assert np.array_equal(carried, np.nonzero(born & (last_child > t))[0])
        assert info["live_before"] == len(live)
        pf, pm = a["fam_father_slot"], a["fam_mother_slot"]
        for s in np.concatenate([pf[pf >= 0], pm[pm >= 0]]):
            assert a["live_flags"][s] & 1, f"layer {t}: a parent is not live"
        assert not np.intersect1d(a["member_slot"], live).size
        for s, x in zip(a["member_slot"], ind):
            occupant[int(s)] = int(x)
        born[ind] = True
        if t == plan.n_layers - 1:
            assert not (a["live_flags"] & 2).any(), "a row is live after the last layer"
    assert np.array_equal(born, member)


@pytest.mark.parametrize("case", SHAPE_CASES)
def test_streamed_plan_equals_the_plan_made_in_one_piece(gen, case, monkeypatch):
    """The plan published layer by layer (what genlib_f runs while it plans) is the plan made in one piece, also
    when a bound does not hold and the planner finishes with exact sizes."""
    father, mother, ranks = make_case(gen, case)
    for world in (1, 2):
        whole = f_plan(gen, father, mother, ranks, world)
        ref = gen.lib().genlib_plan_digest(whole._h, 0)
        for slack in (None, "-1"):
            if slack is None:
                monkeypatch.delenv("GENLIB_STREAM_SLACK_PCT", raising=False)
            else:
                monkeypatch.setenv("GENLIB_STREAM_SLACK_PCT", slack)
            p = f_plan(gen, father, mother, ranks, world, stream=True)
            assert gen.lib().genlib_plan_digest(p._h, 0) == ref, (world, slack)
    monkeypatch.delenv("GENLIB_STREAM_SLACK_PCT", raising=False)


@pytest.mark.parametrize("case", SHAPE_CASES)
def test_two_ranks_own_every_father_row(gen, case):
    """With world = 2 the couples are split over the ranks; the father row of every couple has an owner, which
    is the rank that reads that couple's Psi[father, mother]."""
    father, mother, ranks = make_case(gen, case)
    plan = f_plan(gen, father, mother, ranks, world=2)
    for t in range(plan.n_layers):
        a, sh = plan.layer_arrays(t), plan.layer_shard(t)
        has = a["fam_father_slot"] >= 0
        assert np.array_equal(sh["fam_father_owner"] >= 0, has)
        assert ((sh["fam_father_owner"][has] < 2) & (sh["fam_father_lrow"][has] >= 0)).all()
        assert (sh["fam_father_lrow"][has] < np.array([plan.rank_rows(g) for g in sh["fam_father_owner"][has]])).all()


@pytest.mark.parametrize("case", ["geneaJi", "random0", "random1", "random2", "ladder"])
def test_replay_reads_the_exact_inbreeding(gen, case):
    """The Float64 replay of the plan, reading Psi[father, mother] of each couple in its layer, gives the exact
    kinship of the parents (Karigl's recursion in rationals)."""
    father, mother, ranks = make_case(gen, case)
    plan = f_plan(gen, father, mother, ranks)
    got = replay_f(plan, father, mother, ranks)
    assert_exact(got, father, mother, ranks)
    if case == "ladder":
        assert (got > 0).any() and got[got > 0].min() < 2.0 ** -150          # values far below Float32's range


def test_frontier_stays_near_the_live_peak(gen):
    """C3 at 5 %, every individual listed: the frontier width is within a few percent of the most rows any layer
    needs at once (live before the layer + born in it)."""
    father, mother, ranks = make_case(gen, "C3x0.05")
    plan = f_plan(gen, father, mother, ranks)
    peak = max(i["live_before"] + i["n_new"] for i in plan.layers())
    assert peak <= plan.capacity <= 1.04 * peak + 128, (plan.capacity, peak)


def test_f_without_a_device(gen):
    """What needs no device: an empty list, a list without an individual that has both parents (zeros, duplicates
    kept), an unknown ID or rank (KeyError), and an engine on a gen.f plan (it has no matrix to fetch)."""
    ped = gen.genealogy(gen.geneaJi)
    assert gen.f(ped, []).shape == (0,)
    founders = gen.founder(ped)
    single = [int(ped.ids[r]) for r in range(len(ped.ids)) if (ped.father[r] >= 0) != (ped.mother[r] >= 0)]
    got = gen.f(ped, np.concatenate([founders, founders[:2], single]))
    assert got.dtype == np.float32 and not got.any() and len(got) == len(founders) + 2 + len(single)
    got, stats = gen.f_arrays(ped.father, ped.mother, ped.rank_of(founders), dtype=np.float64)
    assert got.dtype == np.float64 and not got.any() and stats["n_unique"] == 0
    with pytest.raises(KeyError):
        gen.f(ped, [1, 123456789])
    with pytest.raises(KeyError):
        gen.f_arrays(ped.father, ped.mother, [0, len(ped.father)])
    plan = f_plan(gen, ped.father, ped.mother, np.arange(len(ped.father)))
    with pytest.raises(gen.GenlibError) as e:
        gen.Engine(plan, "fp64")
    assert e.value.status == 1 and "genlib_f" in str(e.value)


# ---- on the device --------------------------------------------------------------------------------------------

@pytest.mark.gpu
def test_f_geneaji(gen, ob):
    """test/runtests.jl:47-48, and every ID against the oracle's pairwise recursion; duplicates and one-parent IDs."""
    ped = gen.genealogy(gen.geneaJi)
    assert gen.f(ped, [1]).tolist() == [0.18359375] and gen.f(ped, [17]).tolist() == [0.0]
    o = ob.OraclePedigree.from_csv(gen.geneaJi)
    ids = np.concatenate([ped.ids, ped.ids[::-2], [1, 1]])
    got, stats = gen.f(ped, ids, return_stats=True)
    assert got.dtype == np.float32 and len(got) == len(ids)
    for ID, v in zip(ids, got):
        x = ped[int(ID)]
        want = 0.0 if x.father is None or x.mother is None else o.phi_pair(x.father.ID, x.mother.ID)
        assert v == np.float32(want)
    assert stats["n_unique"] == int(((ped.father >= 0) & (ped.mother >= 0)).sum()) and stats["kernel_launches"] > 0
    with pytest.raises(KeyError):
        gen.f(ped, [1, 123456789])


@pytest.mark.gpu
def test_f_genea140_everyone(gen, ob):
    """All 41 523 individuals of genea140: bitwise the Float64 replay of the same plan, and the oracle's pairwise
    recursion on the sampled IDs of test_inbreeding_f_genea140."""
    father, mother, ranks = make_case(gen, "genea140")
    ped = gen.genealogy(gen.genea140)
    got64, stats = gen.f_arrays(father, mother, ranks, dtype=np.float64)
    want = replay_f(f_plan(gen, father, mother, ranks), father, mother, ranks)
    assert np.array_equal(got64, want)
    got = gen.f(ped, ped.ids)
    assert np.array_equal(got, got64.astype(np.float32))
    o = ob.OraclePedigree.from_csv(gen.genea140)
    rng = np.random.default_rng(5)
    deep = np.nonzero((ped.father >= 0) & (ped.mother >= 0))[0]
    for r in rng.choice(deep[-4000:], 40, replace=False):
        x = ped[int(ped.ids[r])]
        assert got[r] == np.float32(o.phi_pair(x.father.ID, x.mother.ID))
    assert stats["row_updates"] == len(father) and stats["capacity"] > 0


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["random0", "random1", "random2", "ladder", "sibship", "C3x0.05", "C5x0.05"])
def test_f_equals_the_replay(gen, case):
    father, mother, ranks = make_case(gen, case)
    got, _ = gen.f_arrays(father, mother, ranks, dtype=np.float64)
    assert np.array_equal(got, replay_f(f_plan(gen, father, mother, ranks), father, mother, ranks))


@pytest.mark.gpu
def test_f_c3_probands_equals_the_parents_matrix(gen):
    """C3's probands: bitwise what the replaced method gives, the Float64 phi matrix of their parents."""
    s = gen.synth.config("C3")
    ped = gen.genealogy(s.as_columns())
    ranks = ped.rank_of(s.probands)
    fa, mo = ped.father[ranks], ped.mother[ranks]
    both = (fa >= 0) & (mo >= 0)
    parents = np.unique(np.concatenate([fa[both], mo[both]]))
    k = gen.phi(ped, ped.ids[parents], numerics="fp64", dtype=np.float64)
    want = np.zeros(len(ranks))
    want[both] = k[np.searchsorted(parents, fa[both]), np.searchsorted(parents, mo[both])]
    got, _ = gen.f_arrays(ped.father, ped.mother, ranks, dtype=np.float64)
    assert np.array_equal(got, want)


@pytest.mark.gpu
def test_f_c3_everyone_on_one_device(gen):
    """All 1 000 000 individuals of C3 on one device: 0 <= F < 1, full siblings equal, and 64 sampled IDs bitwise
    the Float64 phi of their two parents."""
    s = gen.synth.config("C3")
    ped = gen.genealogy(s.as_columns())
    got, stats = gen.f(ped, ped.ids, return_stats=True)
    got64, _ = gen.f_arrays(ped.father, ped.mother, np.arange(len(ped.ids)), dtype=np.float64)
    assert np.array_equal(got, got64.astype(np.float32))
    assert ((got64 >= 0) & (got64 < 1)).all() and (got64 > 0).any()
    both = np.nonzero((ped.father >= 0) & (ped.mother >= 0))[0]
    key = ped.father[both].astype(np.int64) * len(ped.ids) + ped.mother[both]
    order = np.argsort(key, kind="stable")
    same = key[order][1:] == key[order][:-1]
    assert np.array_equal(got64[both[order]][1:][same], got64[both[order]][:-1][same])
    for r in np.random.default_rng(3).choice(both, 64, replace=False):
        k = gen.phi(ped, ped.ids[[ped.father[r], ped.mother[r]]], numerics="fp64", dtype=np.float64)
        assert got64[r] == k[0, 1], r
    assert stats["device_bytes"] < 180e9 and stats["n_unique"] == len(both)


@pytest.mark.gpu
def test_f_two_devices_equal_one(gen):
    if gen.lib().genlib_device_count() < 2:
        pytest.skip("needs two GPUs")
    for case in ("genea140", "C3x0.05", "C5x0.05"):
        father, mother, ranks = make_case(gen, case)
        one, _ = gen.f_arrays(father, mother, ranks, dtype=np.float64, devices=[0])
        two, _ = gen.f_arrays(father, mother, ranks, dtype=np.float64, devices=[0, 1])
        assert np.array_equal(one, two), case
