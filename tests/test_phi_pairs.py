"""gen.phi_pairs: the kinship of each pair of a list, read on the device from one depth-layered sweep (the
GENLIB_SCHEDULE_PAIRS plan: members = the ancestors-or-self of everybody named, pair (a, b) read just before layer
max(depth a, depth b) + 1, both rows live until then), and the scalar gen.phi(ind1, ind2)."""
from fractions import Fraction

import numpy as np
import pytest

from plan_replay import replay
from test_inbreeding import _NoProbandMatrix, make_case
from util import exact_kinship


def ancestors_depth(father, mother, named):
    """The ancestors-or-self of the named ranks, and every individual's depth below the founders."""
    n = len(father)
    member = np.zeros(n, bool)
    member[np.asarray(named)] = True
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


def make_pairs(father, mother, seed=0, n_random=300):
    """Random pairs, and every kind the conventions speak of: self, parent-child both ways, ancestor-descendant
    across many generations, founders, duplicated and reversed pairs (unrelated ones come with the random pairs)."""
    rng = np.random.default_rng(seed)
    n = len(father)
    a, b = list(rng.integers(0, n, n_random)), list(rng.integers(0, n, n_random))
    kids = np.nonzero(father >= 0)[0]
    for x in rng.choice(np.arange(n), min(n, 20), replace=False):
        a.append(x); b.append(x)                                     # self
    for x in rng.choice(kids, min(len(kids), 20), replace=False):
        a += [x, father[x]]; b += [father[x], x]                     # parent-child, both ways
        if mother[x] >= 0:
            a.append(mother[x]); b.append(x)
    deep = np.argsort(-ancestors_depth(father, mother, np.arange(n))[1], kind="stable")[:10]
    for x in deep:                                                   # ancestor-descendant, many generations apart
        y, steps = int(x), 0
        while True:
            p = father[y] if father[y] >= 0 else mother[y]
            if p < 0:
                break
            y, steps = int(p), steps + 1
            if steps in (2, 5, 11) or (father[y] < 0 and mother[y] < 0):
                a.append(x); b.append(y)
    founders = np.nonzero((father < 0) & (mother < 0))[0]
    for x in rng.choice(founders, min(len(founders), 10), replace=False):
        a.append(x); b.append(int(rng.integers(0, n)))
    k = len(a)
    a += a[:15] + b[:15]                                             # duplicated, and reversed
    b += b[:15] + a[:15]
    assert len(a) == k + 30
    return np.array(a, np.int32), np.array(b, np.int32)


def pairs_case(gen, name):
    """(father, mother, a, b)."""
    father, mother, _ = make_case(gen, name)
    if name == "sibship":                                           # the sibship, its parents, unrelated founders
        rng = np.random.default_rng(1)
        a = np.concatenate([rng.integers(3002, 4002, 200), [0, 1, 0, 3002], rng.integers(2, 3002, 100)])
        b = np.concatenate([rng.integers(3002, 4002, 200), [1, 0, 3002, 3002], rng.integers(0, 4002, 100)])
        return father, mother, a.astype(np.int32), b.astype(np.int32)
    a, b = make_pairs(father, mother, n_random=60 if name == "genea140" else 300)
    return father, mother, a, b


def pairs_plan(gen, father, mother, a, b, world=1, stream=False):
    return gen.Plan.pairs(father, mother, a, b, world=world, stream=stream)


def replay_pairs(plan, K):
    """Psi of every list position from the Float64 replay of the plan: A[row slot, column slot] of each read after
    the layer before its own (reads of layer r happen before layer r; r == n_layers: after the last one)."""
    got = np.full(K, np.nan)
    S = plan.n_layers
    assert plan.pair_reads(0)["pos"].size == 0                       # nobody is read before the founders' layer

    def on_layer(t, A, live):
        r = plan.pair_reads(t + 1)
        got[r["pos"]] = A[r["row_slot"], r["col_slot"]]

    replay(_NoProbandMatrix(plan), "fp64", on_layer=on_layer)
    assert sum(plan.pair_reads(t)["pos"].size for t in range(S + 1)) == K
    return got


def assert_exact(got, father, mother, a, b):
    """Exact rationals; equal wherever the value fits 53 bits, within 2^-50 relative elsewhere."""
    phi = exact_kinship(father, mother)
    for v, x, y in zip(got, a, b):
        want = phi(int(x), int(y))
        if Fraction(float(want)) == want:
            assert Fraction(float(v)) == want, (x, y, v, want)
        else:
            assert abs(Fraction(float(v)) - want) <= want * Fraction(1, 2 ** 50), (x, y, v, want)


# ---- the plan, on the CPU -------------------------------------------------------------------------------------

CASES = ["geneaJi", "genea140", "random0", "random1", "random2", "ladder", "sibship"]


@pytest.mark.parametrize("case", CASES)
def test_replay_reads_the_exact_kinship(gen, case):
    """The Float64 replay of the plan, reading each pair in its layer, gives Karigl's recursion in exact rationals:
    self, parent-child, ancestor-descendant, founders, unrelated (exactly 0), duplicated and reversed pairs."""
    father, mother, a, b = pairs_case(gen, case)
    got = replay_pairs(pairs_plan(gen, father, mother, a, b), len(a))
    assert_exact(got, father, mother, a, b)
    if case == "sibship":                            # founders unrelated, parent-child, self, unrelated founders
        assert got[200] == 0 and got[201] == 0 and got[202] == 0.25 and got[203] == 0.5 and (got[204:] == 0).sum() >= 90
    else:                                            # duplicated and reversed pairs
        assert np.array_equal(got[-30:-15], got[:15]) and np.array_equal(got[-15:], got[:15])


@pytest.mark.parametrize("case", CASES)
def test_plan_shape(gen, case, monkeypatch):
    """Members are the ancestors-or-self of everybody named, born in the layer of their depth; each read's two slots
    are live in its layer and its row side is the higher-ranked member; a row is live from the layer after its birth
    to the later of its last child and its last read; after the last layer only rows read there are kept; the plan
    passes the planner's own checks (GENLIB_PLAN_VERIFY)."""
    monkeypatch.setenv("GENLIB_PLAN_VERIFY", "1")
    father, mother, a, b = pairs_case(gen, case)
    member, depth = ancestors_depth(father, mother, np.concatenate([a, b]))
    plan = pairs_plan(gen, father, mother, a, b)
    S = plan.n_layers
    assert plan.n_unique == len(np.unique(np.concatenate([a, b]))) and S == depth[member].max() + 1
    assert plan.row_updates == member.sum()
    read = np.maximum(depth[a], depth[b]) + 1
    last = np.full(len(father), -1)
    for x in np.nonzero(member)[0]:
        for p in (father[x], mother[x]):
            if p >= 0:
                last[p] = max(last[p], depth[x])
    np.maximum.at(last, a, read)
    np.maximum.at(last, b, read)
    born = np.zeros(len(father), bool)
    home = {}
    for t in range(S + 1):
        r = plan.pair_reads(t)
        assert np.array_equal(r["pos"], np.nonzero(read == t)[0])   # bucketed by read layer, list order kept
        hi, lo = np.maximum(a[r["pos"]], b[r["pos"]]), np.minimum(a[r["pos"]], b[r["pos"]])
        assert np.array_equal(r["row_slot"], [home[x] for x in hi]) and np.array_equal(r["col_slot"], [home[x] for x in lo])
        if t == S:
            break
        arr = plan.layer_arrays(t)
        ind = arr["member_ind"]
        assert (depth[ind] == t).all() and member[ind].all() and not born[ind].any()
        live_slots = np.nonzero(arr["live_flags"] & 1)[0]
        assert np.isin(r["row_slot"], live_slots).all() and np.isin(r["col_slot"], live_slots).all()
        occupant = {s: x for x, s in home.items()}
        who = np.sort([occupant[s] for s in live_slots])
        assert np.array_equal(who, np.nonzero(born & (last >= t))[0]), f"layer {t}: live rows"
        carried = np.sort([occupant[s] for s in np.nonzero(arr["live_flags"] & 2)[0]])
        assert np.array_equal(carried, np.nonzero(born & (last > t))[0]), f"layer {t}: carried rows"
        if t == S - 1:                                               # after the last layer: the rows read there only
            assert set(carried.tolist()) <= set(np.concatenate([a[read == S], b[read == S]]).tolist())
        for x in np.nonzero(born & (last == t))[0]:                  # its slot may be taken from the next layer on
            del home[int(x)]
        for s, x in zip(arr["member_slot"], ind):
            home[int(x)] = int(s)
        born[ind] = True
        for x in ind[last[ind] == t]:                                # read by nobody later: never live again
            del home[int(x)]
    assert np.array_equal(born, member)


@pytest.mark.parametrize("case", ["geneaJi", "genea140", "random0", "random1", "random2", "ladder", "sibship"])
def test_streamed_plan_equals_the_plan_made_in_one_piece(gen, case, monkeypatch):
    """The plan published layer by layer (what genlib_phi_pairs runs while it plans) is the plan made in one piece,
    also when a bound does not hold and the planner finishes with exact sizes."""
    father, mother, a, b = pairs_case(gen, case)
    for world in (1, 2):
        whole = pairs_plan(gen, father, mother, a, b, world)
        ref = gen.lib().genlib_plan_digest(whole._h, 0)
        for slack in (None, "-1"):
            if slack is None:
                monkeypatch.delenv("GENLIB_STREAM_SLACK_PCT", raising=False)
            else:
                monkeypatch.setenv("GENLIB_STREAM_SLACK_PCT", slack)
            p = pairs_plan(gen, father, mother, a, b, world, stream=True)
            assert gen.lib().genlib_plan_digest(p._h, 0) == ref, (world, slack)
    monkeypatch.delenv("GENLIB_STREAM_SLACK_PCT", raising=False)


@pytest.mark.parametrize("case", ["geneaJi", "random0", "random2", "ladder", "sibship"])
def test_two_ranks_hold_the_rows_they_read(gen, case):
    """With world = 2 the owner and local row a read records hold the row: the live list's entry in the read's layer,
    or the member's own home for the reads after the last layer."""
    father, mother, a, b = pairs_case(gen, case)
    plan = pairs_plan(gen, father, mother, a, b, world=2)
    S = plan.n_layers
    homes = {}
    for t in range(S):
        r, sh = plan.pair_reads(t), plan.layer_shard(t)
        assert np.array_equal(r["owner"], sh["live_owner"][r["row_slot"]]) and np.array_equal(r["lrow"], sh["live_lrow"][r["row_slot"]])
        arr = plan.layer_arrays(t)
        for s, g, lr in zip(arr["member_slot"], arr["member_owner"], sh["member_lrow"]):
            homes[int(s)] = (int(g), int(lr))
    r = plan.pair_reads(S)
    assert [homes[int(s)] for s in r["row_slot"]] == list(zip(r["owner"].tolist(), r["lrow"].tolist()))
    assert ((r["owner"] >= 0) & (r["owner"] < 2)).all()


def test_schedules_refuse_the_other_input(gen):
    """A pairs plan reads pairs and nothing else; plan inspection of the reads needs a pairs plan."""
    ped = gen.genealogy(gen.geneaJi)
    with pytest.raises(gen.GenlibError):
        gen.Plan(ped.father, ped.mother, [0, 1], schedule="pairs")
    plan = gen.Plan(ped.father, ped.mother, [0, 1], schedule="f")
    with pytest.raises(gen.GenlibError):
        plan.pair_reads(0)
    plan = pairs_plan(gen, ped.father, ped.mother, [0], [1])
    with pytest.raises(gen.GenlibError):
        plan.pair_reads(plan.n_layers + 1)


def test_phi_pairs_without_a_device(gen):
    """What needs no device: an empty list, lists of unequal length (ValueError), an unknown ID or rank (KeyError),
    Individuals of two pedigrees (ValueError), and an engine on a pairs plan (it has no matrix to fetch)."""
    ped = gen.genealogy(gen.geneaJi)
    got, stats = gen.phi_pairs(ped, [], [], return_stats=True)
    assert got.shape == (0,) and got.dtype == np.float64 and stats["n_unique"] == 0
    assert gen.phi_pairs_arrays(ped.father, ped.mother, [], [], dtype=np.float32)[0].dtype == np.float32
    with pytest.raises(ValueError):
        gen.phi_pairs(ped, [1, 2], [1])
    with pytest.raises(KeyError):
        gen.phi_pairs(ped, [1, 123456789], [1, 2])
    with pytest.raises(KeyError):
        gen.phi_pairs_arrays(ped.father, ped.mother, [0, 1], [len(ped.father), 0])
    other = gen.genealogy(gen.geneaJi)
    with pytest.raises(ValueError):
        gen.phi(ped[1], other[2])
    with pytest.raises(ValueError):
        gen.phi(ped[1], 2)
    plan = pairs_plan(gen, ped.father, ped.mother, [0, 1], [1, 2])
    with pytest.raises(gen.GenlibError) as e:
        gen.Engine(plan, "fp64")
    assert e.value.status == 1 and "genlib_phi_pairs" in str(e.value)


# ---- on the device --------------------------------------------------------------------------------------------

def couples_of(father, mother, ranks):
    both = ranks[(father[ranks] >= 0) & (mother[ranks] >= 0)]
    return father[both], mother[both], both


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES)
def test_phi_pairs_equals_the_replay(gen, case):
    father, mother, a, b = pairs_case(gen, case)
    got, stats = gen.phi_pairs_arrays(father, mother, a, b)
    assert np.array_equal(got, replay_pairs(pairs_plan(gen, father, mother, a, b), len(a)))
    assert stats["n_unique"] == len(np.unique(np.concatenate([a, b]))) and stats["kernel_launches"] > 0
    got32, _ = gen.phi_pairs_arrays(father, mother, a, b, dtype=np.float32)
    assert np.array_equal(got32, got.astype(np.float32))


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["C3x0.05", "C5x0.05"])
def test_phi_pairs_equals_the_replay_on_synthetic_populations(gen, case):
    """Couples, and pairs within a generation (sampled), of 5 % of C3 and C5."""
    father, mother, ranks = make_case(gen, case)
    fa, mo, _ = couples_of(father, mother, ranks)
    _, depth = ancestors_depth(father, mother, ranks)
    rng = np.random.default_rng(2)
    a, b = [fa], [mo]
    for d in np.unique(depth)[::7]:
        at = np.nonzero(depth == d)[0]
        a.append(rng.choice(at, 200)); b.append(rng.choice(at, 200))
    a, b = np.concatenate(a).astype(np.int32), np.concatenate(b).astype(np.int32)
    got, _ = gen.phi_pairs_arrays(father, mother, a, b)
    assert np.array_equal(got, replay_pairs(pairs_plan(gen, father, mother, a, b), len(a)))


@pytest.mark.gpu
def test_phi_pairs_genea140_oracle_and_conventions(gen, ob):
    """Sampled genea140 pairs against the oracle's pairwise recursion; phi(a, b) == phi(b, a) bitwise,
    phi(a, a) == 0.5 + 0.5 * F(a) exactly, unrelated individuals exactly 0; the scalar gen.phi(ind1, ind2)."""
    ped = gen.genealogy(gen.genea140)
    o = ob.OraclePedigree.from_csv(gen.genea140)
    rng = np.random.default_rng(7)
    ids1, ids2 = rng.choice(ped.ids, 60), rng.choice(ped.ids[-8000:], 60)
    got = gen.phi_pairs(ped, ids1, ids2)
    for x, y, v in zip(ids1, ids2, got):
        assert v == o.phi_pair(int(x), int(y)), (x, y)
    assert np.array_equal(gen.phi_pairs(ped, ids2, ids1), got)
    everyone = ped.ids
    diag = gen.phi_pairs(ped, everyone, everyone)
    F, _ = gen.f_arrays(ped.father, ped.mother, np.arange(len(everyone)), dtype=np.float64)
    assert np.array_equal(diag, 0.5 + 0.5 * F)
    founders = gen.founder(ped)
    assert not gen.phi_pairs(ped, founders[:-1], founders[1:]).any()
    v = gen.phi(ped[int(ids1[0])], ped[int(ids2[0])])
    assert isinstance(v, float) and v == got[0]
    assert gen.phi(ped[int(ids1[0])], ped[int(ids1[0])]) == diag[ped.rank_of([ids1[0]])[0]]


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["genea140", "C3x0.05", "C5x0.05"])
def test_phi_pairs_of_the_parents_equals_f(gen, case):
    """phi_pairs(father(x), mother(x)) is bitwise gen.f of x, for everyone with two parents: the same depth-layered
    read, also 200 generations deep."""
    father, mother, ranks = make_case(gen, case)
    fa, mo, kids = couples_of(father, mother, ranks)
    got, _ = gen.phi_pairs_arrays(father, mother, fa, mo)
    F, _ = gen.f_arrays(father, mother, kids, dtype=np.float64)
    assert np.array_equal(got, F)


@pytest.mark.gpu
@pytest.mark.parametrize("config", ["genea140", "C3"])
def test_all_pairs_of_probands_equal_the_phi_matrix(gen, config):
    """All pairs of 200 sampled probands (genea140: all 140): bitwise the Float64 gen.phi matrix the pairs list
    replaces."""
    if config == "genea140":
        ped = gen.genealogy(gen.genea140)
        pro = gen.pro(ped)
    else:
        s = gen.synth.config("C3")
        ped, pro = gen.genealogy(s.as_columns()), s.probands
    k = min(200, len(pro))
    ids = np.random.default_rng(11).choice(pro, k, replace=False)
    want = gen.phi(ped, ids, numerics="fp64", dtype=np.float64)
    i, j = np.meshgrid(np.arange(k), np.arange(k), indexing="ij")
    got = gen.phi_pairs(ped, ids[i.ravel()], ids[j.ravel()])
    assert np.array_equal(got.reshape(k, k), want)


@pytest.mark.gpu
def test_c3_every_couple(gen):
    """Every distinct (father, mother) pair of C3, childless couples of the list included, on one device: bitwise
    gen.f of one child per couple."""
    s = gen.synth.config("C3")
    ped = gen.genealogy(s.as_columns())
    fa, mo, kids = couples_of(ped.father, ped.mother, np.arange(len(ped.ids)))
    key = fa.astype(np.int64) * len(ped.ids) + mo
    _, first = np.unique(key, return_index=True)
    got, stats = gen.phi_pairs_arrays(ped.father, ped.mother, fa[first], mo[first])
    F, _ = gen.f_arrays(ped.father, ped.mother, kids[first], dtype=np.float64)
    assert np.array_equal(got, F)
    assert stats["device_bytes"] < 180e9 and stats["d2h_bytes"] == 8 * len(first)


@pytest.mark.gpu
def test_phi_pairs_two_devices_equal_one(gen):
    if gen.lib().genlib_device_count() < 2:
        pytest.skip("needs two GPUs")
    for case in ("genea140", "random1", "C3x0.05"):
        father, mother, ranks = make_case(gen, case)
        a, b = make_pairs(father, mother, seed=3)
        one, _ = gen.phi_pairs_arrays(father, mother, a, b, devices=[0])
        two, _ = gen.phi_pairs_arrays(father, mother, a, b, devices=[0, 1])
        assert np.array_equal(one, two), case
