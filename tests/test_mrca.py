"""gen.findMRCA and gen.findDistance: most recent common ancestors and minimum meioses.

CPU: the gc schedule (genlib_gc_plan_*) replayed with the uint16 (min, saturating +1) rules on a frontier
poisoned with 0 against breadth-first distances, the reference's definitions (restated below with Python sets)
against the child test and the rec-count criterion the library uses, the layer-count bound, and the front
end's errors.  GPU: findMRCA and findDistance against the restatement, the edge cases of the conventions,
the identities that tie the meioses to occ and rec, several devices, long distances and full-size C3."""
import hashlib
import itertools
from collections import deque

import numpy as np
import pytest

from test_gc import CASES, first_order, make_case
from test_occ import exact_case, exact_occ
from util import ladder_pedigree, random_pedigree

NONE = 0xFFFF                   # the device's "no path"


# ---- the reference's definitions, restated --------------------------------------------------------------
def up_distances(father, mother, x):
    """{ancestor-or-self rank of x: minimum meioses from it down to x}, breadth first over the parents."""
    dist, q = {x: 0}, deque([x])
    while q:
        y = q.popleft()
        for p in (father[y], mother[y]):
            if p >= 0 and p not in dist:
                dist[p] = dist[y] + 1
                q.append(p)
    return dist


def bfs_meioses(father, mother, pro, anc):
    """len(pro) x len(anc): d(anc[j], pro[i]) by breadth-first search, -1 where there is no descent path."""
    father, mother = list(map(int, father)), list(map(int, mother))
    up = {int(p): up_distances(father, mother, int(p)) for p in set(map(int, pro))}
    return np.array([[up[int(p)].get(int(a), -1) for a in anc] for p in pro], np.int64).reshape(len(pro), len(anc))


def proper_ancestors(father, mother, starts):
    """Every proper ancestor of any rank in `starts`."""
    seen, stack = set(), [p for s in starts for p in (father[s], mother[s]) if p >= 0]
    while stack:
        y = stack.pop()
        if y not in seen:
            seen.add(y)
            stack.extend(p for p in (father[y], mother[y]) if p >= 0)
    return seen


def mrca_sets(father, mother, ranks):
    """(common, MRCA) rank sets by the definitions: common = the intersection of the IDs' proper-ancestor sets,
    MRCA = common minus every ancestor of a common ancestor."""
    father, mother = list(map(int, father)), list(map(int, mother))
    common = set.intersection(*(proper_ancestors(father, mother, [int(r)]) for r in set(map(int, ranks))))
    return common, common - proper_ancestors(father, mother, common)


def restated_findMRCA(ped, IDs):
    """(ancestors sorted by ID, meioses) of gen.findMRCA by the definitions and breadth-first distances."""
    ranks = ped.rank_of(IDs)
    _, mrca = mrca_sets(ped.father, ped.mother, ranks)
    anc_ids = np.sort(ped.ids[sorted(mrca)]) if mrca else np.zeros(0, np.int64)
    return anc_ids, bfs_meioses(ped.father, ped.mother, ranks, ped.rank_of(anc_ids))


def chain(n):
    """n individuals, each the only child of the previous one (and of a missing other parent)."""
    father = np.arange(-1, n - 1, dtype=np.int32)
    return father, np.full(n, -1, np.int32)


# ---- the plan, replayed ---------------------------------------------------------------------------------
def replay_min_plus(plan, pro, anc):
    """Run the schedule with the kernel's uint16 rules -- acc = min(acc, min(x + 1, 0xFFFF)) over the inputs,
    0 in the row's own column -- on a frontier and output block poisoned with 0: the rules give 0 only in a
    row's own column, so a slot read before it is written shows up as a distance that is too short.  Output
    rows no path reaches are filled with 0xFFFF, as the engine does.  Returns len(pro) x len(anc), -1 = none."""
    info = plan.info()
    W, cap = info["width"], info["capacity"]
    desc = info["direction"] == "descend"
    tgt_list, col_list = (pro, anc) if desc else (anc, pro)
    F = np.zeros((max(cap, 1), W), np.uint16)
    n_tgt = len(set(tgt_list.tolist()))
    O = np.zeros((n_tgt, W), np.uint16)
    written = np.zeros(n_tgt, bool)
    out_rows = 0
    for L in plan.layers():
        ptr_, ins = L["in_ptr"], L["in_slot"]
        acc = np.full((len(L["row_ind"]), W), NONE, np.uint16)
        fan = np.diff(ptr_)
        for k in range(int(fan.max()) if len(fan) else 0):
            r = np.nonzero(fan > k)[0]
            plus1 = np.minimum(F[ins[ptr_[r] + k]].astype(np.uint32) + 1, NONE).astype(np.uint16)
            acc[r] = np.minimum(acc[r], plus1)
        s = np.nonzero(L["row_seed"] >= 0)[0]
        acc[s, L["row_seed"][s]] = 0
        sl, ou = L["row_slot"], L["row_out"]
        F[sl[sl >= 0]] = acc[sl >= 0]
        O[ou[ou >= 0]] = acc[ou >= 0]
        written[ou[ou >= 0]] = True
        out_rows += int((ou >= 0).sum())
    if out_rows < n_tgt:
        O[~written] = NONE
    G = O[first_order(tgt_list)][:, first_order(col_list)].astype(np.int64)
    G[G == NONE] = -1
    return G if desc else G.T


_BFS = {}


def bfs_case(gen, name):
    if name not in _BFS:
        _BFS[name] = bfs_meioses(*make_case(gen, name))
    return _BFS[name]


@pytest.mark.parametrize("direction", ["descend", "ascend"])
@pytest.mark.parametrize("case", CASES)
def test_plan_replay_min_plus_equals_bfs(gen, case, direction, monkeypatch):
    father, mother, pro, anc = make_case(gen, case)
    monkeypatch.setenv("GENLIB_GC_DIRECTION", direction)
    plan = gen.GcPlan(father, mother, pro, anc)
    assert plan.info()["direction"] == direction
    want = bfs_case(gen, case)
    assert np.array_equal(replay_min_plus(plan, pro, anc), want)
    assert want.max(initial=0) <= plan.info()["n_layers"] - 1                  # the sentinel bound


def _id_sets(gen, ped, rng):
    """The ID lists the definitions are compared on: the probands, pairs of them, and random small sets."""
    P = gen.pro(ped)
    sets = [P] + [list(p) for p in itertools.combinations(P[:6], 2)]
    sets += [rng.choice(ped.ids, k, replace=False) for k in (1, 2, 2, 3, 5)]
    return sets


@pytest.mark.parametrize("case", ["geneaJi", "genea140", "random0", "random1", "random2"])
def test_child_test_and_rec_criterion_select_the_set_definition(gen, case):
    """The library's criterion -- rec(a) over the distinct IDs == their number, a not an ID, no common child --
    selects the MRCAs of the set definition (the child test's equivalence, DESIGN.md 2d)."""
    rng = np.random.default_rng(7)
    if case.startswith("random"):
        ped = gen.genealogy(random_pedigree(np.random.default_rng(int(case[-1])), 300, 30))
    else:
        ped = gen.genealogy(gen.geneaJi if case == "geneaJi" else gen.genea140)
    father, mother = ped.father, ped.mother
    children = [[] for _ in range(len(father))]
    for c in range(len(father)):
        for p in (father[c], mother[c]):
            if p >= 0:
                children[p].append(c)
    for IDs in _id_sets(gen, ped, rng):
        ranks = ped.rank_of(IDs)
        uniq = sorted(set(ranks.tolist()))
        common, mrca = mrca_sets(father, mother, ranks)
        # the child test on the set-defined common ancestors
        assert mrca == {a for a in common if not any(c in common for c in children[a])}
        # the rec-count criterion on S = ancestors-or-self of the IDs, from exact path counts
        S = sorted(proper_ancestors(list(map(int, father)), list(map(int, mother)), uniq) | set(uniq))
        reach = (exact_occ(father, mother, uniq, S) > 0).sum(axis=1)
        common_rec = {a for a, r in zip(S, reach) if r == len(uniq) and a not in uniq}
        assert common_rec == common
        parents = {int(p) for a in common_rec for p in (father[a], mother[a]) if p >= 0}
        assert common_rec - parents == mrca


def test_layer_bound_is_refused_before_any_launch(gen):
    """A distance is below the plan's layer count; 0xFFFF layers or more could reach the sentinel."""
    father, mother = chain(0xFFFF)                            # 0xFFFF layers from rank 0 down to the last rank
    with pytest.raises(gen.GenlibOverflowError) as e:
        gen.meioses_arrays(father, mother, [0xFFFF - 1], [0])
    assert e.value.status == 8 and "65535 layers" in str(e.value)
    plan = gen.GcPlan(father[:-1], mother[:-1], [0xFFFF - 2], [0])
    assert plan.info()["n_layers"] == 0xFFFF - 1                                  # one fewer is allowed


def test_front_end_errors_and_empty_lists(gen):
    ped = gen.genealogy(gen.geneaJi)
    with pytest.raises(KeyError):
        gen.findMRCA(ped, [1, 999])
    with pytest.raises(KeyError):
        gen.findDistance(ped, [1, 999], 17)
    with pytest.raises(KeyError):
        gen.findDistance(ped, [1, 2], 999)
    with pytest.raises(KeyError):
        gen.mrca_arrays(ped.father, ped.mother, [0, len(ped.ids)])
    with pytest.raises(KeyError):
        gen.meioses_arrays(ped.father, ped.mother, [0], [len(ped.ids)])
    father, mother = ped.father.copy(), ped.mother.copy()
    father[3] = 10                                            # a parent after its child
    for call in (lambda: gen.mrca_arrays(father, mother, [0, 1]), lambda: gen.meioses_arrays(father, mother, [0], [20])):
        with pytest.raises(gen.GenlibError) as e:
            call()
        assert e.value.status == 3 and "rank 3" in str(e.value)  # GENLIB_EORDER, the first offending rank
    # empty lists: an empty result without a device
    m = gen.findMRCA(ped, [])
    assert isinstance(m, gen.GenMatrix) and m.meioses.shape == (0, 0) and m.meioses.dtype == np.int64
    assert len(m.individuals) == 0 and len(m.ancestors) == 0
    assert gen.findDistance(ped, [], 17) == 0
    r, _ = gen.mrca_arrays(ped.father, ped.mother, [])
    assert r.shape == (0,)
    for got, shape in ((gen.meioses_arrays(ped.father, ped.mother, [], [0, 1])[0], (0, 2)),
                       (gen.meioses_arrays(ped.father, ped.mother, [0, 1], [])[0], (2, 0))):
        assert got.shape == shape and got.dtype == np.int64
    with pytest.raises(ValueError):
        gen.GenMatrix([1, 2], [3], np.zeros((1, 2), np.int64))


def test_no_cpu_fallback(gen):
    if gen.lib().genlib_device_count() > 0:
        pytest.skip("a CUDA device is present")
    ped = gen.genealogy(gen.geneaJi)
    for call in (lambda: gen.findMRCA(ped, [1, 2]), lambda: gen.findDistance(ped, [1, 2], 17),
                 lambda: gen.meioses_arrays(ped.father, ped.mother, [0], [20])):
        with pytest.raises(gen.GenlibError) as e:
            call()
        assert e.value.status == 4                  # GENLIB_ECUDA


# ---- on the GPU ------------------------------------------------------------------------------------------
def _check_findMRCA(gen, ped, IDs, **kw):
    got = gen.findMRCA(ped, IDs, **kw)
    anc, d = restated_findMRCA(ped, IDs)
    assert np.array_equal(got.individuals, np.asarray(IDs, np.int64))
    assert np.array_equal(got.ancestors, anc), (IDs, got.ancestors, anc)
    assert got.meioses.dtype == np.int64 and np.array_equal(got.meioses, d)
    assert (got.meioses >= 1).all()                    # proper ancestors of every ID
    return got


@pytest.mark.gpu
def test_gpu_findMRCA_geneaJi(gen):
    ped = gen.genealogy(gen.geneaJi)
    P = gen.pro(ped)
    _check_findMRCA(gen, ped, P)
    for pair in itertools.combinations(P, 2):
        _check_findMRCA(gen, ped, list(pair))
    rng = np.random.default_rng(3)
    for _ in range(30):
        _check_findMRCA(gen, ped, rng.choice(ped.ids, 2, replace=False))


@pytest.mark.gpu
def test_gpu_findMRCA_genea140(gen):
    ped = gen.genealogy(gen.genea140)
    P = gen.pro(ped)
    m, stats = gen.findMRCA(ped, P, return_stats=True)
    anc, d = restated_findMRCA(ped, P)
    assert np.array_equal(m.ancestors, anc) and np.array_equal(m.meioses, d)
    assert stats["mrca"]["n_pro"] == len(P) and stats["meioses"]["n_anc"] == len(anc)
    rng = np.random.default_rng(140)
    for _ in range(50):
        _check_findMRCA(gen, ped, rng.choice(P, 2, replace=False))


@pytest.mark.gpu
@pytest.mark.parametrize("seed", [0, 1, 2])
def test_gpu_findMRCA_random(gen, seed):
    rng = np.random.default_rng(seed)
    ped = gen.genealogy(random_pedigree(rng, 300, 30, window=60 if seed % 2 else 0))
    _check_findMRCA(gen, ped, gen.pro(ped))
    for k in (1, 2, 2, 3, 4):
        _check_findMRCA(gen, ped, rng.choice(ped.ids, k, replace=False))


@pytest.mark.gpu
def test_gpu_one_id_gives_its_parents(gen):
    ped = gen.genealogy(gen.geneaJi)
    m = _check_findMRCA(gen, ped, [1])
    r = int(ped.rank_of([1])[0])
    assert m.ancestors.tolist() == sorted(int(ped.ids[p]) for p in (ped.father[r], ped.mother[r]) if p >= 0)
    assert m.meioses.tolist() == [[1] * len(m.ancestors)]


@pytest.mark.gpu
def test_gpu_founder_alone_is_empty(gen):
    ped = gen.genealogy(gen.geneaJi)
    m = gen.findMRCA(ped, [17])
    assert m.ancestors.shape == (0,) and m.meioses.shape == (1, 0)


@pytest.mark.gpu
def test_gpu_no_common_ancestor(gen):
    ped = gen.genealogy(gen.geneaJi)
    founders = gen.founder(ped)
    m = gen.findMRCA(ped, [founders[0], founders[1], 1])
    assert m.ancestors.shape == (0,) and m.meioses.shape == (3, 0) and m.meioses.dtype == np.int64
    # two disjoint families: children of different founder couples
    cols = {"ind": np.array([1, 2, 3, 4, 5, 6]), "father": np.array([0, 0, 0, 0, 1, 3]),
            "mother": np.array([0, 0, 0, 0, 2, 4]), "sex": np.array([1, 2, 1, 2, 1, 2])}
    ped2 = gen.genealogy(cols)
    m = gen.findMRCA(ped2, [5, 6])
    assert m.ancestors.shape == (0,) and m.meioses.shape == (2, 0)


@pytest.mark.gpu
def test_gpu_duplicates_kept(gen):
    ped = gen.genealogy(gen.geneaJi)
    a = _check_findMRCA(gen, ped, [1, 29])
    b = _check_findMRCA(gen, ped, [29, 1, 29, 1])
    assert np.array_equal(a.ancestors, b.ancestors)
    assert np.array_equal(b.meioses, a.meioses[[1, 0, 1, 0]])


@pytest.mark.gpu
def test_gpu_ancestor_of_another_is_not_common(gen):
    """For [parent, child] the MRCAs are the parent's parents, not the parent (an individual is not its own
    ancestor)."""
    ped = gen.genealogy(gen.geneaJi)
    child = 1
    r = int(ped.rank_of([child])[0])
    parent = int(ped.ids[ped.father[r]])
    m = _check_findMRCA(gen, ped, [parent, child])
    assert parent not in m.ancestors.tolist()
    pr = int(ped.rank_of([parent])[0])
    gp = sorted(int(ped.ids[p]) for p in (ped.father[pr], ped.mother[pr]) if p >= 0)
    assert set(gp) <= set(m.ancestors.tolist())
    for j, g in enumerate(m.ancestors):
        if int(g) in gp:
            assert m.meioses[:, j].tolist() == [1, 2]


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES)
def test_gpu_meioses_identities(gen, case, monkeypatch):
    """descend == ascend bitwise, == the breadth-first distances, (meioses >= 0) == (occ > 0).T."""
    father, mother, pro, anc = make_case(gen, case)
    res = {}
    for direction in ("descend", "ascend"):
        monkeypatch.setenv("GENLIB_GC_DIRECTION", direction)
        res[direction], st = gen.meioses_arrays(father, mother, pro, anc)
        assert st["direction"] == direction and st["d2h_bytes"] == res[direction].nbytes
        cm, _ = gen.meioses_arrays(father, mother, pro, anc, col_major=True)
        assert cm.flags.f_contiguous and np.array_equal(cm, res[direction])
    assert np.array_equal(res["descend"], res["ascend"])
    assert np.array_equal(res["ascend"], bfs_case(gen, case))
    exact = exact_case(gen, case)
    if max((int(x) for x in exact.ravel()), default=0) < 1 << 63:
        occ, _ = gen.occ_arrays(father, mother, pro, anc)
    else:
        occ = exact
    assert np.array_equal(res["ascend"] >= 0, (occ > 0).T)


@pytest.mark.gpu
def test_gpu_devices(gen, monkeypatch):
    if gen.lib().genlib_device_count() < 2:
        pytest.skip("one device")
    father, mother, pro, anc = make_case(gen, "random1")
    for direction in ("descend", "ascend"):
        monkeypatch.setenv("GENLIB_GC_DIRECTION", direction)
        one, _ = gen.meioses_arrays(father, mother, pro, anc, device=0)
        two, st = gen.meioses_arrays(father, mother, pro, anc, devices=[0, 1])
        assert np.array_equal(one, two) and st["n_dev"] == 2
    ped = gen.genealogy(gen.genea140)
    P = gen.pro(ped)
    a, b = gen.findMRCA(ped, P, device=0), gen.findMRCA(ped, P, devices=[0, 1])
    assert np.array_equal(a.ancestors, b.ancestors) and np.array_equal(a.meioses, b.meioses)


@pytest.mark.gpu
@pytest.mark.parametrize("direction", ["descend", "ascend"])
def test_gpu_long_distances(gen, direction, monkeypatch):
    """Distances above 255 (one byte) and up to the layer bound."""
    monkeypatch.setenv("GENLIB_GC_DIRECTION", direction)
    cols, pro = ladder_pedigree(300)
    ped = gen.genealogy(cols)
    anc = gen.founder(ped)
    got, _ = gen.meioses_arrays(ped.father, ped.mother, ped.rank_of(pro), ped.rank_of(anc))
    want = bfs_meioses(ped.father, ped.mother, ped.rank_of(pro), ped.rank_of(anc))
    assert want.max() > 255 and np.array_equal(got, want)
    father, mother = chain(0xFFFF - 1)                           # 65534 layers: the longest distance allowed
    got, st = gen.meioses_arrays(father, mother, [0xFFFF - 2, 300, 0], [0, 300])
    assert st["n_layers"] == 0xFFFF - 1
    assert got.tolist() == [[0xFFFF - 2, 0xFFFF - 2 - 300], [300, 0], [0, -1]]


@pytest.mark.gpu
def test_gpu_findDistance(gen):
    for path in (gen.geneaJi, gen.genea140):
        ped = gen.genealogy(path)
        P = gen.pro(ped)
        rng = np.random.default_rng(5)
        fa, mo = list(map(int, ped.father)), list(map(int, ped.mother))
        up = {int(r): up_distances(fa, mo, int(r)) for r in ped.rank_of(P)}
        for _ in range(20):
            IDs = rng.choice(P, 2, replace=False)
            ranks = ped.rank_of(IDs)
            common = set(up[int(ranks[0])]) & set(up[int(ranks[1])])
            for a in sorted(common)[:5]:
                want = up[int(ranks[0])][a] + up[int(ranks[1])][a]
                assert gen.findDistance(ped, IDs, int(ped.ids[a])) == want
        m = gen.findMRCA(ped, P[:2])
        for j, a in enumerate(m.ancestors):
            assert gen.findDistance(ped, P[:2], int(a)) == int(m.meioses[:, j].sum())
        # ancestorID among the IDs contributes 0; a founder above nobody raises
        x = next(int(i) for i in P if ped.father[ped.rank_of([i])[0]] >= 0)
        r = int(ped.rank_of([x])[0])
        par = int(ped.ids[ped.father[r]])
        assert gen.findDistance(ped, [x, par], par) == 1
        lonely = [int(f) for f in gen.founder(ped) if int(ped.rank_of([f])[0]) not in up[r]]
        assert lonely, f"every founder is an ancestor of {x}: no ID to exercise the ValueError with"
        with pytest.raises(ValueError) as e:
            gen.findDistance(ped, [P[0], x], lonely[0])
        assert str(x) in str(e.value)


@pytest.mark.gpu
def test_gpu_c3_full_size(gen, monkeypatch):
    s = gen.synth.config("C3", 1.0)
    ped = gen.genealogy(s.as_columns())
    father, mother, pro, anc = ped.father, ped.mother, ped.rank_of(s.probands), ped.rank_of(gen.founder(ped))
    # 64 probands from a fixed seed against the set restatement
    ids = np.random.default_rng(64).choice(s.probands, 64, replace=False)
    m = gen.findMRCA(ped, ids)
    want_anc, want_d = restated_findMRCA(ped, ids)
    assert np.array_equal(m.ancestors, want_anc) and np.array_equal(m.meioses, want_d)
    # all probands x founders: the two directions agree bitwise, and reachability is gen.rec's
    digests = []
    rec, _ = gen.rec_arrays(father, mother, pro, anc)
    for direction in ("ascend", "descend"):
        monkeypatch.setenv("GENLIB_GC_DIRECTION", direction)
        got, st = gen.meioses_arrays(father, mother, pro, anc)
        assert st["direction"] == direction
        digests.append(hashlib.sha256(got.tobytes()).hexdigest())
        assert np.array_equal((got >= 0).sum(axis=0), rec)
        del got
    assert digests[0] == digests[1]
