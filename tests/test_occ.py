"""gen.occ and gen.rec: descent-path counts and proband coverage.

CPU: the gc schedule (genlib_gc_plan_*) replayed with saturating integer sums and with OR on bit-packed words
against exact path counts in Python integers, the reference's path walk (restated below) against the same, a
sibling-mating chain whose counts double every generation, and the front end's errors.  GPU: the engine
against the known answer, the walk and the exact counts, the identities that tie occ, rec and gc together,
overflow, several devices and full-size C3."""
import hashlib

import numpy as np
import pytest

from test_gc import CASES, _synth_case, active_ranks, first_order, make_case

SAT = 1 << 63                      # the engine's saturation sentinel: a count that does not fit an Int64

# gen.occ(geneaJi) with pro = [1, 2, 29], ancestors = [17, 19, 20, 23, 25, 26], by exact recursion
JI_PRO = [1, 2, 29]
JI_ANC = [17, 19, 20, 23, 25, 26]
JI_OCC = np.array([[6, 6, 2], [8, 8, 2], [1, 1, 2], [0, 0, 1], [8, 8, 3], [8, 8, 3]], np.int64)
JI_TOTAL = np.array([14, 18, 4, 1, 19, 19], np.int64)
JI_REC = np.array([3, 3, 3, 1, 3, 3], np.int64)


def exact_occ(father, mother, pro_ranks, anc_ranks):
    """O[a, p] (len(anc) x len(pro), Python ints in an object array) by O[., p] = [p == .] + O[., father(p)] +
    O[., mother(p)], propagated over whichever list has fewer unique entries."""
    father, mother = np.asarray(father), np.asarray(mother)
    n = len(father)
    pro_u, pro_pos = np.unique(np.asarray(pro_ranks, np.int64), return_inverse=True)
    anc_u, anc_pos = np.unique(np.asarray(anc_ranks, np.int64), return_inverse=True)
    if len(anc_u) <= len(pro_u):              # down the generations, one column per ancestor
        col = {int(a): k for k, a in enumerate(anc_u)}
        S = np.zeros((n, len(anc_u)), object)
        for i in range(n):
            if father[i] >= 0:
                S[i] = S[i] + S[father[i]]
            if mother[i] >= 0:
                S[i] = S[i] + S[mother[i]]
            if i in col:
                S[i, col[i]] += 1
        M = S[pro_u][pro_pos][:, anc_pos].T
    else:                                     # up the generations, one column per proband
        col = {int(p): k for k, p in enumerate(pro_u)}
        S = np.zeros((n, len(pro_u)), object)
        for c in range(n - 1, -1, -1):
            if c in col:
                S[c, col[c]] += 1
            if father[c] >= 0:
                S[father[c]] = S[father[c]] + S[c]
            if mother[c] >= 0:
                S[mother[c]] = S[mother[c]] + S[c]
        M = S[anc_u][anc_pos][:, pro_pos]
    return np.array(M, object).reshape(len(anc_ranks), len(pro_ranks))


def occur_walk(father, mother, pro_ranks, anc_ranks):
    """gen.occ by the reference's algorithm (`_occur!`, SURVEY.md 2: src/describe.jl): for every ancestor a
    recursive walk down the `children` lists, adding 1 to O[a, p] whenever the walk reaches proband p -- one
    visit per descent path, duplicates of either list kept.  The checker, not the engine's algorithm."""
    n = len(father)
    children = [[] for _ in range(n)]
    for c in range(n):
        for par in (int(father[c]), int(mother[c])):
            if par >= 0:
                children[par].append(c)
    cols = {}
    for j, p in enumerate(pro_ranks):
        cols.setdefault(int(p), []).append(j)
    out = np.zeros((len(anc_ranks), len(pro_ranks)), np.int64)
    for i, a in enumerate(anc_ranks):
        stack = [int(a)]
        while stack:
            x = stack.pop()
            for j in cols.get(x, ()):
                out[i, j] += 1
            stack.extend(children[x])
    return out


def rec_from_descendants(father, mother, pro_ranks, anc_ranks):
    """gen.rec restated: the number of proband list entries in the descendants-or-self of each ancestor."""
    n = len(father)
    children = [[] for _ in range(n)]
    for c in range(n):
        for par in (int(father[c]), int(mother[c])):
            if par >= 0:
                children[par].append(c)
    out = np.zeros(len(anc_ranks), np.int64)
    for i, a in enumerate(anc_ranks):
        seen, stack = {int(a)}, [int(a)]
        while stack:
            for c in children[stack.pop()]:
                if c not in seen:
                    seen.add(c)
                    stack.append(c)
        out[i] = sum(int(p) in seen for p in pro_ranks)
    return out


def saturated(M):
    return np.array([[min(int(x), SAT) for x in row] for row in M], object).reshape(M.shape)


_EXACT, _WALK = {}, {}


def exact_case(gen, name):
    if name not in _EXACT:
        _EXACT[name] = exact_occ(*make_case(gen, name))
    return _EXACT[name]


def walk_case(gen, name):
    if name not in _WALK:
        _WALK[name] = occur_walk(*make_case(gen, name))
    return _WALK[name]


def sibling_chain(K):
    """A founder couple, then K generations of a brother and a sister who mate: the last generation's two
    members have 2^(K-1) descent paths from each founder.  Returns (father, mother, last two ranks)."""
    father, mother = [-1, -1], [-1, -1]
    a, b = 0, 1
    for _ in range(K):
        father += [a, a]
        mother += [b, b]
        a, b = len(father) - 2, len(father) - 1
    return np.array(father, np.int32), np.array(mother, np.int32), (a, b)


# ---- the plan, replayed -------------------------------------------------------------------------------------
def replay_counts(plan, pro, anc, exact):
    """Run the schedule with integer sums -- int64, or saturating sums of Python ints where the exact counts
    reach 2^62 -- and fail if a layer reads a frontier slot nobody has written; returns the len(anc) x len(pro)
    matrix."""
    info = plan.info()
    W, cap = info["width"], info["capacity"]
    desc = info["direction"] == "descend"
    tgt_list, col_list = (pro, anc) if desc else (anc, pro)
    big = max((int(x) for x in exact.ravel()), default=0) >= 1 << 62
    dt = object if big else np.int64
    F = np.zeros((max(cap, 1), W), dt)
    written = np.zeros(max(cap, 1), bool)
    O = np.zeros((len(set(tgt_list.tolist())), W), dt)
    for L in plan.layers():
        ptr_, ins = L["in_ptr"], L["in_slot"]
        assert written[ins].all(), "a slot is read before it is written"
        acc = np.zeros((len(L["row_ind"]), W), dt)
        fan = np.diff(ptr_)
        for k in range(int(fan.max()) if len(fan) else 0):
            r = np.nonzero(fan > k)[0]
            acc[r] = acc[r] + F[ins[ptr_[r] + k]]
            if big:
                acc[r] = np.minimum(acc[r], SAT)
        s = np.nonzero(L["row_seed"] >= 0)[0]
        acc[s, L["row_seed"][s]] += 1
        if big:
            acc[s] = np.minimum(acc[s], SAT)
        sl, ou = L["row_slot"], L["row_out"]
        F[sl[sl >= 0]] = acc[sl >= 0]
        written[sl[sl >= 0]] = True
        O[ou[ou >= 0]] = acc[ou >= 0]
    G = O[first_order(tgt_list)][:, first_order(col_list)]
    return G.T if desc else G


def replay_reach(plan, pro, anc):
    """Run the schedule with OR on uint64 words, 64 columns per word; slots read before they are written fail.
    Returns the len(anc) x len(pro) boolean reachability matrix."""
    info = plan.info()
    W, cap = info["width"], info["capacity"]
    words = (W + 63) // 64
    desc = info["direction"] == "descend"
    tgt_list, col_list = (pro, anc) if desc else (anc, pro)
    F = np.zeros((max(cap, 1), words), np.uint64)
    written = np.zeros(max(cap, 1), bool)
    O = np.zeros((len(set(tgt_list.tolist())), words), np.uint64)
    for L in plan.layers():
        ptr_, ins = L["in_ptr"], L["in_slot"]
        assert written[ins].all(), "a slot is read before it is written"
        rows = np.zeros((len(L["row_ind"]), words), np.uint64)
        for r in range(len(rows)):
            for k in range(ptr_[r], ptr_[r + 1]):
                rows[r] |= F[ins[k]]
            s = int(L["row_seed"][r])
            if s >= 0:
                rows[r, s >> 6] |= np.uint64(1) << np.uint64(s & 63)
        sl, ou = L["row_slot"], L["row_out"]
        F[sl[sl >= 0]] = rows[sl >= 0]
        written[sl[sl >= 0]] = True
        O[ou[ou >= 0]] = rows[ou >= 0]
    bits = np.unpackbits(O.view(np.uint8), axis=1, bitorder="little")[:, :W].astype(bool)
    G = bits[first_order(tgt_list)][:, first_order(col_list)]
    return G.T if desc else G


@pytest.mark.parametrize("direction", ["descend", "ascend"])
@pytest.mark.parametrize("case", CASES)
def test_plan_replay_counts_and_reachability(gen, case, direction, monkeypatch):
    father, mother, pro, anc = make_case(gen, case)
    monkeypatch.setenv("GENLIB_GC_DIRECTION", direction)
    plan = gen.GcPlan(father, mother, pro, anc)
    assert plan.info()["direction"] == direction
    want = exact_case(gen, case)
    assert want.shape == (len(anc), len(pro))
    assert sorted(r for L in plan.layers() for r in L["row_ind"].tolist()) == active_ranks(father, mother, pro, anc)
    assert np.array_equal(replay_counts(plan, pro, anc, want), saturated(want))
    assert np.array_equal(replay_reach(plan, pro, anc), want > 0)


@pytest.mark.parametrize("case", ["geneaJi", "genea140", "random0", "random1", "random2", "ladder"])
def test_walk_and_descendants_equal_the_exact_counts(gen, case):
    father, mother, pro, anc = make_case(gen, case)
    want = exact_case(gen, case)
    assert np.array_equal(walk_case(gen, case), want.astype(np.int64))
    assert np.array_equal(rec_from_descendants(father, mother, pro, anc), (want > 0).sum(axis=1))


def test_geneaJi_known_answer(gen):
    want = exact_case(gen, "geneaJi").astype(np.int64)
    assert np.array_equal(want, JI_OCC)
    assert np.array_equal(want.sum(axis=1), JI_TOTAL)
    assert np.array_equal((want > 0).sum(axis=1), JI_REC)


@pytest.mark.parametrize("K", [63, 64])
def test_sibling_chain_exact_counts(K):
    father, mother, (a, b) = sibling_chain(K)
    O = exact_occ(father, mother, [a, b], [0, 1])
    assert O.tolist() == [[1 << (K - 1)] * 2] * 2
    assert (max(O.ravel()) < SAT) == (K == 63)


def test_front_end_errors_and_empty_lists(gen):
    ped = gen.genealogy(gen.geneaJi)
    with pytest.raises(ValueError):
        gen.occ(ped, typeOcc="MEAN")
    with pytest.raises(ValueError):
        gen.occ_arrays(ped.father, ped.mother, [0], [20], typeOcc="ind")
    with pytest.raises(KeyError):
        gen.occ(ped, [1, 999])
    with pytest.raises(KeyError):
        gen.rec(ped, [1], [17, 999])
    with pytest.raises(KeyError):
        gen.occ_arrays(ped.father, ped.mother, [0], [len(ped.ids)], typeOcc="TOTAL")
    father, mother = ped.father.copy(), ped.mother.copy()
    father[3] = 10                                  # a parent after its child
    for call in (lambda: gen.occ_arrays(father, mother, [0], [20]), lambda: gen.rec_arrays(father, mother, [0], [20])):
        with pytest.raises(gen.GenlibError) as e:
            call()
        assert e.value.status == 3 and "rank 3" in str(e.value)  # GENLIB_EORDER, the first offending rank
    for got, shape in ((gen.occ(ped, [], [17, 19]), (2, 0)), (gen.occ(ped, [1, 2], []), (0, 2)),
                       (gen.occ(ped, [], [17, 19], typeOcc="TOTAL"), (2, 1)), (gen.occ(ped, [1], [], typeOcc="TOTAL"), (0, 1)),
                       (gen.rec(ped, [], [17, 19]), (2,)), (gen.rec(ped, [1, 2], []), (0,))):
        assert got.shape == shape and got.dtype == np.int64 and not got.any()
    assert issubclass(gen.GenlibOverflowError, gen.GenlibError) and issubclass(gen.GenlibOverflowError, OverflowError)


def test_no_cpu_fallback(gen):
    if gen.lib().genlib_device_count() > 0:
        pytest.skip("a CUDA device is present")
    ped = gen.genealogy(gen.geneaJi)
    for call in (lambda: gen.occ(ped), lambda: gen.occ(ped, typeOcc="TOTAL"), lambda: gen.rec(ped)):
        with pytest.raises(gen.GenlibError) as e:
            call()
        assert e.value.status == 4                  # GENLIB_ECUDA


# ---- on the GPU ------------------------------------------------------------------------------------------
def _run(gen, what, father, mother, pro, anc, direction, monkeypatch, **kw):
    monkeypatch.setenv("GENLIB_GC_DIRECTION", direction)
    if what == "rec":
        got, stats = gen.rec_arrays(father, mother, pro, anc, **kw)
    else:
        got, stats = gen.occ_arrays(father, mother, pro, anc, typeOcc=what, **kw)
    assert stats["direction"] == direction
    return got, stats


@pytest.mark.gpu
def test_gpu_geneaJi_known_answers(gen, monkeypatch):
    ped = gen.genealogy(gen.geneaJi)
    monkeypatch.delenv("GENLIB_GC_DIRECTION", raising=False)
    got, stats = gen.occ(ped, device=0, return_stats=True)
    assert gen.founder(ped).tolist() == JI_ANC and gen.pro(ped).tolist() == JI_PRO
    assert got.dtype == np.int64 and np.array_equal(got, JI_OCC)
    assert stats["kernel_launches"] == stats["n_layers"] > 0 and stats["ms_kernels"] > 0
    for direction in ("descend", "ascend"):
        monkeypatch.setenv("GENLIB_GC_DIRECTION", direction)
        assert np.array_equal(gen.occ(ped, JI_PRO, JI_ANC), JI_OCC)
        assert np.array_equal(gen.occ(ped, JI_PRO, JI_ANC, typeOcc="TOTAL"), JI_TOTAL[:, None])
        assert np.array_equal(gen.rec(ped, JI_PRO, JI_ANC), JI_REC)
        pro, anc = [29, 1, 29, 2], [26, 17, 20, 17, 23]               # reordered, duplicates kept
        ri, ci = [5, 0, 2, 0, 3], [2, 0, 2, 1]
        want = JI_OCC[np.ix_(ri, ci)]
        assert np.array_equal(gen.occ(ped, pro, anc), want)
        assert np.array_equal(gen.occ(ped, pro, anc, typeOcc="TOTAL"), want.sum(axis=1, keepdims=True))
        assert np.array_equal(gen.rec(ped, pro, anc), (want > 0).sum(axis=1))
        cm, _ = gen.occ_arrays(ped.father, ped.mother, ped.rank_of(pro), ped.rank_of(anc), col_major=True)
        assert cm.flags.f_contiguous and np.array_equal(cm, want)
        o = gen.occ(ped, [1, 17, 29], [17, 19])                        # 17 is both: the empty path counts
        assert o[:, 1].tolist() == [1, 0] and np.array_equal(o[:, [0, 2]], JI_OCC[np.ix_([0, 1], [0, 2])])
        assert gen.rec(ped, [1, 17, 29], [17, 19]).tolist() == [3, 2]


@pytest.mark.gpu
@pytest.mark.parametrize("direction", ["descend", "ascend"])
@pytest.mark.parametrize("case", ["genea140", "random0", "random1", "random2", "ladder", "sibship"])
def test_gpu_equals_the_walk_and_the_exact_counts(gen, case, direction, monkeypatch):
    father, mother, pro, anc = make_case(gen, case)
    want = exact_case(gen, case).astype(np.int64)
    assert np.array_equal(walk_case(gen, case), want)
    got, st = _run(gen, "IND", father, mother, pro, anc, direction, monkeypatch)
    assert np.array_equal(got, want) and st["d2h_bytes"] == got.nbytes
    n_unique = len(np.unique(anc))                                     # the reductions fetch one value each
    tot, st = _run(gen, "TOTAL", father, mother, pro, anc, direction, monkeypatch)
    assert np.array_equal(tot[:, 0], want.sum(axis=1)) and st["d2h_bytes"] == 8 * n_unique
    rec, st = _run(gen, "rec", father, mother, pro, anc, direction, monkeypatch)
    assert np.array_equal(rec, (want > 0).sum(axis=1)) and st["d2h_bytes"] == 8 * n_unique


def _fits(M):
    return max((int(x) for x in M.ravel()), default=0) < SAT


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES)
def test_gpu_identities(gen, case, monkeypatch):
    """descend == ascend bitwise; TOTAL == IND.sum(1); rec == (IND > 0).sum(1); (IND > 0) == (gc.T > 0)."""
    father, mother, pro, anc = make_case(gen, case)
    want = exact_case(gen, case)
    totals = want.sum(axis=1)
    res = {}
    for direction in ("descend", "ascend"):
        if _fits(want):
            res["IND", direction] = _run(gen, "IND", father, mother, pro, anc, direction, monkeypatch)[0]
        else:                                                          # the exact counter predicts the overflow
            with pytest.raises(gen.GenlibOverflowError):
                _run(gen, "IND", father, mother, pro, anc, direction, monkeypatch)
        if max(totals, default=0) < SAT:
            res["TOTAL", direction] = _run(gen, "TOTAL", father, mother, pro, anc, direction, monkeypatch)[0]
        else:
            with pytest.raises(gen.GenlibOverflowError):
                _run(gen, "TOTAL", father, mother, pro, anc, direction, monkeypatch)
        res["rec", direction] = _run(gen, "rec", father, mother, pro, anc, direction, monkeypatch)[0]
        monkeypatch.setenv("GENLIB_GC_DIRECTION", direction)
        res["gc", direction] = gen.gc_arrays(father, mother, pro, anc)[0]
    for what in ("IND", "TOTAL", "rec"):
        if (what, "descend") in res:
            assert np.array_equal(res[what, "descend"], res[what, "ascend"])
    assert np.array_equal(res["rec", "ascend"], (want > 0).sum(axis=1))
    assert np.array_equal(res["gc", "ascend"].T > 0, want > 0)
    if ("IND", "ascend") in res:
        ind = res["IND", "ascend"]
        assert np.array_equal(ind, want.astype(np.int64))
        assert np.array_equal(res["rec", "ascend"], (ind > 0).sum(axis=1))
        assert np.array_equal(ind > 0, res["gc", "ascend"].T > 0)
        if ("TOTAL", "ascend") in res:
            assert np.array_equal(res["TOTAL", "ascend"][:, 0], ind.sum(axis=1))


@pytest.mark.gpu
@pytest.mark.parametrize("direction", ["descend", "ascend"])
def test_gpu_overflow(gen, direction, monkeypatch):
    f63, m63, (a63, b63) = sibling_chain(63)
    got, _ = _run(gen, "IND", f63, m63, [a63], [0, 1], direction, monkeypatch)
    assert got.tolist() == [[1 << 62], [1 << 62]]
    got, _ = _run(gen, "TOTAL", f63, m63, [a63], [0, 1], direction, monkeypatch)
    assert got.tolist() == [[1 << 62], [1 << 62]]
    f64, m64, (a64, b64) = sibling_chain(64)
    for what in ("IND", "TOTAL"):
        with pytest.raises(gen.GenlibOverflowError) as e:
            _run(gen, what, f64, m64, [0, a64, b64], [1, 0], direction, monkeypatch)
        assert isinstance(e.value, OverflowError) and e.value.status == 8
        assert (e.value.ancestor_index, e.value.proband_index) == (0, 1)   # (founder 1, a64): first in list order
    assert _run(gen, "rec", f64, m64, [0, a64, b64], [1, 0], direction, monkeypatch)[0].tolist() == [2, 3]
    for pro in ([a63, a63], [a63, b63]):                              # each entry fits, their sum does not
        got, _ = _run(gen, "IND", f63, m63, pro, [0, 1], direction, monkeypatch)
        assert got.tolist() == [[1 << 62] * 2] * 2
        with pytest.raises(gen.GenlibOverflowError) as e:
            _run(gen, "TOTAL", f63, m63, pro, [0, 1], direction, monkeypatch)
        assert (e.value.ancestor_index, e.value.proband_index) == (0, 0)


@pytest.mark.gpu
def test_gpu_overflow_names_ids(gen):
    father, mother, (a, b) = sibling_chain(64)
    ids = np.arange(1, len(father) + 1, dtype=np.int64) * 10
    ped = gen.genealogy({"ind": ids, "father": np.where(father >= 0, ids[father], 0),
                         "mother": np.where(mother >= 0, ids[mother], 0), "sex": 1 + np.arange(len(ids)) % 2})
    with pytest.raises(OverflowError) as e:
        gen.occ(ped, [int(ids[b])], [20])
    assert "ancestor 20" in str(e.value) and f"proband {int(ids[b])}" in str(e.value)


@pytest.mark.gpu
def test_gpu_devices_and_layout(gen, monkeypatch):
    father, mother, pro, anc = make_case(gen, "random1")
    for direction in ("descend", "ascend"):
        ref = {w: _run(gen, w, father, mother, pro, anc, direction, monkeypatch, device=0)[0] for w in ("IND", "TOTAL", "rec")}
        cm, _ = _run(gen, "IND", father, mother, pro, anc, direction, monkeypatch, device=0, col_major=True)
        assert cm.flags.f_contiguous and np.array_equal(cm, ref["IND"])
        if gen.lib().genlib_device_count() < 2:
            continue
        for w in ("IND", "TOTAL", "rec"):
            two, st = _run(gen, w, father, mother, pro, anc, direction, monkeypatch, devices=[0, 1])
            assert np.array_equal(two, ref[w]) and st["n_dev"] == 2
            if direction == "descend":                                 # a width of 1 over two devices
                w1, _ = _run(gen, w, father, mother, pro, anc[:1], direction, monkeypatch, devices=[0, 1])
                assert np.array_equal(w1, ref[w][:1])
            else:
                w1, _ = _run(gen, w, father, mother, pro[:1], anc, direction, monkeypatch, devices=[0, 1])
                want = ref["IND"][:, :1]
                assert np.array_equal(w1, {"IND": want, "TOTAL": want, "rec": (want > 0).sum(axis=1)}[w])


@pytest.mark.gpu
def test_gpu_c3_full_size(gen, monkeypatch):
    father, mother, pro, anc = _synth_case(gen, "C3", 1.0)
    digests = []
    for direction in ("ascend", "descend"):
        got, _ = _run(gen, "IND", father, mother, pro, anc, direction, monkeypatch)
        digests.append(hashlib.sha256(got.tobytes()).hexdigest())
        tot, st = _run(gen, "TOTAL", father, mother, pro, anc, direction, monkeypatch)
        assert st["d2h_bytes"] == tot.nbytes == 8 * len(anc)
        assert np.array_equal(tot[:, 0], got.sum(axis=1))
        rec, st = _run(gen, "rec", father, mother, pro, anc, direction, monkeypatch)
        assert st["d2h_bytes"] == rec.nbytes
        assert np.array_equal(rec, (got > 0).sum(axis=1))
        del got
    assert digests[0] == digests[1]
