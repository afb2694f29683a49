"""gen.gcGroups: gen.gc summed over groups of probands and/or ancestors (genlib_gc_groups).

CPU: the C entry point's errors and empty lists, the Python mapping's conversion, the grouped schedule against
gen.gc's for singleton groups, and the grouped schedule replayed in NumPy against exact sums.  GPU: the engine
against the known answer, bit for bit against exact sums in both directions and every grouping, a deep pedigree, two
devices, and C3 and C4 at full size."""
import ctypes as C
import math

import numpy as np
import pytest

from test_gc import GENEAJI_FOUNDERS, GENEAJI_GC, GENEAJI_PRO, _synth_case, active_ranks, exact_gc, make_case, replay

EINVAL, EKEY, EORDER, ECUDA = 1, 2, 3, 4
GROUPINGS = ["pro", "anc", "both"]


def hashed_groups(ranks, k):
    """Seeded hashed labels of distinct ranks, renumbered 0 .. G-1 so that every group has a member."""
    h = (np.asarray(ranks, np.int64) * 0x9E3779B1 + 20261022) & 0xFFFFFFFF
    _, index = np.unique(h % min(k, max(len(ranks), 1)), return_inverse=True)
    return index.astype(np.int32), int(index.max()) + 1 if len(index) else 0


def distinct(ranks):
    """The ranks without repeats, in order of first occurrence."""
    _, first = np.unique(ranks, return_index=True)
    return np.asarray(ranks)[np.sort(first)].astype(np.int32)


def grouped_case(father, mother, pro, anc, grouping, k=7, pro_group=None, anc_group=None):
    """(pro, pro_group or None, n_pro_groups, anc, anc_group or None, n_anc_groups): the grouped side(s) made distinct
    and put in hashed groups (or the given ones)."""
    pg = ag = None
    npg = nag = 0
    if grouping in ("pro", "both"):
        pro = distinct(pro)
        pg, npg = hashed_groups(pro, k) if pro_group is None else pro_group
    if grouping in ("anc", "both"):
        anc = distinct(anc)
        ag, nag = hashed_groups(anc, k) if anc_group is None else anc_group
    return pro, pg, npg, anc, ag, nag


def group_sum(m, axis, group, n_groups):
    """Sum the rows (axis 0) or columns (axis 1) of m per group; m is an int64 or object array."""
    if group is None:
        return m
    m = np.moveaxis(m, axis, 0)
    out = np.zeros((n_groups,) + m.shape[1:], m.dtype)
    np.add.at(out, group, m)
    return np.moveaxis(out, 0, axis)


def exact_sums(father, mother, pro, pg, npg, anc, ag, nag):
    """(the sums rounded once to float64, exact): the path counts G * 2^D summed per group as integers (Python ints
    where int64 could overflow) and divided by 2^D once.  Beyond 53 generations G itself is rounded, so the sums are
    math.fsum of the rounded values (exact = False)."""
    G, D = exact_gc(father, mother, pro, anc)
    if D > 53:
        def fs(m, axis, group, n_groups):
            if group is None:
                return m
            m = np.moveaxis(m, axis, 0)
            out = np.array([[math.fsum(m[group == g, j]) for j in range(m.shape[1])] for g in range(n_groups)])
            return np.moveaxis(out.reshape((n_groups,) + m.shape[1:]), 0, axis)
        return fs(fs(G, 0, pg, npg), 1, ag, nag), False
    S = np.ldexp(G, D).astype(np.int64)
    assert np.array_equal(np.ldexp(S.astype(np.float64), -D), G)
    if D + math.log2(max(G.size, 2)) >= 62:
        S = S.astype(object)
    T = group_sum(group_sum(S, 0, pg, npg), 1, ag, nag)
    if T.dtype == object:
        return np.array([[int(x) / (1 << D) for x in row] for row in T], np.float64).reshape(T.shape), True
    return np.ldexp(T.astype(np.float64), -D), True


# ---- the C entry point and the schedule, without a device -------------------------------------------------------

def call(gen, f, m, pro, pg, npg, anc, ag, nag, devices=(-1,), out=None):
    from genlib_jl_b200 import _lib
    f, m = np.ascontiguousarray(f, np.int32), np.ascontiguousarray(m, np.int32)
    arr = lambda x: None if x is None else np.ascontiguousarray(x, np.int32)
    pro, pg, anc, ag = arr(pro), arr(pg), arr(anc), arr(ag)
    dv = np.ascontiguousarray(devices, np.int32)
    out = np.full(64, -7.0) if out is None else out
    st = _lib.GcStats()
    rc = gen.lib().genlib_gc_groups(len(f), _lib.ptr(f), _lib.ptr(m), 0 if pro is None else len(pro), _lib.ptr(pro),
                                    _lib.ptr(pg), npg, 0 if anc is None else len(anc), _lib.ptr(anc), _lib.ptr(ag), nag,
                                    _lib.ptr(out), 0, len(dv), _lib.ptr(dv), C.byref(st))
    return rc, out, st


def last_error(gen):
    return gen.lib().genlib_last_error().decode()


def test_c_entry_point_errors(gen):
    """Every argument error is reported before a device is touched (these run without one)."""
    from genlib_jl_b200 import _lib
    ped = gen.genealogy(gen.geneaJi)
    f, m = ped.father, ped.mother
    pro, anc = ped.rank_of(GENEAJI_PRO), ped.rank_of(GENEAJI_FOUNDERS)
    grp = [0, 0, 1]
    p32, g32, a32, dv = (np.asarray(x, np.int32) for x in (pro, grp, anc, [-1]))
    out = np.zeros(64)

    def raw(n, pro_p, n_pro, npg, anc_p, n_anc, out_p):
        return gen.lib().genlib_gc_groups(n, _lib.ptr(f), _lib.ptr(m), n_pro, pro_p, _lib.ptr(g32), npg, n_anc, anc_p,
                                          None, 0, out_p, 0, 1, _lib.ptr(dv), None)

    P, A = _lib.ptr(p32), _lib.ptr(a32)
    for args in ((len(f), None, 3, 2, A, 6, _lib.ptr(out)),                    # a null list with a size
                 (len(f), P, 3, 2, None, 6, _lib.ptr(out)),
                 (-1, P, 3, 2, A, 6, _lib.ptr(out)),                           # negative sizes
                 (len(f), P, -3, 2, A, 6, _lib.ptr(out)),
                 (len(f), P, 3, -2, A, 6, _lib.ptr(out)),
                 (len(f), P, 3, 2, A, -6, _lib.ptr(out))):
        assert raw(*args) == EINVAL and "null pointer or negative size" in last_error(gen)
    assert raw(len(f), P, 3, 2, A, 6, None) == EINVAL and "out is null" in last_error(gen)
    assert (out == 0).all()
    rc = call(gen, f, m, pro, None, 0, anc, None, 0)[0]                        # neither side grouped
    assert rc == EINVAL and "neither side is grouped" in last_error(gen)
    for bad in ([0, 0, 2], [0, -1, 1]):                                        # a group index out of range
        rc = call(gen, f, m, pro, bad, 2, anc, None, 0)[0]
        assert rc == EINVAL and "group index" in last_error(gen)
    rc = call(gen, f, m, pro, grp, 3, anc, None, 0)[0]                         # group 2 has no member
    assert rc == EINVAL and "has no member" in last_error(gen)
    rc = call(gen, f, m, pro, None, 0, anc, [0, 1, 2, 0, 1, 1], 4)[0]
    assert rc == EINVAL and "ancestor group 3 has no member" in last_error(gen)
    rc = call(gen, f, m, [pro[0], pro[1], pro[0]], grp, 2, anc, None, 0)[0]    # a rank listed twice on a grouped side
    assert rc == EINVAL and "duplicate proband rank" in last_error(gen)
    with pytest.raises(ValueError):
        gen.gc_groups_arrays(f, m, [pro[0], pro[0]], anc, pro_group=[0, 0], n_pro_groups=1)
    assert call(gen, f, m, pro, grp, 2, anc, None, 0, devices=())[0] == EINVAL     # no device
    bad = np.append(pro[:2], len(f))
    assert call(gen, f, m, bad, grp, 2, anc, None, 0)[0] == EKEY               # a rank out of range
    assert call(gen, f, m, pro, None, 0, np.append(anc[:5], -1), [0] * 6, 1)[0] == EKEY
    broken = f.copy()
    broken[1] = len(f) - 1                                                     # a parent after its child
    assert call(gen, broken, m, bad, grp, 2, anc, None, 0)[0] == EORDER        # the broken pedigree is reported first


def test_empty_lists_without_a_device(gen):
    ped = gen.genealogy(gen.geneaJi)
    f, m = ped.father, ped.mother
    anc = ped.rank_of(GENEAJI_FOUNDERS)
    rc, out, st = call(gen, f, m, [], [], 0, anc, None, 0)                     # no proband group: 0 x 6
    assert rc == 0 and (out == -7.0).all() and (st.n_pro, st.n_anc, st.d2h_bytes) == (0, 6, 0)
    rc, out, st = call(gen, f, m, ped.rank_of(GENEAJI_PRO), [0, 0, 1], 2, [], None, 0)   # no ancestor: 2 x 0
    assert rc == 0 and (out == -7.0).all() and (st.n_pro, st.n_anc) == (2, 0)
    rc, out, st = call(gen, f, m, [], None, 0, [], [], 0)
    assert rc == 0 and (st.n_pro, st.n_anc) == (0, 0)
    r = gen.gcGroups(ped, {}, GENEAJI_FOUNDERS)
    assert r.total.shape == (0, 6) and r.mean.shape == (0, 6) and r.cols.tolist() == GENEAJI_FOUNDERS
    r = gen.gcGroups(ped, {1: "a"}, [])
    assert r.total.shape == (1, 0) and r.rows.tolist() == ["a"] and "1 x 0" in repr(r)


def test_no_cpu_fallback(gen):
    if gen.lib().genlib_device_count() > 0:
        pytest.skip("a CUDA device is present")
    ped = gen.genealogy(gen.geneaJi)
    with pytest.raises(gen.GenlibError) as e:
        gen.gcGroups(ped, {1: "a", 2: "a", 29: "b"})
    assert e.value.status == ECUDA


def test_mapping_conversion(gen, monkeypatch):
    """A mapping's IDs are sorted and its labels sorted; a list keeps its order.  (The device call is replaced by a
    recorder.)"""
    from genlib_jl_b200 import engine
    ped = gen.genealogy(gen.geneaJi)
    seen = {}

    def fake(father, mother, pr, an, **kw):
        seen.update(pr=np.asarray(pr), an=np.asarray(an), kw=kw)
        R = len(pr) if kw["pro_group"] is None else kw["n_pro_groups"]
        Cn = len(an) if kw["anc_group"] is None else kw["n_anc_groups"]
        return np.arange(R * Cn, dtype=np.float64).reshape(R, Cn), {}

    monkeypatch.setattr(engine, "gc_groups_arrays", fake)
    r = gen.gcGroups(ped, {29: "south", 2: "north", 1: "south"}, devices=[0, 1])
    assert r.rows.tolist() == ["north", "south"] and r.row_size.dtype == np.int64 and r.row_size.tolist() == [1, 2]
    assert np.array_equal(seen["pr"], ped.rank_of([1, 2, 29])) and seen["kw"]["pro_group"].tolist() == [1, 0, 1]
    assert seen["kw"]["n_pro_groups"] == 2 and seen["kw"]["anc_group"] is None
    assert seen["kw"]["device"] == -1 and seen["kw"]["devices"] == [0, 1]
    assert r.cols.tolist() == gen.founder(ped).tolist() and r.col_size.tolist() == [1] * 6     # default ancestors
    assert np.array_equal(r.mean, r.total / np.array([[1.0], [2.0]]))
    r = gen.gcGroups(ped, None, {26: 3, 17: -1, 19: 3})                        # numeric labels sort as numbers
    assert r.rows.tolist() == gen.pro(ped).tolist() and r.cols.tolist() == [-1, 3] and r.col_size.tolist() == [1, 2]
    assert np.array_equal(seen["an"], ped.rank_of([17, 19, 26])) and seen["kw"]["anc_group"].tolist() == [0, 1, 1]
    r = gen.gcGroups(ped, [29, 1, 29], {17: "x"})                              # a list keeps its order and repeats
    assert r.rows.tolist() == [29, 1, 29] and r.cols.tolist() == ["x"] and np.array_equal(r.mean, r.total)
    with pytest.raises(KeyError):
        gen.gcGroups(ped, {1: "a", 123456789: "b"})
    with pytest.raises(KeyError):
        gen.gcGroups(ped, {1: "a"}, [17, 123456789])
    with pytest.raises(TypeError):
        gen.gcGroups(ped, {1: "a", 2: 2, 29: "a"})
    with pytest.raises(ValueError, match="gen.gc"):
        gen.gcGroups(ped, [1, 2], [17, 19])
    with pytest.raises(ValueError, match="gen.gc"):
        gen.gcGroups(ped)


def test_direction_rule_counts_groups(gen, monkeypatch):
    monkeypatch.delenv("GENLIB_GC_DIRECTION", raising=False)
    ped = gen.genealogy(gen.geneaJi)
    f, m, r = ped.father, ped.mother, ped.rank_of
    pro, anc = r(GENEAJI_PRO), r(GENEAJI_FOUNDERS)
    info = lambda **kw: gen.GcPlan(f, m, pro, anc, **kw).info()
    i = info(pro_group=[0, 0, 0], n_pro_groups=1)                             # 1 group < 6 founders
    assert (i["direction"], i["width"], i["n_pro"], i["n_anc"]) == ("ascend", 1, 1, 6)
    i = info(anc_group=[0, 1, 0, 1, 0, 1], n_anc_groups=2)                    # 2 groups < 3 probands
    assert (i["direction"], i["width"], i["n_pro"], i["n_anc"]) == ("descend", 2, 3, 2)
    i = info(pro_group=[0, 1, 1], n_pro_groups=2, anc_group=[0, 1, 0, 1, 0, 1], n_anc_groups=2)   # a tie descends
    assert (i["direction"], i["width"], i["n_pro"], i["n_anc"]) == ("descend", 2, 2, 2)
    i = gen.GcPlan(f, m, np.concatenate([pro, pro]), anc, anc_group=[0, 1, 2, 3, 4, 0], n_anc_groups=5).info()
    assert (i["direction"], i["width"]) == ("ascend", 3)                      # a list counts its unique entries
    monkeypatch.setenv("GENLIB_GC_DIRECTION", "descend")
    assert info(pro_group=[0, 0, 0], n_pro_groups=1)["direction"] == "descend"
    with pytest.raises(gen.GenlibError) as e:
        gen.GcPlan(f, m, pro, anc, pro_group=[0, 0, 0], n_pro_groups=2)
    assert e.value.status == EINVAL


@pytest.mark.parametrize("direction", ["descend", "ascend"])
@pytest.mark.parametrize("case", ["geneaJi", "genea140", "random0", "ladder"])
def test_singleton_groups_plan_is_the_gc_plan(gen, case, direction, monkeypatch):
    """Groups of one, numbered in list order: the same layers, slots, seeds and inputs as gen.gc's plan."""
    father, mother, pro, anc = make_case(gen, case)
    pro, anc = distinct(pro), distinct(anc)
    monkeypatch.setenv("GENLIB_GC_DIRECTION", direction)
    want = gen.GcPlan(father, mother, pro, anc)
    one_p = (np.arange(len(pro), dtype=np.int32), len(pro))
    one_a = (np.arange(len(anc), dtype=np.int32), len(anc))
    for grouping in GROUPINGS:
        _, pg, npg, _, ag, nag = grouped_case(father, mother, pro, anc, grouping, pro_group=one_p, anc_group=one_a)
        got = gen.GcPlan(father, mother, pro, anc, pro_group=pg, n_pro_groups=npg, anc_group=ag, n_anc_groups=nag)
        drop = lambda i: {k: v for k, v in i.items() if k != "device_bytes"}   # (+ the per-group block)
        assert drop(got.info()) == drop(want.info())
        for a, b in zip(got.layers(), want.layers(), strict=True):
            assert a.keys() == b.keys() and all(np.array_equal(a[k], b[k]) for k in a)


@pytest.mark.parametrize("grouping", GROUPINGS)
@pytest.mark.parametrize("direction", ["descend", "ascend"])
@pytest.mark.parametrize("case", ["geneaJi", "genea140", "random0", "random1", "random2", "ladder", "sibship"])
def test_plan_replay_equals_the_exact_sums(gen, case, direction, grouping, monkeypatch):
    father, mother, pro, anc = make_case(gen, case)
    pro, pg, npg, anc, ag, nag = grouped_case(father, mother, pro, anc, grouping)
    monkeypatch.setenv("GENLIB_GC_DIRECTION", direction)
    plan = gen.GcPlan(father, mother, pro, anc, pro_group=pg, n_pro_groups=npg, anc_group=ag, n_anc_groups=nag)
    info = plan.info()
    assert info["direction"] == direction
    # the column side is propagated per group; the target side keeps a row per member and is summed per group here
    pro_col, anc_col = direction == "ascend", direction == "descend"
    pro_arg = np.arange(npg) if pg is not None and pro_col else pro
    anc_arg = np.arange(nag) if ag is not None and anc_col else anc
    block, rows = replay(plan, pro_arg, anc_arg)
    assert rows == active_ranks(father, mother, pro, anc)
    got = group_sum(block, 0, None if pro_col else pg, npg)
    got = group_sum(got, 1, None if anc_col else ag, nag)
    R, Cn = (len(pro) if pg is None else npg), (len(anc) if ag is None else nag)
    assert got.shape == (R, Cn) and (info["n_pro"], info["n_anc"]) == (R, Cn)
    want, exact = exact_sums(father, mother, pro, pg, npg, anc, ag, nag)
    assert exact and np.array_equal(got, want)


# ---- on the GPU -----------------------------------------------------------------------------------------------------

def gc_groups(gen, father, mother, pro, pg, npg, anc, ag, nag, direction, monkeypatch, **kw):
    monkeypatch.setenv("GENLIB_GC_DIRECTION", direction)
    got, stats = gen.gc_groups_arrays(father, mother, pro, anc, pro_group=pg, n_pro_groups=npg, anc_group=ag,
                                      n_anc_groups=nag, **kw)
    assert stats["direction"] == direction
    R, Cn = got.shape
    assert (stats["n_pro"], stats["n_anc"], stats["d2h_bytes"]) == (R, Cn, 8 * R * Cn)
    assert stats["width"] == ((npg if pg is not None else len(set(pro.tolist()))) if direction == "ascend"
                              else (nag if ag is not None else len(set(anc.tolist()))))
    return got, stats


@pytest.mark.gpu
def test_gpu_geneaJi_known_answer(gen, monkeypatch):
    ped = gen.genealogy(gen.geneaJi)
    want = np.array([[40, 28, 8, 0, 14, 14], [8, 4, 16, 16, 10, 10]], np.float64) / 64
    for direction in ("descend", "ascend"):
        monkeypatch.setenv("GENLIB_GC_DIRECTION", direction)
        r, stats = gen.gcGroups(ped, {1: "a", 2: "a", 29: "b"}, return_stats=True)
        assert stats["direction"] == direction and r.rows.tolist() == ["a", "b"] and r.row_size.tolist() == [2, 1]
        assert r.total.tobytes() == want.tobytes() and r.mean.tobytes() == (want / [[2], [1]]).tobytes()
        assert stats["d2h_bytes"] == 2 * 6 * 8 and stats["kernel_launches"] >= stats["n_layers"] > 0
        one = gen.gcGroups(ped, {i: 0 for i in GENEAJI_PRO})                   # one group: gen.gc's column sums
        assert one.total.tobytes() == GENEAJI_GC.sum(axis=0, keepdims=True).tobytes()
        both = gen.gcGroups(ped, {1: "a", 2: "a", 29: "b"}, {17: 0, 19: 1, 20: 0, 23: 1, 25: 0, 26: 1})
        assert both.total.tobytes() == (np.array([[62, 42], [34, 30]], np.float64) / 64).tobytes()
        # an ID on both sides contributes G[p, p] = 1
        g = gen.gc(ped, [1, 17, 29], [17, 19])
        r = gen.gcGroups(ped, {1: "a", 17: "a", 29: "b"}, [17, 19])
        assert r.total.tobytes() == np.array([g[0] + g[1], g[2]]).tobytes() and r.total[0, 0] == 1 + 20 / 64
        r = gen.gcGroups(ped, [1, 17, 29], {17: "x", 19: "x", 2: "y"})       # 2 reaches no listed proband: zeros
        assert r.total.tobytes() == np.stack([g.sum(axis=1), [0.0, 0.0, 0.0]], axis=1).tobytes()


def synth_groups(gen, name, scale, grouping, k=20):
    """C3 by deme (probands and founders each by their own deme), C4 in seeded hashed groups."""
    s = gen.synth.config(name, scale)
    ped = gen.genealogy(s.as_columns())
    pro, anc = ped.rank_of(s.probands), ped.rank_of(gen.founder(ped))
    by = (lambda r: (np.unique(s.deme[ped.ids[r] - 1], return_inverse=True)[1].astype(np.int32),
                     len(np.unique(s.deme[ped.ids[r] - 1])))) if name == "C3" else (lambda r: hashed_groups(r, k))
    return (ped.father, ped.mother) + grouped_case(ped.father, ped.mother, pro, anc, grouping,
                                                   pro_group=by(pro), anc_group=by(anc))


@pytest.mark.gpu
@pytest.mark.parametrize("grouping", GROUPINGS)
@pytest.mark.parametrize("case", ["genea140", "random0", "random1", "random2", "C3x0.02", "C4x0.004"])
def test_gpu_equals_the_exact_sums(gen, case, grouping, monkeypatch):
    if case.startswith("C"):
        name, scale = case.split("x")
        father, mother, pro, pg, npg, anc, ag, nag = synth_groups(gen, name, float(scale), grouping)
    else:
        father, mother, pro, anc = make_case(gen, case)
        pro, pg, npg, anc, ag, nag = grouped_case(father, mother, pro, anc, grouping)
    want, exact = exact_sums(father, mother, pro, pg, npg, anc, ag, nag)
    assert exact
    for direction in ("descend", "ascend"):
        got, _ = gc_groups(gen, father, mother, pro, pg, npg, anc, ag, nag, direction, monkeypatch)
        assert got.tobytes() == want.tobytes(), (direction, np.abs(got - want).max())
        cm, _ = gc_groups(gen, father, mother, pro, pg, npg, anc, ag, nag, direction, monkeypatch, col_major=True)
        assert cm.flags.f_contiguous and np.array_equal(cm, want)


@pytest.mark.gpu
def test_gpu_deep_pedigree(gen, monkeypatch):
    father, mother, pro, anc = _synth_case(gen, "C5", 0.02)
    for grouping in GROUPINGS:
        pro_, pg, npg, anc_, ag, nag = grouped_case(father, mother, pro, anc, grouping)
        want, exact = exact_sums(father, mother, pro_, pg, npg, anc_, ag, nag)
        assert not exact                                                      # beyond 53 generations
        for direction in ("descend", "ascend"):
            a1, _ = gc_groups(gen, father, mother, pro_, pg, npg, anc_, ag, nag, direction, monkeypatch)
            a2, _ = gc_groups(gen, father, mother, pro_, pg, npg, anc_, ag, nag, direction, monkeypatch)
            assert a1.tobytes() == a2.tobytes()                               # the same bits on a repeat
            np.testing.assert_allclose(a1, want, rtol=1e-12, atol=0)


@pytest.mark.gpu
@pytest.mark.parametrize("grouping", GROUPINGS)
def test_gpu_two_devices_give_the_same_bits(gen, grouping, monkeypatch):
    if gen.lib().genlib_device_count() < 2:
        pytest.skip("needs two GPUs")
    for father, mother, pro, pg, npg, anc, ag, nag in (
            (lambda f, m, p, a: (f, m) + grouped_case(f, m, p, a, grouping))(*make_case(gen, "random1")),
            synth_groups(gen, "C3", 0.02, grouping)):
        for direction in ("descend", "ascend"):
            one, _ = gc_groups(gen, father, mother, pro, pg, npg, anc, ag, nag, direction, monkeypatch, devices=[0])
            two, st = gc_groups(gen, father, mother, pro, pg, npg, anc, ag, nag, direction, monkeypatch,
                                devices=[0, 1])
            assert two.tobytes() == one.tobytes() and st["n_dev"] == 2


@pytest.mark.gpu
def test_gpu_c3_full_size_by_deme(gen, monkeypatch):
    """Probands by deme x all 50 000 founders: every sum equals gen.gc's matrix summed exactly (scaled to int64), and
    every deme's total over the founders is its size."""
    monkeypatch.delenv("GENLIB_GC_DIRECTION", raising=False)
    father, mother, pro, pg, npg, anc, _, _ = synth_groups(gen, "C3", 1.0, "pro")
    got, stats = gen.gc_groups_arrays(father, mother, pro, anc, pro_group=pg, n_pro_groups=npg)
    assert got.shape == (20, len(anc)) and stats["direction"] == "ascend" and stats["width"] == 20
    size = np.bincount(pg, minlength=npg)
    assert all(math.fsum(got[g]) == size[g] for g in range(npg))
    dense, _ = gen.gc_arrays(father, mother, pro, anc)
    D = 40                                                                    # C3 has 20 generations: exact in int64
    for g in range(npg):
        S = np.ldexp(dense[pg == g], D)
        assert np.array_equal(S, np.floor(S))
        want = np.ldexp(S.astype(np.int64).sum(axis=0).astype(np.float64), -D)
        assert got[g].tobytes() == want.tobytes(), g


@pytest.mark.gpu
def test_gpu_c4_full_size_one_device(gen, monkeypatch):
    """100 000 probands in 20 seeded hashed groups x every founder on one device, where gen.gc's matrix (133 GB) does
    not fit: every group's total over the founders is its size."""
    monkeypatch.delenv("GENLIB_GC_DIRECTION", raising=False)
    father, mother, pro, pg, npg, anc, _, _ = synth_groups(gen, "C4", 1.0, "pro")
    got, stats = gen.gc_groups_arrays(father, mother, pro, anc, pro_group=pg, n_pro_groups=npg, devices=[0])
    assert got.shape == (npg, len(anc)) and npg == 20 and len(pro) == 100_000
    size = np.bincount(pg, minlength=npg)
    assert all(math.fsum(got[g]) == size[g] for g in range(npg))
    assert 0 < stats["device_bytes"] < 180e9 and stats["width"] == 20
