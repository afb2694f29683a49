"""gen.gc: the proband x ancestor genetic-contribution matrix.

CPU: the schedule (genlib_gc_plan_*) replayed in NumPy against exact path counts, the reference's gene drop
(restated below) against the same, and the front end's errors.  GPU: the engine against the known answer,
the gene drop and the exact values, in both directions, on one and several devices."""
import ctypes as C
import hashlib
import numpy as np
import pytest

from util import ladder_pedigree, random_pedigree

# gen.gc(geneaJi) with pro = [1, 2, 29], ancestors = founder = [17, 19, 20, 23, 25, 26]: an exact-rational
# evaluation of G[p, a] = [p == a] + 1/2 G[father(p), a] + 1/2 G[mother(p), a]
GENEAJI_PRO = [1, 2, 29]
GENEAJI_FOUNDERS = [17, 19, 20, 23, 25, 26]
GENEAJI_GC = np.array([[20, 14, 4, 0, 7, 7], [20, 14, 4, 0, 7, 7], [8, 4, 16, 16, 10, 10]], np.float64) / 64


def exact_gc(father, mother, pro_ranks, anc_ranks):
    """(G correctly rounded to float64, D) by path counting in integers, independent
    of the engine's halving sums: S = G * 2^D with D = the pedigree's depth, S[i] = 2^D [i listed] + (sum of
    S over the neighbours on the other side) / 2 -- every term of S is a multiple of 4 there, so the halving is
    exact.  Propagates over whichever list has fewer unique entries.  While D <= 53 no path is longer than
    52 edges and G is exactly a float64."""
    father, mother = np.asarray(father), np.asarray(mother)
    n = len(father)
    depth = np.ones(n, np.int64)
    for i in range(n):
        if father[i] >= 0:
            depth[i] = max(depth[i], depth[father[i]] + 1)
        if mother[i] >= 0:
            depth[i] = max(depth[i], depth[mother[i]] + 1)
    D = int(depth.max()) if n else 1
    dt = np.int64 if D <= 60 else object
    pro_u, pro_pos = np.unique(pro_ranks, return_inverse=True)
    anc_u, anc_pos = np.unique(anc_ranks, return_inverse=True)
    one = (1 << D) if dt is object else np.int64(1) << D
    if len(anc_u) <= len(pro_u):              # down the generations, one column per ancestor
        col = {int(a): k for k, a in enumerate(anc_u)}
        S = np.zeros((n, len(anc_u)), dt)
        for i in range(n):
            acc = np.zeros(len(anc_u), dt)
            if father[i] >= 0:
                acc = acc + S[father[i]]
            if mother[i] >= 0:
                acc = acc + S[mother[i]]
            S[i] = acc // 2
            if i in col:
                S[i, col[i]] += one
        M = S[pro_u][pro_pos][:, anc_pos]
    else:                                     # up the generations, one column per proband
        col = {int(p): k for k, p in enumerate(pro_u)}
        S = np.zeros((n, len(pro_u)), dt)
        for c in range(n - 1, -1, -1):
            S[c] = S[c] // 2
            if c in col:
                S[c, col[c]] += one
            if father[c] >= 0:
                S[father[c]] = S[father[c]] + S[c]
            if mother[c] >= 0:
                S[mother[c]] = S[mother[c]] + S[c]
        M = S[anc_u][anc_pos][:, pro_pos].T
    if dt is object:                          # int / int is correctly rounded
        return np.array([[int(x) / (1 << D) for x in row] for row in M], np.float64).reshape(M.shape), D
    return np.ldexp(M.astype(np.float64), -D), D


def gene_drop(father, mother, pro_ranks, anc_ranks):
    """gen.gc by the reference's algorithm as SURVEY.md 2 describes it (compute.jl:518-595, `_contribute!`):
    for every ancestor a recursive walk down the `children` lists (children in rank order), adding 0.5^depth
    to G[p, a] whenever the walk reaches proband p -- one visit per descent path, duplicates of either list
    kept.  Row-major len(pro) x len(ancestors) Float64; the checker, not the engine's algorithm."""
    n = len(father)
    children = [[] for _ in range(n)]
    for c in range(n):
        for par in (int(father[c]), int(mother[c])):
            if par >= 0:
                children[par].append(c)
    pushed = [tuple(reversed(ch)) for ch in children]         # popped in rank order
    rows = {}
    for t, p in enumerate(pro_ranks):
        rows.setdefault(int(p), []).append(t)
    out = np.zeros((len(pro_ranks), len(anc_ranks)), np.float64)
    for j, a in enumerate(anc_ranks):
        stack = [(int(a), 0)]
        while stack:
            i, d = stack.pop()
            for t in rows.get(i, ()):
                out[t, j] += 0.5 ** d
            stack.extend((c, d + 1) for c in pushed[i])
    return out


_GENE_DROP = {}


def gene_drop_case(gen, name):
    if name not in _GENE_DROP:
        _GENE_DROP[name] = gene_drop(*make_case(gen, name))
    return _GENE_DROP[name]


def replay(plan, n_pro_list, anc_list):
    """Run the schedule in NumPy on a frontier poisoned with NaN; returns (G, checks)."""
    info = plan.info()
    W, cap = info["width"], info["capacity"]
    desc = info["direction"] == "descend"
    tgt_list, col_list = (n_pro_list, anc_list) if desc else (anc_list, n_pro_list)
    tgt_uid = first_order(tgt_list)
    n_tgt = len(set(tgt_list.tolist()))
    F = np.full((max(cap, 1), W), np.nan)
    O = np.full((n_tgt, W), np.nan)
    seen, inputs, slotted, out_rows, max_slot = [], 0, 0, 0, -1
    for L in plan.layers():
        rows, ptr_, ins = L["row_ind"], L["in_ptr"], L["in_slot"]
        acc = np.zeros((len(rows), W))
        fan = np.diff(ptr_)
        for k in range(int(fan.max()) if len(fan) else 0):    # ((0 + in_1) + in_2) + ...
            r = np.nonzero(fan > k)[0]
            acc[r] = acc[r] + F[ins[ptr_[r] + k]]
        v = 0.5 * acc
        s = np.nonzero(L["row_seed"] >= 0)[0]
        v[s, L["row_seed"][s]] += 1.0
        written = L["row_slot"][L["row_slot"] >= 0]
        assert len(set(written.tolist())) == len(written), "two rows of a layer share a slot"
        assert not set(written.tolist()) & set(ins.tolist()), "a slot is written while the layer reads it"
        F[written] = v[L["row_slot"] >= 0]
        o = L["row_out"] >= 0
        assert not np.isfinite(O[L["row_out"][o]]).any(), "an output row is written twice"
        O[L["row_out"][o]] = v[o]
        seen.extend(rows.tolist())
        inputs += len(ins); slotted += len(written); out_rows += int(o.sum())
        max_slot = max(max_slot, int(written.max()) if len(written) else -1)
    if out_rows < n_tgt:                       # targets no path reaches read 0 (the engine zeroes the block)
        O[~np.isfinite(O).all(axis=1)] = 0.0
    assert len(seen) == len(set(seen)) == info["rows"], "a row is computed twice"
    assert inputs == info["inputs"] and cap == max_slot + 1
    assert info["alg_bytes"] == (inputs + slotted + out_rows) * W * 8
    G = O[tgt_uid][:, first_order(col_list)]
    return (G if desc else G.T), sorted(seen)


def first_order(lst):
    """Replace every entry by the position of its first occurrence (unique numbering by first occurrence)."""
    first = {}
    return np.array([first.setdefault(int(x), len(first)) for x in lst], np.int64)


def active_ranks(father, mother, pro_ranks, anc_ranks):
    n = len(father)
    down, up = np.zeros(n, bool), np.zeros(n, bool)
    down[anc_ranks] = True
    up[pro_ranks] = True
    for i in range(n):
        down[i] |= (father[i] >= 0 and down[father[i]]) or (mother[i] >= 0 and down[mother[i]])
    for i in range(n - 1, -1, -1):
        if up[i]:
            if father[i] >= 0:
                up[father[i]] = True
            if mother[i] >= 0:
                up[mother[i]] = True
    return sorted(np.nonzero(down & up)[0].tolist())


# ---- cases: (father, mother, pro ranks, ancestor ranks) ---------------------------------------------------
def _ped_case(gen, cols, pro_ids=None, anc_ids=None):
    ped = gen.genealogy(cols)
    p = gen.pro(ped) if pro_ids is None else pro_ids
    a = gen.founder(ped) if anc_ids is None else anc_ids
    return ped.father, ped.mother, ped.rank_of(p), ped.rank_of(a)


def _random_case(gen, seed):
    rng = np.random.default_rng(seed)
    cols = random_pedigree(rng, 300, 30, window=60 if seed % 2 else 0)
    ped = gen.genealogy(cols)
    n = len(ped.ids)
    pro = rng.choice(n, 25, replace=False)
    anc = rng.choice(n, 20, replace=False)                    # any individuals, not only founders
    pro = np.concatenate([pro, pro[:3], anc[:2]])            # duplicates and IDs in both lists
    anc = np.concatenate([anc, anc[:2], pro[3:5]])
    return ped.father, ped.mother, pro.astype(np.int32), anc.astype(np.int32)


def _sibship_case():
    n = 3002 + 1000
    father = np.full(n, -1, np.int32); mother = np.full(n, -1, np.int32)
    father[3002:] = 0; mother[3002:] = 1
    return father, mother, np.arange(2, n, dtype=np.int32), np.arange(0, 3002, dtype=np.int32)


def _synth_case(gen, name, scale, n_anc=None):
    s = gen.synth.config(name, scale)
    ped = gen.genealogy(s.as_columns())
    anc = gen.founder(ped)
    if n_anc is not None and n_anc < len(anc):
        anc = np.random.default_rng(1).choice(anc, n_anc, replace=False)
    return ped.father, ped.mother, ped.rank_of(s.probands), ped.rank_of(anc)


CASES = ["geneaJi", "genea140", "random0", "random1", "random2", "ladder", "sibship", "C3x0.005", "C5x0.01"]


def make_case(gen, name):
    if name == "geneaJi":
        return _ped_case(gen, gen.geneaJi, GENEAJI_PRO, GENEAJI_FOUNDERS)
    if name == "genea140":
        return _ped_case(gen, gen.genea140)
    if name.startswith("random"):
        return _random_case(gen, int(name[-1]))
    if name == "ladder":
        cols, pro = ladder_pedigree(10)
        return _ped_case(gen, cols, pro)
    if name == "sibship":
        return _sibship_case()
    if name == "C3x0.005":
        return _synth_case(gen, "C3", 0.005)
    if name == "C5x0.01":
        return _synth_case(gen, "C5", 0.01, n_anc=60)
    raise KeyError(name)


@pytest.mark.parametrize("direction", ["descend", "ascend"])
@pytest.mark.parametrize("case", CASES)
def test_plan_replay_equals_the_exact_values(gen, case, direction, monkeypatch):
    father, mother, pro, anc = make_case(gen, case)
    monkeypatch.setenv("GENLIB_GC_DIRECTION", direction)
    plan = gen.GcPlan(father, mother, pro, anc)
    assert plan.info()["direction"] == direction
    got, rows = replay(plan, pro, anc)
    assert rows == active_ranks(father, mother, pro, anc)
    want, depth = exact_gc(father, mother, pro, anc)
    assert got.shape == (len(pro), len(anc))
    if depth <= 53:
        assert np.array_equal(got, want)
    else:                                                     # beyond 52 generations: the order of the sums shows
        assert np.allclose(got, want, rtol=1e-12, atol=0)


def test_direction_rule(gen, monkeypatch):
    monkeypatch.delenv("GENLIB_GC_DIRECTION", raising=False)
    ped = gen.genealogy(gen.geneaJi)
    f, m = ped.father, ped.mother
    r = ped.rank_of
    info = lambda p, a: gen.GcPlan(f, m, r(p), r(a)).info()
    assert info([1, 2, 29], GENEAJI_FOUNDERS)["direction"] == "ascend"                 # 3 < 6
    assert info([1, 2, 29], [17, 19, 20])["direction"] == "descend"                    # a tie descends
    assert info([1, 2, 29, 1, 1, 1], [17, 19, 20, 17])["direction"] == "descend"       # unique entries count
    assert info([1, 2, 29], [17, 19, 20, 23])["width"] == 3
    monkeypatch.setenv("GENLIB_GC_DIRECTION", "descend")
    assert info([1, 2, 29], GENEAJI_FOUNDERS)["direction"] == "descend"
    assert info([1, 2, 29], GENEAJI_FOUNDERS)["width"] == 6


@pytest.mark.parametrize("case", ["geneaJi", "genea140", "random0", "random1", "random2", "ladder"])
def test_gene_drop_equals_the_exact_values(gen, case):
    father, mother, pro, anc = make_case(gen, case)
    got = gene_drop_case(gen, case)
    want, _ = exact_gc(father, mother, pro, anc)
    assert np.array_equal(got, want)
    if case == "geneaJi":
        assert np.array_equal(got, GENEAJI_GC)
    if case == "genea140":                          # no single parents: every proband is all founders
        assert (got.sum(axis=1) == 1.0).all()


def test_front_end_errors_and_empty_lists(gen):
    from genlib_jl_b200 import _lib
    assert C.sizeof(_lib.GcStats) == 104
    ped = gen.genealogy(gen.geneaJi)
    assert gen.gc(ped, [], [17, 19]).shape == (0, 2)
    assert gen.gc(ped, [1, 2], []).shape == (2, 0)
    assert gen.gc(ped, [], []).dtype == np.float64
    with pytest.raises(KeyError):
        gen.gc(ped, [1, 999])
    with pytest.raises(KeyError):
        gen.gc(ped, [1], [17, 999])
    with pytest.raises(KeyError):
        gen.gc_arrays(ped.father, ped.mother, [0], [len(ped.ids)])
    father, mother = ped.father.copy(), ped.mother.copy()
    father[3] = 10                                  # a parent after its child
    with pytest.raises(gen.GenlibError) as e:
        gen.gc_arrays(father, mother, [0], [20])
    assert e.value.status == 3 and "rank 3" in str(e.value)  # GENLIB_EORDER, the first offending rank
    with pytest.raises(gen.GenlibError) as e:
        gen.GcPlan(father, mother, [0], [20])
    assert e.value.status == 3


def test_no_cpu_fallback(gen):
    if gen.lib().genlib_device_count() > 0:
        pytest.skip("a CUDA device is present")
    ped = gen.genealogy(gen.geneaJi)
    with pytest.raises(gen.GenlibError) as e:
        gen.gc(ped)
    assert e.value.status == 4                      # GENLIB_ECUDA


# ---- on the GPU ------------------------------------------------------------------------------------------
def _gc(gen, father, mother, pro, anc, direction, monkeypatch, **kw):
    monkeypatch.setenv("GENLIB_GC_DIRECTION", direction)
    got, stats = gen.gc_arrays(father, mother, pro, anc, **kw)
    assert stats["direction"] == direction
    return got, stats


@pytest.mark.gpu
def test_gpu_geneaJi_known_answer(gen, monkeypatch):
    ped = gen.genealogy(gen.geneaJi)
    monkeypatch.delenv("GENLIB_GC_DIRECTION", raising=False)
    got, stats = gen.gc(ped, device=0, return_stats=True)
    assert got.dtype == np.float64 and np.array_equal(got, GENEAJI_GC)
    assert stats["kernel_launches"] == stats["n_layers"] > 0 and stats["ms_kernels"] > 0
    for direction in ("descend", "ascend"):
        monkeypatch.setenv("GENLIB_GC_DIRECTION", direction)
        assert np.array_equal(gen.gc(ped, GENEAJI_PRO, GENEAJI_FOUNDERS), GENEAJI_GC)
        pro, anc = [29, 1, 29, 2], [26, 17, 20, 17, 23]               # reordered, duplicates kept
        want = GENEAJI_GC[np.ix_([2, 0, 2, 1], [5, 0, 2, 0, 3])]
        assert np.array_equal(gen.gc(ped, pro, anc), want)
        g = gen.gc(ped, [1, 17, 29], [17, 19])                         # 17 is both: 1 at its own entry
        assert g[1].tolist() == [1.0, 0.0] and np.array_equal(g[[0, 2]], GENEAJI_GC[np.ix_([0, 2], [0, 1])])


@pytest.mark.gpu
@pytest.mark.parametrize("direction", ["descend", "ascend"])
def test_gpu_genea140_equals_the_gene_drop(gen, direction, monkeypatch):
    father, mother, pro, anc = make_case(gen, "genea140")
    got, _ = _gc(gen, father, mother, pro, anc, direction, monkeypatch)
    want = gene_drop_case(gen, "genea140")
    assert np.array_equal(got, want)
    assert (got.sum(axis=1) == 1.0).all()


@pytest.mark.gpu
@pytest.mark.parametrize("direction", ["descend", "ascend"])
@pytest.mark.parametrize("case", ["random0", "random1", "random2", "ladder", "sibship"])
def test_gpu_random_pedigrees_equal_the_gene_drop(gen, case, direction, monkeypatch):
    father, mother, pro, anc = make_case(gen, case)
    got, _ = _gc(gen, father, mother, pro, anc, direction, monkeypatch)
    assert np.array_equal(got, gene_drop_case(gen, case))


@pytest.mark.gpu
@pytest.mark.parametrize("name,scale", [("C3", 0.02), ("C4", 0.004)])
def test_gpu_scaled_configs_are_exact(gen, name, scale, monkeypatch):
    father, mother, pro, anc = _synth_case(gen, name, scale)
    want, _ = exact_gc(father, mother, pro, anc)
    for direction in ("descend", "ascend"):
        got, _ = _gc(gen, father, mother, pro, anc, direction, monkeypatch)
        assert np.array_equal(got, want)


@pytest.mark.gpu
def test_gpu_deep_pedigree_within_tolerance(gen, monkeypatch):
    father, mother, pro, anc = _synth_case(gen, "C5", 0.02)
    want, _ = exact_gc(father, mother, pro, anc)
    a1, _ = _gc(gen, father, mother, pro, anc, "ascend", monkeypatch)
    a2, _ = _gc(gen, father, mother, pro, anc, "ascend", monkeypatch)
    d1, _ = _gc(gen, father, mother, pro, anc, "descend", monkeypatch)
    assert np.array_equal(a1, a2)                                     # deterministic
    for got in (a1, d1):
        assert np.allclose(got, want, rtol=1e-12, atol=0)
    assert np.allclose(a1, d1, rtol=1e-12, atol=0)


@pytest.mark.gpu
def test_gpu_devices_dtype_and_layout(gen, monkeypatch):
    father, mother, pro, anc = make_case(gen, "random1")
    for direction in ("descend", "ascend"):
        ref, st = _gc(gen, father, mother, pro, anc, direction, monkeypatch, device=0)
        f32, _ = _gc(gen, father, mother, pro, anc, direction, monkeypatch, device=0, dtype=np.float32)
        assert f32.dtype == np.float32 and np.array_equal(f32, ref.astype(np.float32))
        cm, _ = _gc(gen, father, mother, pro, anc, direction, monkeypatch, device=0, col_major=True)
        assert cm.flags.f_contiguous and np.array_equal(cm, ref)
        assert st["n_dev"] == 1 and st["d2h_bytes"] == ref.nbytes
        if gen.lib().genlib_device_count() >= 2:
            two, st2 = _gc(gen, father, mother, pro, anc, direction, monkeypatch, devices=[0, 1])
            assert np.array_equal(two, ref) and st2["n_dev"] == 2
            if direction == "descend":                                 # a width of 1 over two devices
                w1, _ = _gc(gen, father, mother, pro, anc[:1], direction, monkeypatch, devices=[0, 1])
                assert np.array_equal(w1, ref[:, :1])
            else:
                w1, _ = _gc(gen, father, mother, pro[:1], anc, direction, monkeypatch, devices=[0, 1])
                assert np.array_equal(w1, ref[:1])


@pytest.mark.gpu
def test_gpu_c3_full_size(gen, monkeypatch):
    father, mother, pro, anc = _synth_case(gen, "C3", 1.0)
    digests = []
    for direction in ("ascend", "descend"):
        got, _ = _gc(gen, father, mother, pro, anc, direction, monkeypatch)
        assert (got.sum(axis=1) == 1.0).all()                       # 50 000 founders, no single parents
        digests.append(hashlib.sha256(got.tobytes()).hexdigest())
        del got
    assert digests[0] == digests[1]
