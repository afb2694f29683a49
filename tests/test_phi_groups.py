"""gen.phiMeanGroups: mean kinship within and between groups of probands, and of each proband with each group, reduced
on the device from the proband rows each device holds (genlib_phi_groups).  The device result must equal the means of
gen.phi's matrix M (widened to float64, diagonal skipped): bit for bit against exact rationals where every partial sum is
a float64 number, and the same bits on one and two devices."""
import ctypes as C
import math
from fractions import Fraction

import numpy as np
import pytest

from util import ladder_pedigree, random_pedigree

EINVAL, EKEY, EORDER, ECUDA = 1, 2, 3, 4


def same(got, want):
    """Equal as float64 numbers, bit for bit, with NaN exactly where the reference has NaN."""
    got, want = np.asarray(got, np.float64), np.asarray(want, np.float64)
    assert got.shape == want.shape
    nan = np.isnan(want)
    assert np.array_equal(np.isnan(got), nan)
    assert got[~nan].tobytes() == want[~nan].tobytes()


def exact_means(m, index, n_groups):
    """The definition in exact rationals: S[i][g] over j != i in group g, T[h][g] over i in group h, each mean
    divided once and rounded once (float(Fraction) rounds to nearest).  Returns (proband_mean, group_mean)."""
    P, G = len(index), n_groups
    fm = [[Fraction(float(x)) for x in row] for row in np.asarray(m, np.float64)]
    size = np.bincount(index, minlength=G)
    S = [[Fraction(0)] * G for _ in range(P)]
    for i in range(P):
        for j in range(P):
            if j != i:
                S[i][index[j]] += fm[i][j]
    T = [[Fraction(0)] * G for _ in range(G)]
    for i in range(P):
        for g in range(G):
            T[index[i]][g] += S[i][g]
    pm = np.empty((P, G))
    for i in range(P):
        for g in range(G):
            d = size[g] - (index[i] == g)
            pm[i, g] = float(S[i][g] / d) if d else np.nan
    gm = np.empty((G, G))
    for h in range(G):
        for g in range(G):
            a, b = min(h, g), max(h, g)
            d = int(size[a]) * int(size[b]) - (size[a] if a == b else 0)
            gm[h, g] = float(T[a][b] / d) if d else np.nan
    return pm, gm


def fsum_means(m, index, n_groups):
    """The same means with math.fsum (correctly rounded sums) for matrices too large for rationals."""
    m = np.asarray(m, np.float64)
    P, G = len(index), n_groups
    members = [np.flatnonzero(index == g) for g in range(G)]
    pm = np.empty((P, G))
    for i in range(P):
        for g in range(G):
            js = members[g][members[g] != i]
            pm[i, g] = math.fsum(m[i, js]) / len(js) if len(js) else np.nan
    gm = np.empty((G, G))
    for h in range(G):
        for g in range(G):
            blk = m[np.ix_(members[h], members[g])].copy()
            if h == g:
                np.fill_diagonal(blk, 0.0)
            d = len(members[h]) * len(members[g]) - (len(members[h]) if h == g else 0)
            gm[h, g] = math.fsum(blk.ravel()) / d if d else np.nan
    return pm, gm


def assert_multiples_of_2_pow_32(m):
    """The exactness precondition: every kinship a multiple of 2**-32 and at most 1, so every partial sum of fewer
    than 2**20 of them is a float64 number."""
    w = np.asarray(m, np.float64) * 2.0 ** 32
    assert np.array_equal(w, np.floor(w)) and (np.asarray(m) <= 1).all()


def labelled(ids, label):
    return {int(i): label(int(i)) for i in ids}


# ---- the C entry point and the Python conversion, without a device ------------------------------------------------

def call(gen, father, mother, pro, group, n_groups, numerics=0, devices=(-1,), pm=None, gm=None):
    from genlib_jl_b200 import _lib
    father, mother = np.ascontiguousarray(father, np.int32), np.ascontiguousarray(mother, np.int32)
    pro = None if pro is None else np.ascontiguousarray(pro, np.int32)
    group = None if group is None else np.ascontiguousarray(group, np.int32)
    dv = np.ascontiguousarray(devices, np.int32)
    n_pro = 0 if pro is None else len(pro)
    pm = np.full((max(n_pro, 1), max(n_groups, 1)), -7.0) if pm is None else pm
    gm = np.full((max(n_groups, 1), max(n_groups, 1)), -7.0) if gm is None else gm
    st = _lib.Stats()
    rc = gen.lib().genlib_phi_groups(len(father), _lib.ptr(father), _lib.ptr(mother), n_pro, _lib.ptr(pro),
                                     _lib.ptr(group), n_groups, numerics, len(dv), _lib.ptr(dv), _lib.ptr(pm),
                                     _lib.ptr(gm), C.byref(st))
    return rc, pm, gm, st


def test_c_entry_point_errors(gen):
    """Every argument error is reported before a device is touched (these run without one)."""
    from genlib_jl_b200 import _lib
    ped = gen.genealogy(gen.geneaJi)
    f, m = ped.father, ped.mother
    pro = ped.rank_of([1, 2, 29])
    grp = [0, 0, 1]
    p32, g32, dv = (np.asarray(x, np.int32) for x in (pro, grp, [-1]))
    out = np.zeros(9)

    def raw(n, pro_p, grp_p, n_pro, pm_p, gm_p):
        return gen.lib().genlib_phi_groups(n, _lib.ptr(f), _lib.ptr(m), n_pro, pro_p, grp_p, 2, 0, 1, _lib.ptr(dv),
                                           pm_p, gm_p, None)

    for args in ((len(f), None, _lib.ptr(g32), 3, _lib.ptr(out), _lib.ptr(out)),     # a null input with a size
                 (len(f), _lib.ptr(p32), None, 3, _lib.ptr(out), _lib.ptr(out)),
                 (len(f), _lib.ptr(p32), _lib.ptr(g32), 3, None, _lib.ptr(out)),     # a null output
                 (len(f), _lib.ptr(p32), _lib.ptr(g32), 3, _lib.ptr(out), None),
                 (-1, _lib.ptr(p32), _lib.ptr(g32), 3, _lib.ptr(out), _lib.ptr(out)),  # negative sizes
                 (len(f), _lib.ptr(p32), _lib.ptr(g32), -3, _lib.ptr(out), _lib.ptr(out))):
        assert raw(*args) == EINVAL and "null pointer or negative size" in gen.lib().genlib_last_error().decode()
    assert (out == 0).all()
    assert call(gen, f, m, pro, grp, -1)[0] == EINVAL                       # negative n_groups
    assert call(gen, f, m, pro, grp, 2, numerics=2)[0] == EINVAL            # unknown numerics
    assert call(gen, f, m, pro, grp, 2, devices=())[0] == EINVAL            # no device
    assert call(gen, f, m, pro, grp, 2, devices=range(17))[0] == EINVAL     # more than 16
    assert call(gen, f, m, pro, grp, 0)[0] == EINVAL                        # probands without groups
    assert call(gen, f, m, pro, [0, 0, 2], 2)[0] == EINVAL                  # group index out of range
    assert call(gen, f, m, pro, [0, -1, 1], 2)[0] == EINVAL
    rc = call(gen, f, m, pro, [0, 0, 1], 3)[0]                              # group 2 has no proband
    assert rc == EINVAL and "no proband" in gen.lib().genlib_last_error().decode()
    rc = call(gen, f, m, [pro[0], pro[1], pro[0]], grp, 2)[0]               # a rank listed twice
    assert rc == EINVAL and "duplicate" in gen.lib().genlib_last_error().decode()
    with pytest.raises(ValueError):
        gen.phi_groups_arrays(f, m, [pro[0], pro[0]], [0, 0], 1)
    bad = np.append(pro[:2], len(f))
    assert call(gen, f, m, bad, grp, 2)[0] == EKEY                          # a rank out of range
    broken = f.copy()
    broken[1] = len(f) - 1                                                   # a parent after its child
    assert call(gen, broken, m, bad, grp, 2)[0] == EORDER                    # the broken pedigree is reported first


def test_zero_and_one_proband_without_a_device(gen):
    ped = gen.genealogy(gen.geneaJi)
    rc, pm, gm, st = call(gen, ped.father, ped.mother, [], [], 0)
    assert rc == 0 and (pm == -7.0).all() and (gm == -7.0).all() and st.n_unique == 0    # nothing written
    rc, pm, gm, st = call(gen, ped.father, ped.mother, ped.rank_of([29]), [0], 1)
    assert rc == 0 and np.isnan(pm).all() and np.isnan(gm).all() and st.n_unique == 1 and st.d2h_bytes == 0
    r, stats = gen.phiMeanGroups(ped, {29: "b"}, return_stats=True)
    assert r.ids.tolist() == [29] and r.groups.tolist() == ["b"] and r.size.tolist() == [1]
    assert r.mean.shape == (1, 1) and r.proband.shape == (1, 1) and np.isnan(r.mean).all() and np.isnan(r.proband).all()
    assert stats["d2h_bytes"] == 0
    e = gen.phiMeanGroups(ped, {})
    assert len(e.ids) == 0 and len(e.groups) == 0 and e.mean.shape == (0, 0) and e.proband.shape == (0, 0)
    assert e.size.dtype == np.int64 and "0 probands in 0 groups" in repr(e)


def test_mapping_conversion(gen, monkeypatch):
    """Probands are the mapping's IDs sorted, groups its labels sorted; the record carries both and the group sizes.
    (The device call is replaced by a recorder.)"""
    from genlib_jl_b200 import engine
    ped = gen.genealogy(gen.genea140)
    ids = gen.pro(ped)
    seen = {}

    def fake(father, mother, ranks, index, n_groups, **kw):
        seen.update(ranks=np.asarray(ranks), index=np.asarray(index), n_groups=n_groups, kw=kw)
        return np.zeros((len(ranks), n_groups)), np.zeros((n_groups, n_groups)), {}

    monkeypatch.setattr(engine, "phi_groups_arrays", fake)
    picks = [int(ids[k]) for k in (40, 3, 17, 99, 5)]
    groups = {picks[0]: "north", picks[1]: "south", picks[2]: "east", picks[3]: "north", picks[4]: "east"}
    r = gen.phiMeanGroups(ped, groups, numerics="fp64", devices=[0, 1])
    order = sorted(picks)
    assert r.ids.dtype == np.int64 and r.ids.tolist() == order
    assert r.groups.tolist() == ["east", "north", "south"] and r.size.tolist() == [2, 2, 1]
    assert np.array_equal(seen["ranks"], ped.rank_of(order)) and seen["n_groups"] == 3
    assert [r.groups[k] for k in seen["index"]] == [groups[i] for i in order]
    assert seen["kw"] == {"numerics": "fp64", "device": -1, "devices": [0, 1]}
    r = gen.phiMeanGroups(ped, {picks[0]: 3, picks[1]: -1, picks[2]: 3})     # numeric labels sort as numbers
    assert r.groups.tolist() == [-1, 3] and r.size.tolist() == [1, 2]
    with pytest.raises(KeyError):
        gen.phiMeanGroups(ped, {picks[0]: "a", 123456789: "b"})
    with pytest.raises(TypeError):
        gen.phiMeanGroups(ped, {picks[0]: "a", picks[1]: 2, picks[2]: "a"})


def test_synthetic_pedigrees_keep_their_demes(gen):
    s = gen.synth.config("C3", 0.01)
    assert s.deme.shape == s.ind.shape and np.issubdtype(s.deme.dtype, np.integer)
    assert s.deme.min() >= 0 and s.deme.max() < 20 and len(np.unique(s.deme[s.ind.searchsorted(s.probands)])) > 1
    assert (gen.synth.config("C4", 0.001).deme == 0).all()


def test_no_cpu_fallback(gen):
    if gen.lib().genlib_device_count() > 0:
        pytest.skip("a CUDA device is present")
    ped = gen.genealogy(gen.geneaJi)
    with pytest.raises(gen.GenlibError) as e:
        gen.phiMeanGroups(ped, {1: "a", 2: "a", 29: "b"})
    assert e.value.status == ECUDA


# ---- on the device ------------------------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("numerics", ["reference", "fp64"])
def test_geneaJi_known_answer(gen, numerics):
    """From the reference's 3 x 3 matrix (test/runtests.jl:50-52)."""
    ped = gen.genealogy(gen.geneaJi)
    r, stats = gen.phiMeanGroups(ped, {29: "b", 2: "a", 1: "a"}, numerics=numerics, return_stats=True)
    assert r.ids.tolist() == [1, 2, 29] and r.groups.tolist() == ["a", "b"] and r.size.tolist() == [2, 1]
    same(r.mean, [[0.37109375, 0.072265625], [0.072265625, np.nan]])
    same(r.proband, [[0.37109375, 0.072265625], [0.37109375, 0.072265625], [0.072265625, np.nan]])
    assert stats["d2h_bytes"] == 3 * 2 * 8 and stats["n_unique"] == 3


def genea140_labels(ids):
    """Seven groups from a seeded hash of the ID."""
    return labelled(ids, lambda i: f"pop{((i * 0x9E3779B1 + 20261022) & 0xFFFFFFFF) % 7}")


@pytest.mark.gpu
@pytest.mark.parametrize("numerics", ["reference", "fp64"])
def test_genea140_against_exact_rationals(gen, numerics):
    ped = gen.genealogy(gen.genea140)
    groups = genea140_labels(gen.pro(ped))
    r = gen.phiMeanGroups(ped, groups, numerics=numerics)
    assert len(r.groups) == 7 and r.size.sum() == 140
    m = gen.phi(ped, r.ids, numerics=numerics, dtype=np.float32 if numerics == "reference" else np.float64)
    assert_multiples_of_2_pow_32(m)
    index = np.searchsorted(r.groups, [groups[int(i)] for i in r.ids])
    pm, gm = exact_means(m, index, 7)
    same(r.proband, pm)
    same(r.mean, gm)
    assert np.array_equal(r.mean, r.mean.T)


@pytest.mark.gpu
@pytest.mark.parametrize("numerics", ["reference", "fp64"])
def test_one_group_is_phi_mean(gen, numerics):
    """One group: its mean is Engine.phi_mean's (both exact on genea140), every proband's the mean of its row."""
    ped = gen.genealogy(gen.genea140)
    ids = np.sort(gen.pro(ped))
    r = gen.phiMeanGroups(ped, labelled(ids, lambda i: "all"), numerics=numerics)
    eng = gen.Engine(gen.Plan(ped.father, ped.mother, ped.rank_of(ids)), numerics=numerics, device=0)
    try:
        eng.run()
        want = eng.phi_mean()
    finally:
        eng.close()
    same(r.mean, [[want]])
    m = gen.phi(ped, ids, numerics=numerics, dtype=np.float64)
    same(r.proband[:, 0], (m.sum(1) - np.diag(m)) / 139)


def assert_singleton_groups(gen, ped, ids, **kw):
    """Every proband its own group (G = P): off the diagonal the group means are gen.phi's matrix widened, bit for
    bit, and so is every proband's row; the diagonal is NaN."""
    r, stats = gen.phiMeanGroups(ped, labelled(ids, lambda i: i), return_stats=True, **kw)
    m = gen.phi(ped, r.ids, **kw).astype(np.float64)
    np.fill_diagonal(m, np.nan)
    assert r.groups.tolist() == r.ids.tolist()
    same(r.proband, m)
    upper = np.triu(m, 1)                                   # both halves of the group means come from the upper
    same(r.mean, np.where(np.eye(len(m), dtype=bool), np.nan, upper + upper.T))
    P = len(ids)
    assert stats["d2h_bytes"] == P * P * 8
    return stats


@pytest.mark.gpu
def test_every_proband_its_own_group(gen):
    ped = gen.genealogy(gen.genea140)
    assert_singleton_groups(gen, ped, gen.pro(ped))


@pytest.mark.gpu
def test_rows_in_several_staging_blocks(gen):
    """3 000 probands in 3 000 groups: 72 MB of rows, more than one 64 MB staging buffer."""
    s = gen.synth.config("C3", 0.3)
    assert len(s.probands) == 3000 and 3000 * 3000 * 8 > 64 << 20
    assert_singleton_groups(gen, gen.genealogy(s.as_columns()), s.probands, devices=[0])


@pytest.mark.gpu
@pytest.mark.parametrize("seed", [0, 1, 2, 3])
def test_random_pedigrees_against_exact_rationals(gen, seed):
    """Single parents, late founders, unsorted IDs, groups of one to many members."""
    rng = np.random.default_rng(seed)
    cols = random_pedigree(rng, 300, 30, p_single=0.2, p_none=0.05)
    ped = gen.genealogy(cols)
    ids = rng.choice(cols["ind"][100:], 60, replace=False)
    labels = rng.integers(0, 5, len(ids))
    labels[:5] = np.arange(5)
    groups = {int(i): int(g) for i, g in zip(ids, labels)}
    groups[int(ids[5])] = 9                                                  # a group of one
    for numerics, dtype in (("reference", np.float32), ("fp64", np.float64)):
        r = gen.phiMeanGroups(ped, groups, numerics=numerics)
        m = gen.phi(ped, r.ids, numerics=numerics, dtype=dtype)
        index = np.searchsorted(r.groups, [groups[int(i)] for i in r.ids])
        pm, gm = exact_means(m, index, len(r.groups))
        same(r.proband, pm)
        same(r.mean, gm)
        assert np.isnan(r.mean[-1, -1]) and np.isnan(r.proband[list(r.ids).index(int(ids[5])), -1])


def c3_demes(gen, scale):
    s = gen.synth.config("C3", scale)
    return s, gen.genealogy(s.as_columns()), {int(i): int(s.deme[i - 1]) for i in s.probands}


@pytest.mark.gpu
def test_c3_demes_one_and_two_devices(gen):
    s, ped, groups = c3_demes(gen, 0.1)
    one, stats = gen.phiMeanGroups(ped, groups, devices=[0], return_stats=True)
    P, G = len(one.ids), len(one.groups)
    assert G == 20 and stats["d2h_bytes"] == P * G * 8
    m = gen.phi(ped, one.ids)
    index = np.searchsorted(one.groups, [groups[int(i)] for i in one.ids])
    pm, gm = fsum_means(m, index, G)
    np.testing.assert_allclose(one.proband, pm, rtol=1e-12, atol=0)
    np.testing.assert_allclose(one.mean, gm, rtol=1e-12, atol=0)
    assert np.array_equal(one.mean, one.mean.T)
    for h in range(G):                                                       # demes are more related inside
        assert all(one.mean[h, h] > one.mean[h, g] for g in range(G) if g != h), h
    if gen.lib().genlib_device_count() < 2:
        pytest.skip("needs two GPUs")
    two, stats2 = gen.phiMeanGroups(ped, groups, devices=[0, 1], return_stats=True)
    same(two.mean, one.mean)
    same(two.proband, one.proband)
    assert stats2["d2h_bytes"] == P * G * 8


@pytest.mark.gpu
def test_float32_subnormal_kinships_are_summed(gen):
    """A deep ladder: the kinships between its lineages are Float32 subnormals; they are widened, not flushed."""
    cols, probands = ladder_pedigree(70)
    ped = gen.genealogy(cols)
    A_last, B_last, C3 = probands[12], probands[13], probands[9:12]
    groups = labelled(probands, lambda i: "c" if i in C3 else "ab" if i in (A_last, B_last) else "d")
    r = gen.phiMeanGroups(ped, groups)
    m = gen.phi(ped, r.ids)
    tiny = np.finfo(np.float32).tiny
    assert ((m > 0) & (m < tiny)).any()
    index = np.searchsorted(r.groups, [groups[int(i)] for i in r.ids])
    pm, gm = fsum_means(m, index, len(r.groups))
    np.testing.assert_allclose(r.proband, pm, rtol=1e-12, atol=0)
    np.testing.assert_allclose(r.mean, gm, rtol=1e-12, atol=0)
    c, ab = list(r.groups).index("c"), list(r.groups).index("ab")
    rows = [list(r.ids).index(int(i)) for i in C3]
    assert (r.proband[rows, ab] > 0).all() and (r.proband[rows, ab] < tiny).all()
    assert 0 < r.mean[c, ab] < tiny


@pytest.mark.gpu
def test_restart_path_gives_the_same_bits(gen, monkeypatch):
    """GENLIB_STREAM_SLACK_PCT < 0: the streamed plan's bounds do not hold and the call starts over on the finished plan."""
    s, ped, groups = c3_demes(gen, 0.03)
    want = gen.phiMeanGroups(ped, groups)
    monkeypatch.setenv("GENLIB_STREAM_SLACK_PCT", "-40")
    got = gen.phiMeanGroups(ped, groups)
    monkeypatch.delenv("GENLIB_STREAM_SLACK_PCT")
    same(got.mean, want.mean)
    same(got.proband, want.proband)
