"""gen.phiProduct: the proband kinship matrix times a block of vectors, Y = M X, formed on the device from the proband
rows each device holds (genlib_phi_product, genlib_engine_phi_product).  Every result is compared with gen.phi's matrix
M fetched in the same numerics: bit for bit against exact sums where every product and partial sum is a float64
number, within the error bound of a reordered float64 sum elsewhere, and the same bits whatever the number of columns,
devices or entry point."""
import ctypes as C
import math
from fractions import Fraction

import numpy as np
import pytest

from util import ladder_pedigree, random_pedigree

EINVAL, EKEY, EORDER, ECUDA = 1, 2, 3, 4
EPS = 2.0 ** -53


def same(got, want):
    got, want = np.asarray(got, np.float64), np.asarray(want, np.float64)
    assert got.shape == want.shape
    assert got.tobytes() == want.tobytes()


def exact_product(m, X):
    """M X in exact rationals, each entry rounded once to float64, and sum_j |M_ij X_jc| (float64)."""
    m, X = np.asarray(m, np.float64), np.asarray(X, np.float64)
    fm = [[Fraction(float(v)) for v in row] for row in m]
    fx = [[Fraction(float(v)) for v in row] for row in X]
    P, k = X.shape
    Y = np.array([[float(sum(fm[i][j] * fx[j][c] for j in range(P))) for c in range(k)] for i in range(P)]).reshape(P, k)
    return Y, np.abs(m) @ np.abs(X)


def integer_product(m, X):
    """M X for kinships that are multiples of 2**-32 and integer X: exact int64 arithmetic, then one exact scaling."""
    w = np.asarray(m, np.float64) * 2.0 ** 32
    assert np.array_equal(w, np.floor(w)) and (np.asarray(m) <= 1).all()
    Xi = np.asarray(X, np.int64)
    assert np.array_equal(Xi, X) and len(Xi) * max(1, np.abs(Xi).max()) <= 2 ** 21
    Yi = w.astype(np.int64) @ Xi
    assert np.abs(Yi).max() < 2 ** 53
    return Yi.astype(np.float64) / 2.0 ** 32


def documented_order(m, X):
    """M X summed in the documented order: column j into partial j mod 256, ascending j, then in each warp of 32
    partials the tree s[l] += s[l + o] for o = 16, 8, 4, 2, 1, then the eight warps' totals in order.  Exact
    emulation of the device's FMAs when every product M[i, j] X[j][c] is a float64 number."""
    m, X = np.asarray(m, np.float64), np.asarray(X, np.float64)
    P = m.shape[1]
    Y = np.empty((m.shape[0], X.shape[1]))
    for c in range(X.shape[1]):
        prod = m * X[:, c]
        part = np.zeros((m.shape[0], 256))
        for j0 in range(0, P, 256):
            n = min(256, P - j0)
            part[:, :n] = part[:, :n] + prod[:, j0:j0 + n]
        w = part.reshape(-1, 8, 32)
        for o in (16, 8, 4, 2, 1):
            w[:, :, :o] = w[:, :, :o] + w[:, :, o:2 * o]
        t = w[:, 0, 0].copy()
        for u in range(1, 8):
            t = t + w[:, u, 0]
        Y[:, c] = t
    return Y


def within_reordered_sum(Y, want, bound, P, factor=1.0):
    assert np.all(np.abs(np.asarray(Y) - want) <= factor * P * EPS * bound)


# ---- the C entry points and the Python checks, without a device ----------------------------------------------------

def call(gen, father, mother, pro, X, k, numerics=0, devices=(-1,), out=None, diag=None, use_diag=False):
    from genlib_jl_b200 import _lib
    father, mother = np.ascontiguousarray(father, np.int32), np.ascontiguousarray(mother, np.int32)
    pro = None if pro is None else np.ascontiguousarray(pro, np.int32)
    n_pro = 0 if pro is None else len(pro)
    dv = np.ascontiguousarray(devices, np.int32)
    X = None if X is None else np.ascontiguousarray(X, np.float64)
    out = np.full(max(n_pro, 1) * max(k, 1), -7.0) if out is None else out
    diag = (np.full(max(n_pro, 1), -7.0) if use_diag else None) if diag is None else diag
    st = _lib.Stats()
    rc = gen.lib().genlib_phi_product(len(father), _lib.ptr(father), _lib.ptr(mother), n_pro, _lib.ptr(pro), k,
                                      _lib.ptr(X), numerics, len(dv), _lib.ptr(dv), _lib.ptr(out), _lib.ptr(diag),
                                      C.byref(st))
    return rc, out, diag, st


def test_c_entry_point_errors(gen):
    """Every argument error is reported before a device is touched (these run without one)."""
    from genlib_jl_b200 import _lib
    ped = gen.genealogy(gen.geneaJi)
    f, m = ped.father, ped.mother
    pro = np.asarray(ped.rank_of([1, 2, 29]), np.int32)
    X = np.ones((3, 2))
    out = np.zeros(6)
    dv = np.asarray([-1], np.int32)

    def raw(n, pro_p, n_pro, k, x_p, out_p):
        return gen.lib().genlib_phi_product(n, _lib.ptr(f), _lib.ptr(m), n_pro, pro_p, k, x_p, 0, 1, _lib.ptr(dv),
                                            out_p, None, None)

    for args in ((len(f), None, 3, 2, _lib.ptr(X), _lib.ptr(out)),          # a null input with a size
                 (len(f), _lib.ptr(pro), 3, 2, None, _lib.ptr(out)),
                 (len(f), _lib.ptr(pro), 3, 2, _lib.ptr(X), None),          # a null output
                 (-1, _lib.ptr(pro), 3, 2, _lib.ptr(X), _lib.ptr(out)),     # negative sizes
                 (len(f), _lib.ptr(pro), -3, 2, _lib.ptr(X), _lib.ptr(out)),
                 (len(f), _lib.ptr(pro), 3, -1, _lib.ptr(X), _lib.ptr(out))):  # k < 0
        assert raw(*args) == EINVAL and "null pointer or negative size" in gen.lib().genlib_last_error().decode()
    assert (out == 0).all()
    assert gen.lib().genlib_phi_product(len(f), None, _lib.ptr(m), 3, _lib.ptr(pro), 2, _lib.ptr(X), 0, 1, _lib.ptr(dv),
                                        _lib.ptr(out), None, None) == EINVAL   # null parents
    assert call(gen, f, m, pro, X, 2, numerics=2)[0] == EINVAL              # unknown numerics
    assert call(gen, f, m, pro, X, 2, devices=())[0] == EINVAL              # no device
    assert call(gen, f, m, pro, X, 2, devices=range(17))[0] == EINVAL       # more than 16
    rc = call(gen, f, m, [pro[0], pro[1], pro[0]], X, 2)[0]                 # a rank listed twice
    assert rc == EINVAL and "duplicate" in gen.lib().genlib_last_error().decode()
    bad = np.append(pro[:2], len(f))
    assert call(gen, f, m, bad, X, 2)[0] == EKEY                            # a rank out of range
    assert call(gen, f, m, [-1, pro[1], pro[2]], X, 2)[0] == EKEY
    broken = f.copy()
    broken[1] = len(f) - 1                                                   # a parent after its child
    assert call(gen, broken, m, bad, X, 2)[0] == EORDER                      # the broken pedigree is reported first
    # the engine-level call
    y = np.zeros(3)
    assert gen.lib().genlib_engine_phi_product(None, 1, _lib.ptr(X), _lib.ptr(y), None) == EINVAL


def test_nothing_to_compute_needs_no_device(gen):
    ped = gen.genealogy(gen.geneaJi)
    f, m = ped.father, ped.mother
    rc, out, _, st = call(gen, f, m, [], None, 3)                            # no proband
    assert rc == 0 and (out == -7.0).all() and st.n_unique == 0 and st.d2h_bytes == 0
    rc, out, _, st = call(gen, f, m, [], None, 0, use_diag=True)
    assert rc == 0 and st.n_unique == 0
    rc, out, _, st = call(gen, f, m, ped.rank_of([1, 2, 29]), None, 0)      # k == 0 and no diagonal
    assert rc == 0 and (out == -7.0).all() and st.n_unique == 3 and st.d2h_bytes == 0
    broken = f.copy()
    broken[1] = len(f) - 1
    assert call(gen, broken, m, [], None, 0)[0] == EORDER                    # still a checked pedigree
    y = gen.phiProduct(ped, np.zeros((3, 0)), [1, 2, 29])
    assert y.shape == (3, 0)
    e = gen.phiProduct(ped, np.zeros(0), [])
    assert e.shape == (0,)


def test_python_arguments_are_checked_before_any_device_work(gen, monkeypatch):
    from genlib_jl_b200 import engine
    ped = gen.genealogy(gen.genea140)
    ids = gen.pro(ped)
    seen = {}

    def fake(father, mother, ranks, X, **kw):
        seen.update(ranks=np.asarray(ranks), X=np.asarray(X), kw=kw)
        return np.asarray(X) * 2, (np.arange(len(ranks), dtype=np.float64) if kw["diagonal"] else None), {"d2h_bytes": 0}

    monkeypatch.setattr(engine, "phi_product_arrays", fake)
    with pytest.raises(ValueError, match="duplicate"):
        gen.phiProduct(ped, np.ones(3), [int(ids[0]), int(ids[1]), int(ids[0])])
    with pytest.raises(ValueError, match="rows"):
        gen.phiProduct(ped, np.ones(139))                                    # one row short
    with pytest.raises(ValueError, match="rows"):
        gen.phiProduct(ped, np.ones((140, 2, 2)))
    with pytest.raises(KeyError):
        gen.phiProduct(ped, np.ones(2), [int(ids[0]), 123456789])
    assert not seen                                                          # none of these reached the device call
    picks = [int(ids[k]) for k in (40, 3, 17)]
    y = gen.phiProduct(ped, [1, 2, 3], picks, numerics="fp64", devices=[0, 1])
    assert y.shape == (3,) and y.tolist() == [2.0, 4.0, 6.0]                 # 1-D in, 1-D out
    assert np.array_equal(seen["ranks"], ped.rank_of(picks)) and seen["X"].shape == (3, 1)
    assert seen["kw"] == {"numerics": "fp64", "device": -1, "devices": [0, 1], "diagonal": False}
    (y, d), stats = gen.phiProduct(ped, np.ones((140, 4)), return_diagonal=True, return_stats=True)
    assert y.shape == (140, 4) and d.shape == (140,) and "d2h_bytes" in stats
    assert np.array_equal(seen["ranks"], ped.rank_of(ids))                   # probandIDs default to pro(ped)


def test_no_cpu_fallback(gen):
    if gen.lib().genlib_device_count() > 0:
        pytest.skip("a CUDA device is present")
    ped = gen.genealogy(gen.geneaJi)
    with pytest.raises(gen.GenlibError) as e:
        gen.phiProduct(ped, np.ones(3), [1, 2, 29])
    assert e.value.status == ECUDA
    rc = call(gen, ped.father, ped.mother, ped.rank_of([1, 2, 29]), None, 0, use_diag=True)[0]
    assert rc == ECUDA                                                       # k == 0 with the diagonal needs a device


# ---- on the device ------------------------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("numerics", ["reference", "fp64"])
def test_geneaJi_known_answer(gen, numerics):
    """The reference's 3 x 3 matrix (test/runtests.jl:50-52) times small integers: exact."""
    ped = gen.genealogy(gen.geneaJi)
    m = np.array([[0.591796875, 0.37109375, 0.072265625], [0.37109375, 0.591796875, 0.072265625],
                  [0.072265625, 0.072265625, 0.53515625]])                  # test/runtests.jl:51-52
    X = np.array([[1.0, -2.0], [3.0, 0.0], [-5.0, 7.0]])
    (y, d), stats = gen.phiProduct(ped, X, [1, 2, 29], numerics=numerics, return_diagonal=True, return_stats=True)
    same(y, [[0.591796875 + 3 * 0.37109375 - 5 * 0.072265625, -2 * 0.591796875 + 7 * 0.072265625],
             [0.37109375 + 3 * 0.591796875 - 5 * 0.072265625, -2 * 0.37109375 + 7 * 0.072265625],
             [0.072265625 + 3 * 0.072265625 - 5 * 0.53515625, -2 * 0.072265625 + 7 * 0.53515625]])   # (all exact)
    same(y, integer_product(m, X))
    same(d, np.diag(m))
    assert stats["d2h_bytes"] == 3 * 2 * 8 + 3 * 8 and stats["n_unique"] == 3
    same(gen.phiProduct(ped, X[:, 1], [1, 2, 29], numerics=numerics), y[:, 1])


@pytest.mark.gpu
@pytest.mark.parametrize("numerics", ["reference", "fp64"])
def test_genea140_integer_blocks_are_exact(gen, numerics):
    """k = 1, 3, 37, 64, 65: one, several and part of a column block, and a block and one more."""
    ped = gen.genealogy(gen.genea140)
    ids = gen.pro(ped)
    m = gen.phi(ped, ids, numerics=numerics, dtype=np.float32 if numerics == "reference" else np.float64)
    rng = np.random.default_rng(140)
    for k in (1, 3, 37, 64, 65):
        X = rng.integers(-1000, 1001, (len(ids), k)).astype(np.float64)
        (y, d), stats = gen.phiProduct(ped, X, numerics=numerics, return_diagonal=True, return_stats=True)
        same(y, integer_product(m, X))
        same(d, np.diag(m).astype(np.float64))
        assert stats["d2h_bytes"] == 140 * (k + 1) * 8
    eng = gen.Engine(gen.Plan(ped.father, ped.mother, ped.rank_of(ids)), numerics=numerics, device=0)
    try:                                                                     # X = 1: the row sums of the same run
        eng.run()
        y, d = eng.phi_product(np.ones(len(ids)), return_diagonal=True)
        sums = eng.row_sums()
    finally:
        eng.close()
    same(y, sums[:, 0])
    same(d, sums[:, 1])


def check_against_rationals(gen, ped, ids, X, numerics, dtype):
    m = gen.phi(ped, ids, numerics=numerics, dtype=dtype)
    y = gen.phiProduct(ped, X, ids, numerics=numerics)
    want, bound = exact_product(m, X)
    within_reordered_sum(y, want, bound, len(ids))
    w = np.asarray(m, np.float64) * 2.0 ** 32
    if np.array_equal(w, np.floor(w)):                                      # every partial sum a float64 number
        same(y, want)
    return m, y


@pytest.mark.gpu
@pytest.mark.parametrize("seed", [0, 1, 2, 3])
def test_random_pedigrees_against_exact_rationals(gen, seed):
    """Single parents, late founders, unsorted IDs."""
    rng = np.random.default_rng(seed)
    cols = random_pedigree(rng, 300, 30, p_single=0.2, p_none=0.05)
    ped = gen.genealogy(cols)
    ids = rng.choice(cols["ind"][100:], 60, replace=False)
    X = rng.integers(-50, 51, (60, 5)).astype(np.float64)
    for numerics, dtype in (("reference", np.float32), ("fp64", np.float64)):
        check_against_rationals(gen, ped, ids, X, numerics, dtype)


@pytest.mark.gpu
def test_float32_subnormal_kinships_are_multiplied(gen):
    """A deep ladder: the kinships between its lineages are Float32 subnormals; they are widened, not flushed."""
    cols, probands = ladder_pedigree(70)
    ped = gen.genealogy(cols)
    rng = np.random.default_rng(70)
    m = gen.phi(ped, probands)
    tiny = np.finfo(np.float32).tiny
    i, j = np.argwhere((m > 0) & (m < tiny))[0]
    X = rng.integers(1, 9, (len(probands), 3)).astype(np.float64)
    X[:, 2] = 0
    X[j, 2] = 1                                                              # column 2 picks the subnormal M[:, j]
    m, y = check_against_rationals(gen, ped, probands, X, "reference", np.float32)
    assert y[i, 2] == np.float64(m[i, j]) and 0 < y[i, 2] < tiny


def c3(gen, scale):
    s = gen.synth.config("C3", scale)
    return s, gen.genealogy(s.as_columns())


@pytest.mark.gpu
def test_c3_random_normal_against_fsum(gen):
    s, ped = c3(gen, 0.1)
    P = len(s.probands)
    rng = np.random.default_rng(3)
    X = rng.standard_normal((P, 4))
    y = gen.phiProduct(ped, X, s.probands)
    m = gen.phi(ped, s.probands).astype(np.float64)
    for c in range(X.shape[1]):
        prod = m * X[:, c]
        want = np.array([math.fsum(row) for row in prod])
        bound = np.abs(prod).sum(1)
        assert np.all(np.abs(y[:, c] - want) <= P * EPS * bound), c


@pytest.mark.gpu
def test_order_contract(gen):
    """Columns of a 37-column call and 1-column calls, a repeat, and the engine-level call (twice on one engine)
    against the one-shot call: the same bits.  X = 1 on one engine gives Engine.row_sums' sums, through both kernels."""
    s, ped = c3(gen, 0.1)
    P = len(s.probands)
    rng = np.random.default_rng(37)
    X = rng.standard_normal((P, 37))
    (y, d), stats = gen.phiProduct(ped, X, s.probands, devices=[0], return_diagonal=True, return_stats=True)
    assert stats["d2h_bytes"] == P * 38 * 8
    for c in range(37):
        same(gen.phiProduct(ped, X[:, c], s.probands, devices=[0]), y[:, c])
    same(gen.phiProduct(ped, X, s.probands, devices=[0]), y)
    eng = gen.Engine(gen.Plan(ped.father, ped.mother, ped.rank_of(s.probands)), device=0)
    try:
        eng.run()
        e1, ed = eng.phi_product(X, return_diagonal=True)
        e2 = eng.phi_product(X)
        ones = eng.phi_product(np.ones(P))
        ones8 = eng.phi_product(np.ones((P, 8)))                             # (the 8-column kernel)
        sums = eng.row_sums()
    finally:
        eng.close()
    same(e1, y)
    same(e2, y)
    same(ed, d)
    same(ones, sums[:, 0])
    same(ones8, np.repeat(sums[:, :1], 8, axis=1))


@pytest.mark.gpu
def test_the_documented_order_bit_for_bit(gen):
    """X of float32 values and Float32 kinships: every product is a float64 number, so each FMA is one rounding of a
    sum and the host can replay the documented order exactly.  The sums are not exact (another order gives other
    bits), so the one-column and the 8-column kernels must follow that order to match."""
    s, ped = c3(gen, 0.1)
    P = len(s.probands)
    X = np.random.default_rng(5).standard_normal((P, 9)).astype(np.float32).astype(np.float64)
    m = gen.phi(ped, s.probands)
    want = documented_order(m, X)
    assert not np.array_equal(want, np.cumsum(m.astype(np.float64)[:, :, None] * X[None, :, :], 1)[:, -1, :])
    same(gen.phiProduct(ped, X, s.probands), want)
    same(gen.phiProduct(ped, X[:, 4], s.probands), want[:, 4])


@pytest.mark.gpu
def test_one_and_two_devices_give_the_same_bits(gen):
    if gen.lib().genlib_device_count() < 2:
        pytest.skip("needs two GPUs")
    s, ped = c3(gen, 0.1)
    X = np.random.default_rng(37).standard_normal((len(s.probands), 37))
    y, d = gen.phiProduct(ped, X, s.probands, devices=[0], return_diagonal=True)
    y2, d2 = gen.phiProduct(ped, X, s.probands, devices=[0, 1], return_diagonal=True)
    same(y2, y)
    same(d2, d)


@pytest.mark.gpu
def test_rows_in_several_staging_blocks(gen):
    """C3 at full size with k = 1000 (and the diagonal): 80 MB of rows, more than one 64 MB staging buffer."""
    s, ped = c3(gen, 1.0)
    P, k = len(s.probands), 1000
    assert P == 10000 and P * k * 8 > 64 << 20
    rng = np.random.default_rng(1000)
    X = rng.standard_normal((P, k))
    (y, d), stats = gen.phiProduct(ped, X, s.probands, return_diagonal=True, return_stats=True)
    assert stats["d2h_bytes"] == P * (k + 1) * 8
    m = gen.phi(ped, s.probands).astype(np.float64)
    same(d, np.diag(m))
    within_reordered_sum(y, m @ X, m @ np.abs(X), P, factor=2.0)           # (M >= 0: |M| = M)


@pytest.mark.gpu
def test_restart_path_gives_the_same_bits(gen, monkeypatch):
    """GENLIB_STREAM_SLACK_PCT < 0: the streamed plan's bounds do not hold and the call starts over on the finished plan."""
    s, ped = c3(gen, 0.03)
    X = np.random.default_rng(4).standard_normal((len(s.probands), 9))
    want = gen.phiProduct(ped, X, s.probands)
    monkeypatch.setenv("GENLIB_STREAM_SLACK_PCT", "-40")
    got = gen.phiProduct(ped, X, s.probands)
    monkeypatch.delenv("GENLIB_STREAM_SLACK_PCT")
    same(got, want)
