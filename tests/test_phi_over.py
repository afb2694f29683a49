"""gen.phiOver: the proband pairs whose kinship reaches a threshold.  The host form selects from a matrix already in
host memory (GENLIB's phiOver(phiMatrix, threshold)); the device form (genlib_phi_over) runs gen.phi's plan and
layers and selects from the proband rows each device holds, and must give the host form's answer on gen.phi's matrix
bit for bit."""
import ctypes as C

import numpy as np
import pytest

from util import ladder_pedigree

EINVAL, EKEY, EORDER, ECUDA, EOVERFLOW = 1, 2, 3, 4, 8


def assert_same(got, want):
    assert np.array_equal(got.line, want.line) and np.array_equal(got.column, want.column)
    assert np.array_equal(got.pro1, want.pro1) and np.array_equal(got.pro2, want.pro2)
    assert got.kinship.dtype == want.kinship.dtype and got.kinship.tobytes() == want.kinship.tobytes()


# ---- the host form, on hand-made matrices ---------------------------------------------------------------------

def test_host_form_strict_upper_triangle_order_and_equality(gen):
    """(i, j) with i < j and M[i, j] >= t, ordered by i then j; the diagonal and the lower triangle are never read;
    an entry equal to the threshold is selected."""
    m = np.array([[0.50, 0.25, 0.00, 0.125],
                  [0.90, 0.50, 0.125, 0.0625],
                  [0.90, 0.90, 0.75, 0.25],
                  [0.90, 0.90, 0.90, 0.50]], np.float32)
    r = gen.phiOver(m, 0.125)
    assert r.line.tolist() == [0, 0, 1, 2] and r.column.tolist() == [1, 3, 2, 3]
    assert r.kinship.dtype == np.float32 and r.kinship.tolist() == [0.25, 0.125, 0.125, 0.25]
    assert r.pro1.tolist() == r.line.tolist() and r.pro2.tolist() == r.column.tolist() and len(r) == 4
    assert "4 pairs" in repr(r)
    assert len(gen.phiOver(m, 0.5)) == 0                          # only diagonal / lower entries reach 0.5
    rng = np.random.default_rng(0)
    a = rng.choice(np.array([0, 2.0 ** -6, 2.0 ** -4, 2.0 ** -3, 0.3], np.float64), (37, 37))
    for t in (0.0, 2.0 ** -6, 2.0 ** -4, 0.29, 0.3):
        r = gen.phiOver(a, t)
        i, j = np.nonzero(np.triu(a >= t, 1))
        assert np.array_equal(r.line, i) and np.array_equal(r.column, j) and np.array_equal(r.kinship, a[i, j])
        assert r.kinship.dtype == np.float64


def test_host_form_special_thresholds(gen):
    m = np.full((5, 5), 0.0, np.float32)
    assert len(gen.phiOver(m, float("inf"))) == 0
    assert len(gen.phiOver(m, float("-inf"))) == 10 and len(gen.phiOver(m, 0.0)) == 10 and len(gen.phiOver(m, -1)) == 10
    with pytest.raises(ValueError):
        gen.phiOver(m, float("nan"))
    with pytest.raises(ValueError):
        gen.phiOver(np.zeros((2, 3)), 0.1)


def test_host_form_compares_float32_widened(gen):
    """A Float32 entry is compared as the binary64 number it is, not against a threshold rounded to Float32, and
    subnormals are not flushed."""
    x = np.float32(0.1)                                           # 0.100000001490116...
    m = np.array([[0.5, x], [x, 0.5]], np.float32)
    assert len(gen.phiOver(m, 0.1)) == 1
    assert len(gen.phiOver(m, float(x))) == 1
    assert len(gen.phiOver(m, np.nextafter(float(x), 1.0))) == 0   # rounds to x in Float32, above x in binary64
    tiny = np.float32(2.0 ** -140)                                # a Float32 subnormal
    m = np.array([[0.5, tiny], [tiny, 0.5]], np.float32)
    assert len(gen.phiOver(m, 2.0 ** -149)) == 1 and len(gen.phiOver(m, 2.0 ** -139)) == 0


def test_host_form_proband_ids(gen):
    """probandIDs name the rows as gen.phi orders them: duplicates collapse onto their first occurrence."""
    m = np.array([[0.5, 0.25, 0.0], [0.25, 0.5, 0.3], [0.0, 0.3, 0.5]])
    r = gen.phiOver(m, 0.2, [17, 5, 17, 9, 5])
    assert r.pro1.tolist() == [17, 5] and r.pro2.tolist() == [5, 9]
    with pytest.raises(ValueError):
        gen.phiOver(m, 0.2, [1, 2])


# ---- the C entry point, without a device -------------------------------------------------------------------------

def call(gen, father, mother, pro, threshold, max_pairs=-1, devices=(-1,)):
    from genlib_jl_b200 import _lib
    father, mother = np.ascontiguousarray(father, np.int32), np.ascontiguousarray(mother, np.int32)
    pro, dv = np.ascontiguousarray(pro, np.int32), np.ascontiguousarray(devices, np.int32)
    out, st = _lib.KinshipPairs(), _lib.Stats()
    rc = gen.lib().genlib_phi_over(len(father), _lib.ptr(father), _lib.ptr(mother), len(pro), _lib.ptr(pro), threshold,
                                   max_pairs, 0, 0, len(dv), _lib.ptr(dv), C.byref(out), C.byref(st))
    n, empty = out.n, not out.row and not out.col and not out.value
    assert gen.lib().genlib_kinship_pairs_free(C.byref(out)) == 0 and out.n == 0 and not out.row
    return rc, n, empty, st


def test_c_entry_point_errors(gen):
    ped = gen.genealogy(gen.geneaJi)
    pro = ped.rank_of(gen.pro(ped))
    rc, n, empty, _ = call(gen, ped.father, ped.mother, pro, float("nan"))
    assert rc == EINVAL and n == 0 and empty and "NaN" in gen.lib().genlib_last_error().decode()
    bad = np.append(pro, len(ped.father))
    assert call(gen, ped.father, ped.mother, bad, 0.1)[0] == EKEY
    broken = ped.father.copy()
    broken[1] = len(ped.father) - 1                               # a parent after its child
    assert call(gen, broken, ped.mother, bad, 0.1)[0] == EORDER   # the broken pedigree is reported first
    assert gen.lib().genlib_kinship_pairs_free(None) == 0


def test_c_entry_point_fewer_than_two_probands(gen):
    """One distinct proband (listed twice) or none: n = 0, nothing allocated, no device needed."""
    ped = gen.genealogy(gen.geneaJi)
    for pro in ([], [3], [3, 3]):
        rc, n, empty, st = call(gen, ped.father, ped.mother, pro, 0.0, max_pairs=0)
        assert rc == 0 and n == 0 and empty and st.n_unique == len(set(pro))
    r, stats = gen.phiOver(ped, -1.0, [gen.pro(ped)[0]] * 3, return_stats=True)
    assert len(r) == 0 and r.kinship.dtype == np.float32 and stats["d2h_bytes"] == 0
    with pytest.raises(KeyError):
        gen.phiOver(ped, 0.1, [1, 123456789])
    with pytest.raises(ValueError):
        gen.phiOver(ped, float("nan"))


def test_no_cpu_fallback(gen):
    if gen.lib().genlib_device_count() > 0:
        pytest.skip("a CUDA device is present")
    ped = gen.genealogy(gen.geneaJi)
    rc, n, empty, _ = call(gen, ped.father, ped.mother, ped.rank_of(gen.pro(ped)), 0.1)
    assert rc == ECUDA and n == 0 and empty
    with pytest.raises(gen.GenlibError) as e:
        gen.phiOver(ped, 0.1)
    assert e.value.status == ECUDA


# ---- on the device: gen.phiOver(ped, ...) == gen.phiOver(gen.phi(ped, ...), ...) -----------------------------------

def against_matrix(gen, ped, ids, thresholds, numerics="reference", dtype=np.float32, **kw):
    """Every threshold on the device against the host form on gen.phi's matrix; returns the device results.  Only the
    per-row counts and the pairs were copied back."""
    ids = gen.pro(ped) if ids is None else ids
    m = gen.phi(ped, ids, numerics=numerics, dtype=dtype)
    out = []
    for t in thresholds:
        got, stats = gen.phiOver(ped, t, ids, numerics=numerics, dtype=dtype, return_stats=True, **kw)
        assert_same(got, gen.phiOver(m, t, ids))
        assert stats["d2h_bytes"] == 8 * m.shape[0] + len(got) * (4 + np.dtype(dtype).itemsize)
        out.append(got)
    return out, m


@pytest.mark.gpu
def test_geneaJi_thresholds_present_in_the_matrix(gen):
    ped = gen.genealogy(gen.geneaJi)
    ids = ped.ids
    m = gen.phi(ped, ids)
    vals = np.unique(m[np.triu_indices(len(ids), 1)]).astype(np.float64)
    ts = sorted(set(vals.tolist()) | set(((vals[:-1] + vals[1:]) / 2).tolist()) | {0.0, float(vals.max()) * 2})
    got, _ = against_matrix(gen, ped, ids, ts)
    assert [len(g) for g in got] == sorted([len(g) for g in got], reverse=True) and len(got[-1]) == 0


@pytest.mark.gpu
def test_genea140_from_all_pairs_to_none(gen):
    ped = gen.genealogy(gen.genea140)
    m = gen.phi(ped)
    top = float(m[np.triu_indices(140, 1)].max())
    got, _ = against_matrix(gen, ped, None, [float("-inf"), 0.0, 1 / 64, 1 / 16, top, np.nextafter(top, 1.0), float("inf")])
    assert len(got[0]) == len(got[1]) == 9730 and len(got[-1]) == len(got[-2]) == 0 and len(got[-3]) >= 1
    assert len(got[2]) >= len(got[3])


@pytest.mark.gpu
def test_unsorted_proband_list_with_duplicates(gen):
    ped = gen.genealogy(gen.genea140)
    rng = np.random.default_rng(5)
    pro = gen.pro(ped)
    ids = np.concatenate([rng.permutation(pro), rng.choice(pro, 30)])
    rng.shuffle(ids)
    got, _ = against_matrix(gen, ped, ids, [0.0, 1 / 64, 1 / 16])
    assert len(got[0]) == 9730


@pytest.mark.gpu
@pytest.mark.parametrize("numerics", ["reference", "fp64"])
@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_numerics_and_dtypes(gen, numerics, dtype):
    ped = gen.genealogy(gen.genea140)
    got, _ = against_matrix(gen, ped, None, [1 / 256, 1 / 64, 0.1], numerics=numerics, dtype=dtype)
    assert all(g.kinship.dtype == dtype for g in got)


@pytest.mark.gpu
def test_float32_subnormal_kinships(gen):
    """A deep ladder: kinships across its lineages are Float32 subnormals; a positive threshold below them keeps
    them (no flush to zero on the device)."""
    cols, probands = ladder_pedigree(70)
    ped = gen.genealogy(cols)
    got, m = against_matrix(gen, ped, probands, [2.0 ** -149, 2.0 ** -130, 2.0 ** -126])
    tiny = np.finfo(np.float32).tiny
    assert ((got[0].kinship > 0) & (got[0].kinship < tiny)).any()
    assert len(got[0]) > len(got[2])


@pytest.mark.gpu
def test_c3_one_and_two_devices(gen):
    s = gen.synth.config("C3", 0.1)
    ped = gen.genealogy(s.as_columns())
    ts = [2.0 ** -8, 1 / 64, 1 / 16]
    one, m = against_matrix(gen, ped, s.probands, ts, devices=[0])
    assert len(one[0]) > len(one[1]) > 0
    if gen.lib().genlib_device_count() < 2:
        pytest.skip("needs two GPUs")
    for t, o in zip(ts, one):
        two = gen.phiOver(ped, t, s.probands, devices=[0, 1])
        assert_same(two, o)


@pytest.mark.gpu
def test_max_pairs(gen):
    ped = gen.genealogy(gen.genea140)
    want = gen.phiOver(ped, 1 / 64)
    assert_same(gen.phiOver(ped, 1 / 64, max_pairs=len(want)), want)
    with pytest.raises(gen.GenlibOverflowError) as e:
        gen.phiOver(ped, 1 / 64, max_pairs=len(want) - 1)
    assert e.value.count == len(want) and isinstance(e.value, OverflowError)
    assert str(len(want)) in str(e.value) and "0.015625" in str(e.value)
    with pytest.raises(gen.GenlibOverflowError) as e:
        gen.phiOver(ped, 0.0, max_pairs=0)
    assert e.value.count == 9730
