"""Every launch shape of the layer kernel (csrc/layer_kernel.cuh) that the engine can choose, for every schedule and
element type.

The layer kernel behind gen.phi (Float32 storage and fp64), gen.sparse_phi, gen.f and gen.phi_pairs is launched in a
shape that shape_layer (csrc/engine.cu) picks per layer: strip width sw, couples per producer item ft, producer warps,
gangs, strip buffers, ring stages and CTAs per role.  The kernel branches on all of them.  The GENLIB_* tuning
variables force each of them; the knob sets below reach every branch.

On the CPU, Plan.launch_shape (genlib_plan_launch_shape) shows every layer's shape without a device: each must keep
the kernel's contract (StripArgs), and together they must reach every branch.  On the device, every knob set runs
every case through every entry point, bit for bit against a reference that does not use the kernel: the oracle
(phi, sparse_phi) or the NumPy replay of the same plan (fp64, f, pairs), itself anchored to exact rationals."""
import hashlib
import json
import os

import numpy as np
import pytest

from plan_replay import replay
from test_inbreeding import _sibship, replay_f
from test_phi_pairs import make_pairs, pairs_case, replay_pairs
from util import exact_kinship, ladder_pedigree, random_pedigree

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "default_launch_shapes.json")
CASES = ["C3x0.03", "C5x0.03", "random", "sibship", "ladder"]
SCHEDULES = ["phi", "sparse_phi", "f", "pairs"]
NUMERICS = ["reference", "fp64"]
# (schedule, numerics) of the engines the entry points create: what reaches the device
DEVICE_RUNS = [("phi", "reference"), ("phi", "fp64"), ("sparse_phi", "reference"), ("f", "fp64"), ("pairs", "fp64")]
SMEM_LIMIT = 227 * 1024 - 2048          # dynamic shared memory a CTA may take next to the kernel's static part
PTILE = 128                             # frontier columns per producer tile (kPTile)

# GENLIB_<name>: the tuning variables shape_layer reads
KNOB_SETS = [
    {},
    {"PROD_WARPS": 4},
    {"PROD_WARPS": 8},
    {"MAX_SW": 32},                                      # Float32: the fast transpose at sw 32, four stages
    {"MAX_SW": 32, "FT": 16, "PROD_WARPS": 8},           # ft = sw / 2: the generic transpose, two items per tile
    {"MAX_SW": 16, "PROD_WARPS": 8},
    {"MAX_SW": 16, "FT": 8, "PROD_WARPS": 4},
    {"MAX_SW": 8, "PROD_WARPS": 8},                      # eight couples per item over eight producer warps
    {"GANGS": 1, "CTAS_PER_ROLE": 5},                    # many strips per CTA
    {"GANGS": 8, "MAX_SW": 16},
    {"GANGS": 16, "MAX_SW": 8, "MAX_NBUF": 2},           # nbuf = 2 G
    {"GANGS": 4, "MAX_NBUF": 2, "STAGES": 2},
    {"GANG_ITEMS": 64, "MIN_NBUF": 4},
    {"STAGES": 3, "DISCARD": 0},
    {"STRIP_BUDGET_MB": 16, "MIN_NBUF": 8, "MAX_NBUF": 3},
    {"MAX_NBUF": 2, "CTAS_PER_ROLE": 37},
    {"CTAS_PER_ROLE": 2, "STAGES": 2, "FT": 8},
    # shapes that broke the kernel's contract: a strip width that is not a power of two, an item width that is
    # neither sw nor sw / 2, fewer CTAs than gangs, and (Float64) a ring whose two stages do not fit shared memory
    {"MAX_SW": 48},
    {"MAX_SW": 32, "FT": 24},
    {"CTAS_PER_ROLE": 1, "GANGS": 4},
    {"CTAS_PER_ROLE": 3},
    {"FT": 32},
]


def knob_id(knobs):
    return ",".join(f"{k}={v}" for k, v in knobs.items()) or "defaults"


def set_knobs(monkeypatch, knobs):
    for k in ("MAX_SW", "FT", "PROD_WARPS", "GANGS", "GANG_ITEMS", "STAGES", "MAX_NBUF", "MIN_NBUF", "STRIP_BUDGET_MB",
              "CTAS_PER_ROLE", "DISCARD", "STREAM"):
        monkeypatch.delenv("GENLIB_" + k, raising=False)
    for k, v in knobs.items():
        monkeypatch.setenv("GENLIB_" + k, str(v))


# ---- the cases: pedigrees, what each entry point is asked, the plans (none depends on the knobs) ----------------

class Case:
    def __init__(self, gen, name):
        self.name, ids = name, None
        if name.startswith(("C3x", "C5x")):
            s = gen.synth.config(name[:2], float(name[3:]))
            ped = gen.genealogy(s.as_columns())
            pro = ped.rank_of(s.probands)
        elif name == "random":                       # shallow: deep enough for every knob, exact in binary64 mostly
            rng = np.random.default_rng(41)
            ped = gen.genealogy(random_pedigree(rng, 1500, 20, p_single=0.1, p_none=0.02, window=200))
            pro = ped.rank_of(rng.permutation(ped.ids)[:200])
        elif name == "ladder":                       # one couple per layer, 80 layers, Float32 subnormals
            cols, pro_ids = ladder_pedigree(80)
            ped = gen.genealogy(cols)
            pro = ped.rank_of(pro_ids)
        elif name == "sibship":                      # a 1000-child sibship and 3000 unrelated founders
            ped = None
        else:
            raise KeyError(name)
        if ped is None:
            self.father, self.mother, _ = _sibship()
            self.pro = np.arange(2, len(self.father), dtype=np.int32)
            _, _, self.a, self.b = pairs_case(gen, "sibship")
        else:
            self.father, self.mother, ids = ped.father, ped.mother, ped.ids
            self.pro = np.asarray(pro, np.int32)
            self.a, self.b = make_pairs(self.father, self.mother, n_random=300)
        self.ids = ids
        self.f_ranks = np.arange(len(self.father), dtype=np.int32)
        self.plans = {
            "phi": gen.Plan(self.father, self.mother, self.pro),
            "sparse_phi": gen.Plan(self.father, self.mother, self.pro, schedule="sparse_phi", ids=ids),
            "f": gen.Plan(self.father, self.mother, self.f_ranks, schedule="f"),
            "pairs": gen.Plan.pairs(self.father, self.mother, self.a, self.b),
        }
        self.layers = {k: layer_facts(p) for k, p in self.plans.items()}


def layer_facts(plan, rank=0):
    """Per layer what the shape of `rank` follows from: born, the rank's couples, live rows and live tiles before the
    layer."""
    out = []
    for t in range(plan.n_layers):
        info, flags = plan.layer_info(t), plan.layer_arrays(t)["live_flags"]
        fam_base = plan.layer_shard(t)["fam_base"]
        live = np.nonzero(flags & 1)[0]
        out.append({"n_new": info["n_new"], "n_fam": int(fam_base[rank + 1] - fam_base[rank]),
                    "live_before": info["live_before"], "live_tiles": len(np.unique(live // PTILE))})
    return out


@pytest.fixture(scope="module")
def cases(gen):
    made = {}

    def get(name):
        if name not in made:
            made[name] = Case(gen, name)
        return made[name]
    return get


# ---- the CPU view of the shapes --------------------------------------------------------------------------------

def check_shape(sh, numerics, fact, where):
    """The contract of the layer kernel's StripArgs for one layer's shape."""
    if fact["n_new"] == 0 or fact["n_fam"] == 0:
        assert sh["grid"] == 0 and sh["sw"] == 0, where
        return
    es = 8 if numerics == "fp64" else 4
    sw, ft, G, pw = sh["sw"], sh["ft"], sh["gangs"], sh["prod_warps"]
    assert sw in ((8, 16, 32, 64) if es == 4 else (8, 16, 32)), (where, sh)
    assert ft in (8, 16, 32) and ft in (sw, sw // 2), (where, sh)
    assert pw in (4, 8) and 2 * ft % pw == 0 and ft % pw == 0, (where, sh)
    assert sh["n_strips"] == -(-fact["n_fam"] // sw), (where, sh)
    live_tiles = fact["live_tiles"] if fact["live_before"] > 0 else 0
    assert sh["n_pitems"] == (sw // ft) * live_tiles, (where, sh, fact)
    assert sh["n_citems"] >= 1, (where, sh)
    assert G >= 1 and sh["nbuf"] % G == 0 and 2 * G <= sh["nbuf"] <= 8 * G, (where, sh)
    assert sh["n_prod"] % G == 0 and sh["n_cons"] % G == 0, (where, sh)
    assert (sh["n_prod"] >= G) if sh["n_pitems"] > 0 else sh["n_prod"] == 0, (where, sh)
    assert sh["n_cons"] >= G, (where, sh)
    assert sh["grid"] == max(sh["n_prod"], sh["n_cons"]) > 0, (where, sh)
    assert 2 <= sh["stages"] <= 4, (where, sh)
    assert sh["stages"] * 2 * ft * (PTILE * es + 16) < sh["smem"] <= SMEM_LIMIT, (where, sh)
    assert sh["fast_transpose"] == int(es == 4 and ft == 32 and sw in (32, 64) and sh["n_pitems"] > 0), (where, sh)


def shapes_of(case, schedule, numerics, sm_count=148):
    plan = case.plans[schedule]
    return [plan.launch_shape(t, numerics, sm_count=sm_count) for t in range(plan.n_layers)]


def check_knob_set(cases, sm_count=148):
    """Every layer of every case and schedule, under both numerics, keeps the contract; the shapes that reach the
    device are returned: (element type, stored, shape, layer facts)."""
    ran = []
    for name in CASES:
        c = cases(name)
        for schedule in SCHEDULES:
            for numerics in NUMERICS:
                for t, (sh, fact) in enumerate(zip(shapes_of(c, schedule, numerics, sm_count), c.layers[schedule])):
                    check_shape(sh, numerics, fact, (name, schedule, numerics, t))
                    if (schedule, numerics) in DEVICE_RUNS and sh["grid"] > 0:
                        ran.append(("double" if numerics == "fp64" else "float", schedule == "sparse_phi", sh, fact))
    return ran


@pytest.mark.parametrize("knobs", KNOB_SETS, ids=knob_id)
def test_every_shape_keeps_the_kernel_contract(cases, monkeypatch, knobs):
    """sw a power of two, ft in {sw, sw / 2} and in {8, 16, 32}, producer items (sw / ft) per live tile, nbuf a
    multiple of the gangs in [2 G, 8 G], at least one CTA of each role per gang, a kernel for every layer in which
    the rank has couples, two to four ring stages and shared memory within the limit -- whatever the knobs say."""
    set_knobs(monkeypatch, knobs)
    check_knob_set(cases)


def combos(ran):
    return sorted({(T, stored, sh["sw"], sh["ft"], sh["prod_warps"], sh["gangs"], sh["stages"]) for T, stored, sh, _ in ran})


def test_the_knob_sets_reach_every_branch(cases, monkeypatch):
    """Together, the shapes the knob sets launch on the device take every branch of the kernel."""
    ran = []
    for knobs in KNOB_SETS:
        set_knobs(monkeypatch, knobs)
        ran += check_knob_set(cases)
    flo = [sh for T, _, sh, _ in ran if T == "float"]
    dbl = [sh for T, _, sh, _ in ran if T == "double"]
    need = {
        "Float32 fast transpose, sw 64": any(s["fast_transpose"] and s["sw"] == 64 for s in flo),
        "Float32 fast transpose, sw 32": any(s["fast_transpose"] and s["sw"] == 32 for s in flo),
        "Float32 generic transpose, ft 16": any(s["n_pitems"] and not s["fast_transpose"] and s["ft"] == 16 for s in flo),
        "Float32 generic transpose, ft 8": any(s["n_pitems"] and not s["fast_transpose"] and s["ft"] == 8 for s in flo),
        "Float32 ft = sw / 2": any(s["n_pitems"] and s["ft"] == s["sw"] // 2 and s["sw"] <= 32 for s in flo),
        "Float64 ft 8": any(s["n_pitems"] and s["ft"] == 8 for s in dbl),
        "Float64 ft 16": any(s["n_pitems"] and s["ft"] == 16 for s in dbl),
        "Float64 ft = sw / 2": any(s["n_pitems"] and s["ft"] == s["sw"] // 2 for s in dbl),
        "one gang": any(sh["gangs"] == 1 and sh["n_pitems"] for _, _, sh, _ in ran),
        "two or more gangs": any(sh["gangs"] >= 2 for _, _, sh, _ in ran),
        "eight or more gangs": any(sh["gangs"] >= 8 for _, _, sh, _ in ran),
        "nbuf == 2 G, G > 1": any(sh["gangs"] > 1 and sh["nbuf"] == 2 * sh["gangs"] for _, _, sh, _ in ran),
        "a partial last strip": any(f["n_fam"] % sh["sw"] and sh["n_strips"] > 1 for _, _, sh, f in ran),
        "a single-strip layer": any(sh["n_strips"] == 1 and sh["n_pitems"] for _, _, sh, _ in ran),
        "a consumer-only layer": any(f["live_before"] == 0 for _, _, _, f in ran),
        "more strips than CTAs of a role": any(sh["n_strips"] > 4 * max(sh["n_prod"], 1) for _, _, sh, _ in ran),
    }
    for stages in (2, 3, 4):
        need[f"{stages} ring stages"] = any(sh["stages"] == stages and sh["n_pitems"] for _, _, sh, _ in ran)
    for T, stored, label in (("float", True, "sparse_phi"), ("float", False, "phi Float32"), ("double", False, "Float64")):
        for pw in (4, 8):
            need[f"{label}, {pw} producer warps"] = any(
                t == T and st == stored and sh["prod_warps"] == pw and sh["n_pitems"] for t, st, sh, _ in ran)
    missing = [k for k, hit in need.items() if not hit]
    assert not missing, missing


SHAPE_FIELDS = ["sw", "ft", "prod_warps", "gangs", "nbuf", "stages", "n_strips", "n_pitems", "n_citems", "n_prod",
                "n_cons", "grid", "fast_transpose", "smem"]


def default_shapes(cases):
    """{"case/schedule/numerics": {"layers": count, "sha256": of the JSON list of every layer's fields}}, 148 SMs."""
    out = {}
    for name in CASES:
        for schedule in SCHEDULES:
            for numerics in NUMERICS:
                rows = [[sh[k] for k in SHAPE_FIELDS] for sh in shapes_of(cases(name), schedule, numerics)]
                out[f"{name}/{schedule}/{numerics}"] = {
                    "layers": len(rows), "sha256": hashlib.sha256(json.dumps(rows, separators=(",", ":")).encode()).hexdigest()}
    return out


def test_default_shapes_are_unchanged(cases, monkeypatch):
    """Without knobs every layer of every case gets the shape it had before the knobs were made to give legal shapes
    only (tests/golden/default_launch_shapes.json, 148 SMs): the fix changes no default shape."""
    set_knobs(monkeypatch, {})
    want = json.load(open(GOLDEN))
    got = default_shapes(cases)
    assert sorted(got) == sorted(want)
    assert [k for k in want if got[k] != want[k]] == []


def test_launch_shape_arguments(cases):
    plan = cases("ladder").plans["phi"]
    assert plan.launch_shape(0) == plan.launch_shape(0, "reference", rank=0, sm_count=148)
    for bad in ({"layer": plan.n_layers}, {"layer": -1}, {"layer": 0, "rank": 1}, {"layer": 0, "sm_count": 0}):
        with pytest.raises(Exception):
            plan.launch_shape(bad.pop("layer"), **bad)
    # fewer SMs: fewer CTAs per role, never fewer than one per gang
    for sms in (1, 3, 16):
        for t in range(plan.n_layers):
            sh = plan.launch_shape(t, sm_count=sms)
            assert sh["grid"] <= max(sms, sh["gangs"]) and (sh["grid"] > 0) == (sh["sw"] > 0)


# ---- on the device --------------------------------------------------------------------------------------------

def assert_bits(got, want, where):
    assert got.dtype == want.dtype and got.shape == want.shape, (where, got.dtype, got.shape, want.shape)
    u = np.uint32 if got.dtype == np.float32 else np.uint64
    bad = np.argwhere(got.view(u) != want.view(u))
    assert len(bad) == 0, f"{where}: {len(bad)} of {got.size} entries differ; first at {tuple(bad[0])}: " \
                          f"{got[tuple(bad[0])]!r} vs {want[tuple(bad[0])]!r}"


class References:
    """What each entry point must return, computed once per case without the layer kernel."""

    def __init__(self, ob, c):
        self.phi = ob.phi_ranks(c.father, c.mother, c.pro)[0]
        self.fp64 = replay(c.plans["phi"], "fp64")
        self.sparse_phi = ob.sparse_phi_ranks(c.father, c.mother, c.pro, ids=c.ids)[0]
        self.f = replay_f(c.plans["f"], c.father, c.mother, c.f_ranks)
        self.pairs = replay_pairs(c.plans["pairs"], len(c.a))
        self.exact = None
        if c.name == "random":                       # exact rationals, where every partial sum fits binary64
            ex = exact_kinship(c.father, c.mother)
            rows = np.arange(0, len(c.pro), 7)
            vals = np.array([[ex(int(c.pro[i]), int(c.pro[j])) for j in range(len(c.pro))] for i in rows], object)
            fits = np.vectorize(lambda v: v.denominator.bit_length() <= 50)(vals)
            self.exact = (rows, np.vectorize(float)(vals).astype(np.float64), fits)
            assert fits.mean() > 0.5
            self.check_exact(self.fp64, "replay")

    def check_exact(self, got, where):
        if self.exact is not None:
            rows, vals, fits = self.exact
            assert np.array_equal(got[rows][fits], vals[fits]), f"{where}: differs from the exact kinship"


@pytest.fixture(scope="module")
def refs(cases, ob):
    made = {}

    def get(name):
        if name not in made:
            made[name] = References(ob, cases(name))
        return made[name]
    return get


@pytest.fixture(scope="module")
def sm_count():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def engine_run(gen, plan, numerics, sm_count, where):
    """The Engine on the finished plan; each layer's strip width is what Plan.launch_shape predicts."""
    eng = gen.Engine(plan, numerics)
    try:
        eng.run()
        for t in range(plan.n_layers):
            assert eng.layer_info(t)["strip_width"] == plan.launch_shape(t, numerics, sm_count=sm_count)["sw"], (where, t)
        return eng.fetch(dtype=np.float64 if numerics == "fp64" else np.float32)
    finally:
        eng.close()


@pytest.mark.gpu
@pytest.mark.parametrize("knobs", KNOB_SETS, ids=knob_id)
def test_every_entry_point_under_every_shape(gen, cases, refs, sm_count, monkeypatch, knobs):
    set_knobs(monkeypatch, knobs)
    check_knob_set(cases, sm_count)                  # no shape outside the kernel's contract is launched
    for name in CASES:
        c, want = cases(name), refs(name)
        for numerics, dtype, ref in (("reference", np.float32, want.phi), ("fp64", np.float64, want.fp64)):
            got, _ = gen.phi_arrays(c.father, c.mother, c.pro, numerics=numerics, dtype=dtype)
            assert_bits(got, ref, (name, "phi", numerics, "one call"))
            got = engine_run(gen, c.plans["phi"], numerics, sm_count, (name, "phi", numerics))
            assert_bits(got, ref, (name, "phi", numerics, "engine"))
            if numerics == "fp64":
                want.check_exact(got, (name, "phi fp64"))
        got = engine_run(gen, c.plans["sparse_phi"], "reference", sm_count, (name, "sparse_phi"))
        assert_bits(got, want.sparse_phi, (name, "sparse_phi", "engine"))
        for stream in ("1", "0"):                    # the plan streamed to the device, and made first
            monkeypatch.setenv("GENLIB_STREAM", stream)
            got, _ = gen.f_arrays(c.father, c.mother, c.f_ranks, dtype=np.float64)
            assert_bits(got, want.f, (name, "f", "stream", stream))
            got, _ = gen.phi_pairs_arrays(c.father, c.mother, c.a, c.b)
            assert_bits(got, want.pairs, (name, "pairs", "stream", stream))
        monkeypatch.delenv("GENLIB_STREAM")


@pytest.mark.gpu
@pytest.mark.parametrize("knobs", [{}, {"MAX_SW": 8, "PROD_WARPS": 8}, {"GANGS": 4, "MAX_NBUF": 2, "STAGES": 2}, {"FT": 32}],
                         ids=knob_id)
def test_two_devices_under_forced_shapes(gen, cases, refs, monkeypatch, knobs):
    """gen.f and gen.phi_pairs sharded over two devices (each rank shapes its own couples) give the same bits."""
    if gen.lib().genlib_device_count() < 2:
        pytest.skip("needs two GPUs")
    set_knobs(monkeypatch, knobs)
    for name in ("C3x0.03", "C5x0.03", "random"):
        c, want = cases(name), refs(name)
        for schedule, plan in (("f", gen.Plan(c.father, c.mother, c.f_ranks, world=2, schedule="f")),
                               ("pairs", gen.Plan.pairs(c.father, c.mother, c.a, c.b, world=2))):
            for rank in (0, 1):
                for t, fact in enumerate(layer_facts(plan, rank)):
                    check_shape(plan.launch_shape(t, "fp64", rank=rank), "fp64", fact, (name, schedule, rank, t))
        got, _ = gen.f_arrays(c.father, c.mother, c.f_ranks, dtype=np.float64, devices=[0, 1])
        assert_bits(got, want.f, (name, "f", "two devices"))
        got, _ = gen.phi_pairs_arrays(c.father, c.mother, c.a, c.b, devices=[0, 1])
        assert_bits(got, want.pairs, (name, "pairs", "two devices"))
