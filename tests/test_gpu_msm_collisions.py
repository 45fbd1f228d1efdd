"""Every reduction path of the MSM on inputs where bucket sums, running sums, window sums and Horner steps collide.

The tails of the bucket method (running sums, group and window sums, the Horner combination, the marginals of the precomputed
path, the block trees of the fixed-base tables) add points that are almost never equal or opposite when the inputs are random.
Here every point is a small multiple m*G (m in 0, +-1..+-16, 2^c) and every scalar is small: |k| < 0.55 * 2^128,
written as k or q - k.  Below about 0.56 * 2^128 the GLV split of glv.cuh rounds both lattice coefficients to zero, so the
k2 half is 0 and the signed c-bit digits are exactly those of k (negated for q - k): the digits, and with them which sums
meet, are chosen by the test.  The exact answer is (sum k_i m_i mod q) * G, one scalar multiplication.

Case kinds: tiny (every bucket a small multiple of G), deep (a few points repeated thousands of times with one scalar: P + P
in the accumulation, buckets over more than 64 and more than 2048 chunks), cancel (result O), spread (random small scalars,
bit 127 set in some), top (bit 127 set: top digits above 2^(c-1) land in the second bucket unit when c divides 128), horner
(the Horner step at window w adds a window sum equal or opposite to the accumulator), units (the two units of the top window
are equal or opposite) and phi (scalars +-s * lambda: k1 = 0, k2 = +-s, so the same collisions happen on the phi sub-terms).
test_case_expectations_match_the_oracle checks every case's closed form and intended collision on the CPU."""
import ctypes
import functools
import os
import random
import re

import pytest

from oracle import ecc
from python_bulletproofs_b200 import _native as nat

Q, P = ecc.Q, ecc.P
gpu = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIMIT = 55 * 2 ** 128 // 100                        # scalars (as k or q - k) stay below this


# ---- the GLV split of glv.cuh, restated on Python ints from the constants in that file -------------------------------------
def _glv_constants():
    with open(os.path.join(ROOT, "python_bulletproofs_b200", "csrc", "glv.cuh")) as f:
        src = f.read()

    def limbs(pattern):
        body = re.search(pattern + r"\s*=?\s*\{\{?([^}]*)\}", src).group(1)
        return sum(int(x.strip().rstrip("u"), 16) << (32 * i) for i, x in enumerate(body.split(",")))
    return {"g1": limbs(r"glv_g1\(\) \{ Fq r"), "g2": limbs(r"glv_g2\(\) \{ Fq r"), "A1": limbs(r"A1\[4\]"),
            "MB1": limbs(r"MB1\[4\]"), "A2": limbs(r"A2\[5\]"), "beta": limbs(r"#define BP_BETA_LIMBS")}


GLV = _glv_constants()
LAMBDA = 0x5363AD4CC05C30E0A5261C028812645A122E22EA20816678DF02967C1B23BD72       # lambda * (x, y) = (beta * x, y)


def glv_split(k):
    """(k1, k2) as glv_split computes them: k = k1 + k2 * lambda (mod q), signed."""
    k %= Q
    c1 = (k * GLV["g1"] + (1 << 383)) >> 384
    c2 = (k * GLV["g2"] + (1 << 383)) >> 384
    return k - c1 * GLV["A1"] - c2 * GLV["A2"], c1 * GLV["MB1"] - c2 * GLV["A1"]


def shape(c):
    """(W, H, dbl) of msm_shape for window c: W windows over 128 bits, H buckets per unit, dbl = the top window owns two units."""
    return -(-128 // c), 1 << (c - 1), int(128 % c == 0)


def digits(mag, c):
    """Signed c-bit digits of a GLV half of magnitude mag, as k_digits recodes them (the top window keeps its digit)."""
    W, H, _ = shape(c)
    out, carry = [], 0
    for w in range(W):
        d = ((mag >> (w * c)) & ((1 << c) - 1)) + carry
        if w + 1 < W and d > H:
            out.append(d - 2 * H); carry = 1
        else:
            out.append(d); carry = 0
    return out


def auto_c(n, nmsm):
    """The window msm_shape picks for nmsm MSMs of n terms each (bp_msm_last_window reports it)."""
    best, bestc = 1, None
    for c in range(1, 17):
        W, H = (128 + c - 1) // c, float(1 << (c - 1))
        if nmsm <= 8:
            pick = 5 if n <= 64 else (10 if n < 1024 else (13 if n <= 65536 else 16))
            cost = 0.0 if c == pick else 1.0
        else:
            cost = 2.0 * n * W * 10 + 2 * W * H * 14 + c * (W - 1) * 9.0 + W * 14
        if bestc is None or cost < bestc:
            best, bestc = c, cost
    return best


def pre_auto_c(n):
    return 13 if n < (1 << 13) else (15 if n < (1 << 15) else (17 if n < (1 << 19) else 18))


# ---- cases -------------------------------------------------------------------------------------------------------------
@functools.lru_cache(maxsize=None)
def _pt(m):
    return ecc.pack_point(ecc.py_mul(ecc.G, m % Q))


class Case:
    """One MSM over points m_i * G with scalars k_i; `event` = the collision the case is built to cause (checked on the CPU)."""

    def __init__(self, name, terms, event=None):
        self.name, self.terms, self.event = name, terms, event
        self.total = sum(k * m for m, k in terms) % Q

    def __len__(self):
        return len(self.terms)

    def __repr__(self):
        return "Case(%s, %d terms)" % (self.name, len(self.terms))

    @property
    def pts(self):
        return b"".join(_pt(m) for m, _ in self.terms)

    @property
    def sc(self):
        return b"".join(k.to_bytes(32, "little") for _, k in self.terms)

    @property
    def want(self):
        return ecc.py_mul(ecc.G, self.total)


def _sgn(rng, v):
    return v % Q if rng.getrandbits(1) else (Q - v) % Q


def _m(rng, top=4):
    return rng.choice([s * i for i in range(1, top + 1) for s in (1, -1)])


def tiny(rng, n):
    return Case("tiny", [(rng.choice([0] + [s * i for i in range(1, 5) for s in (1, -1)]),
                          rng.randrange(8) if rng.getrandbits(1) else Q - rng.randrange(1, 8)) for _ in range(n)])


def spread(rng, n):
    return Case("spread", [(_m(rng, 16), _sgn(rng, rng.randrange(1 << 127, LIMIT) if i % 3 == 0 else rng.randrange(1, 1 << 127)))
                           for i in range(n)])


def top(rng, n):
    return Case("top", [(_m(rng, 16), _sgn(rng, rng.randrange(1 << 127, LIMIT))) for _ in range(n)])


def phi(rng, n):
    return Case("phi", [(_m(rng), _sgn(rng, (rng.randrange(1, 8) if i % 2 else rng.randrange(1, 1 << 20)) * LAMBDA))
                        for i in range(n)])


def deep_len(reps):
    return reps + reps // 4 + reps // 2 + reps // 8 + 1


def deep(rng, reps):
    """Three points with one shared scalar and a fourth with its own, each repeated: deep buckets of P + P and P + 2P."""
    K1, K2 = _sgn(rng, rng.randrange(1, LIMIT)), _sgn(rng, rng.randrange(1, 1 << 40))
    terms = [(1, K1)] * reps + [(2, K1)] * (reps // 4) + [(-1, K2)] * (reps // 2) + [(3, K2)] * (reps // 8 + 1)
    rng.shuffle(terms)
    return Case("deep", terms)


def cancel(rng, n):
    half = tiny(rng, n // 2).terms[: n // 4] + spread(rng, n // 2).terms[: n // 2 - n // 4]
    terms = half + [(-m, k) if i % 2 else (m, (Q - k) % Q) for i, (m, k) in enumerate(half)]
    rng.shuffle(terms)
    return Case("cancel", terms)


def horner(rng, c, where, opp):
    """Two terms whose window sums meet in the Horner chain: G with digit A at window w + 1 (the only non-zero window above w)
    and 2^c G with digit A (or -A) at window w, so that the step at w adds A 2^c G to the accumulator A 2^c G (or its negative).
    where = "top": w + 1 is the top window; "mid": a window in the middle.  A third term, the identity point, adds nothing."""
    W, H, _ = shape(c)
    w = W - 2 if where == "top" else max(0, W // 2 - 1)
    amax = min(H, (LIMIT - 1) >> (c * (w + 1)))
    A = rng.randrange(1, amax + 1)
    s2 = A << (c * w)
    return Case("horner_%s_%s" % (where, "opp" if opp else "dbl"),
                [(1, A << (c * (w + 1))), (1 << c, (Q - s2) if opp else s2), (0, rng.randrange(1, Q))], ("opp" if opp else "dbl", w))


def units(rng, c, opp):
    """c divides 128: the top window's digit H + 1 (reached through a carry) lands in its second bucket unit, and 3 G with digit
    (H + 1) / 3 fills the first unit with the same point (or its negative): the two units meet where the top window is summed."""
    W, H, dbl = shape(c)
    assert dbl and (H + 1) % 3 == 0
    k = (H << (c * (W - 1))) + ((H + 1) << (c * (W - 2)))
    s2 = ((H + 1) // 3) << (c * (W - 1))
    return Case("units_%s" % ("opp" if opp else "dbl"), [(1, k), (3, (Q - s2) if opp else s2), (0, 5)],
                ("units_opp" if opp else "units_dbl", W - 1))


UNIT_WINDOWS = (4, 8, 16)          # c dividing 128 with a top digit above H in reach of |k| < 0.55 * 2^128


def collision_cases(rng, c):
    out = [horner(rng, c, where, opp) for where in ("top", "mid") for opp in (False, True)]
    if c in UNIT_WINDOWS:
        out += [units(rng, c, opp) for opp in (False, True)]
    return out


def single_cases(c):
    """Cases of one MSM each at window c (0: automatic -- the collision cases are then built for the window of a 3-term MSM)."""
    rng = random.Random(1000 + c)
    common = [tiny(rng, 300), deep(rng, 17000), cancel(rng, 400), spread(rng, 300), top(rng, 200), phi(rng, 300)]
    return common + collision_cases(rng, c or auto_c(3, 1))


BATCH_KINDS = ["horner_top_dbl", "tiny", "horner_top_opp", "empty", "units_dbl", "horner_mid_dbl", "phi", "one", "horner_mid_opp",
               "cancel", "units_opp", "spread", "top", "deep"]


def batch_cases(nmsm, c):
    """nmsm MSMs whose neighbours are of different kinds (so that each warp of the combination holds quads with different
    exceptional cases), empty and one-term MSMs among them, and one long MSM in the middle.  Returns (cases, window)."""
    rng = random.Random(nmsm * 100 + c)
    sizes = {"horner_top_dbl": 3, "horner_top_opp": 3, "horner_mid_dbl": 3, "horner_mid_opp": 3, "units_dbl": 3, "units_opp": 3,
             "tiny": 5, "empty": 0, "phi": 4, "one": 1, "cancel": 6, "spread": 5, "top": 4, "deep": deep_len(8),
             "long": deep_len(1700) + 500}
    kinds = [BATCH_KINDS[(j * 5 + j // len(BATCH_KINDS)) % len(BATCH_KINDS)] for j in range(nmsm)]
    kinds[nmsm // 2] = "long"
    T = sum(sizes[k] for k in kinds)
    cw = c or auto_c(-(-T // nmsm), nmsm)
    out = []
    for kind in kinds:
        if kind.startswith("horner"):
            _, where, what = kind.split("_")
            out.append(horner(rng, cw, where, what == "opp"))
        elif kind.startswith("units"):
            out.append(units(rng, cw, kind.endswith("opp")) if cw in UNIT_WINDOWS else top(rng, 3))
        elif kind == "empty":
            out.append(Case("empty", []))
        elif kind == "one":
            out.append(Case("one", [(_m(rng), _sgn(rng, rng.randrange(1, 1 << 20)))]))
        elif kind == "deep":
            out.append(deep(rng, 8))
        elif kind == "long":
            out.append(Case("long", deep(rng, 1700).terms + tiny(rng, 400).terms + top(rng, 100).terms))
        else:
            out.append({"tiny": tiny, "phi": phi, "cancel": cancel, "spread": spread, "top": top}[kind](rng, sizes[kind]))
    assert [len(x) for x in out] == [sizes[k] for k in kinds]
    return out, cw


BATCH_PARAMS = [(nmsm, c) for nmsm in (2, 9, 2047, 2048, 4096) for c in (0, 4, 10, 11)]


def table_points():
    """A point list with repeats, P / -P pairs and an identity (for the fixed-base tables)."""
    ms = [1, 1, -1, 2, -2, 2, 0, 3, 4, -4, 5, 5, 5, -5, 6, 7, -7, 8, 16, -16, 1, 3, -3, 9, 10, -10, 11, 12, 13, -13, 14, 15]
    return ms * 3


def table_scalar_sets(ms, count, seed):
    """count scalar vectors over the point list ms: tiny, spread, all equal, pairwise cancelling and exactly cancelling."""
    rng = random.Random(seed)
    out = []
    for j in range(count):
        kind = j % 5
        if kind == 0:
            ks = [c.terms[0][1] for c in (tiny(rng, 1) for _ in ms)]
        elif kind == 1:
            ks = [k for _, k in spread(rng, len(ms)).terms]
        elif kind == 2:
            ks = [_sgn(rng, rng.randrange(1, 9))] * len(ms)
        elif kind == 3:
            ks = [(abs(m) * 7 + 3 + j) % 11 for m in ms]                          # one scalar for P and -P
        else:
            ks = [rng.randrange(1, 8) for _ in ms]
            j0 = ms.index(1)
            ks[j0] = 0
            ks[j0] = (-sum(k * m for k, m in zip(ks, ms))) % Q                   # exact cancellation through one term
        out.append(Case("table%d" % kind, list(zip(ms, ks))))
    return out


def partial_slices():
    """A vector of equal-length slices whose MSMs are X, X, -X, O, 2X, -X, ... (X a fixed small multiple of G)."""
    rng = random.Random(77)
    base = tiny(rng, 24).terms
    while sum(k * m for m, k in base) % Q == 0:
        base = tiny(rng, 24).terms
    neg = [(m, (Q - k) % Q) for m, k in base]
    zero = cancel(rng, 24).terms
    dbl = [(m, 2 * k % Q) for m, k in base]
    pattern = [base, base, neg, zero, dbl, neg, neg, base, zero, zero, base, dbl, neg, neg, base, base]
    slices = [pattern[i % len(pattern)] for i in range(64)]
    return slices


def all_cpu_checked_cases():
    """(where, case, window of its collision) for every case the GPU legs run (the table legs' first sets)."""
    for c in range(0, 17):
        for case in single_cases(c):
            yield ("single", c), case, c or auto_c(3, 1)
    for nmsm, c in BATCH_PARAMS:
        cases, cw = batch_cases(nmsm, c)
        for case in cases:
            yield ("batch", nmsm, c), case, cw
    yield ("parts",), parts_case(), None
    for case in slot_cases():
        yield ("slots",), case, None
    ms = table_points()
    for case in table_scalar_sets(ms, 10, 5):
        yield ("table",), case, None
    for i, s in enumerate(partial_slices()[:16]):
        yield ("partial", i), Case("slice", s), None


def parts_case():
    """>= 2^17 terms: bp_msm uploads and sorts such an MSM in parts (msm_run_parts)."""
    rng = random.Random(17)
    terms = deep(rng, 40000).terms + tiny(rng, 30000).terms
    terms += spread(rng, (1 << 17) + 5 - len(terms)).terms
    rng.shuffle(terms)
    return Case("parts", terms)


def slot_cases():
    rng = random.Random(18)
    return [deep(rng, 17000), spread(rng, 6000), Case("tiny", tiny(rng, 5000).terms), cancel(rng, 6000)]


# ---- the expectation itself (no GPU) --------------------------------------------------------------------------------------
def _horner_events(case, c):
    """Collisions of the Horner chain over the window sums (as multiples of G) of a case whose scalars all split to k2 = 0."""
    W, H, dbl = shape(c)
    S = [0] * W
    second = 0
    for m, k in case.terms:
        if m == 0:                                       # the identity point adds nothing, whatever its scalar
            continue
        k1, k2 = glv_split(k)
        assert k2 == 0
        for w, d in enumerate(digits(abs(k1), c)):
            d = -d if k1 < 0 else d
            S[w] += d * m
            if w == W - 1 and abs(d) > H:
                second += d * m
    ev = []
    first = (S[W - 1] - second) % Q
    if dbl and first and second % Q:
        ev += [("units_dbl", W - 1)] if first == second % Q else ([("units_opp", W - 1)] if first == (-second) % Q else [])
    acc = S[W - 1] % Q
    for w in range(W - 2, -1, -1):
        acc = acc * (1 << c) % Q
        s = S[w] % Q
        if acc and s:
            ev += [("dbl", w)] if s == acc else ([("opp", w)] if s == (-acc) % Q else [])
        acc = (acc + s) % Q
    return ev


def test_case_expectations_match_the_oracle():
    """CPU only: every generated case's closed form (sum k_i m_i) G equals the oracle's MSM; the GLV split of glv.cuh gives
    k2 = 0 (k1 = +-k) for the small scalars and k1 = 0, k2 = +-s for the phi scalars; the collision each horner / units case
    is built for happens in the Horner chain of its window; top digits above H occur for the windows that have a second unit."""
    assert ecc.py_mul(ecc.G, LAMBDA) == (GLV["beta"] * ecc.GX % P, ecc.GY)
    seen_second_unit, checked = set(), set()
    items = list(all_cpu_checked_cases())
    wants = ecc.scalar_mul_batch([ecc.G] * len(items), [case.total for _, case, _ in items])
    for (where, case, cw), want in zip(items, wants):
        assert ecc.msm([ecc.unpack_point(_pt(m)) for m, _ in case.terms], [k for _, k in case.terms]) == want, (where, case)
        if where[0] != "batch":
            assert case.want == want, (where, case)                  # the pure-Python scalar multiplication the GPU legs use
        for m, k in set(case.terms) - checked:
            checked.add((m, k))
            k1, k2 = glv_split(k)
            assert (k1 + k2 * LAMBDA - k) % Q == 0
            if case.name == "phi":
                s = k * pow(LAMBDA, -1, Q) % Q
                assert (k1, k2) == (0, s if s < LIMIT else s - Q), (where, case)
            elif m != 0 and case.name != "table4":
                assert k2 == 0 and k1 == (k if k < LIMIT else k - Q), (where, case, k)
                seen_second_unit.update(c for c in UNIT_WINDOWS if digits(abs(k1), c)[-1] > 1 << (c - 1))
        if case.event is not None:
            assert case.event in _horner_events(case, cw), (where, case, _horner_events(case, cw))
    assert seen_second_unit == set(UNIT_WINDOWS)


def test_auto_window_mirror_matches_known_picks():
    """CPU only: the window picks the tests predict (auto_c) agree with the ones msm_shape documents."""
    assert [auto_c(n, 1) for n in (3, 64, 65, 1023, 1024, 65536, 65537)] == [5, 5, 10, 10, 13, 13, 16]
    for nmsm, c in BATCH_PARAMS:
        assert 1 <= batch_cases(nmsm, c)[1] <= 16


# ---- GPU legs ------------------------------------------------------------------------------------------------------------
@pytest.fixture
def lib():
    nat.init(0)
    return nat.load()


@pytest.fixture
def fb(lib):
    """Fixed-base table mode for one test: bucket-method legs set 0, table legs 2.  Restores the default (1) and drops the tables."""
    nat.check(lib.bp_fb_clear())

    def set_mode(m):
        nat.check(lib.bp_fb_set_mode(m))
    yield set_mode
    nat.check(lib.bp_fb_set_mode(1))
    nat.check(lib.bp_fb_clear())


def _stats(lib):
    v = [ctypes.c_uint64() for _ in range(4)]
    nat.check(lib.bp_fb_stats(*[ctypes.byref(x) for x in v]))
    return [x.value for x in v]


class _Window:
    def __init__(self, lib, c):
        self.lib, self.c = lib, c

    def __enter__(self):
        nat.check(self.lib.bp_msm_set_window(self.c))

    def __exit__(self, *exc):
        self.lib.bp_msm_set_window(0)


def _upload(lib, case):
    hp, hs = ctypes.c_uint64(), ctypes.c_uint64()
    nat.check(lib.bp_points_upload(case.pts, len(case), ctypes.byref(hp)))
    nat.check(lib.bp_scalars_upload(case.sc, len(case), ctypes.byref(hs)))
    return hp, hs


def _free(lib, *hs):
    for h in hs:
        nat.check(lib.bp_handle_free(h))


def _out():
    return ctypes.create_string_buffer(64)


@gpu
@pytest.mark.parametrize("c", [0] + list(range(1, 17)))
def test_single_resident_msm(lib, fb, c):
    """bp_msm_hh at the automatic window and at every forced c: the quad first level (c <= 14), k_reduce_seg_plain (c >= 15),
    k_reduce_grp, k_window_sum in one and in two steps (c = 16: 1024 groups), k_combine, k_fixup_mid and k_fixup_big."""
    fb(0)
    out = _out()
    with _Window(lib, c):
        for case in single_cases(c):
            hp, hs = _upload(lib, case)
            nat.check(lib.bp_msm_hh(hp, hs, len(case), out))
            _free(lib, hp, hs)
            assert ecc.unpack_point(out.raw) == case.want, (c, case)
            assert lib.bp_msm_last_window() == (c or auto_c(len(case), 1)), (c, case)


@gpu
@pytest.mark.parametrize("host_finish", [1, 0])
@pytest.mark.parametrize("c", [0, 1, 4, 8, 13, 16])
def test_host_operand_msm(lib, fb, c, host_finish):
    """bp_msm: the Horner chain on the host (horner_host, Jacobian) or on the device (k_combine)."""
    fb(0)
    try:
        nat.check(lib.bp_msm_set_host_finish(host_finish))
        with _Window(lib, c):
            for case in single_cases(c):
                assert ecc.unpack_point(nat.msm_bytes(case.pts, case.sc, len(case))) == case.want, (c, host_finish, case)
                assert lib.bp_msm_last_window() == (c or auto_c(len(case), 1)), (c, case)
    finally:
        lib.bp_msm_set_host_finish(1)


@gpu
@pytest.mark.parametrize("host_finish", [1, 0])
def test_host_operand_msm_in_parts(lib, fb, host_finish):
    """>= 2^17 host terms: sorted and accumulated in parts (msm_run_parts), finished on the host or the device."""
    fb(0)
    case = parts_case()
    try:
        nat.check(lib.bp_msm_set_host_finish(host_finish))
        assert ecc.unpack_point(nat.msm_bytes(case.pts, case.sc, len(case))) == case.want
    finally:
        lib.bp_msm_set_host_finish(1)


@gpu
@pytest.mark.parametrize("mode", [2, 1])
def test_slot_sort_plain_and_precomputed(lib, fb, mode):
    """bp_msm_set_pre_slots(2, 4096): 8 slots per bucket, every bucket overflows and the exact counting sort runs as the fallback;
    (1, 4096): the slot sort itself wherever no bucket overflows.  Plain resident path and precomputed path."""
    from python_bulletproofs_b200.device import DevicePoints
    fb(0)
    out = _out()
    try:
        nat.check(lib.bp_msm_set_pre_slots(mode, 4096))
        for case in slot_cases():
            dp, dq = DevicePoints(raw=case.pts), DevicePoints(raw=case.pts).precompute(0)
            for h, what in ((dp, "plain"), (dq, "pre")):
                nat.check(lib.bp_msm_h(h.handle, case.sc, len(case), out))
                assert ecc.unpack_point(out.raw) == case.want, (mode, what, case)
            dp.free(); dq.free()
    finally:
        lib.bp_msm_set_pre_slots(1, 1 << 18)


@gpu
@pytest.mark.parametrize("c", [8, 11, 16, 0])
def test_precomputed_vectors(lib, fb, c):
    """Precomputed window multiples: each MSM three times with small graphs on (eager, captured, replayed) and once with them
    off; bp_msm_hh_partial of a slice."""
    from python_bulletproofs_b200.device import DevicePoints, DeviceScalars
    fb(0)
    out, part = _out(), ctypes.create_string_buffer(128)
    rng = random.Random(c)
    cases = [tiny(rng, 300), deep(rng, 17000), cancel(rng, 400), spread(rng, 300), top(rng, 200), phi(rng, 300)]
    try:
        for case in cases:
            dp, ds = DevicePoints(raw=case.pts).precompute(c), DeviceScalars(raw=case.sc)
            cw = c or pre_auto_c(len(case))
            for graphs in (1, 0):
                nat.check(lib.bp_msm_set_small_graphs(graphs))
                for call in range(3 if graphs else 1):
                    nat.check(lib.bp_msm_h(dp.handle, case.sc, len(case), out))
                    assert ecc.unpack_point(out.raw) == case.want, (c, graphs, call, case)
                    assert lib.bp_msm_last_window() == cw
                    nat.check(lib.bp_msm_hh(dp.handle, ds.handle, len(case), out))
                    assert ecc.unpack_point(out.raw) == case.want, (c, graphs, call, case, "hh")
                lo, hi = len(case) // 3, len(case) - 7
                nat.check(lib.bp_msm_hh_partial(dp.handle, ds.handle, lo, hi - lo, part))
                nat.check(lib.bp_xyzz_sum(part.raw, 1, out))
                assert ecc.unpack_point(out.raw) == Case("slice", case.terms[lo:hi]).want, (c, graphs, case, "partial")
            dp.free(); ds.free()
    finally:
        lib.bp_msm_set_small_graphs(1)


@gpu
@pytest.mark.parametrize("nmsm,c", BATCH_PARAMS)
def test_batch(lib, fb, nmsm, c):
    """bp_msm_batch: with >= 2048 MSMs and c <= 10 the thread-per-unit tails (k_reduce_unit_plain with the second-unit weighting
    at c = 4, k_combine_plain); c = 11 and fewer MSMs the quad tails and k_combine, whose warps hold neighbouring MSMs of
    different kinds."""
    fb(0)
    cases, cw = batch_cases(nmsm, c)
    offsets = [0]
    for case in cases:
        offsets.append(offsets[-1] + len(case))
    pts = b"".join(case.pts for case in cases)
    sc = b"".join(case.sc for case in cases)
    with _Window(lib, c):
        raw = nat.msm_batch_bytes(pts, sc, offsets)
    assert lib.bp_msm_last_window() == cw
    want = ecc.scalar_mul_batch([ecc.G] * nmsm, [case.total for case in cases])
    got = ecc.unpack_points(raw, nmsm)
    bad = [(j, cases[j].name) for j in range(nmsm) if got[j] != want[j]]
    assert not bad, (nmsm, c, cw, len(bad), bad[:12])


@gpu
def test_fixed_base_tables_single(lib, fb):
    """Mode 2: bp_msm over a point list with repeats, P / -P pairs and an identity builds its table at first use, then hits."""
    fb(2)
    ms = table_points()
    cases = table_scalar_sets(ms, 10, 5)
    hits0, builds0 = _stats(lib)[2:]
    for i, case in enumerate(cases):
        assert ecc.unpack_point(nat.msm_bytes(case.pts, case.sc, len(case))) == case.want, (i, case)
        assert _stats(lib)[2:] == [hits0 + i, builds0 + 1]


@gpu
@pytest.mark.parametrize("nmsm", [3, 64, 65, 1000])
def test_fixed_base_tables_batch(lib, fb, nmsm):
    """Mode 2: bp_msm_batch over one repeated point list -- finished on the host up to 64 MSMs, on the device (fb_msm_run) above."""
    fb(2)
    ms = table_points()
    cases = table_scalar_sets(ms, nmsm, nmsm)
    pts = cases[0].pts * nmsm
    sc = b"".join(case.sc for case in cases)
    offsets = [len(ms) * j for j in range(nmsm + 1)]
    hits0, builds0 = _stats(lib)[2:]
    for call in range(2):
        got = ecc.unpack_points(nat.msm_batch_bytes(pts, sc, offsets), nmsm)
        want = ecc.scalar_mul_batch([ecc.G] * nmsm, [case.total for case in cases])
        bad = [(j, cases[j].name) for j in range(nmsm) if got[j] != want[j]]
        assert not bad, (nmsm, call, bad[:12])
        assert _stats(lib)[2:] == [hits0 + call, builds0 + 1]


@gpu
@pytest.mark.parametrize("pre", [0, 8])
def test_partials_equal_opposite_and_identity(lib, fb, pre):
    """bp_msm_hh_partial over slices whose results are X, X, -X, O, 2X, ...; bp_xyzz_sum over up to 64 of them."""
    from python_bulletproofs_b200.device import DevicePoints, DeviceScalars
    fb(0)
    slices = partial_slices()
    L = len(slices[0])
    whole = Case("all", [t for s in slices for t in s])
    dp, ds = DevicePoints(raw=whole.pts), DeviceScalars(raw=whole.sc)
    if pre:
        dp.precompute(pre)
    part, out = ctypes.create_string_buffer(128), _out()
    parts = []
    for j in range(len(slices)):
        nat.check(lib.bp_msm_hh_partial(dp.handle, ds.handle, j * L, L, part))
        parts.append(part.raw)
        nat.check(lib.bp_xyzz_sum(part.raw, 1, out))
        assert ecc.unpack_point(out.raw) == Case("slice", slices[j]).want, (pre, j)
    for cnt in (2, 3, 4, 5, 6, 17, 64):
        nat.check(lib.bp_xyzz_sum(b"".join(parts[:cnt]), cnt, out))
        assert ecc.unpack_point(out.raw) == Case("sum", [t for s in slices[:cnt] for t in s]).want, (pre, cnt)
    dp.free(); ds.free()
