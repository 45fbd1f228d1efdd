"""The inner-product argument through its C ABI (bp_ipa_prove_hs, bp_ipa_verify_eq_hs, bp_ipa_verify1_eq_hs,
bp_ipa_statement) and the table MSMs past 2048 terms, compared with the CPU oracle at every length, round form and table
path the library chooses between.

Which path a proof takes depends on its length and the switches:
  - table rounds, fast form: one k_ipa_round per round plus a final k_ipa_round_prep (table present: 2 <= n <= 2048);
  - table rounds, four-launch form: k_round_fold, k_build_lr_sv, k_fb_msm, k_fb_finish per round, plus a final fold;
  - bucket rounds: k_round_fold, k_build_lr_sv and a bucket MSM per round (tables off, first sighting, and always for
    n >= 4096, where 2n + 1 points exceed the largest table);
and each of them under graph mode 0 (one synchronisation per round), 1 (mapped-flag handshake) or 2 (one captured CUDA
graph per length and table, replayed).  Every proof is compared byte for byte with protocol_oracle.ipa_prove2, and the
table statistics and launch counts show which path ran, so that a fall-back cannot pass unnoticed.

Points and scalars cross the ABI as packed bytes, so that Python marshalling stays small at n = 8192.
"""
import contextlib
import ctypes
import io
import random

import pytest

from oracle import ecc, protocol_oracle as po
from python_bulletproofs_b200 import _native as nat

Q, P = ecc.Q, ecc.P
SIZES = [1, 2, 4, 8, 16, 32, 64, 128, 256, 512, 1024, 2048, 4096, 8192]
MAX_TABLE_POINTS = 4200            # FbCache::max_points: the largest point set that gets a table
NPOOL = 2 * 8192 + 1 + 8


# ---- oracle side: generators, inputs and proofs, computed once per module ----------------------------------------------
_pool = []


def pool():
    """NPOOL random multiples of G (one batch of scalar multiplications: far cheaper than lifting x coordinates)."""
    if not _pool:
        rng = random.Random(0x1BA2048)
        _pool.extend(ecc.scalar_mul_batch([ecc.G] * NPOOL, [rng.getrandbits(256) for _ in range(NPOOL)]))
    return _pool


class Gens:
    """A generator set (g, h, u) of length n, with its packed bytes."""

    def __init__(self, g, h, u):
        self.g, self.h, self.u = list(g), list(h), u
        self.gb, self.hb, self.ub = ecc.pack_points(self.g), ecc.pack_points(self.h), ecc.pack_point(u)


_gens = {}


def gens(n, variant="A"):
    """Set A: pool[0:n], pool[n:2n], pool[2n]; set B: the same shifted by one point.  The degenerate variants start
    from set A: h = g; g_{k+i} = -g_i (k = n/2); u = g_{n/3}; one identity generator (h_{n-1})."""
    key = (n, variant)
    if key not in _gens:
        pts = pool()
        off = 1 if variant == "B" else 0
        g, h, u = pts[off:off + n], pts[off + n:off + 2 * n], pts[off + 2 * n]
        if variant == "h_eq_g":
            h = list(g)
        elif variant == "g_neg":
            k = n // 2
            g = g[:k] + [ecc.point_neg(p) for p in g[:k]]
        elif variant == "u_eq_g":
            u = g[n // 3]
        elif variant == "ident_gen":
            h = h[:-1] + [None]
        _gens[key] = Gens(g, h, u)
    return _gens[key]


def _sc(ks):
    """Raw 32-byte little-endian words: values in [q, 2^256) stay unreduced, for the library to reduce."""
    return b"".join(int(k).to_bytes(32, "little") for k in ks)


class Case:
    """Inputs of one proof: a, b (raw, possibly >= q), an optional h scale (raw), a transcript prefix, and the
    oracle's proof over the same inputs, packed as the ABI returns it."""

    def __init__(self, S, a, b, hsc=None, tr=None):
        self.S, self.n = S, len(a)
        self.a, self.b, self.hsc, self.tr = a, b, hsc, tr
        self.ab, self.bb = _sc(a), _sc(b)
        self.hsb = _sc(hsc) if hsc is not None else None
        self._want = None

    @property
    def hsp(self):
        return self.S.h if self.hsc is None else ecc.scalar_mul_batch(self.S.h, self.hsc)

    @property
    def want(self):
        if self._want is None:
            self.proof = po.ipa_prove2(self.S.g, self.hsp, self.S.u, self.a, self.b, self.tr)
            self._want = pack_proof(self.proof)
        return self._want


def pack_proof(p):
    return (ecc.pack_points(p["Ls"]), ecc.pack_points(p["Rs"]), _sc(p["xs"]), _sc([p["a"]]), _sc([p["b"]]), p["transcript"])


def _rand(rng, n):
    return [rng.getrandbits(256) % Q for _ in range(n)]


_cases = {}


def case(n, kind="random", variant="A"):
    """Cached inputs of each kind:
      random      uniform a, b < q, no scale (on set A or B);
      unreduced   zeros and words >= q (v + q for small v, and raw 256-bit values) in a and b;
      L_identity  a_lo = 0 and b_hi = 0: round 0's L is the identity (transcript slot AA==);
      R_identity  the mirror case: a_hi = 0 and b_lo = 0;
      h_eq_g / g_neg / u_eq_g / ident_gen   degenerate generator sets (see gens);
      scale_yinv / scale_raw / scale_zeros  h scale y^-i, unreduced random 256-bit words, or words with zeros."""
    key = (n, kind, variant)
    if key in _cases:
        return _cases[key]
    rng = random.Random("%d/%s/%s" % key)
    a, b, hsc = _rand(rng, n), _rand(rng, n), None
    k = n // 2
    S = gens(n, variant if kind in ("random",) else "A")
    if kind == "unreduced":
        for i in range(n):
            r = i % 5
            if r == 0:
                a[i] = 0
            elif r == 1:
                a[i] = rng.randrange(1, 1000) + Q
            elif r == 2:
                b[i] = rng.getrandbits(256) | (1 << 255)
            elif r == 3:
                b[i] = 0 if i % 2 else Q
        a[-1], b[0] = 2 ** 256 - 1, Q + 1
    elif kind == "L_identity":
        a[:k], b[k:] = [0] * k, [0] * (n - k)
    elif kind == "R_identity":
        a[k:], b[:k] = [0] * (n - k), [0] * k
    elif kind in ("h_eq_g", "g_neg", "u_eq_g", "ident_gen"):
        S = gens(n, kind)
    elif kind == "scale_yinv":
        yinv = pow(po.mod_hash(b"y%d" % n), -1, Q)
        hsc = [pow(yinv, i, Q) for i in range(n)]
    elif kind == "scale_raw":
        hsc = [rng.getrandbits(256) for _ in range(n)]
    elif kind == "scale_zeros":
        hsc = [0 if i % 3 == 1 else rng.getrandbits(256) for i in range(n)]
    else:
        assert kind == "random", kind
    tr = None if n % 3 else b"%d&" % (n * 7919)          # a Protocol-1 style transcript prefix on some lengths
    _cases[key] = Case(S, a, b, hsc, tr)
    return _cases[key]


# ---- GPU side ------------------------------------------------------------------------------------------------------------
def lib():
    return nat.load()


def fb_stats():
    v = [ctypes.c_uint64() for _ in range(4)]
    nat.check(lib().bp_fb_stats(*[ctypes.byref(x) for x in v]))
    return dict(zip(("tables", "bytes", "hits", "builds"), (x.value for x in v)))


def launches():
    v = ctypes.c_uint64()
    nat.check(lib().bp_launch_count(ctypes.byref(v)))
    return v.value


@pytest.fixture
def ipa_lib():
    L = lib()
    nat.init(0)
    nat.check(L.bp_fb_clear())
    yield L
    nat.check(L.bp_fb_set_mode(1))
    nat.check(L.bp_ipa_set_graphs(1))
    nat.check(L.bp_ipa_set_fast_rounds(1))
    nat.check(L.bp_msm_set_window(0))
    nat.check(L.bp_fb_clear())


def set_modes(L, tm, gm, fast):
    nat.check(L.bp_fb_set_mode(tm))
    nat.check(L.bp_ipa_set_graphs(gm))
    nat.check(L.bp_ipa_set_fast_rounds(fast))


def gpu_prove(c):
    n = c.n
    L = n.bit_length() - 1
    start = po.transcript_start() + (c.tr or b"")
    cap = len(start) + L * (2 * 45 + 80) + 16
    Ls, Rs, xs = (ctypes.create_string_buffer(w * max(L, 1)) for w in (64, 64, 32))
    ao, bo, t = ctypes.create_string_buffer(32), ctypes.create_string_buffer(32), ctypes.create_string_buffer(cap)
    tl = ctypes.c_size_t(0)
    nat.check(lib().bp_ipa_prove_hs(c.S.gb, c.S.hb, c.hsb, c.S.ub, c.ab, c.bb, n, start, len(start), Ls, Rs, xs, ao, bo, t, cap,
                                    ctypes.byref(tl)))
    return (Ls.raw[:64 * L], Rs.raw[:64 * L], xs.raw[:32 * L], ao.raw, bo.raw, t.raw[:tl.value])


def table_possible(n):
    return n > 1 and 2 * n + 1 <= MAX_TABLE_POINTS


def expected_table(n, tm, rep):
    """(table used, table built by this proof) for the rep-th proof of one generator set after bp_fb_clear."""
    if tm == 0 or not table_possible(n):
        return False, False
    if tm == 2:
        return True, rep == 0
    return rep >= 1, rep == 1                              # mode 1: first sighting takes the bucket method, the second builds


def prove_checked(c, tm, fast, rep):
    """One proof, compared with the oracle, with the path it must have taken asserted from the table statistics and the
    launch count.  Launches per proof (bp_ipa_prove_hs, enqueue_proof): 2 k_reduce_scalars + k_fill_one_mont (+ k_to_mont with
    a scale), k_fb_build per 256 table points when the table is built, then
      fast form         one k_ipa_round per round + the final k_ipa_round_prep;
      four-launch form  k_round_fold + k_build_lr_sv + k_fb_msm + k_fb_finish per round + the final k_round_fold;
      bucket form       k_round_fold + k_build_lr_sv + at least one bucket-MSM launch per round + the final k_round_fold.
    Graph mode 2 counts the kernels of a replayed graph at every launch, so the counts do not depend on the graph mode."""
    n = c.n
    rounds = n.bit_length() - 1
    s0, l0 = fb_stats(), launches()
    got = gpu_prove(c)
    s1, l1 = fb_stats(), launches()
    assert got == c.want, (n, tm, fast, rep, [i for i in range(6) if got[i] != c.want[i]])
    tab, built = expected_table(n, tm, rep)
    assert s1["builds"] - s0["builds"] == int(built), (n, tm, rep)
    assert s1["hits"] - s0["hits"] == int(tab and not built), (n, tm, rep)
    base = 3 + (c.hsc is not None)
    nl = l1 - l0 - (-(-(2 * n + 1) // 256) if built else 0)
    if n == 1:
        assert nl == base
    elif tab and fast:
        assert nl == base + rounds + 1, (n, nl)
    elif tab:
        assert nl == base + 4 * rounds + 1, (n, nl)
    else:
        assert nl >= base + 3 * rounds + 1, (n, nl)
    return got


def run_config(L, c, tm, gm, fast, reps=4):
    """reps proofs in a row under one configuration: graph mode 2 runs its eager, capture and replay proofs (after a
    first-sighting proof in table mode 1), graph mode 1 its first-sighting, build and hit proofs."""
    nat.check(L.bp_fb_clear())
    set_modes(L, tm, gm, fast)
    for rep in range(reps):
        prove_checked(c, tm, fast, rep)


FULL = [(tm, gm, fast) for tm in (0, 1, 2) for gm in (0, 1, 2) for fast in (0, 1)]
MID = [(2, 1, 1), (2, 2, 1), (2, 0, 0), (1, 1, 1), (1, 2, 0), (0, 2, 1)]
KIND_CONFIGS = [(2, 1, 1), (2, 2, 0), (1, 2, 1), (0, 0, 1)]


# ---- 1. prover matrix ----------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("n", SIZES)
def test_prover_matrix(ipa_lib, n):
    if n >= 4096:        # bucket rounds only: graph modes x scale on / off
        for kind in ("random", "scale_yinv"):
            for gm in (0, 1, 2):
                run_config(ipa_lib, case(n, kind), 2, gm, 1)
        return
    configs = FULL if n <= 64 or n == 2048 else MID
    for tm, gm, fast in configs:
        run_config(ipa_lib, case(n), tm, gm, fast)


KIND_SIZES = [("unreduced", n) for n in (1, 8, 64, 2048)] + \
             [(k, n) for k in ("L_identity", "R_identity") for n in (2, 16, 2048)] + \
             [(k, n) for k in ("h_eq_g", "g_neg", "u_eq_g", "ident_gen") for n in (2, 32, 2048)] + \
             [("scale_yinv", n) for n in (8, 256, 2048)] + [("scale_raw", n) for n in (4, 64, 2048, 8192)] + \
             [("scale_zeros", n) for n in (16, 1024, 2048, 4096)]


@pytest.mark.gpu
@pytest.mark.parametrize("kind,n", KIND_SIZES)
def test_prover_input_kinds(ipa_lib, kind, n):
    c = case(n, kind)
    c.want
    if kind in ("L_identity", "R_identity"):                # round 0's L (R) is the identity: transcript slot 1 (2) is AA==
        slot = 1 if kind == "L_identity" else 2
        assert c.proof["Ls" if slot == 1 else "Rs"][0] is None and c.want[5].split(b"&")[slot] == b"AA=="
    for tm, gm, fast in (KIND_CONFIGS if n <= 2048 else [(2, gm, 1) for gm in (0, 1, 2)]):
        run_config(ipa_lib, c, tm, gm, fast)


# ---- 2. graph and table caches -------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("gm", [1, 2])
def test_prover_cache_sequence(ipa_lib, gm):
    """Graph mode 2 keys its captured proofs on (n, round form, table) and drops them when a workspace moves or a table is
    freed; this sequence changes each of those between proofs, and every proof must still equal the oracle."""
    L = ipa_lib
    A, B, As = case(2048, "random", "A"), case(2048, "random", "B"), case(2048, "scale_yinv")
    small = case(64)
    set_modes(L, 2, gm, 1)
    for fast in (1, 0):                                     # 1. sets A and B alternating, both round forms
        nat.check(L.bp_ipa_set_fast_rounds(fast))
        for c in (A, A, B, A, B, B, A):
            assert gpu_prove(c) == c.want, fast
    nat.check(L.bp_ipa_set_fast_rounds(1))
    for c in (As, A, As, A, As):                            # 2. scale on and off alternating
        assert gpu_prove(c) == c.want
    nat.check(L.bp_fb_clear())                              # 3. tables freed between two proofs
    for c in (A, B, A):
        assert gpu_prove(c) == c.want
    rng = random.Random(17)                                 # 4. a 2^17-term MSM grows the shared workspaces
    nbig = 1 << 17
    pts = (pool() * (nbig // NPOOL + 1))[:nbig]
    ks = [rng.getrandbits(256) for _ in range(nbig)]
    got = ecc.unpack_point(nat.msm_bytes(ecc.pack_points(pts), _sc(ks), nbig))
    assert got == ecc.msm(pts, ks, "bucket", ecc.max_threads())
    for c in (A, B, A):
        assert gpu_prove(c) == c.want
    for c in (small, A, small, A, small, A):                # 5. n = 2048 -> 64 -> 2048
        assert gpu_prove(c) == c.want


# ---- 3. verifiers --------------------------------------------------------------------------------------------------------
class _Lhs:
    cache = {}


def oracle_eq(S, hsc, u, Pt, n, a, b, xs, Ls, Rs):
    """Verifier2's equation (inner_product_verifier.py:127-143) without the transcript checks: the same decision the
    ABI makes.  Raises when a challenge is 0 mod q."""
    xs = [x % Q for x in xs]
    a, b = a % Q, b % Q
    key = (id(S), None if hsc is None else id(hsc), u, n, a, b, tuple(xs))
    lhs = _Lhs.cache.get(key)
    if lhs is None:
        ss = po.ss_vector(xs, n)
        hs = hsc if hsc is not None else [1] * n
        lhs = ecc.msm(S.g + S.h + [u], [a * s % Q for s in ss] + [b * po.inv(s) * hs[i] % Q for i, s in enumerate(ss)] + [a * b % Q],
                      "bucket", ecc.max_threads())
        _Lhs.cache[key] = lhs
    rhs = ecc.point_add(Pt, ecc.msm(list(Ls) + list(Rs), [x * x % Q for x in xs] + [po.inv(x) ** 2 % Q for x in xs]))
    return lhs == rhs


def statement(c):
    """P = sum a_i g_i + sum b_i hscale_i h_i + <a, b> u  (the point the IPA proves)."""
    a, b = [x % Q for x in c.a], [x % Q for x in c.b]
    hs = c.hsc if c.hsc is not None else [1] * c.n
    return ecc.msm(c.S.g + c.S.h + [c.S.u], a + [b[i] * hs[i] % Q for i in range(c.n)] + [po.dot(a, b)], "bucket", ecc.max_threads())


def gpu_verify(c, u, Pt, a, b, xs, Ls, Rs, p1=None):
    n = c.n
    acc = ctypes.c_int(-1)
    common = (n, _sc([a]), _sc([b]), _sc(xs), ecc.pack_points(Ls), ecc.pack_points(Rs), ctypes.byref(acc))
    if p1 is None:
        nat.check(lib().bp_ipa_verify_eq_hs(c.S.gb, c.S.hb, c.hsb, ecc.pack_point(u), ecc.pack_point(Pt), *common))
    else:
        P0, u0, xc, x = p1
        nat.check(lib().bp_ipa_verify1_eq_hs(c.S.gb, c.S.hb, c.hsb, ecc.pack_point(u0), ecc.pack_point(P0), _sc([xc]), _sc([x]),
                                             ecc.pack_point(u), ecc.pack_point(Pt), *common))
    assert acc.value in (0, 1)
    return acc.value == 1


def forgeries(c, Pt, rounds_all):
    """(label, P, a, b, xs, Ls, Rs) of the honest proof and of forged ones."""
    p, n = c.proof, c.n
    a, b, xs, Ls, Rs = p["a"], p["b"], list(p["xs"]), list(p["Ls"]), list(p["Rs"])
    L = len(xs)
    idx = range(L) if rounds_all else sorted({0, L // 2, L - 1})
    other = pool()[-3]
    out = [("honest", Pt, a, b, xs, Ls, Rs)]
    for i in (idx if L else ()):
        for nm, arr in (("L", Ls), ("R", Rs)):
            for how, pt in (("other", other), ("neg", ecc.point_neg(arr[i])), ("identity", None)):
                f = list(arr)
                f[i] = pt
                out.append(("%s%d_%s" % (nm, i, how), Pt, a, b, xs, f if nm == "L" else Ls, f if nm == "R" else Rs))
        sl, sr = list(Ls), list(Rs)
        sl[i], sr[i] = Rs[i], Ls[i]
        out.append(("swap%d" % i, Pt, a, b, xs, sl, sr))
        for how, x in (("x+1", (xs[i] + 1) % Q), ("q-x", Q - xs[i])):
            f = list(xs)
            f[i] = x
            out.append(("x%d_%s" % (i, how), Pt, a, b, f, Ls, Rs))
    for nm, da, db in (("a+1", 1, 0), ("a-1", -1, 0), ("b+1", 0, 1), ("b-1", 0, -1)):
        out.append((nm, Pt, (a + da) % Q, (b + db) % Q, xs, Ls, Rs))
    out.append(("a<->b", Pt, b, a, xs, Ls, Rs))
    out.append(("P+u", ecc.point_add(Pt, c.S.u), a, b, xs, Ls, Rs))
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("n", SIZES)
def test_verifiers(ipa_lib, n):
    """bp_ipa_verify_eq_hs and bp_ipa_verify1_eq_hs on the honest proof and on forgeries of every part of it, each
    decision compared with the oracle's equation; Protocol 1's two checks are wrapped honestly around the same proof."""
    rng = random.Random(n)
    for kind in ("random", "scale_yinv"):
        c = case(n, kind)
        c.want
        Pt = statement(c)
        x, xc = rng.randrange(1, Q), rng.randrange(Q)
        u0 = ecc.scalar_mul(c.S.u, po.inv(x))                # u_new = x * u0
        P0 = ecc.point_add(Pt, ecc.point_neg(ecc.scalar_mul(u0, xc)))     # P_new = P0 + xc * u0
        decisions = []
        for label, Pf, a, b, xs, Ls, Rs in forgeries(c, Pt, n <= 64):
            want = oracle_eq(c.S, c.hsc, c.S.u, Pf, n, a, b, xs, Ls, Rs)
            assert gpu_verify(c, c.S.u, Pf, a, b, xs, Ls, Rs) is want, (kind, label)
            assert gpu_verify(c, c.S.u, Pf, a, b, xs, Ls, Rs, (P0, u0, xc, x)) is want, (kind, label)
            decisions.append(want)
        assert decisions[0] is True and decisions.count(True) == 1, decisions
        if n > 1:                                            # a challenge of 0 mod q has no inverse: an error, not a decision
            p = c.proof
            for zero in (0, Q):
                xs = list(p["xs"])
                xs[-1] = zero
                with pytest.raises(nat.BpGpuError):
                    gpu_verify(c, c.S.u, Pt, p["a"], p["b"], xs, p["Ls"], p["Rs"])
                with pytest.raises(nat.BpGpuError):
                    gpu_verify(c, c.S.u, Pt, p["a"], p["b"], xs, p["Ls"], p["Rs"], (P0, u0, xc, x))


def protocol1_checks(c, Pt, P0, u0, xc, x, a, b):
    """Verifier1's three checks (inner_product_verifier.py:51-52 and Verifier2), without the transcript checks."""
    p = c.proof
    return (Pt == ecc.point_add(P0, ecc.scalar_mul(u0, xc)), c.S.u == ecc.scalar_mul(u0, x),
            oracle_eq(c.S, c.hsc, c.S.u, Pt, c.n, a, b, p["xs"], p["Ls"], p["Rs"]))


@pytest.mark.gpu
@pytest.mark.parametrize("n", [8, 4096])
def test_verify1_isolated_protocol1_forgeries(ipa_lib, n):
    """Each forgery breaks exactly one of the three checks bp_ipa_verify1_eq_hs fuses: u_new != x*u with an honest proof for
    (u_new, P_new) and P = P_new - xc*u; P not matching P_new; a wrong xc; a wrong a (Verifier2's equation)."""
    rng = random.Random(n + 1)
    c = case(n, "scale_yinv")
    c.want
    Pt = statement(c)
    p = c.proof
    x, xc = rng.randrange(1, Q), rng.randrange(Q)
    u_honest = ecc.scalar_mul(c.S.u, po.inv(x))
    u_wrong = pool()[-5]
    minus = lambda pt, k, base: ecc.point_add(pt, ecc.point_neg(ecc.scalar_mul(base, k)))     # noqa: E731
    cases = [
        ("honest", minus(Pt, xc, u_honest), u_honest, xc, p["a"], (True, True, True)),
        ("u_new != x*u", minus(Pt, xc, u_wrong), u_wrong, xc, p["a"], (True, False, True)),
        ("P_new wrong", ecc.point_add(minus(Pt, xc, u_honest), ecc.G), u_honest, xc, p["a"], (False, True, True)),
        ("xc wrong", minus(Pt, xc, u_honest), u_honest, (xc + 1) % Q, p["a"], (False, True, True)),
        ("a wrong", minus(Pt, xc, u_honest), u_honest, xc, (p["a"] + 1) % Q, (True, True, False)),
    ]
    for label, P0, u0, xcv, a, checks in cases:
        assert protocol1_checks(c, Pt, P0, u0, xcv, x, a, p["b"]) == checks, label
        got = gpu_verify(c, c.S.u, Pt, a, p["b"], p["xs"], p["Ls"], p["Rs"], (P0, u0, xcv, x))
        assert got is all(checks), label
        assert gpu_verify(c, c.S.u, Pt, a, p["b"], p["xs"], p["Ls"], p["Rs"]) is checks[2], label


# ---- 4. statement --------------------------------------------------------------------------------------------------------
def gpu_statement(S, a, bs, cc, n):
    out = ctypes.create_string_buffer(64)
    nat.check(lib().bp_ipa_statement(S.gb, S.hb, S.ub, _sc(a), _sc(bs), _sc([cc]), n, out))
    return ecc.unpack_point(out.raw)


EDGE = [0, 1, Q - 1, Q, Q + 1, 2 ** 256 - 1, 2 ** 255]


@pytest.mark.gpu
@pytest.mark.parametrize("tm", [0, 1, 2])
@pytest.mark.parametrize("n", [1, 2, 3, 1023, 1024, 2048, 2099, 2100])
def test_statement(ipa_lib, n, tm):
    """bp_ipa_statement = c*u + sum a_i g_i + sum bs_i h_i against ecc.msm; at 2099 / 2100 the 2n + 1 points fall on either
    side of the largest table (4200 points)."""
    nat.check(ipa_lib.bp_fb_clear())
    nat.check(ipa_lib.bp_fb_set_mode(tm))
    pts = pool()
    S = Gens(pts[:n], pts[n:2 * n], pts[2 * n])
    rng = random.Random(n * 3 + tm)
    for rep in range(3):
        a, bs = [rng.getrandbits(256) for _ in range(n)], [rng.getrandbits(256) for _ in range(n)]
        for i, e in enumerate(EDGE):
            a[(5 * i + rep) % n], bs[(3 * i + 2 * rep) % n] = e, EDGE[(i + rep) % len(EDGE)]
        cc = EDGE[(rep * 2 + 1) % len(EDGE)]
        s0 = fb_stats()
        got = gpu_statement(S, a, bs, cc, n)
        s1 = fb_stats()
        assert got == ecc.msm([S.u] + S.g + S.h, [x % Q for x in [cc] + a + bs], "bucket", ecc.max_threads()), (n, tm, rep)
        tab, built = expected_table(n, tm, rep)
        assert (s1["builds"] - s0["builds"], s1["hits"] - s0["hits"]) == (int(built), int(tab and not built)), (n, tm, rep)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [64, 2048])
def test_statement_and_prover_share_one_table(ipa_lib, n):
    """The statement and the prover key the table on the same point set [u | g | h]: each hits the table the other built."""
    L = ipa_lib
    c = case(n)
    S = c.S
    a, bs, cc = [x % Q for x in c.a], [x % Q for x in c.b], po.dot([x % Q for x in c.a], [x % Q for x in c.b])
    want_P = statement(c)
    for first in ("statement", "prover"):
        nat.check(L.bp_fb_clear())
        set_modes(L, 2, 1, 1)
        steps = ["statement", "prover"] if first == "statement" else ["prover", "statement"]
        for i, step in enumerate(steps):
            s0 = fb_stats()
            if step == "statement":
                assert gpu_statement(S, a, bs, cc, n) == want_P
            else:
                assert gpu_prove(c) == c.want
            s1 = fb_stats()
            assert (s1["builds"] - s0["builds"], s1["hits"] - s0["hits"]) == ((1, 0) if i == 0 else (0, 1)), (first, step)
    # table mode 1: the prover's sighting and the statement's add up to the build
    nat.check(L.bp_fb_clear())
    set_modes(L, 1, 1, 1)
    s0 = fb_stats()
    assert gpu_prove(c) == c.want
    assert gpu_statement(S, a, bs, cc, n) == want_P
    assert gpu_prove(c) == c.want
    s1 = fb_stats()
    assert (s1["builds"] - s0["builds"], s1["hits"] - s0["hits"]) == (1, 1)


# ---- 5. table MSMs past 2048 terms ----------------------------------------------------------------------------------------
def adversarial_points(n):
    pts = list(pool()[:n])
    pts[1] = pts[0]                                          # repeated point
    pts[2] = ecc.point_neg(pts[0])                           # and its negation
    pts[17] = None                                           # identity among the generators
    pts[-1] = pts[-2]
    return pts


MSM_EDGE = [0, 1, 2, 255, 256, 0xFF00, 2 ** 248, 2 ** 255, Q - 1, Q, Q + 1, 2 ** 256 - 1, (Q - 1) // 2]


@pytest.mark.gpu
@pytest.mark.parametrize("n", [2049, 2112, 4096, 4200, 4201])
def test_table_msm_past_2048_terms(ipa_lib, n):
    """bp_msm over a table of more than 2048 points: the block sums (more than 64) go through the serial steps of the
    ticketed tail.  4201 points get no table and take the bucket method."""
    nat.check(ipa_lib.bp_fb_set_mode(2))
    pts = adversarial_points(n)
    pb = ecc.pack_points(pts)
    rng = random.Random(n)
    for trial in range(3):
        ks = [rng.getrandbits(256) for _ in range(n)]
        for i, e in enumerate(MSM_EDGE):
            ks[(i * 97 + trial) % n] = e
        if trial == 2:
            ks = [0] * n
            ks[64 * 32] = Q - 1                              # one term, in block 64 only
        s0 = fb_stats()
        got = ecc.unpack_point(nat.msm_bytes(pb, _sc(ks), n))
        s1 = fb_stats()
        assert got == ecc.msm(pts, [k % Q for k in ks], "bucket", ecc.max_threads()), (n, trial)
        tab = n <= MAX_TABLE_POINTS
        assert (s1["builds"] - s0["builds"], s1["hits"] - s0["hits"]) == ((int(trial == 0), int(trial > 0)) if tab else (0, 0))


@pytest.mark.gpu
@pytest.mark.parametrize("nmsm", [2, 64, 65])
def test_table_msm_batch_past_2048_terms(ipa_lib, nmsm):
    """bp_msm_batch of nmsm MSMs of 2049 terms over one point list (one table): up to 64 MSMs are finished by their last
    block (fb_msm_run_host), more go through k_fb_finish, which then loops over 65 block sums."""
    nat.check(ipa_lib.bp_fb_set_mode(2))
    n = 2049
    pts = adversarial_points(n)
    rng = random.Random(nmsm)
    kss = [[rng.getrandbits(256) for _ in range(n)] for _ in range(nmsm)]
    for j, ks in enumerate(kss):
        ks[j % n] = MSM_EDGE[j % len(MSM_EDGE)]
        if j % 7 == 3:
            kss[j] = [0] * (n - 1) + [Q + 5]                 # only the last term, in block 64
    s0 = fb_stats()
    raw = nat.msm_batch_bytes(ecc.pack_points(pts) * nmsm, b"".join(_sc(ks) for ks in kss), [n * j for j in range(nmsm + 1)])
    s1 = fb_stats()
    for j, ks in enumerate(kss):
        assert ecc.unpack_point(raw[64 * j:64 * j + 64]) == ecc.msm(pts, [k % Q for k in ks], "bucket", ecc.max_threads()), j
    assert (s1["builds"] - s0["builds"], s1["hits"] - s0["hits"]) == (1, 0)


# ---- 6. end to end -------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("m", [32, 64])
def test_aggregated_range_proof_2048_and_4096_generators(ipa_lib, m):
    """AggregNIRangeProver with 64-bit values: m = 32 gives an IPA of n = 2048 (table rounds), m = 64 one of n = 4096 (bucket
    rounds; AggregRangeVerifier then takes Verifier1 -> bp_ipa_verify1_eq_hs).  Proofs equal po.range_prove; decisions equal
    po.range_verify, for the proof and for a wrong V."""
    import test_gpu_protocols as tp
    from helpers import gens as hgens
    from python_bulletproofs_b200 import secp256k1
    from python_bulletproofs_b200.rangeproofs import AggregNIRangeProver, AggregRangeVerifier
    n = 64
    seeds = ["ipa_e2e%d_%d" % (m, i) for i in range(7)]
    ogs, ohs, og, oh, ou = hgens(n * m, seeds)
    gs, hs, g, h, u = [tp.P_(t) for t in ogs], [tp.P_(t) for t in ohs], tp.P_(og), tp.P_(oh), tp.P_(ou)
    rng = random.Random(m)
    vs = [rng.getrandbits(n) for _ in range(m)]
    vs[0], vs[-1] = 0, 2 ** n - 1
    gammas = [po.mod_hash(b"g%d" % j) for j in range(m)]
    want = po.range_prove(vs, n, og, oh, ogs, ohs, gammas, ou, seeds[6].encode())
    oVs = [po.commit(og, oh, v, gm) for v, gm in zip(vs, gammas)]
    for rep in range(2):
        proof = AggregNIRangeProver([tp.M_(v) for v in vs], n, g, h, gs, hs, [tp.M_(x) for x in gammas], u, secp256k1,
                                    seeds[6].encode()).prove()
        assert tp.range_json(proof) == po.range_to_json(want), rep
    Vs = [tp.P_(V) for V in oVs]
    Vbad = Vs[:-1] + [Vs[-1] + h]
    assert po.range_verify(oVs, og, oh, ogs, ohs, ou, want) is True
    assert po.range_verify(oVs[:-1] + [ecc.point_add(oVs[-1], oh)], og, oh, ogs, ohs, ou, want) is False
    for _ in range(2):
        assert tp.quiet(AggregRangeVerifier(Vs, g, h, gs, hs, u, proof).verify) is True
        assert tp.quiet(AggregRangeVerifier(Vbad, g, h, gs, hs, u, proof).verify) is False


# ---- oracle-side self-check (no GPU) -------------------------------------------------------------------------------------
def test_oracle_side_cases_are_what_they_claim():
    """The inputs above cause what they are built for: L or R of round 0 is the identity (slot AA==); x -> q - x keeps
    every x^2; the honest proof satisfies the oracle equation and the forgeries do not; a degenerate set is degenerate."""
    for kind, slot in (("L_identity", 1), ("R_identity", 2)):
        c = case(16, kind)
        c.want
        assert (c.proof["Ls"] if kind == "L_identity" else c.proof["Rs"])[0] is None
        assert c.proof["transcript"].split(b"&")[slot] == b"AA=="
    c = case(8, "scale_yinv")
    c.want
    Pt = statement(c)
    decisions = {}
    for label, Pf, a, b, xs, Ls, Rs in forgeries(c, Pt, True):
        decisions[label] = oracle_eq(c.S, c.hsc, c.S.u, Pf, c.n, a, b, xs, Ls, Rs)
        if label.endswith("q-x"):
            assert [x * x % Q for x in xs] == [x * x % Q for x in c.proof["xs"]]
    assert decisions.pop("honest") is True and not any(decisions.values())
    g = gens(8, "g_neg")
    assert ecc.msm(g.g, [1] * 8) is None
    u = case(8, "unreduced")
    assert any(x >= Q for x in u.a) and any(x >= Q for x in u.b) and 0 in u.a and 0 in u.b
    with contextlib.redirect_stdout(io.StringIO()):
        assert po.ipa_verify2(c.S.g, c.hsp, c.S.u, Pt, c.proof)
