"""Known-answer tests of the device arithmetic (fp.cuh, fq.cuh, ec.cuh) against Python big ints
and the CPU oracle.  Bit-exact."""
import random

import pytest

from oracle import ecc
from gpu_util import call_test

pytestmark = pytest.mark.gpu
P, Q = ecc.P, ecc.Q


def _le(vals):
    return b"".join(v.to_bytes(32, "little") for v in vals)


def _un(b):
    return [int.from_bytes(b[i:i + 32], "little") for i in range(0, len(b), 32)]


EDGE = [0, 1, 2, 977, 2 ** 32, 2 ** 32 + 977, P - 1, P - 2, P, P + 1, 2 ** 256 - 1, 2 ** 256 - 2, 2 ** 255, 2 ** 255 - 1,
        2 ** 256 - 2 ** 32 - 978, (1 << 224) - 1, 0xFFFFFFFF, 0xFFFFFFFF00000000, Q, Q - 1]


def _pairs(rng, n_rand, mod=None):
    a = list(EDGE) + [rng.getrandbits(256) for _ in range(n_rand)]
    pairs = [(x, y) for x in EDGE for y in EDGE] + [(a[rng.randrange(len(a))], rng.getrandbits(256)) for _ in range(n_rand)]
    return [p[0] for p in pairs], [p[1] for p in pairs]


@pytest.mark.parametrize("op,fn", [(0, lambda a, b: a * b % P), (1, lambda a, b: (a + b) % P), (2, lambda a, b: (a - b) % P),
                                   (4, lambda a, b: (-a) % P), (5, lambda a, b: a * a % P)])
def test_fp_ops_lazy_inputs(op, fn):
    """Inputs are arbitrary 256-bit residues (the device keeps lazy values in [0, 2^256))."""
    rng = random.Random(100 + op)
    a, b = _pairs(rng, 4000)
    got = _un(call_test("bp_test_fp", op, _le(a), _le(b), len(a), 32))
    assert got == [fn(x, y) for x, y in zip(a, b)]


def test_fp_inv():
    rng = random.Random(5)
    a = [1, 2, P - 1, P - 2, 977, 2 ** 255] + [rng.getrandbits(256) % P or 1 for _ in range(300)]
    got = _un(call_test("bp_test_fp", 3, _le(a), _le(a), len(a), 32))
    assert got == [pow(x, -1, P) for x in a]


def test_fp_inv_binary_gcd_and_sqrt():
    """fp_inv_gcd (single-thread tails) on canonical, lazy (>= p) and degenerate inputs; (sqrt(x^2))^2 == x^2."""
    rng = random.Random(6)
    a = [0, P, 1, 2, 3, P - 1, P - 2, P + 1, 2 ** 256 - 1, 977, 2 ** 255, 2 ** 32 + 977, (P + 1) // 2] + \
        [rng.getrandbits(256) for _ in range(600)] + [1 << k for k in range(0, 256, 7)]
    got = _un(call_test("bp_test_fp", 6, _le(a), _le(a), len(a), 32))
    assert got == [pow(x % P, -1, P) if x % P else 0 for x in a]
    got = _un(call_test("bp_test_fp", 7, _le(a), _le(a), len(a), 32))
    assert got == [x * x % P for x in a]


@pytest.mark.parametrize("dev", [0, 1])
@pytest.mark.parametrize("op,fn", [(0, lambda a, b: a * b % Q), (1, lambda a, b: (a + b) % Q), (2, lambda a, b: (a - b) % Q),
                                   (4, lambda a, b: (-a) % Q)])
def test_fq_ops(op, fn, dev):
    rng = random.Random(200 + op)
    a, b = _pairs(rng, 1500)
    got = _un(call_test("bp_test_fq", op, _le(a), _le(b), len(a), 32, dev))
    assert got == [fn(x % Q, y % Q) for x, y in zip(a, b)]


@pytest.mark.parametrize("dev", [0, 1])
def test_fq_inv(dev):
    rng = random.Random(6)
    a = [1, 2, Q - 1] + [rng.getrandbits(256) % Q or 1 for _ in range(100)]
    got = _un(call_test("bp_test_fq", 3, _le(a), _le(a), len(a), 32, dev))
    assert got == [pow(x, -1, Q) for x in a]


def test_fq_device_standard_form_arithmetic():
    """fqdev.cuh: product / square with the pseudo-Mersenne folds (q = 2^256 - c) and the windowed inversion, on operands
    chosen to exercise every fold (all-ones limbs, values just below q, products just above multiples of 2^256)."""
    rng = random.Random(77)
    edge = [0, 1, 2, Q - 1, Q - 2, (Q + 1) // 2, 2 ** 128, 2 ** 128 - 1, 2 ** 255, Q - 2 ** 128, 2 ** 256 - Q, 2 ** 129 + 12345]
    a = edge + [rng.getrandbits(256) % Q for _ in range(3000)]
    b = [Q - 1] * len(edge) + [rng.getrandbits(256) % Q for _ in range(3000)]
    a += edge; b += edge[::-1]
    got = _un(call_test("bp_test_fq", 5, _le(a), _le(b), len(a), 32, 1))
    assert got == [x * y % Q for x, y in zip(a, b)]
    got = _un(call_test("bp_test_fq", 7, _le(a), _le(a), len(a), 32, 1))
    assert got == [x * x % Q for x in a]
    inv_in = [1, 2, Q - 1, Q - 2, 2 ** 128] + [rng.getrandbits(256) % Q or 1 for _ in range(200)]
    got = _un(call_test("bp_test_fq", 6, _le(inv_in), _le(inv_in), len(inv_in), 32, 1))
    assert got == [pow(x, -1, Q) for x in inv_in]
    inv_in = [0] + inv_in + [1 << k for k in range(0, 256, 5)]                  # binary extended GCD form (0 -> 0)
    got = _un(call_test("bp_test_fq", 8, _le(inv_in), _le(inv_in), len(inv_in), 32, 1))
    assert got == [pow(x % Q, -1, Q) if x % Q else 0 for x in inv_in]


def test_ec_ops_including_exceptional_cases():
    rng = random.Random(9)
    base = [ecc.py_mul(ecc.G, rng.getrandbits(256)) for _ in range(24)]
    A, B = [], []
    for i, p in enumerate(base):
        q = base[(i + 7) % len(base)]
        A += [p, p, p, None, p, None]
        B += [q, p, ecc.point_neg(p), q, None, None]      # generic, doubling, inverse, identities
    pa, pb = ecc.pack_points(A), ecc.pack_points(B)
    n = len(A)
    want_add = [ecc.py_add(a, b) for a, b in zip(A, B)]
    for op in (0, 1, 10, 11):           # mixed add, full add, each also from a re-projected accumulator
        got = ecc.unpack_points(call_test("bp_test_ec", op, pa, pb, n, 64), n)
        assert got == want_add, op
    for op in (2, 12):
        got = ecc.unpack_points(call_test("bp_test_ec", op, pa, pb, n, 64), n)
        assert got == [ecc.py_add(a, a) for a in A], op
    got = ecc.unpack_points(call_test("bp_test_ec", 3, pa, pb, n, 64), n)
    assert got == [ecc.point_neg(a) for a in A]


def test_coop_ops_per_warp_case_mix():
    """coop_add / coop_dbl (coop4.cuh), one quad per pair, 8 quads per warp.  The doubling pass runs for the whole warp when any
    quad adds a point to itself, so the pairs are laid out warp by warp: all generic; one doubling quad (first, middle, last)
    among generic ones; all doublings; doubling, opposite, O + b, a + O and O + O side by side; and a last, partial warp that
    the kernel pads with identity pairs."""
    rng = random.Random(44)
    pool = [ecc.py_mul(ecc.G, rng.getrandbits(256)) for _ in range(40)]
    pick = lambda: pool[rng.randrange(len(pool))]            # noqa: E731

    def pair(kind):
        a = pick()
        if kind == "gen":
            b = pick()
            while b in (a, ecc.point_neg(a)):
                b = pick()
            return a, b
        return {"dbl": (a, a), "opp": (a, ecc.point_neg(a)), "Ob": (None, a), "aO": (a, None), "OO": (None, None)}[kind]

    warps = [["gen"] * 8] + [["gen"] * p + ["dbl"] + ["gen"] * (7 - p) for p in (0, 3, 7)] + [["dbl"] * 8]
    warps += [["dbl", "opp", "Ob", "aO", "OO", "gen", "dbl", "opp"], ["opp", "gen", "OO", "dbl", "aO", "gen", "Ob", "opp"],
              ["opp"] * 4 + ["Ob", "aO", "OO", "gen"], ["dbl", "Ob", "opp", "aO", "OO"]]
    A, B = [], []
    for w in warps:
        for kind in w:
            a, b = pair(kind)
            A.append(a); B.append(b)
    pa, pb, n = ecc.pack_points(A), ecc.pack_points(B), len(A)
    assert n % 8 == 5
    for op in (4, 14):
        got = ecc.unpack_points(call_test("bp_test_ec", op, pa, pb, n, 64), n)
        bad = [i for i in range(n) if got[i] != ecc.py_add(A[i], B[i])]
        assert not bad, (op, [(i // 8, warps[i // 8][i % 8]) for i in bad])
    for op in (5, 15):
        got = ecc.unpack_points(call_test("bp_test_ec", op, pa, pb, n, 64), n)
        assert got == [ecc.py_add(a, a) for a in A], op


# ---- batched lift-x / decompression / generator derivation (SURVEY 8(f) N4) -------------------------------------
def test_lift_x_batch_matches_big_int_square_roots():
    from python_bulletproofs_b200 import _native as nat
    rng = random.Random(0x11F7)
    xs = [rng.getrandbits(256) for _ in range(700)] + [0, 1, 2, P - 1, P, P + 5, 2 ** 256 - 1, ecc.GX]
    want = bytes(rng.randrange(4) for _ in xs)
    got = nat.lift_x_batch(xs, want)
    n_on = 0
    for x, w, xy in zip(xs, want, got):
        rhs = (x * x * x + 7) % P
        y = pow(rhs, (P + 1) // 4, P)
        if x >= P or y * y % P != rhs:
            assert xy is None, hex(x)
            continue
        n_on += 1
        if w == 0:
            y = y if y % 2 == 0 else P - y
        elif w == 1:
            y = y if y % 2 == 1 else P - y
        elif w == 3:
            y = P - y
        assert xy == (x, y), hex(x)
    assert 250 < n_on < 500                                    # about half of all x are on the curve
    assert nat.lift_x_batch([ecc.GX], None) in ([(ecc.GX, ecc.GY)], [(ecc.GX, P - ecc.GY)])
    assert nat.lift_x_batch([]) == []


def test_elliptic_hash_batch_equals_reference_derivation():
    from oracle import protocol_oracle as po
    from python_bulletproofs_b200.curve import secp256k1
    from python_bulletproofs_b200.utils import elliptic_hash, elliptic_hash_batch
    msgs = [b"seed%d" % (i % 7) + str(i).encode() for i in range(400)] + [b"", b"\x00" * 64]
    got = elliptic_hash_batch(msgs, secp256k1)
    assert len(got) == len(msgs)
    for m, g in zip(msgs, got):
        assert (g.x, g.y) == po.elliptic_hash(m), m            # oracle: pinned by the reference's golden generators
    for m, g in list(zip(msgs, got))[:20]:
        h = elliptic_hash(m, secp256k1)
        assert (g.x, g.y) == (h.x, h.y)


def test_bytes_to_points_decompresses_like_bytes_to_point():
    from python_bulletproofs_b200.utils import bytes_to_point, bytes_to_points, point_to_bytes, point_to_b64, b64_to_points
    from python_bulletproofs_b200.point import Point
    from python_bulletproofs_b200.curve import secp256k1
    from helpers import fast_points
    pts = [Point(x, y, secp256k1) for x, y in fast_points(200, 77)]
    enc = [point_to_bytes(p) for p in pts]
    dec = bytes_to_points(enc)
    assert [(p.x, p.y) for p in dec] == [(p.x, p.y) for p in pts]
    assert [(p.x, p.y) for p in dec[:10]] == [(q.x, q.y) for q in map(bytes_to_point, enc[:10])]
    assert [(p.x, p.y) for p in b64_to_points([point_to_b64(p) for p in pts[:50]])] == [(p.x, p.y) for p in pts[:50]]
    with pytest.raises(ValueError):
        bytes_to_points([b"\x02" + (5).to_bytes(32, "big")])     # x = 5: x^3 + 7 = 132 is not a square mod p


def test_point_add_entry_point_is_complete():
    """bp_point_add (Point.__add__): random pairs and every exceptional case of the group law vs the oracle."""
    from python_bulletproofs_b200 import _native as nat
    from helpers import fast_points
    import ctypes
    pts = fast_points(24, 31337)
    P0, P1 = pts[0], pts[1]
    cases = [(P0, P1), (P0, P0), (P0, (P0[0], P - P0[1])), (None, P0), (P0, None), (None, None)] + list(zip(pts[2:13], pts[13:24]))
    lib = nat.load()
    out = ctypes.create_string_buffer(64)
    for a, b in cases:
        nat.check(lib.bp_point_add(ecc.pack_point(a), ecc.pack_point(b), out))
        assert ecc.unpack_point(out.raw) == ecc.py_add(a, b), (a, b)
