"""Parity of the CUDA multi-scalar multiplication (bp_msm & friends, through the C ABI) with
the golden outputs of the reference's Pippenger.multiexp and with the CPU oracle.  Bit-exact
affine outputs."""
import ctypes
import random

import pytest

from oracle import ecc, protocol_oracle as po
from python_bulletproofs_b200 import _native as nat
from helpers import c3_inputs, explicit_case, fast_points
from gpu_util import gpu_msm, gpu_msm_raw

pytestmark = pytest.mark.gpu
Q = ecc.Q


def test_msm_golden_reference_outputs(golden):
    """Every vector recorded from the unmodified reference (tests/golden/msm.json)."""
    for case in golden("msm")["cases"]:
        pts, ks = c3_inputs(case["lgn"], case["n"]) if case["kind"] == "c3" else explicit_case(case)
        got = gpu_msm(pts, ks)
        assert po.enc_point(got).hex() == case["out"], case.get("name", case.get("lgn"))


@pytest.mark.parametrize("c", [1, 2, 3, 4, 5, 7, 8, 11, 13, 16])
def test_msm_every_window_size(c):
    pts, ks = c3_inputs(7)
    want = ecc.msm(pts, ks)
    lib = nat.load()
    try:
        nat.check(lib.bp_msm_set_window(c))
        assert gpu_msm(pts, ks) == want
        assert lib.bp_msm_last_window() == c
    finally:
        lib.bp_msm_set_window(0)


@pytest.mark.parametrize("n", [1, 2, 5, 31, 32, 33, 255, 256, 257, 1000, 4096, 5000])
def test_msm_vs_oracle_sizes(n):
    rng = random.Random(n)
    pts = fast_points(n, 1000 + n)
    ks = [rng.getrandbits(256) for _ in range(n)]          # unreduced: the device reduces mod q
    assert gpu_msm(pts, ks) == ecc.msm(pts, ks)


def test_msm_adversarial_scalars():
    """Range-proof shaped inputs (rangeproof_prover.py:42-47,83): huge buckets, 0/1/q-1 scalars,
    repeated points, P and -P in one bucket."""
    n = 2048
    pts = fast_points(n, 77)
    rng = random.Random(3)
    z = rng.getrandbits(256) % Q
    cases = {
        "all_same_scalar": [z] * n,
        "bits_and_minus_one": [rng.getrandbits(1) for _ in range(n // 2)] + [Q - 1 if rng.getrandbits(1) else 0 for _ in range(n // 2)],
        "all_zero": [0] * n,
        "all_q_minus_1": [Q - 1] * n,
        "small": [rng.randrange(0, 5) for _ in range(n)],
        "half_q": [(Q // 2) + rng.randrange(-2, 3) for _ in range(n)],
        "pow2": [1 << rng.randrange(0, 256) for _ in range(n)],
    }
    for name, ks in cases.items():
        assert gpu_msm(pts, ks) == ecc.msm(pts, ks), name
    same_pt = [pts[0]] * n
    ks = [rng.getrandbits(256) for _ in range(n)]
    assert gpu_msm(same_pt, ks) == ecc.msm(same_pt, ks)
    cancel = pts[:n // 2] + [ecc.point_neg(p) for p in pts[:n // 2]]
    ks2 = ks[:n // 2] * 2
    assert gpu_msm(cancel, ks2) is None
    with_ident = [None if i % 3 == 0 else p for i, p in enumerate(pts)]
    assert gpu_msm(with_ident, ks) == ecc.msm(with_ident, ks)


@pytest.mark.parametrize("lgn", [14, 16])
def test_msm_large_vs_oracle(lgn):
    n = 1 << lgn
    pts = fast_points(n, lgn)
    pb = ecc.pack_points(pts)
    rng = random.Random(lgn)
    sb = bytes(rng.getrandbits(8) for _ in range(32 * n))
    assert gpu_msm_raw(pb, sb, n) == ecc.msm_bytes(pb, sb, n, "bucket", ecc.max_threads())


@pytest.mark.parametrize("n", [(1 << 17), (1 << 17) + 3, 300001])
def test_host_operand_msm_in_two_halves(n):
    """bp_msm with >= 2^17 host terms uploads its operands in parts and sorts and accumulates each part while the next is on
    the wire (msm_run_parts): same result as the device-resident path and the oracle, odd sizes and hot buckets included."""
    base = fast_points(1 << 10, 777)
    rng = random.Random(n)
    pb = b"".join(ecc.pack_point(base[rng.randrange(len(base))]) for _ in range(n))
    ks = [rng.getrandbits(256) for _ in range(n)]
    for i in range(0, n, 7):
        ks[i] = (1, 0, Q - 1, 2 ** 128, 5)[(i // 7) % 5]           # many equal scalars: giant buckets in every part
    sb = b"".join(k.to_bytes(32, "little") for k in ks)
    got = gpu_msm_raw(pb, sb, n)
    assert got == ecc.msm_bytes(pb, sb, n, "bucket", ecc.max_threads())
    lib = nat.load()
    hp = ctypes.c_uint64()
    nat.check(lib.bp_points_upload(pb, n, ctypes.byref(hp)))
    out = ctypes.create_string_buffer(64)
    nat.check(lib.bp_msm_h(hp, sb, n, out))
    assert ecc.unpack_point(out.raw) == got
    lib.bp_handle_free(hp)


@pytest.mark.parametrize("n", [(1 << 17) + 12345, (1 << 17), 300007])
def test_msm_host_operands_in_parts(n):
    """bp_msm with HOST operands of >= 2^17 terms takes them as K x [scalars | points], sorts every part on a side stream and
    accumulates all parts into one bucket set (msm_run_parts): odd sizes (uneven parts), repeated points (P + P across parts),
    P and -P, identity points, adversarial scalars -- against the oracle."""
    base = fast_points(64, 99)
    rng = random.Random(n)
    pts = [base[rng.randrange(64)] for _ in range(n)]
    for i in range(0, n, 1001):
        pts[i] = None
    for i in range(5, n, 4099):
        pts[i] = ecc.point_neg(pts[i - 1]) if pts[i - 1] is not None else pts[i]
    ks = [rng.getrandbits(256) for _ in range(n)]
    for i in range(0, n, 53):
        ks[i] = [0, 1, Q - 1, Q, 2 ** 256 - 1, 2 ** 128, ks[1]][(i // 53) % 7]
    pb = ecc.pack_points(pts)
    sb = b"".join(k.to_bytes(32, "little") for k in ks)
    want = ecc.msm_bytes(pb, sb, n, "bucket", ecc.max_threads())
    for _ in range(2):
        assert gpu_msm_raw(pb, sb, n) == want


def test_msm_full_size_properties():
    """BASELINE size 2^20: slice additivity + linearity + agreement with the multi-threaded oracle."""
    n = 1 << 20
    base = fast_points(1 << 12, 4242)
    rng = random.Random(20)
    pb = b"".join(ecc.pack_point(base[rng.randrange(len(base))]) for _ in range(n))
    sb = rng.randbytes(32 * n)
    lib = nat.load()
    hp, hs = ctypes.c_uint64(), ctypes.c_uint64()
    nat.check(lib.bp_points_upload(pb, n, ctypes.byref(hp)))
    nat.check(lib.bp_scalars_upload(sb, n, ctypes.byref(hs)))
    out = ctypes.create_string_buffer(64)
    nat.check(lib.bp_msm_hh(hp, hs, n, out))
    full = ecc.unpack_point(out.raw)
    # same through the host-buffer entry point and the host-scalar entry point
    assert gpu_msm_raw(pb, sb, n) == full
    nat.check(lib.bp_msm_h(hp, sb, n, out))
    assert ecc.unpack_point(out.raw) == full
    # slice additivity: sum of 3 uneven XYZZ partials == full
    cuts = [0, 300001, 777777, n]
    parts = b""
    part = ctypes.create_string_buffer(128)
    for lo, hi in zip(cuts, cuts[1:]):
        nat.check(lib.bp_msm_hh_partial(hp, hs, lo, hi - lo, part))
        parts += part.raw
    nat.check(lib.bp_xyzz_sum(parts, 3, out))
    assert ecc.unpack_point(out.raw) == full
    # oracle (bucket method, all host threads)
    assert ecc.msm_bytes(pb, sb, n, "bucket", ecc.max_threads()) == full
    lib.bp_handle_free(hp)
    lib.bp_handle_free(hs)


def test_msm_batch_matches_singles():
    rng = random.Random(8)
    sizes = [0, 1, 2, 12, 129, 64, 0, 257, 5]
    pts, ks, offsets = [], [], [0]
    for s in sizes:
        pts += fast_points(s, 500 + s)
        ks += [rng.getrandbits(256) for _ in range(s)]
        offsets.append(len(pts))
    raw = nat.msm_batch_bytes(ecc.pack_points(pts), b"".join(k.to_bytes(32, "little") for k in ks), offsets)
    for j, s in enumerate(sizes):
        lo, hi = offsets[j], offsets[j + 1]
        assert ecc.unpack_point(raw[64 * j:64 * j + 64]) == ecc.msm(pts[lo:hi], ks[lo:hi]), j


def test_scalar_mul_batch():
    n = 300
    rng = random.Random(12)
    pts = fast_points(n, 13)
    pts[5] = None
    ks = [rng.getrandbits(256) for _ in range(n)]
    ks[0], ks[1], ks[2] = 0, 1, Q - 1
    raw = nat.scalar_mul_batch_bytes(ecc.pack_points(pts), b"".join(k.to_bytes(32, "little") for k in ks), n)
    assert ecc.unpack_points(raw, n) == ecc.scalar_mul_batch(pts, ks)


def test_pippenger_dropin_api():
    """Same call / error behaviour as src/pippenger/pippenger.py:22-29."""
    from python_bulletproofs_b200.pippenger import PipSECP256k1
    from python_bulletproofs_b200 import Point, secp256k1
    from python_bulletproofs_b200.utils import ModP
    pts, ks = c3_inputs(5)
    P = [Point(x, y, secp256k1) for x, y in pts]
    r = PipSECP256k1.multiexp(P, [ModP(k, Q) for k in ks])
    assert (r.x, r.y) == ecc.msm(pts, ks)
    assert PipSECP256k1.multiexp([], []) == Point.IDENTITY_ELEMENT
    with pytest.raises(Exception, match="Different number of group elements and exponents"):
        PipSECP256k1.multiexp(P, ks[:-1])
    assert (P[0] + P[1]) == Point(*ecc.py_add(pts[0], pts[1]), secp256k1)
    assert (5 * P[0]) == (P[0] * 5) == Point(*ecc.py_mul(pts[0], 5), secp256k1)
    assert P[0] + (-P[0]) == Point.IDENTITY_ELEMENT


def test_device_resident_handles_and_forced_windows():
    """DevicePoints / DeviceScalars through Pippenger.multiexp, with the automatic and with forced windows, must return the
    oracle's point."""
    from python_bulletproofs_b200.pippenger import PipSECP256k1
    from python_bulletproofs_b200.device import DevicePoints, DeviceScalars
    from python_bulletproofs_b200 import Point, secp256k1
    n = 1 << 15
    pts = fast_points(n, 31)
    rng = random.Random(32)
    ks = [rng.getrandbits(256) for _ in range(n)]
    want = ecc.msm(pts, ks, "bucket", ecc.max_threads())
    dp = DevicePoints(raw=ecc.pack_points(pts))
    ds = DeviceScalars(ks)
    r = PipSECP256k1.multiexp(dp, ds)
    assert (r.x, r.y) == want
    r = PipSECP256k1.multiexp(dp, ks)
    assert (r.x, r.y) == want
    lib = nat.load()
    try:
        for c in (8, 13, 16):
            nat.check(lib.bp_msm_set_window(c))
            r = PipSECP256k1.multiexp(dp, ds)
            assert (r.x, r.y) == want, c
    finally:
        lib.bp_msm_set_window(0)
    dp.free(); ds.free()


@pytest.mark.parametrize("c", [0, 8, 11, 16, 19, 20])
def test_msm_precomputed_window_multiples(c):
    """bp_points_precompute: the MSM over a handle that carries 2^(c*w) * P_i (one shared bucket unit, no doublings) returns
    the same canonical point as the plain path and the oracle -- full vector, slices, adversarial scalars, identity points."""
    from python_bulletproofs_b200.device import DevicePoints, DeviceScalars
    n = 3000
    pts = fast_points(n, 4242)
    pts[7] = None                                        # an identity among the points
    pts[100] = pts[101]                                  # a repeated point
    pts[200] = ecc.point_neg(pts[201])                   # P and -P
    rng = random.Random(c)
    lib = nat.load()
    dp = DevicePoints(raw=ecc.pack_points(pts)).precompute(c)
    wb, nw, nbytes = ctypes.c_int(), ctypes.c_int(), ctypes.c_uint64()
    nat.check(lib.bp_points_pre_info(dp.handle, ctypes.byref(wb), ctypes.byref(nw), ctypes.byref(nbytes)))
    assert wb.value == (c or wb.value) and nw.value == (257 + wb.value - 1) // wb.value and nbytes.value == nw.value * n * 64
    out = ctypes.create_string_buffer(64)
    scalar_sets = {
        "uniform": [rng.getrandbits(256) for _ in range(n)],                      # unreduced: reduced on the device
        "edge": [[0, 1, Q - 1, Q, Q + 1, 2 ** 256 - 1, 2 ** 255, (Q - 1) // 2, (Q + 1) // 2, 2 ** 128][i % 10] for i in range(n)],
        "same": [rng.getrandbits(256) % Q] * n,
        "top_window": [(Q - 1) - rng.randrange(0, 1 << 20) for _ in range(n)],
        "pow2": [1 << rng.randrange(0, 256) for _ in range(n)],
    }
    for name, ks in scalar_sets.items():
        sb = b"".join(int(k % 2 ** 256).to_bytes(32, "little") for k in ks)
        want = ecc.msm(pts, [k % Q for k in ks])
        nat.check(lib.bp_msm_h(dp.handle, sb, n, out))
        assert ecc.unpack_point(out.raw) == want, name
        assert lib.bp_msm_last_window() == wb.value
        ds = DeviceScalars(raw=sb)
        nat.check(lib.bp_msm_hh(dp.handle, ds.handle, n, out))
        assert ecc.unpack_point(out.raw) == want, name
        # a slice in the middle of the vector (XYZZ partial) and a prefix
        part = ctypes.create_string_buffer(128)
        nat.check(lib.bp_msm_hh_partial(dp.handle, ds.handle, 500, 1234, part))
        nat.check(lib.bp_xyzz_sum(part.raw, 1, out))
        assert ecc.unpack_point(out.raw) == ecc.msm(pts[500:1734], [k % Q for k in ks[500:1734]]), name
        nat.check(lib.bp_msm_hh(dp.handle, ds.handle, 33, out))
        assert ecc.unpack_point(out.raw) == ecc.msm(pts[:33], [k % Q for k in ks[:33]]), name
        ds.free()
    # a forced window switches back to the plain bucket method on the same handle
    try:
        nat.check(lib.bp_msm_set_window(13))
        sb = b"".join(int(k).to_bytes(32, "little") for k in scalar_sets["uniform"])
        nat.check(lib.bp_msm_h(dp.handle, sb, n, out))
        assert ecc.unpack_point(out.raw) == ecc.msm(pts, [k % Q for k in scalar_sets["uniform"]])
    finally:
        lib.bp_msm_set_window(0)
    dp.free()


@pytest.mark.parametrize("kind", ["few_values", "pairs_cancel", "uniform", "sparse", "small"])
@pytest.mark.parametrize("c", [8, 11])
def test_msm_precomputed_deep_and_cancelling_buckets(c, kind):
    """Precomputed path on a small vector whose buckets stress the XYZZ accumulation: repeated points with equal scalars (P + P
    in one bucket), P and -P neighbours (sums that cancel to the identity, then identity + point), identity inputs, few distinct
    or all-equal scalars (one deep bucket per window), zero scalars (empty buckets) -- full length and prefixes, against the oracle."""
    from python_bulletproofs_b200.device import DevicePoints
    n = 2500
    pool = fast_points(12, 777)
    rng = random.Random(1000 * c)
    pts = [pool[rng.randrange(12)] for _ in range(n)]                 # 12 distinct points: most pairs inside a bucket are P + P
    for i in range(0, n, 7):
        pts[i] = ecc.point_neg(pts[i - 1]) if i else pts[i]           # P, -P neighbours
    pts[5] = None; pts[6] = None
    lib = nat.load()
    dp = DevicePoints(raw=ecc.pack_points(pts)).precompute(c)
    out = ctypes.create_string_buffer(64)
    few = [rng.getrandbits(256) % Q for _ in range(3)]
    scalar_sets = {
        "few_values": [few[rng.randrange(3)] for _ in range(n)],
        "pairs_cancel": [few[0]] * n,
        "uniform": [rng.getrandbits(256) for _ in range(n)],
        "sparse": [0 if i % 5 else rng.getrandbits(256) for i in range(n)],
        "small": [rng.randrange(0, 4) for _ in range(n)],
    }
    ks = scalar_sets[kind]
    sb = b"".join(int(k % 2 ** 256).to_bytes(32, "little") for k in ks)
    nat.check(lib.bp_msm_h(dp.handle, sb, n, out))
    assert ecc.unpack_point(out.raw) == ecc.msm(pts, [k % Q for k in ks])
    for m in (1, 2, 31, 1025):
        nat.check(lib.bp_msm_h(dp.handle, sb, m, out))
        assert ecc.unpack_point(out.raw) == ecc.msm(pts[:m], [k % Q for k in ks[:m]]), m
    dp.free()


def test_msm_precomputed_2p18_vs_plain_and_oracle():
    n = 1 << 18
    from python_bulletproofs_b200.device import DevicePoints, DeviceScalars
    lib = nat.load()
    rng = random.Random(18)
    base = nat.scalar_mul_batch_bytes(nat.pack_xy(*ecc.G) * n, rng.randbytes(32 * n), n)
    sb = rng.randbytes(32 * n)
    dp, ds = DevicePoints(raw=base), DeviceScalars(raw=sb)
    out = ctypes.create_string_buffer(64)
    nat.check(lib.bp_msm_hh(dp.handle, ds.handle, n, out))
    plain = out.raw
    dp.precompute(0)
    nat.check(lib.bp_msm_hh(dp.handle, ds.handle, n, out))
    assert out.raw == plain
    assert ecc.pack_point(ecc.msm_bytes(base, sb, n, "bucket", ecc.max_threads())) == plain
    dp.free(); ds.free()


def test_msm_2p18_resident_precomputed_host_parts_and_small_graph():
    """One 2^18-term MSM four ways, each bit-identical to the oracle: resident operands on the plain path (nine wide bucket units)
    and on the precomputed path, host operands (uploaded, sorted and accumulated in parts), and an odd-length prefix that takes
    the precomputed vector's small-graph path."""
    n = 1 << 18
    from python_bulletproofs_b200.device import DevicePoints, DeviceScalars
    lib = nat.load()
    rng = random.Random(181)
    base = nat.scalar_mul_batch_bytes(nat.pack_xy(*ecc.G) * n, rng.randbytes(32 * n), n)
    sb = rng.randbytes(32 * n)
    want = ecc.pack_point(ecc.msm_bytes(base, sb, n, "bucket", ecc.max_threads()))
    dp, ds, dq = DevicePoints(raw=base), DeviceScalars(raw=sb), DevicePoints(raw=base).precompute(0)
    out = ctypes.create_string_buffer(64)
    nat.check(lib.bp_msm_hh(dp.handle, ds.handle, n, out)); assert out.raw == want, "plain"
    nat.check(lib.bp_msm_hh(dq.handle, ds.handle, n, out)); assert out.raw == want, "pre"
    nat.check(lib.bp_msm(base, sb, n, out)); assert out.raw == want, "host operands"
    m = (1 << 16) + 77                                                # small-graph path of the precomputed vector, odd length
    nat.check(lib.bp_msm_hh(dq.handle, ds.handle, m, out))
    assert out.raw == ecc.pack_point(ecc.msm_bytes(base, sb, m, "bucket", ecc.max_threads())), m
    dp.free(); ds.free(); dq.free()


def test_msm_slot_sort_and_its_fallback():
    """Sort stage of the precomputed path (msm.cuh, k_scatter_slots_pre / k_accumulate_slots): slot sort on, off, and with 8 slots per
    bucket so that every bucket overflows and the gated exact counting sort does the work; uniform scalars, scalars with thousands
    of equal digits (overflow with the regular slot count), all-zero and single-term corner cases -- bit-identical points."""
    n = 1 << 18
    from python_bulletproofs_b200.device import DevicePoints
    lib = nat.load()
    rng = random.Random(182)
    base = nat.scalar_mul_batch_bytes(nat.pack_xy(*ecc.G) * n, rng.randbytes(32 * n), n)
    few = [rng.getrandbits(256) % Q for _ in range(3)]
    sets = {
        "uniform": rng.randbytes(32 * n),
        "few_values": b"".join(few[rng.randrange(3)].to_bytes(32, "little") for _ in range(n)),          # 3 hot buckets per window
        "small": b"".join(rng.randrange(0, 1 << 20).to_bytes(32, "little") for _ in range(n)),             # only the low windows
        "zero": bytes(32 * n),
    }
    want = {name: ecc.pack_point(ecc.msm_bytes(base, sb, n, "bucket", ecc.max_threads())) for name, sb in sets.items()}
    dq = DevicePoints(raw=base).precompute(0)
    dp = DevicePoints(raw=base)                                          # plain path: k_digits_slots, k_accumulate_slots<true>
    out = ctypes.create_string_buffer(64)
    try:
        for mode in (1, 2, 0):
            nat.check(lib.bp_msm_set_pre_slots(mode, 1 << 12))
            for name, sb in sets.items():
                nat.check(lib.bp_msm_h(dq.handle, sb, n, out)); assert out.raw == want[name], (mode, name)
                nat.check(lib.bp_msm_h(dp.handle, sb, n, out)); assert out.raw == want[name], (mode, name, "plain")
            m = 5000                                                      # short vector, above the lowered threshold
            nat.check(lib.bp_msm_h(dq.handle, sets["uniform"], m, out))
            assert out.raw == ecc.pack_point(ecc.msm_bytes(base, sets["uniform"], m, "bucket", ecc.max_threads())), (mode, m)
    finally:
        lib.bp_msm_set_pre_slots(1, 1 << 18)
    dq.free(); dp.free()
