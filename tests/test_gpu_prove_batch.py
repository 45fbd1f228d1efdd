"""Batch range-proof prover (bp_rp_prove_batch, prove_range_proofs_packed / prove_range_proofs_batch) against the per-proof
provers NIRangeProver / AggregNIRangeProver and the golden proofs recorded from the reference: every field, all three
transcripts, and the packed records byte for byte; then the packed output straight into the batch verifiers."""
import ctypes
import random

import pytest

from oracle import ecc, protocol_oracle as po
from helpers import gens
from python_bulletproofs_b200 import Point, secp256k1, _native as nat
from python_bulletproofs_b200.utils import ModP, commitment, mod_hash
from python_bulletproofs_b200.rangeproofs import (NIRangeProver, AggregNIRangeProver, prove_range_proofs_packed,
                                                   prove_range_proofs_batch)
from python_bulletproofs_b200.rangeproofs.batch import (pack_aggreg_proof, pack_generators, verify_packed, verify_aggreg_packed,
                                                         verify_rlc_packed, verify_stats, unpack_aggreg_proofs)

pytestmark = pytest.mark.gpu
Q = ecc.Q


def P_(t):
    return Point.IDENTITY_ELEMENT if t is None else Point(t[0], t[1], secp256k1)


def T_(p):
    return None if p.curve is None else (p.x, p.y)


def generators(N, tag):
    gs, hs, g, h, u = gens(N, [tag + str(i) for i in range(5)])
    return [P_(t) for t in gs], [P_(t) for t in hs], P_(g), P_(h), P_(u)


def range_json(pr):
    """The golden files' form of a range proof (as tests/test_gpu_protocols.py)."""
    p1, p2 = pr.innerProof, pr.innerProof.proof2
    return {"taux": str(pr.taux.x), "mu": str(pr.mu.x), "t_hat": str(pr.t_hat.x),
            "T1": po.enc_point(T_(pr.T1)).hex(), "T2": po.enc_point(T_(pr.T2)).hex(),
            "A": po.enc_point(T_(pr.A)).hex(), "S": po.enc_point(T_(pr.S)).hex(),
            "transcript": pr.transcript.decode("latin1"),
            "ip": {"u_new": po.enc_point(T_(p1.u_new)).hex(), "P_new": po.enc_point(T_(p1.P_new)).hex(),
                   "transcript": p1.transcript.decode("latin1"),
                   "p2": po.proof2_to_json({"a": p2.a.x, "b": p2.b.x, "xs": [x.x for x in p2.xs], "Ls": [T_(p) for p in p2.Ls],
                                            "Rs": [T_(p) for p in p2.Rs], "transcript": p2.transcript,
                                            "start": p2.start_transcript})}}


def fields(pr):
    """Every field of a proof, reduced where the reference's ModP may carry an unreduced value."""
    p1, p2 = pr.innerProof, pr.innerProof.proof2
    return (pr.taux.x % Q, pr.mu.x % Q, pr.t_hat.x % Q, T_(pr.T1), T_(pr.T2), T_(pr.A), T_(pr.S), pr.transcript,
            T_(p1.u_new), T_(p1.P_new), p1.transcript, p2.a.x % Q, p2.b.x % Q, [x.x % Q for x in p2.xs],
            [T_(p) for p in p2.Ls], [T_(p) for p in p2.Rs], p2.transcript, p2.start_transcript)


def reference(vs, n, g, h, gs, hs, gammas, u, seed):
    if len(vs) == 1:
        return NIRangeProver(vs[0], n, g, h, gs, hs, gammas[0], u, secp256k1, seed).prove()
    return AggregNIRangeProver(vs, n, g, h, gs, hs, gammas, u, secp256k1, seed).prove()


def random_inputs(count, n, m, rng, tag):
    vs = [[ModP(rng.getrandbits(n), Q) for _ in range(m)] for _ in range(count)]
    gammas = [[ModP(rng.getrandbits(256) % Q, Q) for _ in range(m)] for _ in range(count)]
    seeds = [("%s-%d" % (tag, i)).encode() for i in range(count)]
    return vs, gammas, seeds


def check_against_reference(batch, proofs, idx, vs, n, g, h, gs, hs, gammas, u, seeds):
    """Proof idx of a batch equals the per-proof prover's: every field, and its record / transcripts byte for byte."""
    ref = reference(vs[idx], n, g, h, gs, hs, gammas[idx], u, seeds[idx])
    assert fields(proofs[idx]) == fields(ref), idx
    Vs = [commitment(g, h, v, gm) for v, gm in zip(vs[idx], gammas[idx])]
    L = (n * len(vs[idx])).bit_length() - 1
    rec, trio, start = pack_aggreg_proof(Vs, ref, L)
    assert batch.records[idx * batch.stride:(idx + 1) * batch.stride] == rec, idx
    offs = [batch.tr_off[3 * idx + k] for k in range(4)]
    assert tuple(batch.blob[offs[k]:offs[k + 1]] for k in range(3)) == trio, idx
    assert batch.starts[idx] == start


def sample(count):
    return sorted(set(range(0, count, 37)) | {0, count - 1})


# ---- 1. golden proofs at a middle position of a batch ---------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["range_small", "range_c1", "aggreg_small", "aggreg_c4"])
def test_golden_inside_batch(golden, name):
    rng = random.Random(name)
    for case in golden(name)["cases"]:
        n, m = case["n"], case.get("m", 1)
        raw = gens(n * m, case["seeds"])
        gs, hs, g, h, u = [P_(t) for t in raw[0]], [P_(t) for t in raw[1]], P_(raw[2]), P_(raw[3]), P_(raw[4])
        if m == 1 and "vs" not in case:
            vs0, gm0 = [ModP(int(case["v"]), Q)], [mod_hash(case["seeds"][5].encode(), Q)]
            want_V = [case["V"]]
        else:
            vs0, gm0 = [ModP(int(v), Q) for v in case["vs"]], [ModP(int(x), Q) for x in case["gammas"]]
            want_V = case["Vs"]
        vs, gammas, seeds = random_inputs(5, n, m, rng, name)
        vs[2], gammas[2], seeds[2] = vs0, gm0, case["seeds"][6].encode()
        batch = prove_range_proofs_packed(vs, n, g, h, gs, hs, gammas, u, seeds)
        proofs = unpack_aggreg_proofs(batch)
        assert range_json(proofs[2]) == case["proof"]
        got_V = [po.enc_point(T_(Point.from_bytes64(batch.records, 2 * batch.stride + 64 * j))).hex() for j in range(m)]
        assert got_V == want_V
        check_against_reference(batch, proofs, 1, vs, n, g, h, gs, hs, gammas, u, seeds)


# ---- 2. shapes, including (1, 1) with no IPA round -----------------------------------------------------------------------------
@pytest.mark.parametrize("n,m", [(1, 1), (2, 1), (8, 1), (64, 1), (8, 2), (4, 8), (32, 4), (64, 16)])
def test_shapes_equal_per_proof_prover(n, m):
    rng = random.Random(n * 100 + m)
    gs, hs, g, h, u = generators(n * m, "shape%d_%d_" % (n, m))
    vs, gammas, seeds = random_inputs(3, n, m, rng, "shape")
    batch = prove_range_proofs_packed(vs, n, g, h, gs, hs, gammas, u, seeds)
    assert batch.nproofs == 3 and batch.m == m and batch.n == n
    proofs = unpack_aggreg_proofs(batch)
    for i in range(3):
        check_against_reference(batch, proofs, i, vs, n, g, h, gs, hs, gammas, u, seeds)
    # the list-level function returns the same objects
    assert [fields(p) for p in prove_range_proofs_batch(vs, n, g, h, gs, hs, gammas, u, seeds)] == [fields(p) for p in proofs]


# ---- 3. chunk plans: 1, 2 (a last chunk of one proof) and 4 chunks -------------------------------------------------------------
@pytest.mark.parametrize("count,chunks", [(40, 1), (65, 2), (300, 4)])
def test_chunking(count, chunks):
    n = 8
    rng = random.Random(count)
    gs, hs, g, h, u = generators(n, "chunk")
    vs, gammas, seeds = random_inputs(count, n, 1, rng, "chunk%d" % count)
    batch = prove_range_proofs_packed(vs, n, g, h, gs, hs, gammas, u, seeds, packed=pack_generators(g, h, gs, hs, u))
    st = verify_stats()
    assert st["chunks"] == chunks and st["proofs"] == count
    proofs = unpack_aggreg_proofs(batch)
    for i in sample(count):
        check_against_reference(batch, proofs, i, vs, n, g, h, gs, hs, gammas, u, seeds)
    acc, combined = verify_rlc_packed(batch, g, h, gs, hs, u, seed=bytes(32))
    assert combined == 1 and acc == b"\x01" * count


# ---- 4. table paths ---------------------------------------------------------------------------------------------------------------
def test_table_modes_give_identical_bytes():
    """Bucket method (mode 0), table from the second call on (mode 1), table at first sight (mode 2): the same bytes."""
    n, m, count = 16, 2, 70
    rng = random.Random(4)
    gs, hs, g, h, u = generators(n * m, "tables")
    vs, gammas, seeds = random_inputs(count, n, m, rng, "tables")
    lib = nat.load()
    outs = []
    try:
        for mode, want_modes in ((0, [0]), (1, [0, 1]), (2, [1])):
            nat.check(lib.bp_fb_clear())                      # every mode starts from a set no call has seen
            nat.check(lib.bp_fb_set_mode(mode))
            for want in want_modes:
                outs.append(prove_range_proofs_packed(vs, n, g, h, gs, hs, gammas, u, seeds))
                assert verify_stats()["table_mode"] == want, (mode, want)
    finally:
        lib.bp_fb_set_mode(1)
    assert all(b.records == outs[0].records and b.blob == outs[0].blob for b in outs)
    proofs = unpack_aggreg_proofs(outs[0])
    for i in (0, count - 1):
        check_against_reference(outs[0], proofs, i, vs, n, g, h, gs, hs, gammas, u, seeds)


# ---- 5. edge inputs -------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("m", [1, 2])
def test_edge_inputs(m):
    n = 8
    gs, hs, g, h, u = generators(n * m, "edge%d_" % m)
    values = [0, 2 ** n - 1, 2 ** n, 2 ** n + 5, 2 ** 255 + 3, 7, 9, 11]
    gam = [0, Q, Q + 1, 2 ** 256 - 1, 5, 6, 7, 8]
    seeds = [b"", b"s" * 100, b"same", b"same", b"e4", b"e5", b"e6", b"e7"]
    vs = [[ModP(values[(i + j) % 8], Q) for j in range(m)] for i in range(8)]
    gammas = [[ModP(gam[(i + 3 * j) % 8], Q) for j in range(m)] for i in range(8)]
    batch = prove_range_proofs_packed(vs, n, g, h, gs, hs, gammas, u, seeds)
    proofs = unpack_aggreg_proofs(batch)
    for i in range(8):
        check_against_reference(batch, proofs, i, vs, n, g, h, gs, hs, gammas, u, seeds)
    # the same seed gives the same blinding factors: A and S are shared when the bits are (here they differ, so compare S)
    assert T_(proofs[2].S) == T_(proofs[3].S)


# ---- 6. round trip through the batch verifiers -----------------------------------------------------------------------------------
@pytest.mark.parametrize("n,m", [(16, 1), (8, 4)])
def test_round_trip_into_verifiers(n, m):
    count = 24
    rng = random.Random(n + m)
    gs, hs, g, h, u = generators(n * m, "trip%d_%d_" % (n, m))
    pk = pack_generators(g, h, gs, hs, u)
    vs, gammas, seeds = random_inputs(count, n, m, rng, "trip")
    batch = prove_range_proofs_packed(vs, n, g, h, gs, hs, gammas, u, seeds, packed=pk)
    assert verify_rlc_packed(batch, g, h, gs, hs, u, seed=bytes(range(32)), packed=pk) == (b"\x01" * count, 1)
    assert verify_aggreg_packed(batch, g, h, gs, hs, u, packed=pk) == b"\x01" * count
    if m == 1:
        assert verify_packed(batch, g, h, gs, hs, u) == b"\x01" * count
    bad = 13
    vs[bad][m - 1] = ModP(2 ** n + 1, Q)                       # out of range: the same invalid proof as the per-proof prover
    batch = prove_range_proofs_packed(vs, n, g, h, gs, hs, gammas, u, seeds, packed=pk)
    want = bytes(0 if i == bad else 1 for i in range(count))
    assert verify_rlc_packed(batch, g, h, gs, hs, u, seed=bytes(range(32)), packed=pk) == (want, 0)
    assert verify_aggreg_packed(batch, g, h, gs, hs, u, packed=pk) == want
    if m == 1:
        assert verify_packed(batch, g, h, gs, hs, u) == want
    check_against_reference(batch, unpack_aggreg_proofs(batch), bad, vs, n, g, h, gs, hs, gammas, u, seeds)


# ---- 7. no interference with the per-proof prover's graphs and workspaces --------------------------------------------------------
@pytest.mark.parametrize("mode", [0, 1, 2])
def test_single_proofs_unchanged_around_a_batch(golden, mode):
    case = golden("range_c1")["cases"][0]
    n, v = case["n"], int(case["v"])
    raw = gens(n, case["seeds"])
    gs, hs, g, h, u = [P_(t) for t in raw[0]], [P_(t) for t in raw[1]], P_(raw[2]), P_(raw[3]), P_(raw[4])
    gamma = mod_hash(case["seeds"][5].encode(), Q)
    single = lambda: NIRangeProver(ModP(v, Q), n, g, h, gs, hs, gamma, u, secp256k1, case["seeds"][6].encode()).prove()  # noqa: E731
    lib = nat.load()
    try:
        nat.check(lib.bp_ipa_set_graphs(mode))
        for _ in range(2):                                     # mode 2 captures its graph on the second proof
            assert range_json(single()) == case["proof"]
        rng = random.Random(mode)
        vs, gammas, seeds = random_inputs(300, n, 1, rng, "interfere")
        prove_range_proofs_packed(vs, n, g, h, gs, hs, gammas, u, seeds)
        for _ in range(2):
            assert range_json(single()) == case["proof"]
    finally:
        lib.bp_ipa_set_graphs(1)


# ---- 8. errors ----------------------------------------------------------------------------------------------------------------------
def test_errors_and_empty_batch():
    n, m = 8, 1
    gs, hs, g, h, u = generators(n, "err")
    rng = random.Random(8)
    vs, gammas, seeds = random_inputs(3, n, m, rng, "err")
    with pytest.raises(ValueError):
        prove_range_proofs_packed(vs, 3, g, h, gs, hs, gammas, u, seeds)              # N not a power of two
    with pytest.raises(ValueError):
        prove_range_proofs_packed([[ModP(1, Q)] * 2] * 3, 2048, g, h, gs, hs, [[ModP(1, Q)] * 2] * 3, u, seeds)   # N > 2048
    with pytest.raises(ValueError):
        prove_range_proofs_packed(vs[:1] + [vs[1] * 2] + vs[2:], n, g, h, gs, hs, gammas, u, seeds)              # ragged m
    with pytest.raises(ValueError):
        prove_range_proofs_packed(vs, n, g, h, gs, hs, gammas[:2], u, seeds)        # mismatched lengths
    with pytest.raises(ValueError):
        prove_range_proofs_packed(vs, n, g, h, gs, hs, gammas, u, seeds[:2])
    with pytest.raises(ValueError):
        prove_range_proofs_packed(vs, 4, g, h, gs, hs, gammas, u, seeds)              # generator count is not n * m
    # empty batch: no device work
    lib = nat.load()
    before, after = ctypes.c_uint64(), ctypes.c_uint64()
    nat.check(lib.bp_launch_count(ctypes.byref(before)))
    empty = prove_range_proofs_packed([], n, g, h, gs, hs, [], u, [])
    nat.check(lib.bp_launch_count(ctypes.byref(after)))
    assert empty.nproofs == 0 and empty.records == b"" and after.value == before.value
    assert prove_range_proofs_batch([], n, g, h, gs, hs, [], u, []) == []
    # the C entry point: bad N, and a transcript buffer that is too small reports the bytes needed
    gs_b, hs_b, g_b, h_b, u_b = pack_generators(g, h, gs, hs, u)
    vals = b"".join(v[0].x.to_bytes(32, "little") for v in vs)
    gms = b"".join(x[0].x.to_bytes(32, "little") for x in gammas)
    offs = [0]
    for s in seeds:
        offs.append(offs[-1] + len(s))
    stride = lib.bp_rp_aggreg_proof_stride(n, m)

    def call(nn, cap):
        recs, blob, ln = ctypes.create_string_buffer(3 * stride), ctypes.create_string_buffer(max(cap, 1)), ctypes.c_size_t(0)
        tro, sts = (ctypes.c_uint64 * 10)(), (ctypes.c_uint32 * 3)()
        rc = lib.bp_rp_prove_batch(gs_b, hs_b, g_b, h_b, u_b, nn, m, vals, gms, b"".join(seeds), (ctypes.c_uint64 * 4)(*offs), 3,
                                   recs, blob, cap, ctypes.byref(ln), tro, sts)
        return rc, ln.value, recs.raw, blob.raw[:ln.value]
    assert call(3, 1 << 16)[0] != 0
    rc, need, recs, blob = call(n, 1 << 16)
    assert rc == 0 and need > 0
    rc_short, need_short, recs_short, _ = call(n, 10)
    assert rc_short != 0 and need_short == need and recs_short == recs
    ref = prove_range_proofs_packed(vs, n, g, h, gs, hs, gammas, u, seeds)
    assert ref.records == recs and ref.blob == blob
