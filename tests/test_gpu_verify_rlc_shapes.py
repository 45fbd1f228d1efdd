"""bp_rp_verify_mixed_rlc: one random linear combination over a batch of proofs of different shapes (n bits, m values) that use
prefixes of one generator set of nset = 1024 points per side.  Every GPU case runs with the generator tables off and forced on
(bp_fb_set_mode 0 / 2).  Accept bytes are compared with the oracle's decisions (Pool.want of test_gpu_verify_batch, each pool
built over the prefix gs[:n*m], hs[:n*m] of the set); `combined` says whether the combination held.  The packing checks and the
Python-level argument errors need no GPU."""
import ctypes
import random
from types import SimpleNamespace

import pytest

from oracle import ecc
from helpers import gens
from test_gpu_verify_batch import Pool, KINDS, _offsets
from test_gpu_verify_rlc import SETTLED, SEED, TAUX, MU, _rho, _set_scalar, _batch, _exact, _rlc
from test_gpu_protocols import P_, M_, quiet
from python_bulletproofs_b200 import secp256k1, _native as nat
from python_bulletproofs_b200.utils import commitment, mod_hash
from python_bulletproofs_b200.rangeproofs import (NIRangeProver, AggregNIRangeProver, RangeVerifier, AggregRangeVerifier,
                                                  verify_mixed_range_proofs_batch)
from python_bulletproofs_b200.rangeproofs.batch import (PackedMixedBatch, pack_generators, pack_aggreg_proof,
                                                         verify_mixed_rlc_packed)

Q = ecc.Q
NSET = 1024
SHAPES = [(8, 1), (16, 1), (8, 2), (16, 4), (64, 1), (64, 16)]
gpu = pytest.mark.gpu


@pytest.fixture(scope="module")
def mixed():
    """One generator set of NSET points per side and a pool of proofs per shape over its prefixes."""
    nat.init(0)
    ogs, ohs, og, oh, ou = gens(NSET, ["shapes%d" % i for i in range(5)])
    pools = {}
    for n, m in SHAPES:
        N = n * m
        D = 97 if N <= 16 else 79 if N <= 64 else 37
        pools[(n, m)] = Pool(n, m, D, "shp%d_%d_" % (n, m), generators=(ogs[:N], ohs[:N], og, oh, ou))
    st = SimpleNamespace(pools=pools, gens=(og, oh, ogs, ohs, ou), packed=pack_generators(og, oh, ogs, ohs, ou))
    yield st
    nat.check(nat.load().bp_fb_clear())


@pytest.fixture(params=[0, 2], ids=["tables_off", "tables_on"])
def fb_mode(request):
    lib = nat.load()
    nat.init(0)
    nat.check(lib.bp_fb_clear())
    nat.check(lib.bp_fb_set_mode(request.param))
    yield request.param
    nat.check(lib.bp_fb_clear())
    nat.check(lib.bp_fb_set_mode(1))


def _honest(pool):
    return [i for i, k in enumerate(pool.kinds) if k is None]


def _mixed(st, entries, recs=None, nset=NSET):
    """entries: (shape, pool index) in the caller's order; recs: {position: replacement record}.  -> batch, want, kinds"""
    recs = recs or {}
    pools = [st.pools[s] for s, _ in entries]
    batch = PackedMixedBatch(nset, [p.n for p in pools], [p.m for p in pools],
                             [recs.get(k, p.recs[j]) for k, (p, (_, j)) in enumerate(zip(pools, entries))],
                             [p.trs[j] for p, (_, j) in zip(pools, entries)], [p.starts[j] for p, (_, j) in zip(pools, entries)])
    return batch, bytes(p.want[j] for p, (_, j) in zip(pools, entries)), [p.kinds[j] for p, (_, j) in zip(pools, entries)]


def _call(st, batch, seed=SEED, packed=None):
    return verify_mixed_rlc_packed(batch, *st.gens, seed=seed, packed=packed or st.packed)


def _interleaved_honest(st, count, shapes=SHAPES, salt=0):
    """count honest proofs, shapes taken in a scrambled order (never grouped by shape)"""
    rng = random.Random(count * 7 + salt)
    out = []
    for i in range(count):
        s = shapes[rng.randrange(len(shapes))]
        hon = _honest(st.pools[s])
        out.append((s, hon[(5 * i + salt) % len(hon)]))
    return out


def _diff(got, want, kinds):
    return [(i, kinds[i], got[i], want[i]) for i in range(len(want)) if got[i] != want[i]][:16]


@gpu
@pytest.mark.parametrize("count", [1, 33, 1001])
def test_honest_interleaved(fb_mode, mixed, count):
    entries = _interleaved_honest(mixed, count)
    if count > 1:
        assert len({s for s, _ in entries}) == len(SHAPES)
    batch, want, _ = _mixed(mixed, entries)
    assert want == b"\x01" * count
    for call in range(2):
        assert _call(mixed, batch) == (want, 1), (count, call)
    assert verify_mixed_rlc_packed(batch, *mixed.gens, packed=mixed.packed) == (want, 1)     # seed=None: os.urandom


@gpu
@pytest.mark.parametrize("nm", [(8, 2), (64, 1)])
def test_one_shape_equals_batch_rlc(fb_mode, mixed, nm):
    """One shape over a set of exactly n*m points: the mixed call and bp_rp_verify_batch_rlc give the same bytes and flag."""
    pool = mixed.pools[nm]
    N = nm[0] * nm[1]
    for idx in (_honest(pool)[:40], [(3 + 5 * i) % pool.D for i in range(150)]):
        batch = _batch(pool, idx)
        mb, want, kinds = _mixed(mixed, [(nm, j) for j in idx], nset=N)
        got = verify_mixed_rlc_packed(mb, *pool.gens, seed=SEED, packed=pool.packed_gens)
        assert got == _rlc(pool, batch)
        assert got[0] == want, _diff(got[0], want, kinds)
        assert got[1] == (1 if want == b"\x01" * len(idx) else 0)


@gpu
def test_proofs_shorter_than_the_set(fb_mode, mixed):
    """Only shapes with n*m < nset: their Gsum / Hsum terms are spread over their own columns (k_rlc_fold's spread flag)."""
    short = [s for s in SHAPES if s[0] * s[1] < NSET]
    entries = _interleaved_honest(mixed, 120, short, salt=1)
    batch, want, kinds = _mixed(mixed, entries)
    assert _call(mixed, batch) == (want, 1)
    for k in (0, 57):                                   # mu + 1 on one proof
        s, j = entries[k]
        pool = mixed.pools[s]
        rec = _set_scalar(pool.recs[j], _offsets(pool.m, pool.L)["T2"] + MU, lambda v: v + 1)
        batch, _, _ = _mixed(mixed, entries, {k: rec})
        acc, comb = _call(mixed, batch)
        assert comb == 0
        assert acc == bytes(0 if i == k else 1 for i in range(len(entries))), _diff(acc, want, kinds)
    # a single shape shorter than the set
    one = [((8, 2), j) for j in _honest(mixed.pools[(8, 2)])[:30]]
    batch, want, _ = _mixed(mixed, one)
    assert _call(mixed, batch) == (want, 1)


@gpu
def test_one_forgery_of_each_kind(fb_mode, mixed):
    """Every kind of forgery once, each time in a different shape group, among honest proofs of every shape."""
    filler = _interleaved_honest(mixed, 40, salt=2)
    for k, kind in enumerate(KINDS):
        for t in range(len(SHAPES)):
            shape = SHAPES[(k + t) % len(SHAPES)]
            pool = mixed.pools[shape]
            if kind in pool.kinds:
                break
        else:
            pytest.fail("no pool holds a forgery of kind %s" % kind)
        entries = list(filler)
        entries.insert((7 * k) % 41, (shape, pool.kinds.index(kind)))
        batch, want, kinds = _mixed(mixed, entries)
        acc, comb = _call(mixed, batch)
        assert acc == want, (kind, shape, _diff(acc, want, kinds))
        assert comb == (1 if kind in SETTLED else 0), (kind, shape)


@gpu
def test_weights_span_shapes(fb_mode, mixed):
    """tau_x + d on a proof of one shape and tau_x - d rho_0 / rho_1 on a proof of another cancel under the pinned seed's weights:
    one sum with the caller's indices spans the shape groups.  The exact verifiers reject both; any other seed rejects both."""
    a, b = (8, 1), (16, 4)
    entries = [(a, _honest(mixed.pools[a])[0]), (b, _honest(mixed.pools[b])[0])] + _interleaved_honest(mixed, 9, salt=3)
    r0, r1 = _rho(SEED, 0), _rho(SEED, 1)
    d = 987654321
    pa, pb = mixed.pools[a], mixed.pools[b]
    recs = {0: _set_scalar(pa.recs[entries[0][1]], _offsets(pa.m, pa.L)["T2"] + TAUX, lambda v: v + d),
            1: _set_scalar(pb.recs[entries[1][1]], _offsets(pb.m, pb.L)["T2"] + TAUX, lambda v: v - d * r0 * pow(r1, -1, Q))}
    batch, _, _ = _mixed(mixed, entries, recs)
    rest = b"\x01" * (len(entries) - 2)
    for k, (s, j) in enumerate(entries[:2]):           # the exact verifier of each shape, proof by proof
        assert _exact(mixed.pools[s], _batch(mixed.pools[s], [j], {0: recs[k]})) == b"\x00"
    assert _call(mixed, batch) == (b"\x01\x01" + rest, 1)
    for seed in (bytes(32), bytes(range(1, 33))):
        assert _call(mixed, batch, seed) == (b"\x00\x00" + rest, 0)


@gpu
def test_several_groups_over_several_chunks(fb_mode, mixed):
    """Groups of 300 / 200 / 260 / 130 / 65 / 20 proofs (4, 4, 4, 3, 2 and 1 chunks), each pool tiled with its forged proofs,
    shuffled into one caller order: the sum fails, every group goes to its exact verifier, the bytes come back in order."""
    counts = dict(zip(SHAPES, (300, 200, 260, 130, 65, 20)))
    entries = [(s, (11 * s[0] + i) % mixed.pools[s].D) for s in SHAPES for i in range(counts[s])]
    random.Random(5).shuffle(entries)
    batch, want, kinds = _mixed(mixed, entries)
    assert all(b"\x00" in bytes(mixed.pools[s].want[j] for s2, j in entries if s2 == s) for s in SHAPES)
    acc, comb = _call(mixed, batch)
    assert comb == 0
    assert acc == want, _diff(acc, want, kinds)


def _py_items(tag):
    """Python proof objects over prefixes of one 16-point set: bare-V single-value proofs of 8 and 16 bits, aggregated ones of
    2 x 4 and 2 x 8 bits."""
    ogs, ohs, og, oh, ou = gens(16, [tag + "%d" % i for i in range(5)])
    gs, hs, g, h, u = [P_(t) for t in ogs], [P_(t) for t in ohs], P_(og), P_(oh), P_(ou)
    rng = random.Random(tag)
    items = []
    for i, (n, m) in enumerate([(8, 1), (4, 2), (16, 1), (8, 2), (8, 1), (16, 1), (4, 2), (8, 2)]):
        N = n * m
        vs = [M_(rng.getrandbits(n)) for _ in range(m)]
        gammas = [mod_hash(b"%s_g%d_%d" % (tag.encode(), i, j), Q) for j in range(m)]
        Vs = [commitment(g, h, vs[j], gammas[j]) for j in range(m)]
        if m == 1:
            pr = NIRangeProver(vs[0], n, g, h, gs[:N], hs[:N], gammas[0], u, secp256k1, b"%s_p%d" % (tag.encode(), i)).prove()
            items.append((Vs[0], pr))
        else:
            pr = AggregNIRangeProver(vs, n, g, h, gs[:N], hs[:N], gammas, u, secp256k1, b"%s_p%d" % (tag.encode(), i)).prove()
            items.append((Vs, pr))
    return (g, h, gs, hs, u), items


def _one_by_one(gset, items):
    g, h, gs, hs, u = gset
    out = []
    for V, pr in items:
        N = 1 << len(pr.innerProof.proof2.xs)
        cls = AggregRangeVerifier if isinstance(V, list) else RangeVerifier
        out.append(quiet(lambda: cls(V, g, h, gs[:N], hs[:N], u, pr).verify()))
    return out


@gpu
def test_list_level(fb_mode):
    """verify_mixed_range_proofs_batch equals RangeVerifier / AggregRangeVerifier item by item over the prefixes, with a forged
    proof and one whose IPA challenge is unreduced (deferred to the Python classes)."""
    gset, items = _py_items("mixl")
    assert verify_mixed_range_proofs_batch(items, *gset, seed=SEED) == [True] * len(items)
    items[1][1].taux = items[1][1].taux + M_(1)
    p2 = items[5][1].innerProof.proof2
    p2.xs[0] = M_(p2.xs[0].x + Q)
    assert PackedMixedBatch.from_items(items, 16).starts[5] == 0xFFFFFFFF
    want = _one_by_one(gset, items)
    assert want[1] is False and want[5] is False and want.count(True) == len(items) - 2
    assert verify_mixed_range_proofs_batch(items, *gset, seed=SEED) == want
    assert verify_mixed_range_proofs_batch(items, *gset) == want


@gpu
def test_errors(mixed):
    entries = _interleaved_honest(mixed, 6, salt=4)
    batch, _, _ = _mixed(mixed, entries)
    lib = nat.load()
    acc = ctypes.create_string_buffer(max(batch.nproofs, 1))
    comb = ctypes.c_int(-1)

    def call(nset=NSET, ns=None, ms=None, nbytes=None, seed=SEED, nproofs=None, gens_=None):
        ns = ns or batch.ns_arr
        ms = ms or batch.ms_arr
        rc = lib.bp_rp_verify_mixed_rlc(*(gens_ or mixed.packed), nset, ns, ms, batch.records,
                                        len(batch.records) if nbytes is None else nbytes, batch.nproofs if nproofs is None else nproofs,
                                        batch.blob, batch.tr_off, batch.starts, seed, acc, ctypes.byref(comb))
        return rc, lib.bp_last_error().decode()
    assert call()[0] == 0 and comb.value == 1 and acc.raw[:6] == b"\x01" * 6
    rc, msg = call(seed=None)
    assert rc != 0 and "seed" in msg
    rc, msg = call(nset=4096)
    assert rc != 0 and "2048" in msg
    u32s = lambda v: (ctypes.c_uint32 * 6)(*v)          # noqa: E731
    for ns, ms in (([3] + batch.ns[1:], batch.ms), ([8] * 6, [0] + [1] * 5), ([2048] + batch.ns[1:], [1] + batch.ms[1:])):
        rc, msg = call(ns=u32s(ns), ms=u32s(ms))
        assert rc != 0 and "power of two" in msg and "nset" in msg, (ns, ms, msg)
    rc, msg = call(nbytes=len(batch.records) - 1)
    assert rc != 0 and "proofs_bytes" in msg
    # 2^20 proofs of 2048 values x 1 bit: 2^20 x (2048 + 6 + 22) proof points >= 2^31
    big = 1 << 20
    full = ctypes.c_uint32 * big
    gens_2048 = (bytes(64 * 2048), bytes(64 * 2048)) + mixed.packed[2:]
    rc, msg = call(nset=2048, ns=full(*([1] * big)), ms=full(*([2048] * big)), nproofs=big, gens_=gens_2048)
    assert rc != 0 and "too large" in msg
    empty = PackedMixedBatch(NSET, [], [], [], [], [])
    assert _call(mixed, empty) == (b"", 1)


# ---- packing and argument errors, no GPU ------------------------------------------------------------------------------------
def _fake_proof(L, tag=0):
    """A proof object with the attributes the packer reads (points on the curve, arbitrary scalars)."""
    pt = lambda k: ecc.py_mul(ecc.G, 1000 * tag + k)      # noqa: E731
    p2 = SimpleNamespace(a=11 + tag, b=12, xs=[100 + j for j in range(L)], Ls=[pt(20 + j) for j in range(L)],
                         Rs=[pt(40 + j) for j in range(L)], transcript=b"p2-%d" % tag, start_transcript=3 + tag)
    ip = SimpleNamespace(u_new=pt(2), P_new=pt(3), transcript=b"ip-%d" % tag, proof2=p2)
    return SimpleNamespace(A=pt(4), S=pt(5), T1=pt(6), T2=pt(7), taux=8, mu=9, t_hat=10, transcript=b"rp-%d" % tag, innerProof=ip)


def test_packing_of_mixed_shapes():
    lib = nat.load()
    V = ecc.py_mul(ecc.G, 77)
    shapes = [(8, 1), (4, 2), (64, 16), (16, 1), (2, 8)]            # (n, m): N = n m
    items = []
    for t, (n, m) in enumerate(shapes):
        L = (n * m).bit_length() - 1
        items.append((V if m == 1 else [V] * m, _fake_proof(L, t)))
    b = PackedMixedBatch.from_items(items, NSET)
    assert (b.nproofs, b.nset, b.ns, b.ms) == (5, NSET, [n for n, _ in shapes], [m for _, m in shapes])
    assert list(b.ns_arr) == b.ns and list(b.ms_arr) == b.ms
    sizes = [lib.bp_rp_aggreg_proof_stride(n, m) for n, m in shapes]
    assert b.offsets == [sum(sizes[:k]) for k in range(5)] and len(b.records) == sum(sizes)
    for k, ((V_, pr), (n, m)) in enumerate(zip(items, shapes)):
        rec = pack_aggreg_proof(V_ if isinstance(V_, list) else [V_], pr, (n * m).bit_length() - 1)[0]
        assert b.records[b.offsets[k]:b.offsets[k] + sizes[k]] == rec
    assert sizes[0] == lib.bp_rp_proof_stride(8)                     # m = 1: the single-value record
    assert list(b.starts)[:5] == [3, 4, 5, 6, 7]
    tr = list(b.tr_off)
    assert len(tr) == 16 and b.blob[tr[3]:tr[6]] == b"rp-1ip-1p2-1"
    items[2][1].innerProof.proof2.xs[0] = Q + 5                      # unreduced challenge: deferred to Python
    assert PackedMixedBatch.from_items(items, NSET).starts[2] == 0xFFFFFFFF


def test_python_argument_errors():
    V = ecc.py_mul(ecc.G, 77)
    with pytest.raises(ValueError, match="larger than the set"):
        PackedMixedBatch.from_items([(V, _fake_proof(3)), ([V] * 16, _fake_proof(10))], 512)
    with pytest.raises(ValueError, match="shape"):
        PackedMixedBatch.from_items([([V] * 3, _fake_proof(3))], NSET)
    bad = _fake_proof(3)
    bad.innerProof.proof2.Ls.pop()
    with pytest.raises(ValueError, match="shape"):
        PackedMixedBatch.from_items([(V, bad)], NSET)
    gs = [ecc.py_mul(ecc.G, 2 + i) for i in range(8)]
    with pytest.raises(ValueError, match="larger than the set"):
        verify_mixed_range_proofs_batch([(V, _fake_proof(4))], V, V, gs, gs, V)
    batch = PackedMixedBatch.from_items([(V, _fake_proof(3))], 8)
    with pytest.raises(ValueError, match="seed"):
        verify_mixed_rlc_packed(batch, V, V, gs, gs, V, seed=b"short")
    with pytest.raises(ValueError, match="set of 8"):
        verify_mixed_rlc_packed(batch, V, V, gs[:4], gs[:4], V, seed=SEED)
