"""bp_rp_verify_rlc_locate: the random linear combination of bp_rp_verify_mixed_rlc, and when it fails, per-leaf sub-combinations
that send only the proofs of failing leaves to the exact verifier.  Every GPU case runs with the generator tables off and forced on
(bp_fb_set_mode 0 / 2) and compares the accept bytes with the oracle's decisions (Pool.want of test_gpu_verify_batch) and with
verify_rlc_packed / verify_mixed_rlc_packed on the same batch and seed, `combined` with their flag.  The leaf statistics are
checked against a restatement of the chunk and leaf plan below.  The Python-level argument checks need no GPU."""
import ctypes
import random

import pytest

from oracle import ecc
from test_gpu_verify_batch import Pool, KINDS, _offsets
from test_gpu_verify_rlc import SETTLED, SEED, TAUX, MU, _set_scalar, _batch, _rlc
from test_gpu_verify_rlc_shapes import mixed, NSET, SHAPES, _mixed, _interleaved_honest, _py_items, _one_by_one  # noqa: F401
from test_gpu_protocols import _small_batch, M_
from python_bulletproofs_b200 import secp256k1, _native as nat
from python_bulletproofs_b200.utils import commitment, mod_hash
from python_bulletproofs_b200.rangeproofs import (AggregNIRangeProver, verify_range_proofs_batch, verify_aggreg_range_proofs_batch,
                                                  verify_mixed_range_proofs_batch)
from python_bulletproofs_b200.rangeproofs.batch import (PackedBatch, PackedMixedBatch, verify_rlc_packed, verify_mixed_rlc_packed,
                                                         verify_rlc_locate_packed, rlc_locate_stats)

Q = ecc.Q
THAT = 128                       # t_hat's offset after T2 in a record (include/bp_gpu.h)
FORGE = (TAUX, MU, THAT)         # the algebraic forgeries: tau_x, mu or t_hat + 1
# kinds whose proofs stay out of the sum (the host or point checks give 0 or 2); the other kinds enter it
OUT = SETTLED - {"y_slot_leading_zeros"}
gpu = pytest.mark.gpu


@pytest.fixture(scope="module")
def pools():
    nat.init(0)
    made = {}

    def get(n, m=1):
        if (n, m) not in made:
            made[(n, m)] = Pool(n, m, 97 if n * m <= 16 else 79, "loc%d_%d_" % (n, m))
        return made[(n, m)]
    yield get
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


# ---- the chunk and leaf plan, restated -----------------------------------------------------------------------------------------
def auto_leaf(shapes):
    """The leaf size the library picks: the smallest power of two >= sqrt(512 nproofs^2 / sum of n m), within [8, 256]."""
    sum_n = sum(n * m for n, m in shapes)
    leaf = 8
    while leaf < 256 and leaf * leaf * sum_n < 512 * len(shapes) ** 2:
        leaf *= 2
    return leaf


def plan_leaves(shapes, leaf):
    """shapes[p] = (n, m) of proof p in the caller's order -> leaves as lists of caller indices, in processing order: grouped by
    (n m, m) (stable), chunks of clamp(ceil(cnt / 4), 64, 2048) <= cnt proofs per group, leaves of `leaf` proofs per chunk."""
    order = sorted(range(len(shapes)), key=lambda p: (shapes[p][0] * shapes[p][1], shapes[p][1]))
    groups = {}
    for p in order:
        groups.setdefault((shapes[p][0] * shapes[p][1], shapes[p][1]), []).append(p)
    leaves = []
    for key in sorted(groups):
        idx = groups[key]
        ch = min(min(max((len(idx) + 3) // 4, 64), 2048), len(idx))
        for lo in range(0, len(idx), ch):
            chunk = idx[lo:lo + ch]
            leaves += [chunk[k:k + leaf] for k in range(0, len(chunk), leaf)]
    return leaves


def expected_stats(shapes, kinds, leaf):
    """-> (leaves, failing leaves, proofs decided exactly).  A leaf fails when it holds an
    algebraic forgery (a kind that enters the sum and is rejected); its proofs that entered the sum are decided exactly."""
    leaves = plan_leaves(shapes, leaf)
    bad = lambda k: k is not None and k not in SETTLED          # noqa: E731
    failing = [lf for lf in leaves if any(bad(kinds[p]) for p in lf)]
    entered = sum(1 for lf in failing for p in lf if kinds[p] not in OUT)
    return len(leaves), len(failing), entered


def _locate(pool, batch, seed=SEED, leaf=0):
    return verify_rlc_locate_packed(batch, *pool.gens, seed=seed, packed=pool.packed_gens, leaf=leaf)


def _honest(pool):
    return [i for i, k in enumerate(pool.kinds) if k is None]


def _diff(got, want, kinds):
    return [(i, kinds[i], got[i], want[i]) for i in range(len(want)) if got[i] != want[i]][:16]


def _check(pool, batch, want, kinds, leaf=0):
    """locate against the oracle and against verify_rlc_packed; the statistics against the restated plan"""
    got = _locate(pool, batch, leaf=leaf)
    st = rlc_locate_stats()
    assert got[0] == want, _diff(got[0], want, kinds)
    assert got == _rlc(pool, batch)
    shapes = [(pool.n, pool.m)] * batch.nproofs
    used = leaf or auto_leaf(shapes)
    assert st["leaf"] == used
    if got[1] == 1:
        assert st["leaves"] == st["failing_leaves"] == st["exact_proofs"] == 0
    else:
        nleaves, nfail, entered = expected_stats(shapes, kinds, used)
        assert st["failing_leaves"] >= 1
        assert (st["leaves"], st["failing_leaves"], st["exact_proofs"]) == (nleaves, nfail, entered), st
    return got, st


# ---- one shape ------------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("nm", [(8, 1), (64, 1), (8, 2), (64, 16)])
def test_honest_batches(fb_mode, pools, nm):
    pool = pools(*nm)
    hon = _honest(pool)
    for count in (1, 33, 1031):
        idx = [hon[(7 * i) % len(hon)] for i in range(count)]
        got, st = _check(pool, _batch(pool, idx), b"\x01" * count, [None] * count)
        assert got[1] == 1 and st["leaves"] == 0
    assert verify_rlc_locate_packed(_batch(pool, idx), *pool.gens)[0] == b"\x01" * count      # seed=None


@gpu
@pytest.mark.parametrize("nm", [(8, 1), (8, 2)])
@pytest.mark.parametrize("count", [40, 600], ids=["one_chunk", "four_chunks"])
def test_one_forgery(fb_mode, pools, nm, count):
    """tau_x, mu or t_hat + 1 on the first, a middle and the last proof: one failing leaf, and only its proofs are re-decided."""
    pool = pools(*nm)
    hon = _honest(pool)
    idx = [hon[(5 * i) % len(hon)] for i in range(count)]
    T2 = _offsets(pool.m, pool.L)["T2"]
    for t, pos in enumerate((0, count // 2 + 3, count - 1)):
        batch = _batch(pool, idx, {pos: _set_scalar(pool.recs[idx[pos]], T2 + FORGE[t], lambda v: v + 1)})
        kinds = [None] * count
        kinds[pos] = "forged"
        want = bytes(0 if k == pos else 1 for k in range(count))
        for leaf in (0, 8):
            got, st = _check(pool, batch, want, kinds, leaf=leaf)
            lf = [lf for lf in plan_leaves([nm] * count, st["leaf"]) if pos in lf][0]
            assert got[1] == 0 and st["failing_leaves"] == 1 and st["exact_proofs"] == len(lf)


@gpu
@pytest.mark.parametrize("nm", [(8, 1), (8, 2)])
def test_forgeries_of_every_kind_in_every_chunk(fb_mode, pools, nm):
    """The pool tiled over 1031 proofs (4 chunks): a third forged, settled kinds next to algebraic forgeries in the same leaves."""
    pool = pools(*nm)
    batch, want, kinds = pool.tile(1031, 13)
    for leaf in (0, 4):
        got, st = _check(pool, batch, want, kinds, leaf=leaf)
        assert got[1] == 0 and st["failing_leaves"] > 1


@gpu
def test_every_proof_forged(fb_mode, pools):
    pool = pools(8, 2)
    hon = _honest(pool)
    count = 150
    idx = [hon[i % len(hon)] for i in range(count)]
    T2 = _offsets(pool.m, pool.L)["T2"]
    batch = _batch(pool, idx, {k: _set_scalar(pool.recs[j], T2 + FORGE[k % 3], lambda v: v + 1) for k, j in enumerate(idx)})
    got, st = _check(pool, batch, b"\x00" * count, ["forged"] * count)
    assert got[1] == 0 and st["failing_leaves"] == st["leaves"] and st["exact_proofs"] == count


@gpu
@pytest.mark.parametrize("leaf", [1, 3, 8, 200, 10 ** 6], ids=["1", "3", "fold_group", "past_a_chunk", "past_the_batch"])
def test_explicit_leaf(fb_mode, pools, leaf):
    """Leaf boundaries placed by the caller over 600 proofs (4 chunks of 150): one proof per leaf, leaves that are not a power of
    two, exactly one fold group, one leaf per chunk."""
    pool = pools(8, 1)
    batch, want, kinds = pool.tile(600, 29)
    got, st = _check(pool, batch, want, kinds, leaf=leaf)
    assert got[1] == 0 and st["leaves"] == 4 * -(-150 // min(leaf, 150))


@gpu
def test_more_leaves_than_one_table_launch(fb_mode, pools):
    """70000 one-proof leaves, more than the 65535 MSMs one launch of the block-tree table MSM could take: the leaf pass uses
    one-dimensional grids and takes them in one pass."""
    pool = pools(8, 1)
    hon = _honest(pool)
    count = 70000
    idx = [hon[i % len(hon)] for i in range(count)]
    T2 = _offsets(pool.m, pool.L)["T2"]
    pos = (3, 65600)
    batch = _batch(pool, idx, {p: _set_scalar(pool.recs[idx[p]], T2 + MU, lambda v: v + 1) for p in pos})
    kinds = [None] * count
    for p in pos:
        kinds[p] = "forged"
    got, st = _check(pool, batch, bytes(0 if k in pos else 1 for k in range(count)), kinds, leaf=1)
    assert st["leaves"] == count and st["failing_leaves"] == 2 and st["exact_proofs"] == 2


# ---- mixed shapes ---------------------------------------------------------------------------------------------------------------
def _mixed_check(st, batch, want, kinds, shapes, leaf=0):
    got = verify_rlc_locate_packed(batch, *st.gens, seed=SEED, packed=st.packed, leaf=leaf)
    stats = rlc_locate_stats()
    assert got[0] == want, _diff(got[0], want, kinds)
    assert got == verify_mixed_rlc_packed(batch, *st.gens, seed=SEED, packed=st.packed)
    used = leaf or auto_leaf(shapes)
    assert stats["leaf"] == used
    if got[1] == 1:
        assert stats["leaves"] == 0
    else:
        assert stats["failing_leaves"] >= 1
        assert (stats["leaves"], stats["failing_leaves"], stats["exact_proofs"]) == expected_stats(shapes, kinds, used), stats
    return got, stats


@gpu
@pytest.mark.parametrize("leaf", [0, 5, 64])
def test_mixed_shapes(fb_mode, mixed, leaf):   # noqa: F811
    """Proofs of every shape interleaved (groups of sizes that are no multiple of the leaf); all valid, then algebraic
    forgeries in three shape groups next to settled kinds."""
    entries = _interleaved_honest(mixed, 301, salt=7)
    shapes = [s for s, _ in entries]
    batch, want, kinds = _mixed(mixed, entries)
    got, stats = _mixed_check(mixed, batch, want, kinds, shapes, leaf)
    assert got == (b"\x01" * 301, 1)
    for kind in ("offcurve_A", "ipa_transcript_digit", "y_slot_non_numeric"):
        s = next(s for s in SHAPES if kind in mixed.pools[s].kinds)
        entries.insert(151, (s, mixed.pools[s].kinds.index(kind)))
        shapes.insert(151, s)
    recs = {}
    for k, pos in enumerate((0, 150, len(entries) - 1)):
        s, j = entries[pos]
        pool = mixed.pools[s]
        recs[pos] = _set_scalar(pool.recs[j], _offsets(pool.m, pool.L)["T2"] + FORGE[k], lambda v: v + 1)
    batch, want, kinds = _mixed(mixed, entries, recs)
    want = bytes(0 if p in recs else w for p, w in enumerate(want))
    kinds = ["forged" if p in recs else k for p, k in enumerate(kinds)]
    got, stats = _mixed_check(mixed, batch, want, kinds, shapes, leaf)
    assert got[1] == 0 and got[0].count(0) >= 4


# ---- argument errors, list level -----------------------------------------------------------------------------------------------
@gpu
def test_errors(pools):
    pool = pools(8)
    batch = _batch(pool, _honest(pool)[:6])
    lib = nat.load()
    acc = ctypes.create_string_buffer(6)
    comb = ctypes.c_int(-1)
    u32s = lambda v: (ctypes.c_uint32 * 6)(*v)          # noqa: E731

    def call(leaf=0, seed=SEED, nset=8, ns=(8,) * 6, ms=(1,) * 6, nbytes=None):
        rc = lib.bp_rp_verify_rlc_locate(*pool.packed_gens, nset, u32s(ns), u32s(ms), batch.records,
                                         len(batch.records) if nbytes is None else nbytes, 6, batch.blob, batch.tr_off, batch.starts,
                                         seed, leaf, acc, ctypes.byref(comb))
        return rc, lib.bp_last_error().decode()
    assert call()[0] == 0 and comb.value == 1 and acc.raw == b"\x01" * 6
    assert call(leaf=(1 << 32) - 1)[0] == 0 and comb.value == 1
    rc, msg = call(leaf=1 << 32)
    assert rc != 0 and "leaf" in msg and "32 bits" in msg
    rc, msg = call(seed=None)
    assert rc != 0 and "seed" in msg and "bp_rp_verify_rlc_locate" in msg
    rc, msg = call(nset=4096)
    assert rc != 0 and "2048" in msg
    rc, msg = call(ns=(3,) + (8,) * 5)
    assert rc != 0 and "power of two" in msg
    rc, msg = call(nset=4)
    assert rc != 0 and "nset" in msg
    rc, msg = call(nbytes=len(batch.records) - 1)
    assert rc != 0 and "proofs_bytes" in msg
    assert _locate(pool, PackedBatch(8, [], [], [])) == (b"", 1)


@gpu
def test_list_level(fb_mode):
    """locate=True on the three list functions gives the lists of their default paths, with a forged proof and one whose IPA
    challenge is unreduced (deferred to the Python classes)."""
    n = 8
    gs, hs, g, h, u, Vs, proofs = _small_batch(n, 6, "locl")
    proofs[2].taux = proofs[2].taux + M_(1)
    p2 = proofs[4].innerProof.proof2
    p2.xs[0] = M_(p2.xs[0].x + Q)
    want = verify_range_proofs_batch(Vs, g, h, gs, hs, u, proofs)
    assert want[2] is False and want[4] is False and want.count(True) == 4
    assert verify_range_proofs_batch(Vs, g, h, gs, hs, u, proofs, locate=True) == want
    assert verify_range_proofs_batch(Vs, g, h, gs, hs, u, proofs, locate=True, seed=SEED) == want
    m = 2
    Vs_list, aps = [], []
    for i in range(5):
        vs = [M_((5 * i + j) % 16) for j in range(m)]
        gammas = [mod_hash(b"locga%d_%d" % (i, j), Q) for j in range(m)]
        Vs_list.append([commitment(g, h, vs[j], gammas[j]) for j in range(m)])
        aps.append(AggregNIRangeProver(vs, n // m, g, h, gs, hs, gammas, u, secp256k1, b"locap%d" % i).prove())
    aps[1].mu = aps[1].mu + M_(1)
    p2 = aps[3].innerProof.proof2
    p2.xs[1] = M_(p2.xs[1].x + Q)
    want = verify_aggreg_range_proofs_batch(Vs_list, g, h, gs, hs, u, aps)
    assert want[1] is False and want[3] is False and want.count(True) == 3
    assert verify_aggreg_range_proofs_batch(Vs_list, g, h, gs, hs, u, aps, locate=True) == want
    gset, items = _py_items("locm")
    items[1][1].taux = items[1][1].taux + M_(1)
    p2 = items[5][1].innerProof.proof2
    p2.xs[0] = M_(p2.xs[0].x + Q)
    want = _one_by_one(gset, items)
    assert want[1] is False and want[5] is False
    assert verify_mixed_range_proofs_batch(items, *gset, seed=SEED, locate=True) == want
    assert verify_mixed_range_proofs_batch(items, *gset, locate=True) == want


def test_python_argument_errors():
    V = ecc.py_mul(ecc.G, 77)
    gs = [ecc.py_mul(ecc.G, 2 + i) for i in range(8)]
    batch = PackedBatch(8, [], [], [])
    with pytest.raises(ValueError, match="seed"):
        verify_rlc_locate_packed(batch, V, V, gs, gs, V, seed=b"short")
    with pytest.raises(ValueError, match="leaf"):
        verify_rlc_locate_packed(batch, V, V, gs, gs, V, seed=SEED, leaf=-1)
    with pytest.raises(ValueError, match="set of 8"):
        verify_rlc_locate_packed(batch, V, V, gs[:4], gs[:4], V, seed=SEED)
    mb = PackedMixedBatch(16, [], [], [], [], [])
    with pytest.raises(ValueError, match="set of 16"):
        verify_rlc_locate_packed(mb, V, V, gs, gs, V, seed=SEED)


def test_leaf_plan_restatement():
    """The restated plan: chunks of a quarter of the group within 64 .. 2048, leaves per chunk, groups by (n m, m)."""
    assert auto_leaf([(64, 1)] * 8192) == 256 and auto_leaf([(64, 16)] * 2048) == 32 and auto_leaf([(64, 1)]) == 8
    assert auto_leaf([(64, 1)] * 2048 + [(64, 16)] * 2048) == 64
    leaves = plan_leaves([(8, 1)] * 600, 64)
    assert [len(lf) for lf in leaves] == [64, 64, 22] * 4 and sum(leaves, []) == list(range(600))
    shapes = [(8, 2), (16, 1), (8, 1), (16, 1)]
    assert plan_leaves(shapes, 1) == [[2], [1], [3], [0]]
    assert plan_leaves([(8, 1)] * 10, 4) == [[0, 1, 2, 3], [4, 5, 6, 7], [8, 9]]
