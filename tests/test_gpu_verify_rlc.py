"""bp_rp_verify_batch_rlc: one random linear combination per batch, the exact verifier when it fails.  Every case runs with the
generator tables off and forced on (bp_fb_set_mode 0 / 2).  Accept bytes are compared with the oracle's decisions (Pool.want of
test_gpu_verify_batch); `combined` says whether the combination held."""
import ctypes
import hashlib

import pytest

from oracle import ecc
from test_gpu_verify_batch import Pool, KINDS, _offsets
from test_gpu_protocols import _small_batch, M_
from python_bulletproofs_b200 import secp256k1, _native as nat
from python_bulletproofs_b200.utils import commitment, mod_hash
from python_bulletproofs_b200.rangeproofs import AggregNIRangeProver
from python_bulletproofs_b200.rangeproofs.batch import (PackedBatch, PackedAggregBatch, verify_packed, verify_aggreg_packed,
                                                         verify_rlc_packed, verify_range_proofs_batch,
                                                         verify_aggreg_range_proofs_batch)

pytestmark = pytest.mark.gpu
Q = ecc.Q
SEED = bytes(range(32))
# kinds that the transcript or point checks settle (0 or 2) before the combination, and the one that is a valid proof
SETTLED = {"ipa_transcript_digit", "challenge_leading_zero", "y_slot_non_numeric", "y_slot_leading_zeros"} | \
          {k for k in KINDS if k.startswith("offcurve_")}


@pytest.fixture(scope="module")
def pools():
    nat.init(0)
    made = {}

    def get(n, m=1):
        if (n, m) not in made:
            made[(n, m)] = Pool(n, m, 97 if n * m <= 16 else 79, "rlc%d_%d_" % (n, m))
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


def _batch(pool, idx, recs=None):
    recs = recs or {}
    r = [recs.get(k, pool.recs[j]) for k, j in enumerate(idx)]
    t, s = [pool.trs[j] for j in idx], [pool.starts[j] for j in idx]
    return PackedBatch(pool.n, r, t, s) if pool.m == 1 else PackedAggregBatch(pool.n, pool.m, r, t, s)


def _exact(pool, batch):
    return verify_packed(batch, *pool.gens) if pool.m == 1 else verify_aggreg_packed(batch, *pool.gens, packed=pool.packed_gens)


def _rlc(pool, batch, seed=SEED):
    return verify_rlc_packed(batch, *pool.gens, seed=seed, packed=pool.packed_gens)


def _honest(pool):
    return [i for i, k in enumerate(pool.kinds) if k is None]


def _rho(seed, p):
    r = int.from_bytes(hashlib.sha256(seed + p.to_bytes(8, "little")).digest(), "little") % Q
    return r or 1


def _set_scalar(rec, off, fn):
    rec = bytearray(rec)
    rec[off:off + 32] = (fn(int.from_bytes(rec[off:off + 32], "little")) % Q).to_bytes(32, "little")
    return bytes(rec)


TAUX, MU = 64, 96                # scalar offsets after T2 in a record (include/bp_gpu.h)


@pytest.mark.parametrize("nm", [(8, 1), (64, 1), (8, 2), (64, 16)])
def test_honest_batches(fb_mode, pools, nm):
    pool = pools(*nm)
    hon = _honest(pool)
    for count in (1, 33, 1031):
        batch = _batch(pool, [hon[(7 * i) % len(hon)] for i in range(count)])
        for call in range(2):
            acc, comb = _rlc(pool, batch)
            assert (acc, comb) == (b"\x01" * count, 1), (count, call, comb, acc.count(1))
    acc, comb = verify_rlc_packed(batch, *pool.gens)                  # seed=None: a fresh seed from os.urandom
    assert (acc, comb) == (b"\x01" * batch.nproofs, 1)


@pytest.mark.parametrize("nm", [(8, 1), (8, 2)])
def test_one_forgery_of_each_kind(fb_mode, pools, nm):
    pool = pools(*nm)
    hon = _honest(pool)
    seen = set()
    for j, kind in enumerate(pool.kinds):
        if kind is None or kind in seen:
            continue
        seen.add(kind)
        idx = [hon[i % len(hon)] for i in range(40)]
        idx.insert(len(seen) % 40, j)
        batch = _batch(pool, idx)
        want = bytes(pool.want[i] for i in idx)
        acc, comb = _rlc(pool, batch)
        assert acc == want, (kind, [(i, acc[i], want[i]) for i in range(len(acc)) if acc[i] != want[i]])
        assert comb == (1 if kind in SETTLED else 0), kind
    assert seen == set(KINDS)


@pytest.mark.parametrize("nm", [(8, 1), (8, 2)])
def test_mixed_pool_over_several_chunks(fb_mode, pools, nm):
    pool = pools(*nm)
    batch, want, kinds = pool.tile(1031, 13)
    acc, comb = _rlc(pool, batch)
    assert comb == 0
    assert acc == want, [(i, kinds[i], acc[i], want[i]) for i in range(len(acc)) if acc[i] != want[i]][:16]


@pytest.mark.parametrize("nm", [(8, 1), (8, 2)])
@pytest.mark.parametrize("off", [TAUX, MU], ids=["taux", "mu"])
def test_errors_of_two_proofs_do_not_cancel(fb_mode, pools, nm, off):
    """tau_x + d on one proof and tau_x - d on another (E1), or the same with mu (E2): with equal weights the two errors would cancel."""
    pool = pools(*nm)
    hon = _honest(pool)
    idx = hon[:20]
    o = _offsets(pool.m, pool.L)["T2"] + off
    d = 123456789
    batch = _batch(pool, idx, {3: _set_scalar(pool.recs[idx[3]], o, lambda v: v + d),
                               11: _set_scalar(pool.recs[idx[11]], o, lambda v: v - d)})
    acc, comb = _rlc(pool, batch)
    assert comb == 0
    assert acc == bytes(0 if k in (3, 11) else 1 for k in range(20))


@pytest.mark.parametrize("nm", [(8, 1), (8, 2)])
def test_weights_follow_the_seed(fb_mode, pools, nm):
    """With the weights of a known seed two invalid proofs can be made to cancel: the combination holds and both are accepted,
    while the exact verifier rejects both.  Under any other seed the same pair fails the combination."""
    pool = pools(*nm)
    hon = _honest(pool)
    idx = hon[:2] + hon[2:9]
    r0, r1 = _rho(SEED, 0), _rho(SEED, 1)
    d = 987654321
    o = _offsets(pool.m, pool.L)["T2"] + TAUX
    batch = _batch(pool, idx, {0: _set_scalar(pool.recs[idx[0]], o, lambda v: v + d),
                               1: _set_scalar(pool.recs[idx[1]], o, lambda v: v - d * r0 * pow(r1, -1, Q))})
    assert _exact(pool, batch) == b"\x00\x00" + b"\x01" * 7
    assert _rlc(pool, batch) == (b"\x01" * 9, 1)
    assert _rlc(pool, batch, bytes(32)) == (b"\x00\x00" + b"\x01" * 7, 0)


def test_list_level_combine(fb_mode):
    """combine=True gives the lists of the default path, single-value and aggregated, with a forged proof and one whose IPA
    challenge is unreduced (deferred to the Python classes)."""
    n = 8
    gs, hs, g, h, u, Vs, proofs = _small_batch(n, 6, "rlcl")
    proofs[2].taux = proofs[2].taux + M_(1)
    p2 = proofs[4].innerProof.proof2
    p2.xs[0] = M_(p2.xs[0].x + Q)
    want = verify_range_proofs_batch(Vs, g, h, gs, hs, u, proofs)
    assert want[2] is False and want[4] is False and want.count(True) == 4
    assert verify_range_proofs_batch(Vs, g, h, gs, hs, u, proofs, combine=True) == want
    assert verify_range_proofs_batch(Vs, g, h, gs, hs, u, proofs, combine=True, seed=SEED) == want
    good = [0, 1, 3, 5]
    assert verify_range_proofs_batch([Vs[i] for i in good], g, h, gs, hs, u, [proofs[i] for i in good], combine=True) == [True] * 4
    # aggregated, m = 2
    m = 2
    gs2, hs2 = gs[:n // m * m], hs[:n // m * m]
    Vs_list, aps = [], []
    for i in range(5):
        vs = [M_((5 * i + j) % 16) for j in range(m)]
        gammas = [mod_hash(b"rlcga%d_%d" % (i, j), Q) for j in range(m)]
        Vs_list.append([commitment(g, h, vs[j], gammas[j]) for j in range(m)])
        aps.append(AggregNIRangeProver(vs, n // m, g, h, gs2, hs2, gammas, u, secp256k1, b"rlcap%d" % i).prove())
    aps[1].mu = aps[1].mu + M_(1)
    p2 = aps[3].innerProof.proof2
    p2.xs[1] = M_(p2.xs[1].x + Q)
    want = verify_aggreg_range_proofs_batch(Vs_list, g, h, gs2, hs2, u, aps)
    assert want[1] is False and want[3] is False and want.count(True) == 3
    assert verify_aggreg_range_proofs_batch(Vs_list, g, h, gs2, hs2, u, aps, combine=True) == want


def test_errors(pools):
    pool = pools(8)
    batch = _batch(pool, _honest(pool)[:4])
    lib = nat.load()
    acc = ctypes.create_string_buffer(4)
    comb = ctypes.c_int(-1)

    def call(n, m, stride, seed):
        rc = lib.bp_rp_verify_batch_rlc(*pool.packed_gens, n, m, batch.records, stride, batch.nproofs, batch.blob, batch.tr_off,
                                        batch.starts, seed, acc, ctypes.byref(comb))
        return rc, lib.bp_last_error().decode()
    assert call(8, 1, batch.stride, SEED)[0] == 0 and comb.value == 1 and acc.raw == b"\x01" * 4
    rc, msg = call(8, 1, batch.stride, None)
    assert rc != 0 and "seed" in msg
    for n, m in ((3, 1), (1, 3), (4096, 1), (64, 64)):
        rc, msg = call(n, m, batch.stride, SEED)
        assert rc != 0 and "power of two" in msg, (n, m, msg)
    rc, msg = call(8, 1, batch.stride - 1, SEED)
    assert rc != 0 and "proof_stride" in msg
    empty = PackedBatch(8, [], [], [])
    assert verify_rlc_packed(empty, *pool.gens, seed=SEED) == (b"", 1)
