"""The batch verifiers at the sizes they are used at: batches of thousands of proofs cut into several chunks, every chunk plan
and kernel form of bp_rp_verify_batch (forced chunk lengths, both inversion forms, k_sv_comb2 and k_sv_comb2q, the two-chunk plan
of few host threads, 16-bit lookups with three and four warps), the one-rank gather, and bp_rp_verify_aggreg_batch over several
chunks.  Every accept byte is compared with the oracle verifier's decision on the same bytes.

The proofs come from small pools of distinct proofs (a prime number of them, so that no chunk length is a multiple of the pool
and every chunk of a large batch sees the pool at a different phase); about a third of each pool is forged, one kind of forgery
per proof.  Large batches are the pool's packed records tiled at the byte level, from a different starting offset per leg.  A
buffer, flag or verdict that leaks from one chunk into another then changes the decision pattern instead of repeating it."""
import copy
import ctypes
import functools
import os
import pickle
import random
import subprocess
import sys

import pytest

from oracle import ecc, protocol_oracle as po
from helpers import gens
from gpu_util import gpu_msm_raw
from test_gpu_protocols import range_json, P_, M_
from python_bulletproofs_b200 import secp256k1, _native as nat
from python_bulletproofs_b200.utils import commitment, mod_hash
from python_bulletproofs_b200.rangeproofs import NIRangeProver, AggregNIRangeProver
from python_bulletproofs_b200.rangeproofs.batch import (PackedBatch, PackedAggregBatch, pack_proof, pack_aggreg_proof,
                                                         pack_generators, verify_packed, verify_packed_sharded,
                                                         verify_aggreg_packed, verify_stats)

pytestmark = pytest.mark.gpu
Q, P = ecc.Q, ecc.P
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# One kind of forgery per forged proof.  The first group edits the proof and is judged by the oracle; "offcurve_*" puts a point
# that is not on secp256k1 into the packed record (rejected: fastecdsa could never build it); the last three edit transcript
# slots the way the reference compares them (a non-numeric y slot makes the reference raise: accept byte 2, "defer").
KINDS = ["t_hat_digit", "V_plus_g", "a_plus_1", "ipa_transcript_digit", "mu_plus_1", "u_new_plus_g", "taux_plus_1", "b_plus_1",
         "P_new_plus_h", "u_new_neg", "P_new_neg", "u_new_identity", "P_new_identity", "V_swapped",
         "offcurve_V", "offcurve_A", "offcurve_S", "offcurve_T1", "offcurve_T2", "offcurve_u_new", "offcurve_P_new",
         "offcurve_L0", "offcurve_R_last", "y_slot_non_numeric", "challenge_leading_zero", "y_slot_leading_zeros"]


def _offsets(m, L):
    """Byte offsets of the proof points in a packed record (include/bp_gpu.h; m = 1 is the single-value layout)."""
    v = 64 * m
    return {"V": 0, "A": v, "S": v + 64, "T1": v + 128, "T2": v + 192, "u_new": v + 352, "P_new": v + 416,
            "L0": v + 544 + 32 * L, "R_last": v + 544 + 160 * L - 64}


def _digit(v):
    s = str(v)
    return int(s[:-1] + ("1" if s[-1] != "1" else "2"))


def _edit_slot(tr, slot, fn):
    parts = tr.split(b"&")
    parts[slot] = fn(parts[slot])
    return b"&".join(parts)


def _neg(pt):
    return (pt[0], P - pt[1])


def _forge(kind, oVs, pr, other_V, og, oh):
    """Apply one oracle-visible forgery to (commitments, oracle proof dict), in place."""
    ip, p2 = pr["ip"], pr["ip"]["p2"]
    if kind == "t_hat_digit":
        pr["t_hat"] = _digit(pr["t_hat"])
    elif kind == "V_plus_g":
        oVs[-1] = ecc.point_add(oVs[-1], og)
    elif kind == "a_plus_1":
        p2["a"] = (p2["a"] + 1) % Q
    elif kind == "ipa_transcript_digit":
        t = bytearray(p2["transcript"])
        t[-5] = ord("1") if t[-5] != ord("1") else ord("2")
        p2["transcript"] = bytes(t)
    elif kind == "mu_plus_1":
        pr["mu"] = (pr["mu"] + 1) % Q
    elif kind == "u_new_plus_g":
        ip["u_new"] = ecc.point_add(ip["u_new"], og)
    elif kind == "taux_plus_1":
        pr["taux"] = (pr["taux"] + 1) % Q
    elif kind == "b_plus_1":
        p2["b"] = (p2["b"] + 1) % Q
    elif kind == "P_new_plus_h":
        ip["P_new"] = ecc.point_add(ip["P_new"], oh)
    elif kind == "u_new_neg":
        ip["u_new"] = _neg(ip["u_new"])
    elif kind == "P_new_neg":
        ip["P_new"] = _neg(ip["P_new"])
    elif kind == "u_new_identity":
        ip["u_new"] = None
    elif kind == "P_new_identity":
        ip["P_new"] = None
    elif kind == "V_swapped":
        oVs[0] = other_V
    elif kind == "y_slot_non_numeric":
        pr["transcript"] = _edit_slot(pr["transcript"], 3, lambda s: b"12x4")
    elif kind == "challenge_leading_zero":
        p2["transcript"] = _edit_slot(p2["transcript"], p2["start"] + 2, lambda s: b"0" + s)
    elif kind == "y_slot_leading_zeros":
        pr["transcript"] = _edit_slot(pr["transcript"], 3, lambda s: b"00" + s)
    else:
        assert kind.startswith("offcurve_"), kind


def _pack(oVs, pr):
    """Wire record of an oracle proof dict (same layout as batch.pack_proof / pack_aggreg_proof, points as tuples / None)."""
    le = lambda s: (s % Q).to_bytes(32, "little")          # noqa: E731
    ip, p2 = pr["ip"], pr["ip"]["p2"]
    rec = [ecc.pack_point(V) for V in oVs] + [ecc.pack_point(pr[k]) for k in ("A", "S", "T1", "T2")]
    rec += [le(pr["taux"]), le(pr["mu"]), le(pr["t_hat"]), ecc.pack_point(ip["u_new"]), ecc.pack_point(ip["P_new"]),
            le(p2["a"]), le(p2["b"])]
    rec += [le(x) for x in p2["xs"]] + [ecc.pack_point(p) for p in p2["Ls"]] + [ecc.pack_point(p) for p in p2["Rs"]]
    return b"".join(rec), (pr["transcript"], ip["transcript"], p2["transcript"]), p2["start"]


class Pool:
    """D distinct proofs over one generator set: packed records, transcripts, start indices and the expected accept bytes."""

    def __init__(self, n, m, D, tag, kind_shift=0, generators=None):
        self.n, self.m, self.D = n, m, D
        nm = n * m
        self.L = nm.bit_length() - 1
        self.ogs, self.ohs, self.og, self.oh, self.ou = generators or gens(nm, [tag + "%d" % i for i in range(5)])
        self.gens = (self.og, self.oh, self.ogs, self.ohs, self.ou)          # argument order of verify_packed
        self.packed_gens = pack_generators(self.og, self.oh, self.ogs, self.ohs, self.ou)
        gs, hs, g, h, u = [P_(t) for t in self.ogs], [P_(t) for t in self.ohs], P_(self.og), P_(self.oh), P_(self.ou)
        rng = random.Random(tag)
        honest = []
        for i in range(D):                       # GPU prover, as the reference's API is used
            vs = [M_(rng.getrandbits(n)) for _ in range(m)]
            gammas = [mod_hash(b"%s_g%d_%d" % (tag.encode(), i, j), Q) for j in range(m)]
            Vs = [commitment(g, h, vs[j], gammas[j]) for j in range(m)]
            seed = b"%s_p%d" % (tag.encode(), i)
            if m == 1:
                pr = NIRangeProver(vs[0], n, g, h, gs, hs, gammas[0], u, secp256k1, seed).prove()
                ref = pack_proof(Vs[0], pr, self.L)
            else:
                pr = AggregNIRangeProver(vs, n, g, h, gs, hs, gammas, u, secp256k1, seed).prove()
                ref = pack_aggreg_proof(Vs, pr, self.L)
            oVs, opr = [(V.x, V.y) for V in Vs], po.range_from_json(range_json(pr))
            assert _pack(oVs, opr) == ref                    # this file's packer is the library's packer
            honest.append((oVs, opr))
        off = _offsets(m, self.L)
        self.recs, self.trs, self.starts, self.kinds, want = [], [], [], [], []
        for i, (oVs, opr) in enumerate(honest):
            kind = KINDS[(i // 3 + kind_shift) % len(KINDS)] if i % 3 == 1 else None
            oVs, opr = list(oVs), copy.deepcopy(opr)
            if kind:
                _forge(kind, oVs, opr, honest[(i + 1) % D][0][0], self.og, self.oh)
            rec, trs, st = _pack(oVs, opr)
            if kind and kind.startswith("offcurve_"):
                rec = bytearray(rec)
                base = off[kind[len("offcurve_"):]]
                if i % 2:
                    rec[base + 32] ^= 1                                      # y altered: (x, y') is not on the curve
                else:
                    rec[base:base + 32] = (P + 5).to_bytes(32, "little")     # x >= p: not canonical
                rec, w = bytes(rec), 0
            elif kind == "y_slot_non_numeric":
                with pytest.raises(ValueError):                              # the reference's int() raises
                    po.range_verify(oVs, self.og, self.oh, self.ogs, self.ohs, self.ou, opr)
                w = 2
            else:
                w = int(po.range_verify(oVs, self.og, self.oh, self.ogs, self.ohs, self.ou, opr))
                assert w == (kind in (None, "y_slot_leading_zeros")), (i, kind)
            self.recs.append(rec); self.trs.append(trs); self.starts.append(st); self.kinds.append(kind); want.append(w)
        self.want = bytes(want)
        if D // 3 >= len(KINDS):
            assert set(KINDS) <= set(self.kinds)

    def tile(self, count, start):
        """A batch of `count` proofs: the pool's records from offset `start` on, wrapping around; and its expected bytes."""
        idx = [(start + i) % self.D for i in range(count)]
        recs, trs, sts = [self.recs[j] for j in idx], [self.trs[j] for j in idx], [self.starts[j] for j in idx]
        batch = PackedBatch(self.n, recs, trs, sts) if self.m == 1 else PackedAggregBatch(self.n, self.m, recs, trs, sts)
        return batch, bytes(self.want[j] for j in idx), [self.kinds[j] for j in idx]


def _same(got, want, kinds, what):
    if got != want:
        bad = [(i, kinds[i], got[i], want[i]) for i in range(min(len(got), len(want))) if got[i] != want[i]]
        pytest.fail("%s: %d of %d decisions differ from the oracle (position, forgery, got, want): %s"
                    % (what, len(bad), len(want), bad[:16]))


def _clear_tables():
    nat.check(nat.load().bp_fb_clear())


@pytest.fixture(scope="module")
def pools():
    nat.init(0)
    made = {}

    def get(n, m=1):
        if (n, m) not in made:
            D = 97 if n * m <= 16 else 79
            made[(n, m)] = Pool(n, m, D, "vb%d_%d_" % (n, m))
        return made[(n, m)]
    yield get
    _clear_tables()                 # the 16-bit table of the n = 64 set alone is ~9 GB


@pytest.fixture
def fb_mode():
    lib = nat.load()
    nat.init(0)
    _clear_tables()

    def set_mode(m):
        nat.check(lib.bp_fb_set_mode(m))
    yield set_mode
    _clear_tables()
    nat.check(lib.bp_fb_set_mode(1))


def _verify(pool, batch, first=0, count=None):
    return verify_packed(batch, *pool.gens, first, count)


# ---- single-value verifier ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [8, 64])
def test_table_paths_in_turn(fb_mode, pools, n):
    """Mode 1: first sight of the generator set takes the bucket method, the second the byte tables, the third the 16-bit tables;
    mode 0 the bucket method every time.  One chunk each (the default plan of 300 proofs)."""
    pool = pools(n)
    batch, want, kinds = pool.tile(300, 11)
    fb_mode(1)
    for call, mode in enumerate((0, 1, 2, 2)):
        _same(_verify(pool, batch), want, kinds, "fb mode 1, call %d" % call)
        st = verify_stats()
        assert (st["table_mode"], st["chunks"], st["proofs"]) == (mode, 1, 300), st
    fb_mode(0)
    _same(_verify(pool, batch), want, kinds, "fb mode 0")
    assert verify_stats()["table_mode"] == 0


def test_bucket_method_over_three_chunks(fb_mode, pools):
    """Without tables a batch of >= 4096 proofs runs as chunks of 2048: the third reuses the first one's buffers."""
    pool = pools(8)
    batch, want, kinds = pool.tile(4200, 40)
    fb_mode(0)
    _same(_verify(pool, batch), want, kinds, "bucket method, 2048 + 2048 + 104")
    st = verify_stats()
    assert (st["table_mode"], st["chunks"]) == (0, 3), st


@pytest.mark.parametrize("mode", [2, 0])
@pytest.mark.parametrize("chunk", [1, 7, 8, 9, 31, 32, 33, 65])
def test_forced_chunk_lengths(fb_mode, pools, monkeypatch, chunk, mode):
    """BP_VERIFY_CHUNK: chunks of <= 8 proofs invert on the host, longer ones in k_rp_invert (partial warps at 9, 31, 33, 65);
    from the third chunk on a buffer set is reused; the host verdicts of every chunk are merged at the end."""
    pool = pools(8)
    count = 300
    batch, want, kinds = pool.tile(count, 3 * chunk + mode)
    fb_mode(mode)
    monkeypatch.setenv("BP_VERIFY_CHUNK", str(chunk))
    _same(_verify(pool, batch), want, kinds, "chunks of %d, fb mode %d" % (chunk, mode))
    st = verify_stats()
    assert (st["table_mode"], st["chunks"]) == (mode, -(-count // chunk)), st


def test_long_chunks_take_k_sv_comb2(fb_mode, pools, monkeypatch):
    """Chunks longer than 1536 proofs finish the proof-specific terms in k_sv_comb2, shorter ones in k_sv_comb2q: 1537 + 1537 +
    226 proofs run both in one batch."""
    pool = pools(8)
    batch, want, kinds = pool.tile(3300, 29)
    fb_mode(2)
    monkeypatch.setenv("BP_VERIFY_CHUNK", "1537")
    for call in range(2):                   # the second call finds both tables of the set and skips the generator uploads
        _same(_verify(pool, batch), want, kinds, "chunks of 1537, call %d" % call)
        st = verify_stats()
        assert (st["table_mode"], st["chunks"]) == (2, 3), st


def test_default_plan_at_64_bits(fb_mode, pools):
    """The production shape: 4096 proofs of 64 bits are planned as 512 + 1024 + 2048 + 512 proofs."""
    pool = pools(64)
    batch, want, kinds = pool.tile(4096, 7)
    fb_mode(2)
    for call in range(2):
        _same(_verify(pool, batch), want, kinds, "4096 proofs of 64 bits, call %d" % call)
        st = verify_stats()
        assert (st["table_mode"], st["chunks"], st["proofs"]) == (2, 4, 4096), st


def test_few_host_threads_split_in_two(fb_mode, pools, monkeypatch):
    """One process per GPU sharing every core (LOCAL_WORLD_SIZE >= cores: one host thread): 1024 proofs go as 256 + 768."""
    pool = pools(8)
    batch, want, kinds = pool.tile(1024, 50)
    fb_mode(2)
    monkeypatch.setenv("LOCAL_WORLD_SIZE", "4096")
    _same(_verify(pool, batch), want, kinds, "one host thread")
    st = verify_stats()
    assert (st["table_mode"], st["chunks"], st["host_threads"]) == (2, 2, 1), st


def test_slices_and_one_rank_gather(fb_mode, pools):
    """verify_packed on sub-ranges, bp_rp_verify_batch_gather on one rank (padding past the block, an empty block) and the
    one-rank sharded call all give the bytes of the whole batch's call."""
    pool = pools(8)
    batch, want, kinds = pool.tile(211, 17)
    fb_mode(1)
    full = _verify(pool, batch)
    _same(full, want, kinds, "whole batch")
    for first, count in ((0, 1), (1, 37), (38, 99), (137, 73), (210, 1), (5, 9)):
        assert _verify(pool, batch, first, count) == full[first:first + count], (first, count)

    def gather(b, width):
        out = ctypes.create_string_buffer(max(width, 1))
        nat.check(nat.load().bp_rp_verify_batch_gather(*pool.packed_gens, b.n, b.records, b.stride, b.nproofs, b.blob, b.tr_off,
                                                        b.starts, width, out))
        return out.raw[:width]
    assert gather(batch, batch.nproofs + 5) == full + bytes(5)
    assert gather(PackedBatch(pool.n, [], [], []), 4) == bytes(4)
    # an empty block (a rank with no proofs) is planned as no chunk at all, and the library goes on working afterwards
    rng = random.Random(3)
    ks = [rng.getrandbits(256) % Q for _ in range(pool.n)]
    assert gpu_msm_raw(ecc.pack_points(pool.ogs), b"".join(k.to_bytes(32, "little") for k in ks), pool.n) == ecc.msm(pool.ogs, ks)
    assert verify_packed_sharded(batch, *pool.gens, rank=0, world=1) == full
    assert _verify(pool, batch) == full


# ---- aggregated verifier --------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("count", [65, 300, 1031])
@pytest.mark.parametrize("nm", [(8, 2), (64, 16)])
def test_aggregated_over_several_chunks(fb_mode, pools, nm, count):
    """Chunks of max(64, ceil(count / 4)) proofs (several chunks and a short last one), both host buffer sets, the previous
    chunk finished while the next is on the device; bucket method over the generator rows, then the byte table."""
    pool = pools(*nm)
    batch, want, kinds = pool.tile(count, count % pool.D)
    for mode, calls in ((0, 1), (1, 2)):
        fb_mode(mode)
        for call in range(calls):
            _same(verify_aggreg_packed(batch, *pool.gens, packed=pool.packed_gens), want, kinds,
                  "%d aggregated proofs, fb mode %d, call %d" % (count, mode, call))


# ---- one generator set, three entry points --------------------------------------------------------------------------------
def test_shared_generator_tables_across_entry_points(fb_mode):
    """The single-value verifier at n = 8 and the aggregated one at n = 4, m = 2 use the same 21 table rows (same cache key), and
    bp_msm the same 8 points as a set of its own.  Interleaved calls, with the cache cleared in between, change no decision."""
    sv = Pool(8, 1, 29, "shared", kind_shift=9)
    ag = Pool(4, 2, 23, "shared", kind_shift=19)
    assert sv.packed_gens == ag.packed_gens
    sv_batch, sv_want, sv_kinds = sv.tile(40, 0)
    ag_batch, ag_want, ag_kinds = ag.tile(30, 0)
    rng = random.Random(21)
    fb_mode(1)

    def run(step):
        if step == "sv":
            _same(_verify(sv, sv_batch), sv_want, sv_kinds, "single-value")
        elif step == "agg":
            _same(verify_aggreg_packed(ag_batch, *ag.gens, packed=ag.packed_gens), ag_want, ag_kinds, "aggregated")
        elif step == "msm":
            ks = [rng.getrandbits(256) % Q for _ in range(sv.n)]
            assert gpu_msm_raw(ecc.pack_points(sv.ogs), b"".join(k.to_bytes(32, "little") for k in ks), sv.n) == ecc.msm(sv.ogs, ks)
        else:
            _clear_tables()
    for step in ("sv", "agg", "msm", "sv", "msm", "agg", "sv", "clear", "agg", "sv", "msm", "agg", "sv", "msm", "clear", "sv", "sv",
                 "agg", "sv"):
        run(step)


# ---- knobs read once per process ------------------------------------------------------------------------------------------
_CHILD = r'''
import os, pickle, sys
sys.path.insert(0, sys.argv[1])
from python_bulletproofs_b200 import _native as nat
from python_bulletproofs_b200.rangeproofs.batch import PackedBatch, PackedAggregBatch, verify_packed, verify_aggreg_packed, verify_stats
with open(sys.argv[2], "rb") as f:
    cases = pickle.load(f)
nat.init(0)
lib = nat.load()
for c in cases:
    if c["m"] == 1:
        batch = PackedBatch(c["n"], c["recs"], c["trs"], c["starts"])
        if c["chunk"]:
            os.environ["BP_VERIFY_CHUNK"] = str(c["chunk"])
        nat.check(lib.bp_fb_set_mode(2))
        for call in range(2):
            got = verify_packed(batch, *c["gens"])
            st = verify_stats()
            assert got == c["want"], ("single", c["n"], c["chunk"], [i for i in range(len(got)) if got[i] != c["want"][i]][:16])
            assert (st["table_mode"], st["chunks"]) == (2, c["chunks"]), st
        os.environ.pop("BP_VERIFY_CHUNK", None)
    else:
        batch = PackedAggregBatch(c["n"], c["m"], c["recs"], c["trs"], c["starts"])
        for mode in (0, 1, 1):
            nat.check(lib.bp_fb_set_mode(mode))
            got = verify_aggreg_packed(batch, *c["gens"])
            assert got == c["want"], ("aggregated", mode, [i for i in range(len(got)) if got[i] != c["want"][i]][:16])
    nat.check(lib.bp_fb_clear())
print("OK")
'''


def test_knobs_read_once_per_process(tmp_path, pools):
    """BP_SV_LATENCY_MAX=0 (k_sv_comb2 at every chunk length), BP_RP_WARPS=4 (k_rp_lookup16<128, 4>) and BP_AGG_CHUNK=3 (many
    3-proof aggregated chunks) are read once per process, so they are set for a fresh one."""
    cases = []
    for n, count, start, chunk, chunks in ((8, 301, 2, None, 1), (8, 300, 61, 7, 43), (8, 2100, 5, None, 4), (64, 200, 13, 33, 7)):
        pool = pools(n)
        batch, want, _ = pool.tile(count, start)
        idx = [(start + i) % pool.D for i in range(count)]
        cases.append({"m": 1, "n": n, "recs": [pool.recs[j] for j in idx], "trs": [pool.trs[j] for j in idx],
                      "starts": [pool.starts[j] for j in idx], "want": want, "gens": pool.gens, "chunk": chunk, "chunks": chunks})
    pool = pools(8, 2)
    count, start = 65, 31
    idx = [(start + i) % pool.D for i in range(count)]
    cases.append({"m": 2, "n": 8, "recs": [pool.recs[j] for j in idx], "trs": [pool.trs[j] for j in idx],
                  "starts": [pool.starts[j] for j in idx], "want": pool.tile(count, start)[1], "gens": pool.gens})
    data = tmp_path / "cases.pkl"
    with open(data, "wb") as f:
        pickle.dump(cases, f)
    script = tmp_path / "child.py"
    script.write_text(_CHILD)
    env = dict(os.environ, BP_SV_LATENCY_MAX="0", BP_RP_WARPS="4", BP_AGG_CHUNK="3")
    env.pop("BP_VERIFY_CHUNK", None)
    env.pop("LOCAL_WORLD_SIZE", None)
    out = subprocess.run([sys.executable, str(script), ROOT, str(data)], env=env, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0 and out.stdout.strip().endswith("OK"), (out.stdout[-2000:], out.stderr[-4000:])


# ---- a generator set whose own sums collide -------------------------------------------------------------------------------
def _degenerate_generators(n, tag):
    """gs = [P1, -P1, P2, -P2, ...] (Gsum = O), hs = [Q1, Q1, Q2, Q2, ...] (Hsum a sum of doublings), u = g."""
    base = [po.elliptic_hash(b"%s%d" % (tag, i)) for i in range(n + 2)]
    gs = [p for i in range(n // 2) for p in (base[i], _neg(base[i]))]
    hs = [base[n // 2 + i // 2] for i in range(n)]
    g, h = base[n], base[n + 1]
    return gs, hs, g, h, g


def test_degenerate_generator_set(fb_mode):
    """The verifier's own sums of a generator set (k_sum_points: Gsum, Hsum) on a set where they cancel and double; every accept
    byte against the oracle under table modes 0, 1 and 2, then the set alternated with an ordinary one of the same length in one
    process, so that the Gsum / Hsum kept from one set can never serve the other."""
    n = 16
    gens16 = _degenerate_generators(n, b"degenerate")
    assert functools.reduce(ecc.point_add, gens16[0]) is None
    deg = Pool(n, 1, 64, "degenerate", generators=gens16)
    plain = Pool(n, 1, 31, "ordinary16_")
    deg_batch, deg_want, deg_kinds = deg.tile(64, 0)
    plain_batch, plain_want, plain_kinds = plain.tile(93, 5)
    for mode in (0, 1, 2):
        fb_mode(mode)
        for call in range(2):
            _same(_verify(deg, deg_batch), deg_want, deg_kinds, "degenerate set, fb mode %d, call %d" % (mode, call))
    for mode in (0, 1):
        fb_mode(mode)
        for step in range(6):
            if step % 2:
                _same(_verify(plain, plain_batch), plain_want, plain_kinds, "ordinary set, fb mode %d, step %d" % (mode, step))
            else:
                _same(_verify(deg, deg_batch), deg_want, deg_kinds, "degenerate set, fb mode %d, step %d" % (mode, step))
