"""One mixed-shape call (bp_rp_verify_mixed_rlc) against per-shape calls on the same batch.
usage: python tools/mixed_rlc_probe.py [--out profiles/mixed_rlc_probe.json] [--reps 10]

Workload: 4096 range proofs of 64-bit values with m = 1, 2, 4, 8, 16 values per proof in the proportions 16 : 8 : 4 : 2 : 1
(2114, 1057, 529, 264 and 132 proofs), all over prefixes of one generator set of nset = 1024 points per side, `--distinct` distinct
proofs per shape tiled and shuffled into one caller order.  Arms:
  (a) one bp_rp_verify_mixed_rlc call over the set;
  (b) one bp_rp_verify_batch_rlc call per shape over its prefix set, the decisions scattered back to the caller's order;
  (c) the exact verifiers per shape (bp_rp_verify_batch for m = 1, bp_rp_verify_aggreg_batch otherwise), scattered likewise;
  (d) (a) with mu + 1 on one proof.
Every call is timed on the host around the whole call (packing is done once, outside).  First each arm alone after the generator
tables are cleared: 4 warm-up calls, then bp_fb_stats gives the table bytes that arm keeps.  Then, tables cleared again, 4 warm-up
calls of each arm and `reps` timed calls of each, alternating; median and best wall time, `combined`, and whether the decisions
equal those of the exact per-shape verifiers on the same batch.  The card's name and power limit are read in the same run and
written beside the numbers (one JSON line)."""
import argparse
import ctypes
import json
import os
import random
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

NSET, NBITS = 1024, 64
SHAPE_COUNTS = {1: 2114, 2: 1057, 4: 529, 8: 264, 16: 132}          # m -> proofs (16 : 8 : 4 : 2 : 1 of 4096)


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return out.stdout.strip().splitlines()[0] if out.returncode == 0 and out.stdout.strip() else "unknown"


def make_items(distinct):
    """-> generators (g, h, gs, hs, u) of the set, {m: [(record, transcripts, start)]} of `distinct` valid proofs per shape"""
    from python_bulletproofs_b200 import secp256k1
    from python_bulletproofs_b200.rangeproofs import NIRangeProver, AggregNIRangeProver
    from python_bulletproofs_b200.rangeproofs.batch import pack_aggreg_proof
    from python_bulletproofs_b200.utils import ModP, commitment, mod_hash, elliptic_hash
    q = secp256k1.q
    gs = [elliptic_hash(str(i).encode() + b"mix0", secp256k1) for i in range(NSET)]
    hs = [elliptic_hash(str(i).encode() + b"mix1", secp256k1) for i in range(NSET)]
    g, h, u = (elliptic_hash(s, secp256k1) for s in (b"mix2", b"mix3", b"mix4"))
    rng = random.Random(31)
    made = {}
    for m in SHAPE_COUNTS:
        N = NBITS * m
        out = []
        for i in range(distinct):
            vs = [ModP(rng.getrandbits(NBITS), q) for _ in range(m)]
            gammas = [mod_hash(b"mx%d_%d_%d" % (m, i, j), q) for j in range(m)]
            Vs = [commitment(g, h, vs[j], gammas[j]) for j in range(m)]
            if m == 1:
                pr = NIRangeProver(vs[0], NBITS, g, h, gs[:N], hs[:N], gammas[0], u, secp256k1, b"mp%d_%d" % (m, i)).prove()
            else:
                pr = AggregNIRangeProver(vs, NBITS, g, h, gs[:N], hs[:N], gammas, u, secp256k1, b"mp%d_%d" % (m, i)).prove()
            out.append(pack_aggreg_proof(Vs, pr, N.bit_length() - 1))
        made[m] = out
    return (g, h, gs, hs, u), made


def bump_mu(rec, m):
    """mu + 1 mod q in an aggregated record of m values"""
    from python_bulletproofs_b200 import _native as nat
    o = 64 * m + 288
    rec = bytearray(rec)
    rec[o:o + 32] = ((int.from_bytes(rec[o:o + 32], "little") + 1) % nat.Q).to_bytes(32, "little")
    return bytes(rec)


class Workload:
    """The caller's order of (m, distinct index), the mixed batch and the per-shape batches (with their positions)."""

    def __init__(self, gens_, made, distinct, forged_at=None):
        from python_bulletproofs_b200.rangeproofs.batch import PackedBatch, PackedAggregBatch, PackedMixedBatch, pack_generators
        self.gens = gens_
        g, h, gs, hs, u = gens_
        entries = [(m, i % distinct) for m, c in SHAPE_COUNTS.items() for i in range(c)]
        random.Random(7).shuffle(entries)
        self.n = len(entries)
        recs = [made[m][j][0] for m, j in entries]
        if forged_at is not None:
            recs[forged_at] = bump_mu(recs[forged_at], entries[forged_at][0])
        trs, sts = [made[m][j][1] for m, j in entries], [made[m][j][2] for m, j in entries]
        self.mixed = PackedMixedBatch(NSET, [NBITS] * self.n, [m for m, _ in entries], recs, trs, sts)
        self.packed = pack_generators(g, h, gs, hs, u)
        self.shapes = []
        for m in SHAPE_COUNTS:
            pos = [k for k, (mm, _) in enumerate(entries) if mm == m]
            r, t, s = [recs[k] for k in pos], [trs[k] for k in pos], [sts[k] for k in pos]
            b = PackedBatch(NBITS, r, t, s) if m == 1 else PackedAggregBatch(NBITS, m, r, t, s)
            N = NBITS * m
            self.shapes.append((m, pos, b, (g, h, gs[:N], hs[:N], u), pack_generators(g, h, gs[:N], hs[:N], u)))

    def arm_mixed(self):
        from python_bulletproofs_b200.rangeproofs.batch import verify_mixed_rlc_packed
        return verify_mixed_rlc_packed(self.mixed, *self.gens, packed=self.packed)

    def arm_per_shape(self, combine):
        from python_bulletproofs_b200.rangeproofs.batch import verify_rlc_packed, verify_packed, verify_aggreg_packed
        out = bytearray(self.n)
        comb = 1
        for m, pos, b, gens_, packed in self.shapes:
            if combine:
                acc, c = verify_rlc_packed(b, *gens_, packed=packed)
                comb &= c
            else:
                acc, c = (verify_packed(b, *gens_) if m == 1 else verify_aggreg_packed(b, *gens_, packed=packed)), None
            for k, a in zip(pos, acc):
                out[k] = a
        return bytes(out), (comb if combine else None)


def fb_bytes():
    from python_bulletproofs_b200 import _native as nat
    t, b = ctypes.c_uint64(), ctypes.c_uint64()
    nat.check(nat.load().bp_fb_stats(ctypes.byref(t), ctypes.byref(b), None, None))
    return int(t.value), int(b.value)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "mixed_rlc_probe.json"))
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--distinct", type=int, default=8)
    args = ap.parse_args()
    from python_bulletproofs_b200 import _native as nat
    nat.init(0)
    lib = nat.load()
    gens_, made = make_items(args.distinct)
    ok = Workload(gens_, made, args.distinct)
    bad = Workload(gens_, made, args.distinct, forged_at=ok.n // 3)
    arms = [("(a) one bp_rp_verify_mixed_rlc call", ok.arm_mixed),
            ("(b) one bp_rp_verify_batch_rlc call per shape", lambda: ok.arm_per_shape(True)),
            ("(c) exact verifier per shape", lambda: ok.arm_per_shape(False)),
            ("(d) (a) with mu + 1 on one proof", bad.arm_mixed)]
    want = {id(ok): ok.arm_per_shape(False)[0], id(bad): bad.arm_per_shape(False)[0]}
    ref = [want[id(ok)]] * 3 + [want[id(bad)]]
    tables = []
    for name, fn in arms:                       # each arm alone: the tables it keeps
        nat.check(lib.bp_fb_clear())
        for _ in range(4):
            fn()
        tables.append(fb_bytes())
    nat.check(lib.bp_fb_clear())
    for _ in range(4):
        for _, fn in arms:
            fn()
    all_tables = fb_bytes()
    times = [[] for _ in arms]
    last = [None] * len(arms)
    for _ in range(args.reps):
        for k, (_, fn) in enumerate(arms):
            a = time.perf_counter()
            last[k] = fn()
            times[k].append(time.perf_counter() - a)
    ms = lambda v: round(v * 1e3, 3)            # noqa: E731
    rows = []
    for k, (name, _) in enumerate(arms):
        acc, comb = last[k]
        rows.append({"arm": name, "ms_median": ms(statistics.median(times[k])), "ms_best": ms(min(times[k])), "combined": comb,
                     "decisions_equal_exact": acc == ref[k], "rejected": acc.count(b"\x00"),
                     "tables": tables[k][0], "table_bytes": tables[k][1], "timed_calls": args.reps})
    res = {"tool": "mixed_rlc_probe", "card": card(), "host_threads": os.cpu_count(), "nset": NSET, "bits": NBITS,
           "proofs_per_m": SHAPE_COUNTS, "distinct_per_shape": args.distinct, "tables_all_arms": all_tables[0],
           "table_bytes_all_arms": all_tables[1], "rows": rows}
    line = json.dumps(res)
    print(line)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(line + "\n")


if __name__ == "__main__":
    main()
