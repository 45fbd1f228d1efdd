"""Exact batch verifiers against bp_rp_verify_batch_rlc (one random linear combination per batch) on the same batches.
usage: python tools/rlc_probe.py [--out profiles/rlc_probe.json] [--reps 10]

Workloads: (a) 8192 distinct valid 64-bit single-value proofs (made as bench.py's verify row makes them), (b) (a) with tau_x + 1 on
one proof, (c) 2048 aggregated proofs of 16 x 64 bits, 32 distinct proofs tiled (as bench.py's aggregated row), all valid, (d) (c)
with mu + 1 on one proof.  Per workload: 4 warm-up calls of each (they build the generator tables), then `reps` timed calls of
each, alternating; median and best wall time of each, `combined`, and whether both give the same accept bytes.  The card's name
and power limit are read in the same run and written beside the numbers (one JSON line)."""
import argparse
import json
import os
import random
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return out.stdout.strip().splitlines()[0] if out.returncode == 0 and out.stdout.strip() else "unknown"


def bump(batch, i, off):
    """scalar at byte `off` of record i, plus 1 mod q"""
    from python_bulletproofs_b200 import _native as nat
    rec = bytearray(batch.records)
    o = i * batch.stride + off
    rec[o:o + 32] = ((int.from_bytes(rec[o:o + 32], "little") + 1) % nat.Q).to_bytes(32, "little")
    batch.records = bytes(rec)


def single_value(total):
    from python_bulletproofs_b200 import secp256k1
    from python_bulletproofs_b200.rangeproofs import NIRangeProver
    from python_bulletproofs_b200.rangeproofs.batch import PackedBatch
    from python_bulletproofs_b200.utils import ModP, commitment, mod_hash, elliptic_hash
    q, nbits = secp256k1.q, 64
    seeds = [b"seed%d" % i for i in range(5)]
    gs = [elliptic_hash(str(i).encode() + seeds[0], secp256k1) for i in range(nbits)]
    hs = [elliptic_hash(str(i).encode() + seeds[1], secp256k1) for i in range(nbits)]
    g, h, u = (elliptic_hash(s, secp256k1) for s in seeds[2:5])
    rng = random.Random(5)
    vals = [rng.getrandbits(64) for _ in range(total)]
    Vs, proofs = [], []
    for i in range(total):
        gamma = mod_hash(b"gamma%d" % i, q)
        Vs.append(commitment(g, h, ModP(vals[i], q), gamma))
        proofs.append(NIRangeProver(ModP(vals[i], q), nbits, g, h, gs, hs, gamma, u, secp256k1, b"p%d" % i).prove())
    return PackedBatch.from_proofs(Vs, proofs, nbits), (g, h, gs, hs, u)


def aggregated(total, distinct, m=16, nbits=64):
    from python_bulletproofs_b200 import secp256k1
    from python_bulletproofs_b200.rangeproofs import AggregNIRangeProver
    from python_bulletproofs_b200.rangeproofs.batch import PackedAggregBatch
    from python_bulletproofs_b200.utils import ModP, commitment, mod_hash, elliptic_hash
    q, nm = secp256k1.q, nbits * m
    gs = [elliptic_hash(str(i).encode() + b"agg0", secp256k1) for i in range(nm)]
    hs = [elliptic_hash(str(i).encode() + b"agg1", secp256k1) for i in range(nm)]
    g, h, u = (elliptic_hash(s_, secp256k1) for s_ in (b"agg2", b"agg3", b"agg4"))
    rng = random.Random(16)
    Vl, pl = [], []
    for i in range(distinct):
        vs = [ModP(rng.getrandbits(nbits), q) for _ in range(m)]
        gammas = [mod_hash(b"ag%d_%d" % (i, j), q) for j in range(m)]
        Vl.append([commitment(g, h, vs[j], gammas[j]) for j in range(m)])
        pl.append(AggregNIRangeProver(vs, nbits, g, h, gs, hs, gammas, u, secp256k1, b"y%d" % i).prove())
    return PackedAggregBatch.from_proofs(Vl * (total // distinct), pl * (total // distinct), nbits), (g, h, gs, hs, u)


def measure(name, batch, gens, exact, reps):
    from python_bulletproofs_b200.rangeproofs.batch import pack_generators, verify_rlc_packed
    packed = pack_generators(*gens)
    te, tr, acc_e, acc_r, comb = [], [], b"", b"", None
    for it in range(4 + reps):
        a = time.perf_counter()
        acc_e = exact(batch, *gens)
        b = time.perf_counter()
        acc_r, comb = verify_rlc_packed(batch, *gens, packed=packed)
        c = time.perf_counter()
        if it >= 4:
            te.append(b - a)
            tr.append(c - b)
    ms = lambda v: round(v * 1e3, 3)      # noqa: E731
    return {"workload": name, "proofs": batch.nproofs, "exact_ms_median": ms(statistics.median(te)), "exact_ms_best": ms(min(te)),
            "rlc_ms_median": ms(statistics.median(tr)), "rlc_ms_best": ms(min(tr)), "combined": comb,
            "decisions_equal": acc_e == acc_r, "rejected": acc_e.count(b"\x00"), "timed_calls_each": reps}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "rlc_probe.json"))
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--proofs", type=int, default=8192)
    ap.add_argument("--aggregated", type=int, default=2048)
    args = ap.parse_args()
    from python_bulletproofs_b200 import _native as nat
    from python_bulletproofs_b200.rangeproofs.batch import verify_packed, verify_aggreg_packed
    nat.init(0)
    rows = []
    sv, sv_gens = single_value(args.proofs)
    rows.append(measure("(a) %d distinct 64-bit proofs, all valid" % sv.nproofs, sv, sv_gens, verify_packed, args.reps))
    bump(sv, sv.nproofs // 3, 320)                    # tau_x of the single-value record
    rows.append(measure("(b) (a) with tau_x + 1 on one proof", sv, sv_gens, verify_packed, args.reps))
    ag, ag_gens = aggregated(args.aggregated, 32)
    rows.append(measure("(c) %d aggregated 16 x 64-bit proofs, 32 distinct, all valid" % ag.nproofs, ag, ag_gens, verify_aggreg_packed, args.reps))
    bump(ag, ag.nproofs // 3, 64 * 16 + 288)          # mu of the aggregated record
    rows.append(measure("(d) (c) with mu + 1 on one proof", ag, ag_gens, verify_aggreg_packed, args.reps))
    res = {"tool": "rlc_probe", "card": card(), "host_threads": os.cpu_count(), "rows": rows}
    line = json.dumps(res)
    print(line)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(line + "\n")


if __name__ == "__main__":
    main()
