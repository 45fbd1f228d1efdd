"""bp_rp_prove_batch (prove_range_proofs_packed / prove_range_proofs_batch) against a loop over the per-proof prover classes.
usage: python tools/prove_batch_probe.py [--out profiles/prove_batch_probe.json] [--reps 10]

Workloads:
  (a) 8192 distinct 64-bit single-value proofs (NIRangeProver; the loop arm times 256 proofs and is scaled to the batch);
  (b) 2048 distinct aggregated 16 x 64-bit proofs (AggregNIRangeProver; the loop arm times 32 proofs and is scaled).
Arms: the per-proof class loop; prove_range_proofs_packed (wire-form output, the verifiers' input); prove_range_proofs_batch (the
same call plus the Proof objects).  The generator set's table is warmed first: 4 warm-up calls of each arm, then `reps` timed calls
of each, alternating.  Every call is timed on the host around the whole call (inputs built once, outside).  Per arm: median and
best wall time and proofs/s; for the packed arm the library's statistics of its last call (host ms of the host steps, device span,
chunks, host threads, table mode).  A sample of each batch (every 37th proof, the first and the last) is compared byte for byte
with the per-proof prover inside the probe.  The card's name and power limit are read in the same run (one JSON line)."""
import argparse
import json
import os
import random
import statistics
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import rlc_probe                # noqa: E402  (card())


def inputs(count, m, nbits, tag):
    from python_bulletproofs_b200 import secp256k1
    from python_bulletproofs_b200.utils import ModP, elliptic_hash
    q, nm = secp256k1.q, nbits * m
    gs = [elliptic_hash(str(i).encode() + tag + b"0", secp256k1) for i in range(nm)]
    hs = [elliptic_hash(str(i).encode() + tag + b"1", secp256k1) for i in range(nm)]
    g, h, u = (elliptic_hash(tag + s, secp256k1) for s in (b"2", b"3", b"4"))
    rng = random.Random(tag)
    vs = [[ModP(rng.getrandbits(nbits), q) for _ in range(m)] for _ in range(count)]
    gammas = [[ModP(rng.getrandbits(256) % q, q) for _ in range(m)] for _ in range(count)]
    seeds = [tag + b"-%d" % i for i in range(count)]
    return (g, h, gs, hs, u), vs, gammas, seeds


def per_proof(gens, vs, gammas, seeds, nbits, i):
    from python_bulletproofs_b200 import secp256k1
    from python_bulletproofs_b200.rangeproofs import NIRangeProver, AggregNIRangeProver
    g, h, gs, hs, u = gens
    if len(vs[i]) == 1:
        return NIRangeProver(vs[i][0], nbits, g, h, gs, hs, gammas[i][0], u, secp256k1, seeds[i]).prove()
    return AggregNIRangeProver(vs[i], nbits, g, h, gs, hs, gammas[i], u, secp256k1, seeds[i]).prove()


def identical_sample(batch, gens, vs, gammas, seeds, nbits):
    """every 37th proof, the first and the last: record and transcripts equal to the per-proof prover's"""
    from python_bulletproofs_b200.rangeproofs.batch import pack_aggreg_proof
    from python_bulletproofs_b200.utils import commitment
    g, h = gens[0], gens[1]
    L = (nbits * batch.m).bit_length() - 1
    idx = sorted(set(range(0, batch.nproofs, 37)) | {0, batch.nproofs - 1})
    for i in idx:
        ref = per_proof(gens, vs, gammas, seeds, nbits, i)
        rec, trio, start = pack_aggreg_proof([commitment(g, h, v, gm) for v, gm in zip(vs[i], gammas[i])], ref, L)
        offs = [batch.tr_off[3 * i + k] for k in range(4)]
        if (batch.records[i * batch.stride:(i + 1) * batch.stride] != rec or batch.starts[i] != start
                or tuple(batch.blob[offs[k]:offs[k + 1]] for k in range(3)) != trio):
            return False, len(idx)
    return True, len(idx)


def workload(name, count, m, nbits, loop_count, reps, tag):
    from python_bulletproofs_b200.rangeproofs import prove_range_proofs_packed, prove_range_proofs_batch
    from python_bulletproofs_b200.rangeproofs.batch import pack_generators, verify_stats
    gens, vs, gammas, seeds = inputs(count, m, nbits, tag)
    g, h, gs, hs, u = gens
    packed = pack_generators(g, h, gs, hs, u)
    arms = [("per-proof class loop (%d proofs, scaled x%d)" % (loop_count, count // loop_count),
             lambda: [per_proof(gens, vs, gammas, seeds, nbits, i) for i in range(loop_count)], count // loop_count),
            ("prove_range_proofs_packed", lambda: prove_range_proofs_packed(vs, nbits, g, h, gs, hs, gammas, u, seeds, packed), 1),
            ("prove_range_proofs_batch", lambda: prove_range_proofs_batch(vs, nbits, g, h, gs, hs, gammas, u, seeds, packed), 1)]
    for _ in range(4):
        for _, fn, _ in arms:
            fn()
    times = [[] for _ in arms]
    stats, last = None, None
    for _ in range(reps):
        for k, (label, fn, _) in enumerate(arms):
            a = time.perf_counter()
            out = fn()
            times[k].append(time.perf_counter() - a)
            if label == "prove_range_proofs_packed":
                stats, last = verify_stats(), out
    same, checked = identical_sample(last, gens, vs, gammas, seeds, nbits)
    row = {"workload": name, "proofs": count, "timed_calls_each": reps, "sample_identical": same, "sample_size": checked, "arms": []}
    for k, (label, _, scale) in enumerate(arms):
        med, best = statistics.median(times[k]) * scale, min(times[k]) * scale
        arm = {"arm": label, "ms_median": round(med * 1e3, 3), "ms_best": round(best * 1e3, 3),
               "proofs_per_s_median": round(count / med, 1)}
        if label == "prove_range_proofs_packed":
            arm["stats"] = {k2: (round(v, 3) if isinstance(v, float) else v) for k2, v in stats.items()}
        row["arms"].append(arm)
    print(json.dumps(row), flush=True)
    return row


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "prove_batch_probe.json"))
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--proofs", type=int, default=8192)
    ap.add_argument("--aggregated", type=int, default=2048)
    args = ap.parse_args()
    from python_bulletproofs_b200 import _native as nat
    card = rlc_probe.card()
    nat.init(0)
    rows = [workload("(a) %d distinct 64-bit single-value proofs" % args.proofs, args.proofs, 1, 64, 256, args.reps, b"pb1"),
            workload("(b) %d distinct aggregated 16 x 64-bit proofs" % args.aggregated, args.aggregated, 16, 64, 32, args.reps,
                     b"pb16")]
    res = {"tool": "prove_batch_probe", "card": card, "host_threads": os.cpu_count(), "rows": rows}
    line = json.dumps(res)
    print(line)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(line + "\n")


if __name__ == "__main__":
    main()
