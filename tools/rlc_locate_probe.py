"""bp_rp_verify_rlc_locate against the random-linear-combination verifiers and the exact verifiers on the same batches.
usage: python tools/rlc_locate_probe.py [--out profiles/rlc_locate_probe.json] [--reps 10]

Workloads (the batches of tools/rlc_probe.py and tools/mixed_rlc_probe.py):
  (a) 8192 distinct valid 64-bit single-value proofs: locate against verify_rlc_packed;
  (b) (a) with tau_x + 1 on 1, 8 and 64 proofs spread over the batch, and on every proof: the exact verifier, verify_rlc_packed
      (the exact verifier over the whole batch when the sum fails) and locate;
  (c) 2048 aggregated 16 x 64-bit proofs (32 distinct, tiled), all valid and with mu + 1 on one proof: the same three arms;
  (d) the mixed batch of tools/mixed_rlc_probe.py (4096 proofs, m = 1 ... 16 over one set of 1024 generators), all valid and with
      mu + 1 on one proof: exact verifiers per shape, verify_mixed_rlc_packed and locate;
  (e) leaf-size sweep: locate with leaf = 8 ... 256 on (b) and (c) with one forged proof.
Every call is timed on the host around the whole call (packing is done once, outside).  Per workload: 4 warm-up calls of each arm,
then `reps` timed calls of each, alternating arms on the same batch; median and best wall time, `combined`, the locate statistics
(leaf, leaves, failing leaves, proofs decided exactly) and whether every arm gives the same accept bytes.  The card's name and
power limit are read in the same run and written beside the numbers (one JSON line)."""
import argparse
import json
import os
import statistics
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import rlc_probe                # noqa: E402  (the batches of (a) - (c), card())
import mixed_rlc_probe          # noqa: E402  (the batch of (d))


def forged(batch, positions, off):
    """a copy of `batch` with the scalar at byte `off` of every record in `positions` plus 1 mod q"""
    import copy
    from python_bulletproofs_b200 import _native as nat
    rec = bytearray(batch.records)
    for i in positions:
        o = i * batch.stride + off
        rec[o:o + 32] = ((int.from_bytes(rec[o:o + 32], "little") + 1) % nat.Q).to_bytes(32, "little")
    out = copy.copy(batch)
    out.records = bytes(rec)
    return out


def spread(n, k):
    return [(2 * i + 1) * n // (2 * k) for i in range(k)]


def run(name, arms, reps):
    """arms: [(label, fn -> (accept, combined))]; 4 warm-up calls each, then `reps` rounds of one call of each arm"""
    from python_bulletproofs_b200.rangeproofs.batch import rlc_locate_stats
    for _ in range(4):
        for _, fn in arms:
            fn()
    times = [[] for _ in arms]
    last, stats = [None] * len(arms), {}
    for _ in range(reps):
        for k, (label, fn) in enumerate(arms):
            a = time.perf_counter()
            last[k] = fn()
            times[k].append(time.perf_counter() - a)
            if label.startswith("locate"):
                stats[label] = rlc_locate_stats()
    ms = lambda v: round(v * 1e3, 3)            # noqa: E731
    row = {"workload": name, "decisions_equal": all(acc == last[0][0] for acc, _ in last), "rejected": last[0][0].count(b"\x00"),
           "timed_calls_each": reps, "arms": []}
    for k, (label, _) in enumerate(arms):
        arm = {"arm": label, "ms_median": ms(statistics.median(times[k])), "ms_best": ms(min(times[k])), "combined": last[k][1]}
        if label in stats:
            arm["locate_stats"] = stats[label]
        row["arms"].append(arm)
    print(json.dumps(row), flush=True)
    return row


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "rlc_locate_probe.json"))
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--proofs", type=int, default=8192)
    ap.add_argument("--aggregated", type=int, default=2048)
    args = ap.parse_args()
    from python_bulletproofs_b200 import _native as nat
    from python_bulletproofs_b200.rangeproofs.batch import (pack_generators, verify_packed, verify_aggreg_packed, verify_rlc_packed,
                                                             verify_mixed_rlc_packed, verify_rlc_locate_packed)
    card = rlc_probe.card()
    nat.init(0)
    rows, sweep = [], []

    def arms3(batch, gens, exact, packed):
        return [("exact", lambda: (exact(batch, gens, packed), None)),
                ("rlc", lambda: verify_rlc_packed(batch, *gens, packed=packed)),
                ("locate", lambda: verify_rlc_locate_packed(batch, *gens, packed=packed))]

    def leaf_arms(batch, gens, packed):
        return [("locate leaf=%d" % lf, lambda lf=lf: verify_rlc_locate_packed(batch, *gens, packed=packed, leaf=lf))
                for lf in (8, 16, 32, 64, 128, 256)]

    # (a), (b): single-value proofs, tau_x at byte 320 of the record
    sv, g1 = rlc_probe.single_value(args.proofs)
    p1 = pack_generators(*g1)
    ex1 = lambda b, gens, packed: verify_packed(b, *gens)          # noqa: E731
    rows.append(run("(a) %d distinct 64-bit proofs, all valid" % sv.nproofs,
                    [("rlc", lambda: verify_rlc_packed(sv, *g1, packed=p1)),
                     ("locate", lambda: verify_rlc_locate_packed(sv, *g1, packed=p1))], args.reps))
    for k in (1, 8, 64, sv.nproofs):
        b = forged(sv, spread(sv.nproofs, k) if k < sv.nproofs else range(sv.nproofs), 320)
        rows.append(run("(b) (a) with tau_x + 1 on %s" % ("every proof" if k == sv.nproofs else "%d proofs" % k),
                        arms3(b, g1, ex1, p1), args.reps))
        if k == 1:
            sweep.append(run("(e) sweep on (b), one forged proof", leaf_arms(b, g1, p1), args.reps))
    # (c): aggregated proofs, mu at byte 64 m + 288
    ag, g2 = rlc_probe.aggregated(args.aggregated, 32)
    p2 = pack_generators(*g2)
    ex2 = lambda b, gens, packed: verify_aggreg_packed(b, *gens, packed=packed)      # noqa: E731
    rows.append(run("(c) %d aggregated 16 x 64-bit proofs, all valid" % ag.nproofs, arms3(ag, g2, ex2, p2), args.reps))
    b = forged(ag, [ag.nproofs // 3], 64 * 16 + 288)
    rows.append(run("(c) with mu + 1 on one proof", arms3(b, g2, ex2, p2), args.reps))
    sweep.append(run("(e) sweep on (c), one forged proof", leaf_arms(b, g2, p2), args.reps))
    # (d): mixed shapes
    gens_, made = mixed_rlc_probe.make_items(8)
    for label, at in (("all valid", None), ("mu + 1 on one proof", 4096 // 3)):
        w = mixed_rlc_probe.Workload(gens_, made, 8, forged_at=at)
        rows.append(run("(d) 4096 proofs of mixed shapes, %s" % label,
                        [("exact per shape", lambda w=w: w.arm_per_shape(False)),
                         ("rlc", lambda w=w: verify_mixed_rlc_packed(w.mixed, *w.gens, packed=w.packed)),
                         ("locate", lambda w=w: verify_rlc_locate_packed(w.mixed, *w.gens, packed=w.packed))], args.reps))
    res = {"tool": "rlc_locate_probe", "card": card, "host_threads": os.cpu_count(), "rows": rows, "leaf_sweep": sweep}
    line = json.dumps(res)
    print(line)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(line + "\n")


if __name__ == "__main__":
    main()
