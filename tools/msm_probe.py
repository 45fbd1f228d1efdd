"""Stage-level timing probe of the CUDA MSM (development aid; not part of the test suite).

usage: python tools/msm_probe.py [--lgn 16,18,20] [--c 0,13,14,15,16] [--iters 5]
"""
import argparse
import ctypes
import os
import random
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from python_bulletproofs_b200 import _native as nat   # noqa: E402

GX = 0x79BE667EF9DCBBAC55A06295CE870B07029BFCDB2DCE28D959F2815B16F81798
GY = 0x483ADA7726A3C4655DA4FBFC0E1108A8FD17B448A68554199C47D08FFB10D4B8


def synth_points(n, seed):
    """n distinct points k_i * G, made on the GPU by bp_scalar_mul_batch (seeded k_i)."""
    rng = random.Random(seed)
    g = nat.pack_xy(GX, GY) * n
    ks = rng.randbytes(32 * n)
    return nat.scalar_mul_batch_bytes(g, ks, n)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--lgn", default="16,18,20")
    ap.add_argument("--c", default="0")
    ap.add_argument("--iters", type=int, default=5)
    ap.add_argument("--pre", default="", help="comma list of window widths for bp_points_precompute (0 = automatic); timed after the plain runs")
    args = ap.parse_args()
    lib = nat.load()
    nat.init(0)
    lib.bp_msm_set_pre_slots(int(os.environ.get("BP_PRE_SLOTS", "1")), int(os.environ.get("BP_PRE_SLOTS_MIN", "0")))
    macs, ms = ctypes.c_double(), ctypes.c_float()
    nat.check(lib.bp_imad_peak(4096, ctypes.byref(macs), ctypes.byref(ms)))
    print("imad peak: %.3f T limb-MAC/s (%.2f ms)" % (macs.value / 1e12, ms.value), flush=True)
    nmax = 1 << max(int(x) for x in args.lgn.split(","))
    pts = synth_points(nmax, 1)
    sc = random.Random(2).randbytes(32 * nmax)
    hp, hs = ctypes.c_uint64(), ctypes.c_uint64()
    nat.check(lib.bp_points_upload(pts, nmax, ctypes.byref(hp)))
    nat.check(lib.bp_scalars_upload(sc, nmax, ctypes.byref(hs)))
    out = ctypes.create_string_buffer(64)
    stage = (ctypes.c_float * 7)()
    names = ["digits", "scan", "scatter", "accum", "reduce", "combine", "total"]
    for lgn in [int(x) for x in args.lgn.split(",")]:
        n = 1 << lgn
        for c in [int(x) for x in args.c.split(",")]:
            nat.check(lib.bp_msm_set_window(c))
            times = (ctypes.c_float * args.iters)()
            nat.check(lib.bp_bench_msm(hp, hs, n, 2, args.iters, 1, times, out))
            best = min(times)
            lib.bp_msm_set_profiling(1)
            nat.check(lib.bp_msm_hh(hp, hs, n, out))
            nat.check(lib.bp_msm_stage_ms(stage))
            lib.bp_msm_set_profiling(0)
            print("n=2^%d c=%d: best %.3f ms median %.3f ms -> %.1f Mpts/s | " % (
                lgn, lib.bp_msm_last_window(), best, sorted(times)[len(times) // 2], n / best / 1e3)
                + " ".join("%s=%.3f" % (nm, v) for nm, v in zip(names, stage)), flush=True)
    lib.bp_msm_set_window(0)
    for pc in [int(x) for x in args.pre.split(",") if x != ""]:
        for lgn in [int(x) for x in args.lgn.split(",")]:
            n = 1 << lgn
            hq = ctypes.c_uint64()
            nat.check(lib.bp_points_upload(pts, n, ctypes.byref(hq)))
            nat.check(lib.bp_points_precompute(hq, pc))
            times = (ctypes.c_float * args.iters)()
            nat.check(lib.bp_bench_msm(hq, hs, n, 2, args.iters, 1, times, out))
            best = min(times)
            lib.bp_msm_set_profiling(1)
            nat.check(lib.bp_msm_hh(hq, hs, n, out))
            nat.check(lib.bp_msm_stage_ms(stage))
            lib.bp_msm_set_profiling(0)
            print("PRE n=2^%d c=%d: best %.3f ms median %.3f ms -> %.1f Mpts/s | " % (
                lgn, lib.bp_msm_last_window(), best, sorted(times)[len(times) // 2], n / best / 1e3)
                + " ".join("%s=%.3f" % (nm, v) for nm, v in zip(names, stage)), flush=True)
            lib.bp_handle_free(hq)


if __name__ == "__main__":
    main()
