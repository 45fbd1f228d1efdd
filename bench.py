"""bench.py -- headline benchmark of the hot path on B200.

    python bench.py --gpus N --steps K --warmup W            (N > 1: launched under torchrun)
    python bench.py --impl reference --gpus N --steps K --warmup W
    python bench.py --gpus N --steps K --warmup W --dump-outputs DIR

Metric (BASELINE.json): secp256k1 MSM throughput in Mpts/s at 2^20 points per GPU; a "step" is one
full multi-scalar multiplication over the resident 2^20-term slice (N > 1: slice MSM on every
rank + one ncclAllGather of the 128-byte partials + the N-way sum = one MSM over N * 2^20 terms,
weak scaling).  Secondary, in the same JSON line under "verify": 64-bit range-proof verifies/s
for a batch of 8192 proofs (BASELINE config 5).

No PyTorch on the data path: device work is libbpgpu (ctypes); torch.distributed (gloo) is only the
launcher-side rendezvous for N > 1 (NCCL id exchange, barriers, max-over-ranks of the timings).
The oracle (oracle/) is used here only for the cpu_baseline leg and for the in-bench parity check.
"""
import argparse
import atexit
import ctypes
import json
import os
import random
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True          # the bench writes nothing into the source tree (it may be read-only): no __pycache__
# the batch verifier's OpenMP workers must sleep, not spin, between chunks: with one process per GPU on a shared host the spinning
# pools starve each other (read by libgomp when it is loaded, so it has to be set before any import that pulls it in)
os.environ.setdefault("OMP_WAIT_POLICY", "PASSIVE")

GX = 0x79BE667EF9DCBBAC55A06295CE870B07029BFCDB2DCE28D959F2815B16F81798
GY = 0x483ADA7726A3C4655DA4FBFC0E1108A8FD17B448A68554199C47D08FFB10D4B8
METRIC = "secp256k1 MSM Mpts/s at 2^20"
LIMB_MACS_PER_FIELD_MUL = 136          # SURVEY.md 8(d): 8-limb Montgomery CIOS, the algorithmic unit
FIELD_MULS_PER_MADD = 10               # XYZZ + affine, 8M + 2S
FIELD_MULS_PER_ADD = 14                # XYZZ + XYZZ, 12M + 2S


def synth_inputs(n, seed):
    """Seeded synthetic workload: points k_i * G (made on the GPU by the scalar-mul batch kernel),
    scalars uniform 256-bit (reduced mod q on the device)."""
    from python_bulletproofs_b200 import _native as nat
    rng = random.Random(seed)

    def rb(nbytes, step=1 << 26):       # random.randbytes is limited to < 2^28 bytes per call
        return b"".join(rng.randbytes(min(step, nbytes - o)) for o in range(0, nbytes, step))
    pts = nat.scalar_mul_batch_bytes(nat.pack_xy(GX, GY) * n, rb(32 * n), n)
    return pts, rb(32 * n)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            atexit.register(self.proc.kill)      # a bench that fails before stop() must not leave nvidia-smi sampling behind
            threading.Thread(target=self._pump, daemon=True).start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [c.strip() for c in line.split(",")]))

    def stop(self, t0=None, t1=None):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        rows = [r for t, r in self.rows if (t0 is None or t >= t0 - 0.2) and (t1 is None or t <= t1 + 0.2)] or [r for _, r in self.rows]
        sm = [float(r[0]) for r in rows if r and r[0].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [nm for k, nm in enumerate(names) if any(len(r) > 3 + k and r[3 + k].startswith("Active") for r in rows)]
        return {"sm_mhz": statistics.median(sm) if sm else None,
                "sm_max_mhz": float(rows[0][1]) if rows and rows[0][1].replace(".", "").isdigit() else None,
                "power_w_max": max([float(r[2]) for r in rows if r[2].replace(".", "").isdigit()], default=None),
                "samples": len(rows), "reasons": reasons}


def dist_setup(world):
    if world <= 1:
        return None
    import torch.distributed as dist
    dist.init_process_group("gloo")          # rendezvous only; MASTER_ADDR/PORT, RANK, WORLD_SIZE from torchrun
    return dist


def max_over_ranks(dist, x):
    if dist is None:
        return x
    import torch
    t = torch.tensor([x], dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t[0])


def pinned_copy(nat, data):
    buf = nat.load().bp_host_alloc(len(data))
    if not buf:
        raise RuntimeError("bp_host_alloc failed")
    ctypes.memmove(buf, data, len(data))
    return buf


def ncu_record():
    """Counters of the dominant kernel taken from the committed ncu capture (profiles/r2_ncu_metrics.json, written by
    tools/ncu_metrics.sh from one `ncu --set full` run of this same bench command); None when absent."""
    try:
        with open(os.path.join(ROOT, "profiles", "r2_ncu_metrics.json")) as f:
            return json.load(f)
    except Exception:   # noqa: BLE001
        return None


def launches(lib):
    v = ctypes.c_uint64()
    lib.bp_launch_count(ctypes.byref(v))
    return v.value


def run_ref_runner(argv, timeout=900):
    """oracle/ref_runner.py as a subprocess (fork()-free next to a CUDA context) -> dict, or None when the reference copy is absent."""
    env = dict(os.environ)
    for k in ("OMP_NUM_THREADS", "MKL_NUM_THREADS"):     # torchrun pins these to 1; the CPU arm uses every host core
        env.pop(k, None)
    env["PYTHONDONTWRITEBYTECODE"] = "1"
    try:
        out = subprocess.run([sys.executable, "-m", "oracle.ref_runner"] + argv, cwd=ROOT, env=env, capture_output=True, text=True, timeout=timeout)
    except subprocess.TimeoutExpired:
        return None
    if out.returncode != 0:
        return None
    try:
        return json.loads(out.stdout.strip().splitlines()[-1])
    except Exception:   # noqa: BLE001
        return None


# ------------------------------------------------------------------------------------------------
def run_ours(args):
    from python_bulletproofs_b200 import _native as nat, sharding
    rank, local_rank, world = sharding.env_rank()
    if world != args.gpus and world > 1:
        args.gpus = world
    dist = dist_setup(world)
    nat.init(local_rank)
    lib = nat.load()
    if dist is not None:
        sharding.init_nccl()
    n = 1 << args.lgn

    # IMAD.WIDE issue-rate microbenchmark = the measured roofline denominator (SURVEY.md 8d)
    macs, ms_peak = ctypes.c_double(), ctypes.c_float()
    nat.check(lib.bp_imad_peak(1 << 16, ctypes.byref(macs), ctypes.byref(ms_peak)))

    pts, sc = synth_inputs(n, 0xB2000000 + args.lgn + 1000 * rank)
    hp, hs = ctypes.c_uint64(), ctypes.c_uint64()
    nat.check(lib.bp_points_upload(pts, n, ctypes.byref(hp)))
    nat.check(lib.bp_scalars_upload(sc, n, ctypes.byref(hs)))
    out = ctypes.create_string_buffer(64)

    # plain bucket method first (no per-vector precomputation): reported beside the headline as "value_no_precompute"
    tp = (ctypes.c_float * 5)()
    if dist is not None:
        dist.barrier()
    nat.check(lib.bp_bench_msm_sharded(hp, hs, 0, n, 3, 5, 1, tp, out))
    plain_ms = max_over_ranks(dist, float(sum(tp)) / 5)
    plain_hex = out.raw.hex()
    plain_c = lib.bp_msm_last_window()
    # the resident point vector gets its window multiples (bp_points_precompute): a one-off per vector, outside the timed region
    t_pre = time.perf_counter()
    if not args.no_precompute:
        nat.check(lib.bp_points_precompute(hp, 0))
    pre_s = time.perf_counter() - t_pre
    pre_c, pre_w, pre_bytes = ctypes.c_int(), ctypes.c_int(), ctypes.c_uint64()
    nat.check(lib.bp_points_pre_info(hp, ctypes.byref(pre_c), ctypes.byref(pre_w), ctypes.byref(pre_bytes)))

    # ---- timed region: K resident MSM steps, CUDA events on the library stream, L2 flushed between steps
    sampler = ClockSampler(local_rank)
    times = (ctypes.c_float * args.steps)()
    if dist is not None:
        dist.barrier()
    t0 = time.time()
    l0 = launches(lib)
    nat.check(lib.bp_bench_msm_sharded(hp, hs, 0, n, args.warmup, args.steps, 1, times, out))
    gpu_launches = (launches(lib) - l0) * args.steps // (args.steps + args.warmup)      # kernels of the K timed steps (every step launches the same set)
    t1 = time.time()
    if dist is not None:
        dist.barrier()
    total_ms = max_over_ranks(dist, float(sum(times)))
    result_hex = out.raw.hex()
    assert result_hex == plain_hex, "precomputed-path result differs from the plain bucket method"
    value = world * n * args.steps / (total_ms * 1e-3) / 1e6

    # ---- per-stage device times of one MSM and of the dominant kernel (k_accumulate) alone: CUDA events recorded on
    #      the library stream around the stages / the kernel while profiling mode is on
    stage = (ctypes.c_float * 7)()
    kms = ctypes.c_float()
    acc_ms, stage_rows = [], []
    lib.bp_msm_set_profiling(1)
    for _ in range(5):
        nat.check(lib.bp_msm_hh(hp, hs, n, out))
        nat.check(lib.bp_msm_stage_ms(stage))
        nat.check(lib.bp_msm_accumulate_kernel_ms(ctypes.byref(kms)))
        acc_ms.append(kms.value)
        stage_rows.append(list(stage))
    lib.bp_msm_set_profiling(0)
    med = [statistics.median(r[i] for r in stage_rows) for i in range(7)]
    stages = {k: round(float(v), 4) for k, v in zip(["digits", "scan", "scatter", "accumulate_stage", "reduce", "combine", "total"], med)}
    if pre_c.value > 0 and n >= (1 << 18):
        stages["note"] = ("slot sort: 'digits' is the one scattered pass (k_scatter_slots_pre: digits, slot atomics, entry stores), "
                          "'scatter' the gated fallback that returns at once")
    c = lib.bp_msm_last_window()
    pre = pre_c.value > 0
    # windows: precomputed path = ceil(257 / c) windows of a 256-bit scalar; plain path = GLV halves < 2^128, ceil(128 / c) windows each
    W = pre_w.value if pre else (128 + c - 1) // c
    ent = ctypes.c_uint64()
    nat.check(lib.bp_msm_last_entries(ctypes.byref(ent)))
    acc = statistics.median(acc_ms)
    # Work of one k_accumulate launch = one mixed add (XYZZ + affine, 8M + 2S) per non-zero signed digit; ent.value is
    # that count, read back from the device (~ 2 halves * n * 128 / c).
    #  * issued: this implementation spends 72 IMAD.WIDE per field multiplication (64 + 8, pseudo-Mersenne fold) and 45
    #    per squaring, i.e. 666 32x32->64 multiply-accumulates per mixed add -- the count the IMAD.WIDE pipe peak bounds;
    #  * algorithmic (SURVEY.md 8d units): 10 field multiplications x 136 limb-MAC (8-limb Montgomery CIOS) = 1360.
    issued_macs = ent.value * (8 * 72 + 2 * 45)
    alg_macs = ent.value * FIELD_MULS_PER_MADD * LIMB_MACS_PER_FIELD_MUL
    achieved = issued_macs / (acc * 1e-3) / 1e12
    peak = macs.value / 1e12
    nominal = 148 * 64 * 1965.0 * 1e6 / 1e12
    ncu = ncu_record() or {}
    # the accumulation kernel of this launch: over the slot layout (precomputed path, >= 2^18 terms: msm.cuh slot sort, 4-byte
    # entries) or over the compact sorted list (8-byte entries); same chunks, same mixed additions
    kname = "k_accumulate_slots" if pre and n >= (1 << 18) else "k_accumulate"
    ent_bytes = 4 if kname == "k_accumulate_slots" else 8
    kacc = ncu.get(kname) or ncu.get("k_accumulate", {})
    roofline = {"bound": "imad", "kernel": kname, "achieved": round(achieved, 3), "peak": round(peak, 3),
                "unit": "T IMAD.WIDE (32x32+64 limb-MAC)/s", "frac": round(achieved / peak, 4),
                "traffic": kacc.get("dram_bytes"),
                "traffic_note": "dram__bytes_read.sum + dram__bytes_write.sum of one %s launch from profiles/r2_ncu_metrics.json "
                                "(ncu --set full, cold L2: its default cache flush between replay passes); algorithmic bytes: one gathered 64 B "
                                "point + %d B entry per mixed add = %.2f GB" % (kname, ent_bytes, ent.value * (64 + ent_bytes) / 1e9),
                "peak_source": "measured in this process: bp_imad_peak, data-dependent IMAD.WIDE.U32 stream (SASS checked); "
                               "IMAD.WIDE issues at half the 32-bit IMAD rate on B200, with or without the carry predicate",
                "nominal_imad32_peak": round(nominal, 2),
                "ncu_pipe_fmaheavy_active_pct": kacc.get("pipe_fmaheavy_active_pct"),
                "ncu_source": ncu.get("source"),
                "window_bits": c, "windows": W, "glv": not pre, "mixed_adds_per_launch": ent.value, "kernel_ms": round(acc, 4),
                "share_of_step": round(acc / med[6], 3),
                "whole_step_frac": round(issued_macs / (total_ms / args.steps * 1e-3) / 1e12 / peak, 4),
                "issued_limb_macs_per_launch": issued_macs,
                "algorithmic_limb_macs_per_launch_survey_units": alg_macs,
                "algorithmic_rate_survey_units_T_per_s": round(alg_macs / (acc * 1e-3) / 1e12, 3),
                "whole_msm_algorithmic_limb_macs_per_pt": round((alg_macs + (1 if pre else (W + (1 if 128 % c == 0 else 0))) * (1 << (c - 1)) * 2 * FIELD_MULS_PER_ADD * LIMB_MACS_PER_FIELD_MUL) / n, 1),
                "hbm": {"bound": "hbm", "achieved": round(ent.value * (64 + ent_bytes) / (acc * 1e-3) / 1e9, 1), "unit": "GB/s",
                        "peak": measured_hbm(), "note": "gathered 64 B point + %d B entry per mixed add; not the binding resource" % ent_bytes}}

    # ---- end to end through the C ABI with pinned HOST buffers (H2D + MSM + D2H inside the timed region)
    pp, ps = pinned_copy(nat, pts), pinned_copy(nat, sc)
    e2e_t = []
    for it in range(2 + args.steps):
        if dist is not None:
            dist.barrier()
        a = time.perf_counter()
        nat.check(lib.bp_msm_sharded_host(pp, ps, n, out))
        e2e_t.append(max_over_ranks(dist, time.perf_counter() - a))
    e2e_t = e2e_t[2:]
    assert out.raw.hex() == result_hex, "end-to-end result differs from resident result"
    e2e = {"value": round(world * n / (sum(e2e_t) / len(e2e_t)) / 1e6, 3), "unit": "Mpts/s", "h2d_bytes_per_step": 96 * n,
           "d2h_bytes_per_step": 64, "h2d_gbs_per_rank": round(96 * n / (sum(e2e_t) / len(e2e_t)) / 1e9, 2),
           "api": "bp_msm_sharded_host (C ABI, pinned host buffers)" if world > 1 else "bp_msm / bp_msm_sharded_host (C ABI, pinned host buffers)"}
    lib.bp_host_free(pp)
    lib.bp_host_free(ps)
    clocks = sampler.stop(t0, time.time())       # sampled from the start of the timed region through the e2e loop

    # multi-GPU parity: every rank's own slice result (no NCCL) is gathered through the launcher's process group and
    # summed with the CPU oracle's group law on rank 0; it must equal the point every rank got from the sharded call
    sharded_ok = None
    if dist is not None:
        nat.check(lib.bp_msm_hh(hp, hs, n, out))
        mine = out.raw
        parts = [None] * world
        dist.all_gather_object(parts, mine)
        if rank == 0:
            from oracle import ecc
            tot = None
            for pb in parts:
                tot = ecc.point_add(tot, ecc.unpack_point(pb))
            sharded_ok = ecc.pack_point(tot).hex() == result_hex

    # ---- strong scaling (SURVEY.md 8e: ONE N-point MSM cut into contiguous slices [r*T/R, (r+1)*T/R)): totals 2^a, 2^b
    strong = []
    for lgt in args.strong:
        T = 1 << lgt
        lo, hi = sharding.slice_bounds(T, rank, world)
        m = hi - lo
        if m <= n:
            sp, ss, free = hp, hs, False
        else:
            spts, ssc = synth_inputs(m, 0xB2000000 + lgt + 1000 * rank + 77)
            sp, ss, free = ctypes.c_uint64(), ctypes.c_uint64(), True
            nat.check(lib.bp_points_upload(spts, m, ctypes.byref(sp)))
            nat.check(lib.bp_scalars_upload(ssc, m, ctypes.byref(ss)))
            if not args.no_precompute:
                nat.check(lib.bp_points_precompute(sp, 0))
            del spts, ssc
        st = (ctypes.c_float * 5)()
        if dist is not None:
            dist.barrier()
        nat.check(lib.bp_bench_msm_sharded(sp, ss, 0, m, 3, 5, 1, st, out))
        ms = max_over_ranks(dist, float(sum(st)) / 5)
        strong.append({"terms_total": T, "terms_per_gpu": m, "ms_per_msm": round(ms, 4), "value": round(T / (ms * 1e-3) / 1e6, 2), "unit": "Mpts/s"})
        if free:
            lib.bp_handle_free(sp)
            lib.bp_handle_free(ss)

    line = {"metric": METRIC, "value": round(value, 3), "unit": "Mpts/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": round(total_ms / args.steps, 4), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u32x8 (256-bit modular integer)", "data": "synthetic",
            "config": {"workload": "C3: standalone MSM, 2^%d secp256k1 points + 256-bit scalars resident per GPU" % args.lgn,
                       "terms_per_gpu": n, "terms_total": world * n, "window_bits": c,
                       "resident_points": ("with precomputed window multiples (bp_points_precompute: %d windows, %.2f GB per GPU, built once in %.2f s outside the timed region)"
                                           % (pre_w.value, pre_bytes.value / 1e9, pre_s)) if pre else "plain affine vector",
                       "l2": "flushed between steps (256 MiB memset outside the timed events)",
                       "parallelism": "slice%d" % world, "seed": "0xB2000000+lgn(+1000*rank), points k_i*G"},
            "gpu_launches": gpu_launches,
            "value_no_precompute": round(world * n / (plain_ms * 1e-3) / 1e6, 3), "ms_per_step_no_precompute": round(plain_ms, 4), "window_bits_no_precompute": plain_c,
            "clocks": clocks, "e2e": e2e, "roofline": roofline, "stages_ms": stages, "result": result_hex,
            "strong_scaling": {"scaling": "strong", "note": "one MSM of terms_total terms cut into contiguous slices, one per GPU; "
                               "slice MSM + ncclAllGather of the 128-byte partials + sum, max over ranks", "points": strong}}

    if rank == 0 and world == 1 and not os.environ.get("BP_BENCH_NO_SWEEP"):      # (left out under ncu: tools/ncu_metrics.sh)
        line["sweep"] = msm_sweep(lib, nat, pts, hs, args.lgn, not args.no_precompute)
        line["cpu_baseline"], bit_exact = cpu_baseline(pts, sc, n, result_hex)
        line["bit_exact_vs_oracle"] = bit_exact
    if sharded_ok is not None:
        line["sharded_result_equals_sum_of_slices"] = sharded_ok
    accept = None
    if not args.no_verify:
        try:
            line["verify"], accept = bench_verify(args, nat, dist, rank, world, peak)
        except Exception as e:   # noqa: BLE001  -- the headline metric must still print
            import traceback
            line["verify"] = {"error": repr(e), "trace": traceback.format_exc()[-600:]}
    lib.bp_handle_free(hp)
    lib.bp_handle_free(hs)
    if rank == 0:
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, result_hex, accept)
        print(json.dumps(line), flush=True)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


def dump_outputs(dirname, result_hex, accept):
    """What the timed paths handed their caller in their last step, as arrays on which two builds can be compared:
      msm_result.npy     (2, 8) float64: x and y of the affine MSM result as 32-bit little-endian limbs (exact in float64);
                         the identity is all zero
      verify_accept.npy  (proofs,) float32: the decisions of the last timed batch verification, 1 = accepted, 0 = rejected
                         (absent with --no-verify or when the verify leg failed)"""
    import numpy as np
    os.makedirs(dirname, exist_ok=True)
    limbs = np.frombuffer(bytes.fromhex(result_hex), dtype="<u4").astype(np.float64).reshape(2, 8)
    np.save(os.path.join(dirname, "msm_result.npy"), limbs)
    if accept is not None:
        np.save(os.path.join(dirname, "verify_accept.npy"), np.frombuffer(accept, dtype=np.uint8).astype(np.float32))


def measured_hbm():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return json.load(f)["hbm_gbs"]
    except Exception:   # noqa: BLE001
        return 6650.0


def msm_sweep(lib, nat, pts, hs, lgmax, precompute):
    """BASELINE config 3: the resident MSM at 2^10 ... 2^lgmax terms (prefixes of the same point / scalar vectors), L2 flushed
    between iterations, median of 5 after 2 warm-up calls; per size the plain bucket method and, with `precompute`, the same
    vector carrying its window multiples."""
    out = ctypes.create_string_buffer(64)
    rows = {}
    for lg in range(10, lgmax + 1):
        m = 1 << lg
        h = ctypes.c_uint64()
        nat.check(lib.bp_points_upload(pts, m, ctypes.byref(h)))
        ts = (ctypes.c_float * 5)()
        nat.check(lib.bp_bench_msm(h, hs, m, 2, 5, 1, ts, out))
        ms = statistics.median(ts)
        row = {"ms_plain": round(ms, 4), "mpts_per_s_plain": round(m / ms / 1e3, 2), "window_bits_plain": lib.bp_msm_last_window()}
        if precompute:
            plain_hex = out.raw.hex()
            nat.check(lib.bp_points_precompute(h, 0))
            nat.check(lib.bp_bench_msm(h, hs, m, 2, 5, 1, ts, out))
            ms = statistics.median(ts)
            row.update({"ms": round(ms, 4), "mpts_per_s": round(m / ms / 1e3, 2), "window_bits": lib.bp_msm_last_window(), "same_result": out.raw.hex() == plain_hex})
        else:
            row.update({"ms": row["ms_plain"], "mpts_per_s": row["mpts_per_s_plain"], "window_bits": row["window_bits_plain"]})
        rows[str(lg)] = row
        lib.bp_handle_free(h)
    return rows


def cpu_baseline(pts, sc, n, gpu_hex):
    """CPU baseline of the MSM leg, timed on this box's host cores:
      * kind "reference": the reference's OWN Pippenger.multiexp (unmodified src/ from baseline/_ref over the fastecdsa stand-in),
        one 2^10-term slice of the workload per core -- its best operating point (BASELINE.md 2.1: throughput falls from 2^10
        on) -- plus single calls at 2^12 for the sweep; 2^13 and beyond take > 39 s per call (2^20: 2.3 G table entries,
        cannot run);
      * beside it the oracle port (C, bucket method, all host threads) on the SAME 2^lgn inputs, which also checks the GPU
        result bit for bit, and the reference's subset-table algorithm restated in C at 2^12."""
    from oracle import ecc
    cores = os.cpu_count() or 1
    t = time.perf_counter()
    res = ecc.msm_bytes(pts, sc, n, "bucket", cores)
    dt = time.perf_counter() - t
    bit_exact = ecc.pack_point(res).hex() == gpu_hex
    ns = 1 << 12
    t = time.perf_counter()
    ecc.msm_bytes(pts[:64 * ns], sc[:32 * ns], ns, "subset", 1)
    dts = time.perf_counter() - t
    port = {"value": round(n / dt / 1e6, 4), "unit": "Mpts/s", "cores": cores, "kind": "port",
            "sample": "full workload (2^%d terms) once, oracle/ecc_oracle.c bucket MSM on %d OpenMP threads, %.2f s; "
                      "reference's subset-table algorithm restated in C, 1 thread, 2^12 terms: %.4f Mpts/s"
                      % (n.bit_length() - 1, cores, dt, ns / dts / 1e6)}
    r10 = run_ref_runner(["msm", "--lgn", "10", "--procs", str(cores), "--reps", "3"])
    if not r10:
        return port, bit_exact
    r12 = run_ref_runner(["msm", "--lgn", "12", "--procs", str(cores), "--reps", "1"])
    walls = r10["wall_s"][1:] or r10["wall_s"]
    val = cores * 1024 * len(walls) / sum(walls) / 1e6
    base = {"value": round(val, 6), "unit": "Mpts/s", "cores": cores, "kind": "reference",
            "sample": "reference Pippenger.multiexp (src/pippenger/pippenger.py:22-61, unmodified, plain-Python fastecdsa stand-in), one 2^10-term "
                      "slice of the C3 workload per core on %d processes, %d timed rounds of %.2f s (first round dropped); one core: %.0f pts/s"
                      % (cores, len(walls), sum(walls) / len(walls), r10["pts_per_s_one_core"]),
            "sweep_one_core_pts_per_s": {"10": round(r10["pts_per_s_one_core"], 1)},
            "beyond": "2^13: 39 s per call, 2^14: 100 s (BASELINE.md 2.1, survey container); 2^16 and up impractical, 2^20 impossible (2.3 G table entries)",
            "port": port}
    if r12:
        base["sweep_one_core_pts_per_s"]["12"] = round(4096 / r12["mean_single_call_s"], 1)
    return base, bit_exact


# ---- second half of the metric: batch verification of 64-bit range proofs (config 5) ----------------------
def verify_work_model(n=64):
    """IMAD.WIDE (32x32+64 multiply-accumulates) this implementation issues per verified n-bit proof on the table path:
    72 per field multiplication, 45 per squaring (csrc/fp.cuh); Z_q products 120 (csrc/fqdev.cuh)."""
    L = n.bit_length() - 1
    M, S = 72, 45
    madd, add, jdbl, mdbl = 8 * M + 2 * S, 12 * M + 2 * S, 2 * M + 5 * S, 4 * M + 3 * S
    nfix = (2 * n + 1) + (n + 4) + 1 + 2                       # generator terms of E4, E2, E3, E1
    nv = 5 + 2 * L                                             # proof-specific points with a full scalar
    fixed = nfix * 16 * madd                                   # 16-bit windows: one lookup + mixed add per (term, window)
    fold = (8 * 7 + 3 * 4 * 7 + 7 + 3 * 3 + 4) * add           # lane sums -> one point per equation, + the variable part
    table = nv * (mdbl + 6 * madd) + (nv + 2) * (2 * S + M)    # 2P..8P per point, curve check of all proof points
    main = 2 * nv * 32 * (15 / 16) * add + nv * 32 * (15 / 16) * M      # lane = window: one addition per (sub-term, window); beta*X on the phi half
    comb1 = 3 * 4 * 7 * (4 * jdbl + 3 * M + S + add)
    comb2 = 3 * 3 * (32 * jdbl + 3 * M + S + add) + 3 * madd
    zq = (2 * n * 14 + 334) * 120                              # term scalars (k_rp_expand) + one inversion per proof
    parts = {"fixed_base_lookups": fixed, "fold": fold, "variable_tables": table, "variable_window_sums": main,
             "horner_tails": comb1 + comb2, "scalar_field": zq}
    return {k: int(v) for k, v in parts.items()}, int(sum(parts.values())), nfix, nv


def bench_verify(args, nat, dist, rank, world, imad_peak):
    import contextlib
    import io
    from python_bulletproofs_b200 import Point, secp256k1, sharding
    from python_bulletproofs_b200.rangeproofs import NIRangeProver
    from python_bulletproofs_b200.rangeproofs.batch import PackedBatch, verify_local_gather, verify_stats
    from python_bulletproofs_b200.utils import ModP, commitment, mod_hash, elliptic_hash
    q, nbits = secp256k1.q, 64
    seeds = [b"seed%d" % i for i in range(5)]
    gs = [elliptic_hash(str(i).encode() + seeds[0], secp256k1) for i in range(nbits)]
    hs = [elliptic_hash(str(i).encode() + seeds[1], secp256k1) for i in range(nbits)]
    g, h, u = (elliptic_hash(s, secp256k1) for s in seeds[2:5])
    total = args.verify_proofs
    slices = sharding.all_slices(total, world)
    lo, hi = slices[rank]
    counts = [b - a for a, b in slices]
    rng = random.Random(5)
    vals = [rng.getrandbits(64) for _ in range(total)]         # SURVEY.md 8(d) C5 stream: v_i in index order
    # ---- every proof of the batch is distinct; rank r proves (and verifies) its own block [lo, hi)
    Vs, proofs = [], []
    t = time.perf_counter()
    for i in range(lo, hi):
        gamma = mod_hash(b"gamma%d" % i, q)
        Vs.append(commitment(g, h, ModP(vals[i], q), gamma))
        pr = NIRangeProver(ModP(vals[i], q), nbits, g, h, gs, hs, gamma, u, secp256k1, b"p%d" % i).prove()
        if i % 16 == 15:       # every 16th proof corrupted: flip one decimal digit of t_hat
            s = str(pr.t_hat.x)
            pr.t_hat = ModP(int(s[:-1] + ("1" if s[-1] != "1" else "2")), q)
        proofs.append(pr)
    prove_s = (time.perf_counter() - t) / max(hi - lo, 1)
    local = PackedBatch.from_proofs(Vs, proofs, nbits)
    h2d = len(local.records) + len(local.blob)
    times, spans, hosts = [], [], []
    acc = b""
    lib = nat.load()
    l0 = 0
    for it in range(4 + args.verify_reps):      # the first calls build the generator tables (byte windows, then 16-bit windows)
        if it == 4:
            l0 = launches(lib)
        if dist is not None:
            dist.barrier()
        a = time.perf_counter()
        acc = verify_local_gather(local, g, h, gs, hs, u, counts)
        times.append(max_over_ranks(dist, time.perf_counter() - a))
        st = verify_stats()
        spans.append(max_over_ranks(dist, st["device_span_ms"]))
        hosts.append(st["host_check_ms"])
    nl = (launches(lib) - l0) // max(args.verify_reps, 1)
    times, spans, hosts = times[4:], spans[4:], hosts[4:]
    med, best = statistics.median(times), min(times)
    want = bytes([0 if i % 16 == 15 else 1 for i in range(total)])
    res = {"metric": "64-bit range-proof verifies/s", "value": round(total / med, 1), "unit": "verifies/s", "n_gpus": world,
           "scaling": "strong", "proofs": total, "distinct_proofs": total, "proofs_per_gpu": counts[0],
           "ms_per_batch": round(med * 1e3, 3), "ms_per_batch_best": round(best * 1e3, 3), "value_best": round(total / best, 1),
           "batches_timed": len(times), "decisions_ok": acc == want, "rejected": acc.count(b"\x00"),
           "gpu_launches_per_batch": nl,
           "e2e": {"value": round(total / med, 1), "unit": "verifies/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": total,
                   "api": "bp_rp_verify_batch_gather (C ABI): packed proofs + transcripts in HOST memory -> host transcript checks, H2D, "
                          "device equations, ncclAllGather of the accept bytes, D2H"},
           "device_span_ms": round(statistics.median(spans), 3), "host_check_ms": round(statistics.median(hosts), 3),
           "stats": st,
           "note": "timed region = the whole call from host buffers (max over ranks, median of %d batches after 4 warm-up batches that "
                   "build the generator tables); proofs made by the GPU prover (%.2f ms/proof), all distinct, every 16th corrupted"
                   % (len(times), prove_s * 1e3)}
    # ---- roofline of the verify leg: issued IMAD.WIDE of the table path / device span / measured IMAD.WIDE peak
    parts, per_proof, nfix, nv = verify_work_model(nbits)
    span = statistics.median(spans)
    ach = per_proof * counts[0] / (span * 1e-3) / 1e12         # per GPU (every rank runs the same work over its block)
    res["roofline"] = {"bound": "imad", "kernel": "batch verifier, all kernels of one batch (k_rp_lookup16 dominant)",
                       "achieved": round(ach, 3), "peak": round(imad_peak, 3), "unit": "T IMAD.WIDE (32x32+64 limb-MAC)/s per GPU",
                       "frac": round(ach / imad_peak, 4), "imad_wide_per_proof": per_proof, "imad_wide_per_proof_parts": parts,
                       "generator_terms_per_proof": nfix, "proof_point_terms_per_proof": nv + 4,
                       "gpu_ms": round(span, 3), "gpu_ms_note": "CUDA events on the library stream: first kernel of the first chunk .. last accept kernel "
                       "(includes any wait for host transcript checks between chunks), max over ranks",
                       "kernel_list": "profiles/r2_verify_kernels_v3.csv (ncu --metrics gpu__time_duration.sum of one batch, tools/ncu_verify.sh)", "traffic": None}
    if rank == 0:
        # ---- decisions against the ORACLE verifier: the first 128 proofs of this rank's block (incl. every corrupted one in
        #      the sample), and the prover's output against the oracle prover on 16 proofs (byte-identical transcripts)
        from oracle import protocol_oracle as po
        T_ = lambda p_: None if p_.curve is None else (p_.x, p_.y)      # noqa: E731
        ogs, ohs, og, oh, ou = [T_(x) for x in gs], [T_(x) for x in hs], T_(g), T_(h), T_(u)
        sample = min(128, hi - lo)
        dec_ok, corrupted = True, 0
        for k in range(sample):
            pr = proofs[k]
            ip, p2 = pr.innerProof, pr.innerProof.proof2
            op = {"taux": pr.taux.x % q, "mu": pr.mu.x % q, "t_hat": pr.t_hat.x % q, "T1": T_(pr.T1), "T2": T_(pr.T2), "A": T_(pr.A), "S": T_(pr.S),
                  "transcript": pr.transcript,
                  "ip": {"u_new": T_(ip.u_new), "P_new": T_(ip.P_new), "transcript": ip.transcript,
                         "p2": {"a": p2.a.x % q, "b": p2.b.x % q, "xs": [x.x % q for x in p2.xs], "Ls": [T_(x) for x in p2.Ls],
                                "Rs": [T_(x) for x in p2.Rs], "transcript": p2.transcript, "start": p2.start_transcript}}}
            ok = po.range_verify([T_(Vs[k])], og, oh, ogs, ohs, ou, op)
            corrupted += 0 if ok else 1
            dec_ok = dec_ok and (acc[lo + k] == (1 if ok else 0))
        res["decisions_vs_oracle"] = {"proofs": sample, "rejected_by_oracle": corrupted, "all_equal": dec_ok}
        same = True
        for k in range(min(args.verify_prover_check, hi - lo)):
            i = lo + k
            if i % 16 == 15:
                continue
            gamma = mod_hash(b"gamma%d" % i, q)
            opr = po.range_prove([vals[i]], nbits, og, oh, ogs, ohs, [gamma.x], ou, b"p%d" % i)
            same = same and proofs[k].transcript == opr["transcript"] and proofs[k].innerProof.proof2.transcript == opr["ip"]["p2"]["transcript"]
        res["prover_vs_oracle"] = {"proofs": min(args.verify_prover_check, hi - lo), "byte_identical_transcripts": same}
        if world == 1:
            res["cpu_baseline"] = verify_cpu_baseline(Vs, proofs, og, oh, ogs, ohs, ou, T_, q)
            try:
                res["aggregated"] = bench_verify_aggregated(nat, q)
            except Exception as e:   # noqa: BLE001
                res["aggregated"] = {"error": repr(e)}
    return res, acc


def bench_verify_aggregated(nat, q, m=16, nbits=64, distinct=32, total=2048):
    """Widening row (BASELINE config 4 as a batch): `total` aggregated range proofs (m values x nbits bits, n*m = 1024 generators per
    side) through bp_rp_verify_aggreg_batch in one call -- `distinct` different proofs tiled (proving 1024 of them would take the
    bench 3 s more for nothing: the verifier does the same work per record), every 8th distinct proof corrupted; decisions of the
    distinct proofs checked against the oracle verifier; the class API (AggregRangeVerifier.verify, proof by proof) timed beside it."""
    import contextlib
    import io
    from oracle import protocol_oracle as po
    from python_bulletproofs_b200 import secp256k1
    from python_bulletproofs_b200.rangeproofs import AggregNIRangeProver, AggregRangeVerifier
    from python_bulletproofs_b200.rangeproofs.batch import PackedAggregBatch, pack_generators, verify_aggreg_packed
    from python_bulletproofs_b200.utils import ModP, commitment, mod_hash, elliptic_hash
    nm = nbits * m
    gs = [elliptic_hash(str(i).encode() + b"agg0", secp256k1) for i in range(nm)]
    hs = [elliptic_hash(str(i).encode() + b"agg1", secp256k1) for i in range(nm)]
    g, h, u = (elliptic_hash(s_, secp256k1) for s_ in (b"agg2", b"agg3", b"agg4"))
    rng = random.Random(16)
    Vl, pl = [], []
    t = time.perf_counter()
    for i in range(distinct):
        vs = [ModP(rng.getrandbits(nbits), q) for _ in range(m)]
        gammas = [mod_hash(b"ag%d_%d" % (i, j), q) for j in range(m)]
        Vl.append([commitment(g, h, vs[j], gammas[j]) for j in range(m)])
        pr = AggregNIRangeProver(vs, nbits, g, h, gs, hs, gammas, u, secp256k1, b"y%d" % i).prove()
        if i % 8 == 7:
            pr.mu = ModP((pr.mu.x + 1) % q, q)
        pl.append(pr)
    prove_ms = (time.perf_counter() - t) / distinct * 1e3
    batch = PackedAggregBatch.from_proofs(Vl * (total // distinct), pl * (total // distinct), nbits)
    packed = pack_generators(g, h, gs, hs, u)
    ts, acc = [], b""
    for it in range(3 + 5):                    # the first calls meet the generator set for the first time and build its table
        a = time.perf_counter()
        acc = verify_aggreg_packed(batch, g, h, gs, hs, u, packed)
        ts.append(time.perf_counter() - a)
    med = statistics.median(ts[3:])
    want = bytes([0 if i % 8 == 7 else 1 for i in range(distinct)]) * (total // distinct)
    T_ = lambda p_: None if p_.curve is None else (p_.x, p_.y)      # noqa: E731
    ogs, ohs, og, oh, ou = [T_(x) for x in gs], [T_(x) for x in hs], T_(g), T_(h), T_(u)
    dec_ok = True
    for k in (0, 7):                           # one intact, one corrupted proof against the oracle's AggregRangeVerifier restatement
        pr = pl[k]
        ip, p2 = pr.innerProof, pr.innerProof.proof2
        op = {"taux": pr.taux.x % q, "mu": pr.mu.x % q, "t_hat": pr.t_hat.x % q, "T1": T_(pr.T1), "T2": T_(pr.T2), "A": T_(pr.A), "S": T_(pr.S),
              "transcript": pr.transcript,
              "ip": {"u_new": T_(ip.u_new), "P_new": T_(ip.P_new), "transcript": ip.transcript,
                     "p2": {"a": p2.a.x % q, "b": p2.b.x % q, "xs": [x.x % q for x in p2.xs], "Ls": [T_(x) for x in p2.Ls],
                            "Rs": [T_(x) for x in p2.Rs], "transcript": p2.transcript, "start": p2.start_transcript}}}
        dec_ok = dec_ok and (po.range_verify([T_(V) for V in Vl[k]], og, oh, ogs, ohs, ou, op) == (acc[k] == 1))
    with contextlib.redirect_stdout(io.StringIO()):
        a = time.perf_counter()
        for k in range(4):
            AggregRangeVerifier(Vl[k], g, h, gs, hs, u, pl[k]).verify()
        one_ms = (time.perf_counter() - a) / 4 * 1e3
    # generator terms: 3 * nm + 6 table terms x 32 byte-window lookups, one mixed addition (666 IMAD.WIDE) each
    return {"workload": "%d aggregated range proofs of m = %d values x %d bits (n*m = %d generators per side), %d distinct, one call of "
                        "bp_rp_verify_aggreg_batch from host buffers" % (total, m, nbits, nm, distinct),
            "ms_per_batch": round(med * 1e3, 3), "proofs_per_s": round(total / med, 1), "values_per_s": round(total * m / med, 1),
            "decisions_ok": acc == want, "decisions_vs_oracle_ok": dec_ok, "rejected": acc.count(b"\x00"),
            "class_api_ms_per_proof": round(one_ms, 3), "speedup_vs_class_api": round(one_ms / (med * 1e3 / total), 1),
            "prove_ms_per_proof": round(prove_ms, 3),
            "table_lookups_per_proof": (3 * nm + 6) * 32,
            "imad_wide_T_per_s": round((3 * nm + 6) * 32 * 666 * total / med / 1e12, 3),
            "reference": "AggregRangeVerifier.verify, src/rangeproofs/rangeproof_aggreg_verifier.py:42-108: 20.0 s per proof on one core (BASELINE.md 2.2)"}


def verify_cpu_baseline(Vs, proofs, og, oh, ogs, ohs, ou, T_, q):
    """The reference's own RangeVerifier.verify (unmodified src/ from baseline/_ref, fastecdsa stand-in) fanned out over all host
    cores by proof on a 64-proof sample of the same C5 stream (proved by the reference's own prover in the workers, untimed);
    falls back to the oracle port (protocol_oracle.range_verify, one core) when the reference copy is absent."""
    cores = os.cpu_count() or 1
    r = run_ref_runner(["verify", "--count", "64", "--procs", str(cores)], timeout=1200)
    if r:
        want = "".join("0" if i % 16 == 15 else "1" for i in range(64))
        return {"value": round(r["verifies_per_s"], 3), "unit": "verifies/s", "cores": r["procs"], "kind": "reference",
                "sample": "64 proofs of the C5 stream, reference RangeVerifier.verify (src/rangeproofs/rangeproof_verifier.py:55-86) on %d processes, "
                          "%.1f s; one core: %.3f verifies/s; reference decisions equal the expected pattern: %s"
                          % (r["procs"], r["wall_s"], r["verifies_per_s_one_core"], r["decisions"] == want)}
    from oracle import protocol_oracle as po
    t = time.perf_counter()
    cnt = min(64, len(proofs))
    for k in range(cnt):
        pr = proofs[k]
        ip, p2 = pr.innerProof, pr.innerProof.proof2
        op = {"taux": pr.taux.x % q, "mu": pr.mu.x % q, "t_hat": pr.t_hat.x % q, "T1": T_(pr.T1), "T2": T_(pr.T2), "A": T_(pr.A), "S": T_(pr.S),
              "transcript": pr.transcript,
              "ip": {"u_new": T_(ip.u_new), "P_new": T_(ip.P_new), "transcript": ip.transcript,
                     "p2": {"a": p2.a.x % q, "b": p2.b.x % q, "xs": [x.x % q for x in p2.xs], "Ls": [T_(x) for x in p2.Ls],
                            "Rs": [T_(x) for x in p2.Rs], "transcript": p2.transcript, "start": p2.start_transcript}}}
        po.range_verify([T_(Vs[k])], og, oh, ogs, ohs, ou, op)
    dt = time.perf_counter() - t
    return {"value": round(cnt / dt, 2), "unit": "verifies/s", "cores": 1, "kind": "port",
            "sample": "%d proofs, oracle/protocol_oracle.range_verify over the C oracle, one core" % cnt}


# ------------------------------------------------------------------------------------------------
def run_reference(args):
    """Reference arm: the reference's own CPU implementation of the path on this box's host cores -- the UNMODIFIED Python of
    baseline/_ref (a copy of /root/reference/src made by build(); its absent third-party fastecdsa extension replaced by the
    plain-Python stand-in), every host core busy: one 2^10-term slice of the C3 workload per core and step (the reference is
    single threaded, and 2^10 is where its throughput peaks; at 2^20 its table would need 2.3 G entries).  Same metric, unit
    and JSON keys as the GPU arm; plus a "verify" object for the second half of the metric.  When the reference copy is
    absent the oracle port (C, OpenMP, all cores) is timed instead and says so ("kind": "port")."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    steps, warm = args.steps, args.warmup
    r = run_ref_runner(["msm", "--lgn", "10", "--procs", str(cores), "--reps", str(steps + max(warm, 1))], timeout=3000)
    line = None
    if r:
        walls = r["wall_s"][max(warm, 1):]
        val = round(cores * 1024 * len(walls) / sum(walls) / 1e6, 6)
        sample = ("reference Pippenger.multiexp (unmodified src/pippenger/pippenger.py over the plain-Python fastecdsa stand-in), one 2^10-term slice of the "
                  "2^%d workload per core and step, %d processes" % (args.lgn, cores))
        line = {"impl": "reference", "metric": METRIC, "value": val, "unit": "Mpts/s", "n_gpus": args.gpus, "steps": len(walls),
                "warmup": max(warm, 1), "ms_per_step": round(1e3 * sum(walls) / len(walls), 3), "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "Python int (256-bit modular integer, CPU)", "data": "synthetic",
                "config": {"workload": "C3: standalone MSM, 2^%d secp256k1 points (CPU arm: bounded sample)" % args.lgn, "sample_terms": cores * 1024},
                "cpu_baseline": {"value": val, "unit": "Mpts/s", "cores": cores, "kind": "reference", "sample": sample,
                                 "one_core_pts_per_s": round(r["pts_per_s_one_core"], 1)},
                "e2e": {"value": val, "unit": "Mpts/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        v = run_ref_runner(["verify", "--count", "64", "--procs", str(cores)], timeout=1500)
        if v:
            line["verify"] = {"impl": "reference", "metric": "64-bit range-proof verifies/s", "value": round(v["verifies_per_s"], 3), "unit": "verifies/s",
                              "cores": v["procs"], "kind": "reference", "one_core": round(v["verifies_per_s_one_core"], 3),
                              "sample": "64 proofs of the C5 stream (reference prover, untimed), reference RangeVerifier.verify fanned out by proof over %d "
                                        "processes, %.1f s" % (v["procs"], v["wall_s"])}
    if line is None:
        from oracle import ecc
        lgs = min(args.lgn, 18)
        ns = 1 << lgs
        rng = random.Random(0xB2000000 + args.lgn)
        base = [ecc.py_mul(ecc.G, rng.getrandbits(256)) for _ in range(16)]
        pts_l = ecc.scalar_mul_batch([base[i % 16] for i in range(ns)], [rng.getrandbits(256) for _ in range(ns)])
        pts, sc = ecc.pack_points(pts_l), rng.randbytes(32 * ns)
        ts = []
        for it in range(warm + steps):
            t = time.perf_counter()
            ecc.msm_bytes(pts, sc, ns, "bucket", cores)        # explicit thread count: torchrun exports OMP_NUM_THREADS=1
            ts.append(time.perf_counter() - t)
        ts = ts[warm:]
        val = round(ns * len(ts) / sum(ts) / 1e6, 4)
        sample = "2^%d-term sample of the 2^%d workload per step, oracle/ecc_oracle.c bucket MSM, %d OpenMP threads (reference copy baseline/_ref absent)" % (lgs, args.lgn, cores)
        line = {"impl": "reference", "metric": METRIC, "value": val, "unit": "Mpts/s", "n_gpus": args.gpus, "steps": steps,
                "warmup": warm, "ms_per_step": round(1e3 * sum(ts) / len(ts), 3), "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "u64x4 (256-bit modular integer, CPU)", "data": "synthetic",
                "config": {"workload": "C3: standalone MSM, 2^%d secp256k1 points (CPU arm: bounded sample)" % args.lgn, "sample_terms": ns},
                "cpu_baseline": {"value": val, "unit": "Mpts/s", "cores": cores, "kind": "port", "sample": sample},
                "e2e": {"value": val, "unit": "Mpts/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--lgn", type=int, default=20)
    ap.add_argument("--strong", type=lambda s: [int(x) for x in s.split(",") if x], default=[20, 23])
    ap.add_argument("--verify-proofs", type=int, default=8192)
    ap.add_argument("--verify-reps", type=int, default=12)
    ap.add_argument("--verify-prover-check", type=int, default=16)
    ap.add_argument("--no-verify", action="store_true")
    ap.add_argument("--no-precompute", action="store_true", help="time the plain bucket method as the headline (no per-vector precomputation)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write the outputs of the last step as DIR/<name>.npy "
                    "(same arguments, same inputs: two builds can be compared output for output)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
