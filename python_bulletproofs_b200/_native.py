"""ctypes binding of libbpgpu.so (include/bp_gpu.h) and the byte packers at the boundary.

There is deliberately NO fallback: if the shared library is missing, or no sm_100 GPU is
visible, the first call raises.  Points cross the boundary as 64-byte little-endian affine
(x || y), the identity as 64 zero bytes; scalars as 32-byte little-endian.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libbpgpu.so")

Q = 0xFFFFFFFFFFFFFFFFFFFFFFFFFFFFFFFEBAAEDCE6AF48A03BBFD25E8CD0364141
P = 0xFFFFFFFFFFFFFFFFFFFFFFFFFFFFFFFFFFFFFFFFFFFFFFFFFFFFFFFEFFFFFC2F

c_u8p = ctypes.c_char_p
c_sz = ctypes.c_size_t
c_h = ctypes.c_uint64

# name -> (restype, argtypes): every symbol include/bp_gpu.h declares
PROTOTYPES = {
    "bp_init": (ctypes.c_int, [ctypes.c_int]),
    "bp_shutdown": (ctypes.c_int, []),
    "bp_last_error": (ctypes.c_char_p, []),
    "bp_device_count": (ctypes.c_int, []),
    "bp_device_info": (ctypes.c_int, [ctypes.c_char_p, c_sz, ctypes.POINTER(ctypes.c_int), ctypes.POINTER(ctypes.c_int), ctypes.POINTER(ctypes.c_int)]),
    "bp_msm": (ctypes.c_int, [c_u8p, c_u8p, c_sz, c_u8p]),
    "bp_points_upload": (ctypes.c_int, [c_u8p, c_sz, ctypes.POINTER(c_h)]),
    "bp_scalars_upload": (ctypes.c_int, [c_u8p, c_sz, ctypes.POINTER(c_h)]),
    "bp_handle_free": (ctypes.c_int, [c_h]),
    "bp_points_precompute": (ctypes.c_int, [c_h, ctypes.c_int]),
    "bp_msm_set_pre_slots": (ctypes.c_int, [ctypes.c_int, c_sz]),
    "bp_msm_set_host_finish": (ctypes.c_int, [ctypes.c_int]),
    "bp_msm_set_small_graphs": (ctypes.c_int, [ctypes.c_int]),
    "bp_points_pre_info": (ctypes.c_int, [c_h, ctypes.POINTER(ctypes.c_int), ctypes.POINTER(ctypes.c_int), ctypes.POINTER(ctypes.c_uint64)]),
    "bp_msm_h": (ctypes.c_int, [c_h, c_u8p, c_sz, c_u8p]),
    "bp_msm_hh": (ctypes.c_int, [c_h, c_h, c_sz, c_u8p]),
    "bp_msm_hh_partial": (ctypes.c_int, [c_h, c_h, c_sz, c_sz, c_u8p]),
    "bp_xyzz_sum": (ctypes.c_int, [c_u8p, c_sz, c_u8p]),
    "bp_msm_batch": (ctypes.c_int, [c_u8p, c_u8p, ctypes.POINTER(ctypes.c_uint32), c_sz, c_u8p]),
    "bp_msm_set_window": (ctypes.c_int, [ctypes.c_int]),
    "bp_msm_last_window": (ctypes.c_int, []),
    "bp_msm_last_entries": (ctypes.c_int, [ctypes.POINTER(ctypes.c_uint64)]),
    "bp_msm_set_profiling": (ctypes.c_int, [ctypes.c_int]),
    "bp_launch_count": (ctypes.c_int, [ctypes.POINTER(ctypes.c_uint64)]),
    "bp_msm_stage_ms": (ctypes.c_int, [ctypes.POINTER(ctypes.c_float)]),
    "bp_msm_accumulate_kernel_ms": (ctypes.c_int, [ctypes.POINTER(ctypes.c_float)]),
    "bp_scalar_mul_batch": (ctypes.c_int, [c_u8p, c_u8p, c_sz, c_u8p]),
    "bp_point_add": (ctypes.c_int, [c_u8p, c_u8p, c_u8p]),
    "bp_lift_x_batch": (ctypes.c_int, [c_u8p, c_u8p, c_sz, c_u8p, c_u8p]),
    "bp_rp_verifier_scalars": (ctypes.c_int, [c_sz, c_sz, c_u8p, c_u8p, c_u8p, c_u8p, c_u8p]),
    "bp_rp_prover_poly1": (ctypes.c_int, [c_u8p, c_u8p, c_u8p, c_sz, c_sz, c_u8p, c_u8p, c_u8p, c_u8p]),
    "bp_rp_prover_poly2": (ctypes.c_int, [c_u8p, c_u8p, c_u8p, c_sz, c_sz, c_u8p, c_u8p, c_u8p, c_u8p, c_u8p, c_u8p, c_u8p, c_u8p, c_u8p]),
    "bp_ipa_statement": (ctypes.c_int, [c_u8p, c_u8p, c_u8p, c_u8p, c_u8p, c_u8p, c_sz, c_u8p]),
    "bp_fb_set_mode": (ctypes.c_int, [ctypes.c_int]),
    "bp_fb_stats": (ctypes.c_int, [ctypes.POINTER(ctypes.c_uint64)] * 4),
    "bp_fb_clear": (ctypes.c_int, []),
    "bp_ipa_fold_round": (ctypes.c_int, [c_u8p, c_u8p, c_u8p, c_u8p, c_sz, c_u8p, c_u8p, c_u8p, c_u8p, c_u8p]),
    "bp_ipa_prove": (ctypes.c_int, [c_u8p, c_u8p, c_u8p, c_u8p, c_u8p, c_sz, c_u8p, c_sz, c_u8p, c_u8p, c_u8p, c_u8p, c_u8p,
                                    c_u8p, c_sz, ctypes.POINTER(c_sz)]),
    "bp_ipa_set_graphs": (ctypes.c_int, [ctypes.c_int]),
    "bp_ipa_set_fast_rounds": (ctypes.c_int, [ctypes.c_int]),
    "bp_ipa_prove_hs": (ctypes.c_int, [c_u8p, c_u8p, c_u8p, c_u8p, c_u8p, c_u8p, c_sz, c_u8p, c_sz, c_u8p, c_u8p, c_u8p, c_u8p, c_u8p,
                                       c_u8p, c_sz, ctypes.POINTER(c_sz)]),
    "bp_ipa_verify1_eq_hs": (ctypes.c_int, [c_u8p, c_u8p, c_u8p, c_u8p, c_u8p, c_u8p, c_u8p, c_u8p, c_u8p, c_sz, c_u8p, c_u8p, c_u8p, c_u8p, c_u8p,
                                            ctypes.POINTER(ctypes.c_int)]),
    "bp_ipa_verify_eq_hs": (ctypes.c_int, [c_u8p, c_u8p, c_u8p, c_u8p, c_u8p, c_sz, c_u8p, c_u8p, c_u8p, c_u8p, c_u8p, ctypes.POINTER(ctypes.c_int)]),
    "bp_ipa_verify_eq": (ctypes.c_int, [c_u8p, c_u8p, c_u8p, c_u8p, c_sz, c_u8p, c_u8p, c_u8p, c_u8p, c_u8p, ctypes.POINTER(ctypes.c_int)]),
    "bp_rp_verify_batch": (ctypes.c_int, [c_u8p, c_u8p, c_u8p, c_u8p, c_u8p, c_sz, c_u8p, c_sz, c_sz, c_u8p,
                                          ctypes.POINTER(ctypes.c_uint64), ctypes.POINTER(ctypes.c_uint32), c_u8p]),
    "bp_rp_proof_stride": (c_sz, [c_sz]),
    "bp_rp_verify_batch_gather": (ctypes.c_int, [c_u8p, c_u8p, c_u8p, c_u8p, c_u8p, c_sz, c_u8p, c_sz, c_sz, c_u8p,
                                                 ctypes.POINTER(ctypes.c_uint64), ctypes.POINTER(ctypes.c_uint32), c_sz, c_u8p]),
    "bp_rp_verify_stats": (ctypes.c_int, [ctypes.POINTER(ctypes.c_double)]),
    "bp_rp_aggreg_proof_stride": (c_sz, [c_sz, c_sz]),
    "bp_rp_verify_aggreg_batch": (ctypes.c_int, [c_u8p, c_u8p, c_u8p, c_u8p, c_u8p, c_sz, c_sz, c_u8p, c_sz, c_sz, c_u8p,
                                                 ctypes.POINTER(ctypes.c_uint64), ctypes.POINTER(ctypes.c_uint32), c_u8p]),
    "bp_rp_verify_batch_rlc": (ctypes.c_int, [c_u8p, c_u8p, c_u8p, c_u8p, c_u8p, c_sz, c_sz, c_u8p, c_sz, c_sz, c_u8p,
                                              ctypes.POINTER(ctypes.c_uint64), ctypes.POINTER(ctypes.c_uint32), c_u8p, c_u8p,
                                              ctypes.POINTER(ctypes.c_int)]),
    "bp_rp_verify_mixed_rlc": (ctypes.c_int, [c_u8p, c_u8p, c_u8p, c_u8p, c_u8p, c_sz, ctypes.POINTER(ctypes.c_uint32),
                                              ctypes.POINTER(ctypes.c_uint32), c_u8p, c_sz, c_sz, c_u8p, ctypes.POINTER(ctypes.c_uint64),
                                              ctypes.POINTER(ctypes.c_uint32), c_u8p, c_u8p, ctypes.POINTER(ctypes.c_int)]),
    "bp_rp_verify_rlc_locate": (ctypes.c_int, [c_u8p, c_u8p, c_u8p, c_u8p, c_u8p, c_sz, ctypes.POINTER(ctypes.c_uint32),
                                               ctypes.POINTER(ctypes.c_uint32), c_u8p, c_sz, c_sz, c_u8p, ctypes.POINTER(ctypes.c_uint64),
                                               ctypes.POINTER(ctypes.c_uint32), c_u8p, c_sz, c_u8p, ctypes.POINTER(ctypes.c_int)]),
    "bp_rp_rlc_locate_stats": (ctypes.c_int, [ctypes.POINTER(ctypes.c_uint64)]),
    "bp_rp_prove_batch": (ctypes.c_int, [c_u8p, c_u8p, c_u8p, c_u8p, c_u8p, c_sz, c_sz, c_u8p, c_u8p, c_u8p,
                                         ctypes.POINTER(ctypes.c_uint64), c_sz, c_u8p, c_u8p, c_sz, ctypes.POINTER(c_sz),
                                         ctypes.POINTER(ctypes.c_uint64), ctypes.POINTER(ctypes.c_uint32)]),
    "bp_mod_hash": (ctypes.c_int, [c_u8p, c_sz, c_u8p]),
    "bp_mod_hash_indexed": (ctypes.c_int, [c_u8p, c_sz, ctypes.c_uint32, ctypes.c_uint32, c_u8p]),
    "bp_sha256": (ctypes.c_int, [c_u8p, c_sz, c_u8p]),
    "bp_sha256_set_portable": (ctypes.c_int, [ctypes.c_int]),
    "bp_point_to_b64": (ctypes.c_int, [c_u8p, c_u8p, ctypes.POINTER(c_sz)]),
    "bp_bench_msm": (ctypes.c_int, [c_h, c_h, c_sz, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.POINTER(ctypes.c_float), c_u8p]),
    "bp_imad_peak": (ctypes.c_int, [ctypes.c_int, ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_float)]),
    "bp_pipe_probe": (ctypes.c_int, [ctypes.c_int, ctypes.c_int, ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_float)]),
    "bp_test_fp": (ctypes.c_int, [ctypes.c_int, c_u8p, c_u8p, c_sz, c_u8p]),
    "bp_test_ec": (ctypes.c_int, [ctypes.c_int, c_u8p, c_u8p, c_sz, c_u8p]),
    "bp_test_fq": (ctypes.c_int, [ctypes.c_int, ctypes.c_int, c_u8p, c_u8p, c_sz, c_u8p]),
    "bp_test_xyzz_to_affine_host": (ctypes.c_int, [c_u8p, c_sz, c_u8p]),
    "bp_test_affine_sum_host": (ctypes.c_int, [c_u8p, c_sz, c_u8p]),
    "bp_test_horner_host": (ctypes.c_int, [c_u8p, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, c_u8p]),
    "bp_nccl_unique_id": (ctypes.c_int, [c_u8p]),
    "bp_nccl_init": (ctypes.c_int, [ctypes.c_int, ctypes.c_int, c_u8p]),
    "bp_msm_sharded": (ctypes.c_int, [c_h, c_h, c_sz, c_sz, c_u8p]),
    "bp_allgather_bytes": (ctypes.c_int, [c_u8p, c_sz, c_u8p]),
    "bp_bench_msm_sharded": (ctypes.c_int, [c_h, c_h, c_sz, c_sz, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.POINTER(ctypes.c_float), c_u8p]),
    "bp_msm_sharded_host": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, c_sz, c_u8p]),
    "bp_host_alloc": (ctypes.c_void_p, [c_sz]),
    "bp_host_free": (ctypes.c_int, [ctypes.c_void_p]),
}

_lib = None


class BpGpuError(RuntimeError):
    """Raised when libbpgpu reports a failure (missing GPU, CUDA error, bad arguments)."""


def load():
    """dlopen libbpgpu.so and attach prototypes.  Does not touch the GPU."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise BpGpuError(
                "libbpgpu.so not built (%s): run `python -c 'import __graft_entry__ as g; g.build()'` "
                "or `make -C python_bulletproofs_b200/csrc`; there is no CPU fallback" % LIB_PATH)
        # The batch verifier's host checks run on an OpenMP worker pool.  libgomp's idle workers spin by default; with one
        # process per GPU sharing the host (torchrun) the spinning pools of eight ranks starve each other's main threads and the
        # batch time jitters by milliseconds.  libgomp reads this at load time, so it has to be in the environment before dlopen.
        os.environ.setdefault("OMP_WAIT_POLICY", "PASSIVE")
        lib = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in PROTOTYPES.items():
            fn = getattr(lib, name)
            fn.restype, fn.argtypes = res, args
        _lib = lib
    return _lib


def check(rc):
    if rc != 0:
        raise BpGpuError(load().bp_last_error().decode(errors="replace"))


def init(device=None):
    """Bind this process to one GPU (LOCAL_RANK by default)."""
    if device is None:
        device = int(os.environ.get("LOCAL_RANK", "0"))
    check(load().bp_init(device))


# ---- packers -------------------------------------------------------------------------------
_ZERO64 = bytes(64)


def pack_xy(x, y):
    return x.to_bytes(32, "little") + y.to_bytes(32, "little")


def pack_point(pt):
    """Any object with .x/.y/.curve (fastecdsa-style; curve None = identity) or an (x, y) tuple / None."""
    if pt is None:
        return _ZERO64
    if isinstance(pt, tuple):
        if not (0 <= pt[0] < P and 0 <= pt[1] < P and (pt[1] * pt[1] - pt[0] * pt[0] * pt[0] - 7) % P == 0):
            raise ValueError("coordinates are not on curve <secp256k1>")
        return pack_xy(pt[0], pt[1])
    if getattr(pt, "curve", True) is None:
        return _ZERO64
    pk = getattr(pt, "_pk", None)          # this package's Point caches its wire form (generators are packed on every call)
    if pk is not None and pk[0] is pt.x and pk[1] is pt.y:
        return pk[2]
    b = pack_xy(pt.x, pt.y)
    try:
        pt._pk = (pt.x, pt.y, b)
    except AttributeError:                 # foreign point types (fastecdsa) have no such slot
        pass
    return b


def pack_points(pts):
    out = []
    add = out.append
    for p in pts:      # fast path inlined: a cached wire form that still matches the point's coordinates
        pk = getattr(p, "_pk", None)
        if pk is not None and pk[0] is p.x and pk[1] is p.y:
            add(pk[2])
        else:
            add(pack_point(p))
    return b"".join(out)


def unpack_xy(b, off=0):
    """-> (x, y) or None for the identity."""
    chunk = b[off:off + 64]
    if chunk == _ZERO64:
        return None
    return int.from_bytes(chunk[:32], "little"), int.from_bytes(chunk[32:], "little")


def pack_scalar(k):
    """ints / ModP / anything supporting `% int`  ->  32-byte LE of (k mod q)  (pippenger.py:26)."""
    return (k % Q).to_bytes(32, "little")


def pack_scalars(ks):
    """32-byte little-endian wire form of a scalar list (ints or ModP-like objects with .x), reduced mod q."""
    try:                # the common case -- every value already in [0, 2^256): no big-int division per element
        return b"".join([getattr(k, "x", k).to_bytes(32, "little") for k in ks]) if _all_reduced(ks) else _pack_scalars_slow(ks)
    except (OverflowError, AttributeError):
        return _pack_scalars_slow(ks)


def _all_reduced(ks):
    q = Q
    for k in ks:
        v = getattr(k, "x", k)
        if not (0 <= v < q):
            return False
    return True


def _pack_scalars_slow(ks):
    return b"".join([(int(getattr(k, "x", k)) % Q).to_bytes(32, "little") for k in ks])


def unpack_scalars(b, n):
    return [int.from_bytes(b[32 * i:32 * i + 32], "little") for i in range(n)]


# ---- thin call helpers ---------------------------------------------------------------------
def msm_bytes(pts_b, sc_b, n):
    out = ctypes.create_string_buffer(64)
    check(load().bp_msm(pts_b, sc_b, n, out))
    return out.raw


def msm_batch_bytes(pts_b, sc_b, offsets):
    nmsm = len(offsets) - 1
    if len(pts_b) != 64 * offsets[-1] or len(sc_b) != 32 * offsets[-1]:     # the C side copies offsets[-1] records
        raise AssertionError("msm_batch_bytes: %d point bytes / %d scalar bytes for %d terms" % (len(pts_b), len(sc_b), offsets[-1]))
    out = ctypes.create_string_buffer(64 * max(nmsm, 1))
    off = (ctypes.c_uint32 * len(offsets))(*offsets)
    check(load().bp_msm_batch(pts_b, sc_b, off, nmsm, out))
    return out.raw[:64 * nmsm]


def mod_hash_indexed_raw(suffix, first, count):
    """mod_hash(str(i).encode() + suffix, q) for i in range(first, first + count), as count 32-byte LE scalars (hashed in C)."""
    out = ctypes.create_string_buffer(32 * max(count, 1))
    check(load().bp_mod_hash_indexed(suffix, len(suffix), first, count, out))
    return out.raw[:32 * count]


def mod_hash_indexed(suffix, first, count):
    raw = mod_hash_indexed_raw(suffix, first, count)
    return [int.from_bytes(raw[32 * i:32 * i + 32], "little") for i in range(count)]


def rp_verifier_scalars(n, m, y, z):
    """(y^-i packed, (z + zz_i y^-i) packed, delta as int) -- bp_rp_verifier_scalars."""
    nm = n * m
    yinv, hsc, delta = ctypes.create_string_buffer(32 * nm), ctypes.create_string_buffer(32 * nm), ctypes.create_string_buffer(32)
    check(load().bp_rp_verifier_scalars(n, m, (y % Q).to_bytes(32, "little"), (z % Q).to_bytes(32, "little"), yinv, hsc, delta))
    return yinv.raw, hsc.raw, int.from_bytes(delta.raw, "little")


def rp_prover_poly1(bits, sL_b, sR_b, n, m, y, z):
    """(t1, t2) of the range-proof polynomial, computed in C (bp_rp_prover_poly1)."""
    t1, t2 = ctypes.create_string_buffer(32), ctypes.create_string_buffer(32)
    check(load().bp_rp_prover_poly1(bits, sL_b, sR_b, n, m, (y % Q).to_bytes(32, "little"), (z % Q).to_bytes(32, "little"), t1, t2))
    return int.from_bytes(t1.raw, "little"), int.from_bytes(t2.raw, "little")


def rp_prover_poly2(bits, sL_b, sR_b, n, m, y, z, x):
    """(ls, rs, y^-i, z + zz_i y^-i) as packed scalar vectors, t_hat as an int, then rs_i y^-i packed (bp_rp_prover_poly2)."""
    nm = n * m
    ls, rs, yinv, hsc, rsy = (ctypes.create_string_buffer(32 * nm) for _ in range(5))
    that = ctypes.create_string_buffer(32)
    check(load().bp_rp_prover_poly2(bits, sL_b, sR_b, n, m, (y % Q).to_bytes(32, "little"), (z % Q).to_bytes(32, "little"),
                                    (x % Q).to_bytes(32, "little"), ls, rs, yinv, hsc, rsy, that))
    return ls.raw, rs.raw, yinv.raw, hsc.raw, int.from_bytes(that.raw, "little"), rsy.raw


def lift_x_batch(xs, want=None):
    """[(x, y) or None] for candidate x coordinates; want[i] in {0: even y, 1: odd y, 2: principal root, 3: its negation}."""
    n = len(xs)
    if n == 0:
        return []
    xb = b"".join(int(x).to_bytes(32, "little") for x in xs)
    out = ctypes.create_string_buffer(64 * n)
    ok = ctypes.create_string_buffer(n)
    check(load().bp_lift_x_batch(xb, bytes(want) if want is not None else None, n, out, ok))
    raw = out.raw
    return [(int.from_bytes(raw[64 * i:64 * i + 32], "little"), int.from_bytes(raw[64 * i + 32:64 * i + 64], "little"))
            if ok.raw[i] else None for i in range(n)]


def scalar_mul_batch_bytes(pts_b, sc_b, n):
    out = ctypes.create_string_buffer(64 * max(n, 1))
    check(load().bp_scalar_mul_batch(pts_b, sc_b, n, out))
    return out.raw[:64 * n]
