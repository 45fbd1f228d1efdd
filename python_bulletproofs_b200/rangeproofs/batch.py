"""Batch verification of independent single-value range proofs over one generator set
(BASELINE config 5).  Not an API of the reference -- it is the data-parallel form of calling
`RangeVerifier(V_i, g, h, gs, hs, u, proof_i).verify()` for every i, with the same decisions.

Packing of a proof follows include/bp_gpu.h (bp_rp_verify_batch); the per-proof transcript
checks run in C on host threads, the scalar algebra and all point equations on the GPU.
"""
import ctypes
import os

from .. import _native as nat
from .rangeproof_verifier import RangeVerifier


def pack_proof(V, proof, log_n):
    ip = proof.innerProof
    p2 = ip.proof2
    le = lambda s: (s % nat.Q).to_bytes(32, "little")          # noqa: E731
    rec = [nat.pack_point(V), nat.pack_point(proof.A), nat.pack_point(proof.S), nat.pack_point(proof.T1),
           nat.pack_point(proof.T2), le(proof.taux), le(proof.mu), le(proof.t_hat),
           nat.pack_point(ip.u_new), nat.pack_point(ip.P_new), le(p2.a), le(p2.b)]
    rec += [le(x) for x in p2.xs[:log_n]]
    rec += [nat.pack_point(L) for L in p2.Ls[:log_n]] + [nat.pack_point(R) for R in p2.Rs[:log_n]]
    return b"".join(rec), (proof.transcript, ip.transcript, p2.transcript), p2.start_transcript


class PackedBatch:
    """A batch in the wire layout of bp_rp_verify_batch (struct-of-records + transcript blob)."""

    def __init__(self, n, records, transcripts, starts):
        self.n = n
        self.nproofs = len(records)
        self.records = b"".join(records)
        self.stride = len(records[0]) if records else nat.load().bp_rp_proof_stride(n)
        offs, blob, pos = [0], [], 0
        for trio in transcripts:
            for t in trio:
                blob.append(t)
                pos += len(t)
                offs.append(pos)
        self.blob = b"".join(blob)
        self.tr_off = (ctypes.c_uint64 * len(offs))(*offs)
        self.starts = (ctypes.c_uint32 * max(len(starts), 1))(*starts)

    @classmethod
    def from_proofs(cls, Vs, proofs, n):
        log_n = n.bit_length() - 1
        recs, trs, sts = [], [], []
        for V, pr in zip(Vs, proofs):
            if len(pr.innerProof.proof2.xs) != log_n or len(pr.innerProof.proof2.Ls) != log_n or len(pr.innerProof.proof2.Rs) != log_n:
                raise ValueError("proof shape does not match the generator count")
            r, t, s = pack_proof(V, pr, log_n)
            # The C transcript check compares the decimal of the REDUCED challenge with the transcript slot; the reference
            # compares str(xs[i]) of the raw ModP.x (inner_product_verifier.py:121-125).  An unreduced xs[i] (= hash + q)
            # is therefore sent down the step-by-step path (start index past the end = verdict "defer").
            if any(not (0 <= int(getattr(x, "x", x)) < nat.Q) for x in pr.innerProof.proof2.xs):
                s = 0xFFFFFFFF
            recs.append(r)
            trs.append(t)
            sts.append(s)
        return cls(n, recs, trs, sts)


def verify_packed(batch: PackedBatch, g, h, gs, hs, u, first=0, count=None):
    """accept bytes (1 accept / 0 reject / 2 defer-to-Python) for proofs [first, first+count)."""
    count = batch.nproofs - first if count is None else count
    accept = ctypes.create_string_buffer(max(count, 1))
    tr_off = ctypes.cast(ctypes.byref(batch.tr_off, 8 * 3 * first), ctypes.POINTER(ctypes.c_uint64))
    starts = ctypes.cast(ctypes.byref(batch.starts, 4 * first), ctypes.POINTER(ctypes.c_uint32))
    recs = ctypes.c_char_p(batch.records[first * batch.stride:(first + count) * batch.stride])
    nat.check(nat.load().bp_rp_verify_batch(
        nat.pack_points(gs), nat.pack_points(hs), nat.pack_point(g), nat.pack_point(h), nat.pack_point(u), batch.n,
        recs, batch.stride, count, batch.blob, tr_off, starts, accept))
    return accept.raw[:count]


def verify_local_gather(local: PackedBatch, g, h, gs, hs, u, counts):
    """This rank's block `local` (counts[rank] proofs) is verified, then the accept bytes of all ranks are all-gathered on the
    device (the one ncclAllGather inside bp_rp_verify_batch_gather) -> accept bytes of the WHOLE batch, on every rank.
    More than one rank needs sharding.init_nccl() first."""
    width = max(counts) if counts else 0
    out = ctypes.create_string_buffer(max(width * len(counts), 1))
    nat.check(nat.load().bp_rp_verify_batch_gather(
        nat.pack_points(gs), nat.pack_points(hs), nat.pack_point(g), nat.pack_point(h), nat.pack_point(u), local.n,
        local.records, local.stride, local.nproofs, local.blob, local.tr_off, local.starts, width, out))
    raw = out.raw
    return b"".join(raw[r * width:r * width + c] for r, c in enumerate(counts))


def verify_packed_sharded(batch: PackedBatch, g, h, gs, hs, u, rank, world):
    """Proof-sharded batch (SURVEY.md 8e) from a batch every rank holds in full: rank r verifies the contiguous block
    sharding.slice_bounds(nproofs, r, world); returns the accept bytes of the whole batch."""
    from ..sharding import all_slices
    slices = all_slices(batch.nproofs, world)
    first, last = slices[rank]
    count = last - first
    width = max(b - a for a, b in slices) if slices else 0
    out = ctypes.create_string_buffer(max(width * world, 1))
    tr_off = ctypes.cast(ctypes.byref(batch.tr_off, 8 * 3 * first), ctypes.POINTER(ctypes.c_uint64))
    starts = ctypes.cast(ctypes.byref(batch.starts, 4 * first), ctypes.POINTER(ctypes.c_uint32))
    recs = ctypes.c_char_p(batch.records[first * batch.stride:(first + count) * batch.stride])
    nat.check(nat.load().bp_rp_verify_batch_gather(
        nat.pack_points(gs), nat.pack_points(hs), nat.pack_point(g), nat.pack_point(h), nat.pack_point(u), batch.n,
        recs, batch.stride, count, batch.blob, tr_off, starts, width, out))
    raw = out.raw
    return b"".join(raw[r * width:r * width + (b - a)] for r, (a, b) in enumerate(slices))


def verify_stats():
    """dict of the last batch call's measurements (bp_rp_verify_stats)."""
    v = (ctypes.c_double * 7)()
    nat.check(nat.load().bp_rp_verify_stats(v))
    return {"wall_ms": v[0], "host_check_ms": v[1], "device_span_ms": v[2], "chunks": int(v[3]), "host_threads": int(v[4]),
            "table_mode": int(v[5]), "proofs": int(v[6])}


def verify_range_proofs_batch(Vs, g, h, gs, hs, u, proofs, combine=False, seed=None):
    """-> list[bool].  A proof the C layer cannot classify (exotic numeric transcript slot) is replayed
    through RangeVerifier so that the reference's exception type (ValueError / IndexError) surfaces.
    combine=True checks one random linear combination of the whole batch first (verify_rlc_packed; seed as there)."""
    n = len(gs)
    if len(Vs) != len(proofs):
        raise Exception('Different number of commitments and proofs')
    batch = PackedBatch.from_proofs(Vs, proofs, n)
    acc = verify_rlc_packed(batch, g, h, gs, hs, u, seed)[0] if combine else verify_packed(batch, g, h, gs, hs, u)
    out = []
    for i, a in enumerate(acc):
        if a == 2:
            try:
                import contextlib, io
                with contextlib.redirect_stdout(io.StringIO()):
                    out.append(bool(RangeVerifier(Vs[i], g, h, gs, hs, u, proofs[i]).verify()))
            except Exception as e:      # noqa: BLE001
                if str(e) != "Proof invalid":
                    raise
                out.append(False)
        else:
            out.append(a == 1)
    return out


# ---- aggregated proofs (m values per proof) ---------------------------------------------------------------------------------
def pack_aggreg_proof(Vs, proof, log_nm):
    """One aggregated proof in the wire layout of bp_rp_verify_aggreg_batch (include/bp_gpu.h)."""
    ip = proof.innerProof
    p2 = ip.proof2
    le = lambda s: (s % nat.Q).to_bytes(32, "little")          # noqa: E731
    rec = [nat.pack_point(V) for V in Vs]
    rec += [nat.pack_point(proof.A), nat.pack_point(proof.S), nat.pack_point(proof.T1), nat.pack_point(proof.T2),
            le(proof.taux), le(proof.mu), le(proof.t_hat), nat.pack_point(ip.u_new), nat.pack_point(ip.P_new), le(p2.a), le(p2.b)]
    rec += [le(x) for x in p2.xs[:log_nm]]
    rec += [nat.pack_point(L) for L in p2.Ls[:log_nm]] + [nat.pack_point(R) for R in p2.Rs[:log_nm]]
    return b"".join(rec), (proof.transcript, ip.transcript, p2.transcript), p2.start_transcript


class PackedAggregBatch(PackedBatch):
    """A batch of aggregated proofs, each over m commitments of n bits (n * m generators per side)."""

    def __init__(self, n, m, records, transcripts, starts):
        super().__init__(n, records, transcripts, starts)
        self.m = m
        if not records:
            self.stride = nat.load().bp_rp_aggreg_proof_stride(n, m)

    @classmethod
    def from_proofs(cls, Vs_list, proofs, n):
        if not proofs:
            return cls(n, 1, [], [], [])
        m = len(Vs_list[0])
        log_nm = (n * m).bit_length() - 1
        recs, trs, sts = [], [], []
        for Vs, pr in zip(Vs_list, proofs):
            p2 = pr.innerProof.proof2
            if len(Vs) != m:
                raise ValueError("every proof of a batch aggregates the same number of commitments")
            if len(p2.xs) != log_nm or len(p2.Ls) != log_nm or len(p2.Rs) != log_nm:
                raise ValueError("proof shape does not match the generator count")
            r, t, s = pack_aggreg_proof(Vs, pr, log_nm)
            if any(not (0 <= int(getattr(x, "x", x)) < nat.Q) for x in p2.xs):      # unreduced challenge: step-by-step path (see PackedBatch)
                s = 0xFFFFFFFF
            recs.append(r)
            trs.append(t)
            sts.append(s)
        return cls(n, m, recs, trs, sts)


def pack_generators(g, h, gs, hs, u):
    """The five generator arguments in wire form; a caller that verifies many batches over one generator set packs them once."""
    return nat.pack_points(gs), nat.pack_points(hs), nat.pack_point(g), nat.pack_point(h), nat.pack_point(u)


def verify_aggreg_packed(batch: PackedAggregBatch, g, h, gs, hs, u, packed=None):
    """accept bytes (1 accept / 0 reject / 2 defer-to-Python) of a batch of aggregated proofs (packed = pack_generators(...))."""
    accept = ctypes.create_string_buffer(max(batch.nproofs, 1))
    gs_b, hs_b, g_b, h_b, u_b = packed if packed is not None else pack_generators(g, h, gs, hs, u)
    nat.check(nat.load().bp_rp_verify_aggreg_batch(gs_b, hs_b, g_b, h_b, u_b, batch.n, batch.m,
                                                   batch.records, batch.stride, batch.nproofs, batch.blob, batch.tr_off, batch.starts, accept))
    return accept.raw[:batch.nproofs]


def verify_rlc_packed(batch, g, h, gs, hs, u, seed=None, packed=None):
    """-> (accept bytes, combined) of a PackedBatch (m = 1) or PackedAggregBatch through bp_rp_verify_batch_rlc: one random
    linear combination of every proof's equations is checked; combined = 1 when it holds (every proof that passed its
    transcript and point checks is accepted), 0 when it does not (the bytes are then the exact verifier's).
    seed=None draws 32 fresh bytes from os.urandom for this call.  The decisions are the exact verifier's except with
    probability <= 4/q only while the seed is unknown to whoever made the proofs: pass a fixed seed for reproducible tests,
    never for proofs from an untrusted source."""
    if seed is None:
        seed = os.urandom(32)
    if len(seed) != 32:
        raise ValueError("seed must be 32 bytes")
    accept = ctypes.create_string_buffer(max(batch.nproofs, 1))
    combined = ctypes.c_int(0)
    gs_b, hs_b, g_b, h_b, u_b = packed if packed is not None else pack_generators(g, h, gs, hs, u)
    nat.check(nat.load().bp_rp_verify_batch_rlc(gs_b, hs_b, g_b, h_b, u_b, batch.n, getattr(batch, "m", 1), batch.records,
                                                batch.stride, batch.nproofs, batch.blob, batch.tr_off, batch.starts, bytes(seed),
                                                accept, ctypes.byref(combined)))
    return accept.raw[:batch.nproofs], combined.value


def verify_aggreg_range_proofs_batch(Vs_list, g, h, gs, hs, u, proofs, combine=False, seed=None):
    """-> list[bool]: AggregRangeVerifier(Vs_i, g, h, gs, hs, u, proof_i).verify() for every i, in one call
    (rangeproof_aggreg_verifier.py:42-108).  A proof the C layer cannot classify is replayed through AggregRangeVerifier so that
    the reference's exception type surfaces.  combine=True checks one random linear combination of the whole batch first
    (verify_rlc_packed; seed as there)."""
    from .rangeproof_aggreg_verifier import AggregRangeVerifier
    if len(Vs_list) != len(proofs):
        raise Exception('Different number of commitments and proofs')
    if not proofs:
        return []
    m = len(Vs_list[0])
    if len(gs) % m:
        raise ValueError("generator count is not a multiple of the number of commitments")
    batch = PackedAggregBatch.from_proofs(Vs_list, proofs, len(gs) // m)
    acc = verify_rlc_packed(batch, g, h, gs, hs, u, seed)[0] if combine else verify_aggreg_packed(batch, g, h, gs, hs, u)
    out = []
    for i, a in enumerate(acc):
        if a == 2:
            import contextlib, io
            try:
                with contextlib.redirect_stdout(io.StringIO()):
                    out.append(bool(AggregRangeVerifier(Vs_list[i], g, h, gs, hs, u, proofs[i]).verify()))
            except Exception as e:   # noqa: BLE001
                if str(e) == "Proof invalid":
                    out.append(False)
                else:
                    raise
        else:
            out.append(a == 1)
    return out
