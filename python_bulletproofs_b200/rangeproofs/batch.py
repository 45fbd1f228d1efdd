"""Batch verification of independent single-value range proofs over one generator set
(BASELINE config 5).  Not an API of the reference -- it is the data-parallel form of calling
`RangeVerifier(V_i, g, h, gs, hs, u, proof_i).verify()` for every i, with the same decisions.
The batch prover at the end is the same for `NIRangeProver` / `AggregNIRangeProver(...).prove()`.

Packing of a proof follows include/bp_gpu.h (bp_rp_verify_batch); the per-proof transcript
checks run in C on host threads, the scalar algebra and all point equations on the GPU.
"""
import array
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


def pack_transcripts(transcripts, starts):
    """-> (blob, tr_off, starts) of the C ABI: every proof's three transcripts in one blob with 3 * nproofs + 1 offsets."""
    offs, blob, pos = [0], [], 0
    for trio in transcripts:
        for t in trio:
            blob.append(t)
            pos += len(t)
            offs.append(pos)
    return b"".join(blob), (ctypes.c_uint64 * len(offs))(*offs), (ctypes.c_uint32 * max(len(starts), 1))(*starts)


class PackedBatch:
    """A batch in the wire layout of bp_rp_verify_batch (struct-of-records + transcript blob)."""

    def __init__(self, n, records, transcripts, starts):
        self.n = n
        self.nproofs = len(records)
        self.records = b"".join(records)
        self.stride = len(records[0]) if records else nat.load().bp_rp_proof_stride(n)
        self.blob, self.tr_off, self.starts = pack_transcripts(transcripts, starts)

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


def verify_range_proofs_batch(Vs, g, h, gs, hs, u, proofs, combine=False, seed=None, locate=False):
    """-> list[bool].  A proof the C layer cannot classify (exotic numeric transcript slot) is replayed
    through RangeVerifier so that the reference's exception type (ValueError / IndexError) surfaces.
    combine=True checks one random linear combination of the whole batch first (verify_rlc_packed; seed as there).
    locate=True implies it and, when it fails, sends only the proofs of failing leaves to the exact verifier
    (verify_rlc_locate_packed)."""
    n = len(gs)
    if len(Vs) != len(proofs):
        raise Exception('Different number of commitments and proofs')
    batch = PackedBatch.from_proofs(Vs, proofs, n)
    if locate:
        acc = verify_rlc_locate_packed(batch, g, h, gs, hs, u, seed)[0]
    else:
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
    def from_wire(cls, n, m, nproofs, records, blob, tr_off, starts):
        """A batch already in wire form (records back to back, the C ABI's transcript blob, offsets and start indices)."""
        self = cls.__new__(cls)
        self.n, self.m, self.nproofs = n, m, nproofs
        self.stride = nat.load().bp_rp_aggreg_proof_stride(n, m)
        self.records, self.blob, self.tr_off, self.starts = records, blob, tr_off, starts
        return self

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


def verify_aggreg_range_proofs_batch(Vs_list, g, h, gs, hs, u, proofs, combine=False, seed=None, locate=False):
    """-> list[bool]: AggregRangeVerifier(Vs_i, g, h, gs, hs, u, proof_i).verify() for every i, in one call
    (rangeproof_aggreg_verifier.py:42-108).  A proof the C layer cannot classify is replayed through AggregRangeVerifier so that
    the reference's exception type surfaces.  combine=True checks one random linear combination of the whole batch first
    (verify_rlc_packed; seed as there).  locate=True implies it and, when it fails, sends only the proofs of failing leaves to
    the exact verifier (verify_rlc_locate_packed)."""
    from .rangeproof_aggreg_verifier import AggregRangeVerifier
    if len(Vs_list) != len(proofs):
        raise Exception('Different number of commitments and proofs')
    if not proofs:
        return []
    m = len(Vs_list[0])
    if len(gs) % m:
        raise ValueError("generator count is not a multiple of the number of commitments")
    batch = PackedAggregBatch.from_proofs(Vs_list, proofs, len(gs) // m)
    if locate:
        acc = verify_rlc_locate_packed(batch, g, h, gs, hs, u, seed)[0]
    else:
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


# ---- proofs of mixed shapes over prefixes of one generator set ----------------------------------------------------------------
class PackedMixedBatch:
    """A batch in the wire layout of bp_rp_verify_mixed_rlc: proofs of any shape (n bits, m values; n * m a power of two <= nset)
    over the prefixes gs[:n*m], hs[:n*m] of one set of nset generators per side, records back to back in the caller's order."""

    def __init__(self, nset, ns, ms, records, transcripts, starts):
        self.nset = nset
        self.nproofs = len(records)
        self.ns, self.ms = list(ns), list(ms)
        self.offsets, pos = [], 0                  # byte offset of every record
        for r in records:
            self.offsets.append(pos)
            pos += len(r)
        self.records = b"".join(records)
        self.blob, self.tr_off, self.starts = pack_transcripts(transcripts, starts)
        self.ns_arr = (ctypes.c_uint32 * max(len(ns), 1))(*ns)
        self.ms_arr = (ctypes.c_uint32 * max(len(ms), 1))(*ms)

    @classmethod
    def from_items(cls, items, nset):
        """items: (V, proof) or (Vs, proof) pairs; a bare V is a single-value proof (m = 1), a list Vs an aggregated one of m =
        len(Vs) values.  The proof's length N = 2^len(xs) gives n = N / m."""
        ns, ms, recs, trs, sts = [], [], [], [], []
        for V, pr in items:
            Vs = V if isinstance(V, list) else [V]
            p2 = pr.innerProof.proof2
            m, L = len(Vs), len(p2.xs)
            N = 1 << L
            if m == 0 or N % m or len(p2.Ls) != L or len(p2.Rs) != L:
                raise ValueError("proof shape does not match its number of commitments")
            if N > nset:
                raise ValueError("proof of %d generators per side is larger than the set of %d" % (N, nset))
            r, t, s = pack_aggreg_proof(Vs, pr, L)
            if any(not (0 <= int(getattr(x, "x", x)) < nat.Q) for x in p2.xs):      # unreduced challenge: step-by-step path (see PackedBatch)
                s = 0xFFFFFFFF
            ns.append(N // m)
            ms.append(m)
            recs.append(r)
            trs.append(t)
            sts.append(s)
        return cls(nset, ns, ms, recs, trs, sts)


def verify_mixed_rlc_packed(batch: PackedMixedBatch, g, h, gs, hs, u, seed=None, packed=None):
    """-> (accept bytes, combined) of a PackedMixedBatch through bp_rp_verify_mixed_rlc: one random linear combination of every
    proof's equations, whatever its shape; combined = 1 when it holds, 0 when it does not (the bytes are then the exact
    verifiers', one call per shape).  gs, hs: the set of batch.nset generators per side (packed = pack_generators(...) of it).
    seed as for verify_rlc_packed: None draws 32 fresh bytes from os.urandom; a fixed seed only for reproducible tests."""
    if seed is None:
        seed = os.urandom(32)
    if len(seed) != 32:
        raise ValueError("seed must be 32 bytes")
    gs_b, hs_b, g_b, h_b, u_b = packed if packed is not None else pack_generators(g, h, gs, hs, u)
    if len(gs_b) != 64 * batch.nset or len(hs_b) != 64 * batch.nset:
        raise ValueError("the batch was packed for a set of %d generators per side" % batch.nset)
    accept = ctypes.create_string_buffer(max(batch.nproofs, 1))
    combined = ctypes.c_int(0)
    nat.check(nat.load().bp_rp_verify_mixed_rlc(gs_b, hs_b, g_b, h_b, u_b, batch.nset, batch.ns_arr, batch.ms_arr, batch.records,
                                                len(batch.records), batch.nproofs, batch.blob, batch.tr_off, batch.starts, bytes(seed),
                                                accept, ctypes.byref(combined)))
    return accept.raw[:batch.nproofs], combined.value


def verify_rlc_locate_packed(batch, g, h, gs, hs, u, seed=None, packed=None, leaf=0):
    """-> (accept bytes, combined) of a PackedBatch, PackedAggregBatch or PackedMixedBatch through bp_rp_verify_rlc_locate: the
    random linear combination of verify_rlc_packed / verify_mixed_rlc_packed (same weights, same result when it holds,
    combined = 1); when it fails (combined = 0) the batch is cut into leaves of consecutive proofs, each leaf's part of the sum is
    tested, and only the proofs of failing leaves go to the exact verifier.  leaf=0 lets the library pick the leaf size; an
    explicit leaf places the boundaries (for tests).  The decisions are the exact verifier's except with probability
    <= 4 (K + 1)/q for K leaves, only while the seed is unknown to whoever made the proofs: seed=None draws 32 fresh bytes from
    os.urandom; pass a fixed seed for reproducible tests, never for proofs from an untrusted source."""
    if seed is None:
        seed = os.urandom(32)
    if len(seed) != 32:
        raise ValueError("seed must be 32 bytes")
    if leaf < 0:
        raise ValueError("leaf must be >= 0")
    if isinstance(batch, PackedMixedBatch):
        nset, ns_arr, ms_arr = batch.nset, batch.ns_arr, batch.ms_arr
    else:
        m = getattr(batch, "m", 1)
        nset = batch.n * m
        cnt = max(batch.nproofs, 1)
        ns_arr = (ctypes.c_uint32 * cnt).from_buffer(array.array("I", [batch.n]) * cnt)
        ms_arr = (ctypes.c_uint32 * cnt).from_buffer(array.array("I", [m]) * cnt)
    gs_b, hs_b, g_b, h_b, u_b = packed if packed is not None else pack_generators(g, h, gs, hs, u)
    if len(gs_b) != 64 * nset or len(hs_b) != 64 * nset:
        raise ValueError("the batch was packed for a set of %d generators per side" % nset)
    accept = ctypes.create_string_buffer(max(batch.nproofs, 1))
    combined = ctypes.c_int(0)
    nat.check(nat.load().bp_rp_verify_rlc_locate(gs_b, hs_b, g_b, h_b, u_b, nset, ns_arr, ms_arr, batch.records, len(batch.records),
                                                 batch.nproofs, batch.blob, batch.tr_off, batch.starts, bytes(seed), leaf, accept,
                                                 ctypes.byref(combined)))
    return accept.raw[:batch.nproofs], combined.value


def rlc_locate_stats():
    """dict of the last verify_rlc_locate_packed call (bp_rp_rlc_locate_stats): leaf size used, leaves (0 when no leaf pass ran),
    failing leaves, proofs decided by the exact verifier."""
    v = (ctypes.c_uint64 * 4)()
    nat.check(nat.load().bp_rp_rlc_locate_stats(v))
    return {"leaf": v[0], "leaves": v[1], "failing_leaves": v[2], "exact_proofs": v[3]}


def verify_mixed_range_proofs_batch(items, g, h, gs, hs, u, seed=None, locate=False):
    """-> list[bool] in the order of `items`, (V, proof) or (Vs, proof) pairs of any shape over prefixes of one generator set:
    RangeVerifier(V, g, h, gs[:N], hs[:N], u, proof).verify() for a bare V, AggregRangeVerifier(Vs, ...) for a list, N = n * m
    the proof's length -- in one call (one random linear combination, seed as for verify_rlc_packed).  A proof the C layer cannot
    classify is replayed through those classes so that the reference's exception type surfaces.  ValueError: a proof larger than
    the set.  locate=True: when the combination fails, only the proofs of failing leaves go to the exact verifier
    (verify_rlc_locate_packed)."""
    from .rangeproof_aggreg_verifier import AggregRangeVerifier
    batch = PackedMixedBatch.from_items(items, len(gs))
    acc = (verify_rlc_locate_packed if locate else verify_mixed_rlc_packed)(batch, g, h, gs, hs, u, seed)[0]
    out = []
    for i, a in enumerate(acc):
        if a == 2:
            import contextlib, io
            V, pr = items[i]
            N = batch.ns[i] * batch.ms[i]
            cls = AggregRangeVerifier if isinstance(V, list) else RangeVerifier
            try:
                with contextlib.redirect_stdout(io.StringIO()):
                    out.append(bool(cls(V, g, h, gs[:N], hs[:N], u, pr).verify()))
            except Exception as e:   # noqa: BLE001
                if str(e) == "Proof invalid":
                    out.append(False)
                else:
                    raise
        else:
            out.append(a == 1)
    return out


# ---- batch prover ---------------------------------------------------------------------------------------------------------------
def _scalar_bytes(vals, what):
    out = []
    for v in vals:
        x = int(getattr(v, "x", v))
        if not 0 <= x < 1 << 256:
            raise ValueError("%s must lie in [0, 2^256)" % what)
        out.append(x.to_bytes(32, "little"))
    return b"".join(out)


def prove_range_proofs_packed(vs_list, n, g, h, gs, hs, gammas_list, u, seeds, packed=None):
    """-> PackedAggregBatch of AggregNIRangeProver(vs_list[p], n, g, h, gs, hs, gammas_list[p], u, secp256k1, seeds[p]).prove()
    for every p (NIRangeProver for m = 1 values per proof), byte for byte, in the wire form the batch verifiers read: the records
    (V_j = v_j g + gamma_j h first; for m = 1 also a valid PackedBatch) and the three transcripts of every proof, with no Python
    objects in between (bp_rp_prove_batch).  vs_list, gammas_list: one list of m values (ModP or int) per proof, the same m for
    every proof; seeds: one bytes seed per proof; packed = pack_generators(g, h, gs, hs, u), as for the verifiers.
    As in the reference, the blinding factors (alpha, rho, sL, sR, tau1, tau2) derive from the seed alone: proofs that must not
    share them need distinct seeds.  ValueError: ragged m, mismatched lengths, or n*m not a power of two <= 2048 or not len(gs)."""
    nproofs = len(vs_list)
    if len(gammas_list) != nproofs or len(seeds) != nproofs:
        raise ValueError("vs_list, gammas_list and seeds must have one entry per proof")
    m = len(vs_list[0]) if nproofs else 1
    if any(len(vs) != m for vs in vs_list) or any(len(gm) != m for gm in gammas_list):
        raise ValueError("every proof of a batch aggregates the same number of values, with one gamma each")
    N = n * m
    if n < 1 or m < 1 or N & (N - 1) or N > 2048:
        raise ValueError("n * m must be a power of two <= 2048")
    if nproofs == 0:
        return PackedAggregBatch(n, m, [], [], [])
    gs_b, hs_b, g_b, h_b, u_b = packed if packed is not None else pack_generators(g, h, gs, hs, u)
    if len(gs_b) != 64 * N or len(hs_b) != 64 * N:
        raise ValueError("gs and hs must hold n * m = %d points each" % N)
    values = _scalar_bytes([v for vs in vs_list for v in vs], "values")
    gammas = _scalar_bytes([gm for gms in gammas_list for gm in gms], "gammas")
    seed_off = [0]
    for sd in seeds:
        seed_off.append(seed_off[-1] + len(sd))
    L = N.bit_length() - 1
    stride = nat.load().bp_rp_aggreg_proof_stride(n, m)
    # upper bound of the transcripts: seed slot, 4 points of 45 and 3 decimals of <= 79 bytes; Protocol 1 "&x1&" and Protocol 2's
    # start "&&x1&"; per round 2 points and a decimal
    cap = sum(4 * ((len(sd) + 2) // 3) for sd in seeds) + nproofs * (1 + 4 * 45 + 3 * 79 + 81 + 82 + L * (2 * 45 + 79))
    records = ctypes.create_string_buffer(nproofs * stride)
    blob = ctypes.create_string_buffer(cap)
    tr_len = ctypes.c_size_t(0)
    tr_off = (ctypes.c_uint64 * (3 * nproofs + 1))()
    starts = (ctypes.c_uint32 * nproofs)()
    nat.check(nat.load().bp_rp_prove_batch(gs_b, hs_b, g_b, h_b, u_b, n, m, values, gammas, b"".join(seeds),
                                           (ctypes.c_uint64 * (nproofs + 1))(*seed_off), nproofs, records, blob, cap,
                                           ctypes.byref(tr_len), tr_off, starts))
    return PackedAggregBatch.from_wire(n, m, nproofs, records.raw, blob.raw[:tr_len.value], tr_off, starts)


def unpack_aggreg_proofs(batch: PackedAggregBatch):
    """-> list[Proof] of a packed batch (pack_aggreg_proof in reverse; the commitments V_j are not part of a Proof)."""
    from ..innerproduct.inner_product_verifier import Proof1, Proof2
    from ..point import Point
    from ..utils.utils import ModP
    from ._core import Proof
    q, m, stride = nat.Q, batch.m, batch.stride
    L = (batch.n * m).bit_length() - 1
    rec, blob, offs = batch.records, batch.blob, batch.tr_off
    sc = lambda b, o: ModP(int.from_bytes(b[o:o + 32], "little"), q)       # noqa: E731
    out = []
    for p in range(batch.nproofs):
        base = p * stride
        pt = lambda k: Point.from_bytes64(rec, base + 64 * k)               # noqa: E731  (points m, m+1, ... after the V_j)
        A, S, T1, T2 = pt(m), pt(m + 1), pt(m + 2), pt(m + 3)
        o = base + 64 * (m + 4)
        taux, mu, t_hat = sc(rec, o), sc(rec, o + 32), sc(rec, o + 64)
        u_new, P_new = Point.from_bytes64(rec, o + 96), Point.from_bytes64(rec, o + 160)
        o += 224
        a, b = sc(rec, o), sc(rec, o + 32)
        o += 64
        xs = [sc(rec, o + 32 * j) for j in range(L)]
        Ls = [Point.from_bytes64(rec, o + 32 * L + 64 * j) for j in range(L)]
        Rs = [Point.from_bytes64(rec, o + 96 * L + 64 * j) for j in range(L)]
        t0, t1, t2, t3 = (offs[3 * p + k] for k in range(4))
        p2 = Proof2(a, b, xs, Ls, Rs, blob[t2:t3], batch.starts[p])
        out.append(Proof(taux, mu, t_hat, T1, T2, A, S, Proof1(u_new, P_new, p2, blob[t1:t2]), blob[t0:t1]))
    return out


def prove_range_proofs_batch(vs_list, n, g, h, gs, hs, gammas_list, u, seeds, packed=None):
    """-> list[Proof]: the proofs of prove_range_proofs_packed (same arguments, same rules on seeds) as Python objects, equal field
    for field to NIRangeProver / AggregNIRangeProver(...).prove()."""
    return unpack_aggreg_proofs(prove_range_proofs_packed(vs_list, n, g, h, gs, hs, gammas_list, u, seeds, packed))
