/*
 * bp_gpu.h -- C ABI of libbpgpu.so, the B200 (sm_100a) implementation of the data-parallel hot
 * path of wborgeaud/python-bulletproofs.  Plain pointers and sizes only; loaded with ctypes
 * (python_bulletproofs_b200/_native.py).  Every entry point names the reference interface it
 * replaces (paths relative to /root/reference/).
 *
 * Conventions
 *   - return value: 0 = ok, non-zero = error; bp_last_error() describes the last failure of
 *     the calling thread's most recent call.
 *   - affine point  : 64 bytes, x then y, each 32-byte LITTLE-endian, canonical (< p);
 *                     the identity is 64 zero bytes (fastecdsa's Point.IDENTITY_ELEMENT).
 *   - scalar        : 32-byte little-endian, any value < 2^256; reduced mod q on the device
 *                     exactly as `es = [ei % order]` (src/pippenger/pippenger.py:26).
 *   - all buffers are caller-owned host memory unless a handle is used; calls are synchronous
 *     and serialised on one CUDA stream per process; one process drives one GPU (bp_init).
 *   - threading: the library keeps per-process state (workspaces, the table cache of "fixed-base tables", captured
 *     graphs); like the reference it is meant to be called from ONE thread at a time.  It starts host threads of its own
 *     only inside bp_rp_verify_batch (transcript checks of a chunk, joined before the call returns).
 */
#ifndef BP_GPU_H
#define BP_GPU_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef uint64_t bp_handle;   /* device-resident vector of points or scalars */

/* ---- lifetime ------------------------------------------------------------------------------ */
int bp_init(int device);                 /* select GPU `device`, create the stream/workspace */
int bp_shutdown(void);
const char* bp_last_error(void);
int bp_device_count(void);
int bp_device_info(char* name, size_t cap, int* sm_count, int* cc_major, int* cc_minor);

/* ---- multi-scalar multiplication ---------------------------------------------------------------
 * Pippenger.multiexp(gs, es)                      src/pippenger/pippenger.py:22-61
 * (and through it vector_commitment, src/utils/commitments.py:9-13).
 * n = 0 yields the identity (pippenger.py:28-29).  The length check of pippenger.py:23-24 is
 * done by the Python wrapper, which raises the reference's exception text. */
int bp_msm(const uint8_t* pts64, const uint8_t* sc32, size_t n, uint8_t out64[64]);

/* device-resident operands (SURVEY.md 7 "hard part 2": marshalling 2^20 Python Points costs
 * three orders of magnitude more than the kernel) */
int bp_points_upload(const uint8_t* pts64, size_t n, bp_handle* h);
int bp_scalars_upload(const uint8_t* sc32, size_t n, bp_handle* h);
int bp_handle_free(bp_handle h);
/* Precomputed window multiples for a resident point vector (fixed generators: the setting of every Bulletproofs commitment
 * call site, src/utils/commitments.py:9-13): stores 2^(c*w) * P_i for the W = ceil(257/c) windows of a 256-bit scalar
 * (W * 64 bytes per point; window_bits = 0 picks c from the vector length, 19 at 2^20 points = 0.94 GB).  Every later
 * MSM over the handle (bp_msm_h, bp_msm_hh, bp_msm_hh_partial, bp_msm_sharded, bp_bench_msm*) then needs no doublings at
 * all: one shared bucket unit, no Horner chain, 14 instead of 16 mixed additions per point.  Same canonical result.
 * bp_msm_set_window(c > 0) forces the plain bucket method again. */
int bp_points_precompute(bp_handle points, int window_bits);
int bp_points_pre_info(bp_handle points, int* window_bits, int* windows, uint64_t* bytes);
int bp_msm_set_small_graphs(int on);      /* MSMs of <= 2^17 terms over a precomputed vector as replayed CUDA graphs (default on) */
int bp_msm_set_pre_slots(int mode, size_t min_terms);   /* sort stage of one large resident MSM (precomputed path; plain path where a bucket holds >= 48 entries, i.e. from 2^20 terms): 1 (default) = slot sort (one scattered pass; exact counting sort as gated fallback) for MSMs of >= min_terms terms (default 2^18; 0 keeps the value), 0 = exact counting sort only, 2 = test hook, 8 slots per bucket so that the fallback runs */
int bp_msm_set_host_finish(int on);     /* 1 (default): an MSM whose result goes to the host (bp_msm, bp_msm_sharded_host on one rank; bucket method without precomputed multiples) hands its window sums to the host, which runs the Horner chain and the affine conversion; 0 = k_combine on the device */
int bp_msm_h(bp_handle points, const uint8_t* sc32, size_t n, uint8_t out64[64]);     /* scalars from host */
int bp_msm_hh(bp_handle points, bp_handle scalars, size_t n, uint8_t out64[64]);      /* all resident */
/* XYZZ partial (4 x 32-byte LE: X, Y, ZZ, ZZZ) of a point slice, for sharding over GPUs
 * (SURVEY.md 8e); bp_xyzz_sum adds `count` partials and returns the canonical affine point. */
int bp_msm_hh_partial(bp_handle points, bp_handle scalars, size_t first, size_t n, uint8_t out128[128]);
int bp_xyzz_sum(const uint8_t* partials128, size_t count, uint8_t out64[64]);

/* many independent MSMs in one launch sequence: MSM j uses terms offsets[j] .. offsets[j+1]-1
 * (offsets has nmsm+1 entries).  Replaces the per-round / per-proof multiexp calls of
 * src/innerproduct/inner_product_prover.py:98-99, inner_product_verifier.py:134-143,
 * src/rangeproofs/rangeproof_verifier.py:88-97. */
int bp_msm_batch(const uint8_t* pts64, const uint8_t* sc32, const uint32_t* offsets, size_t nmsm, uint8_t* out64);

/* window-size override for experiments (0 = automatic) and per-stage device timings (ms) of the
 * last MSM call: [0]=digits [1]=scan [2]=scatter [3]=accumulate [4]=reduce [5]=combine [6]=total */
int bp_msm_set_window(int c);
int bp_msm_last_window(void);
int bp_msm_last_entries(uint64_t* entries);   /* mixed additions (non-zero signed digits) of the last MSM */
int bp_msm_set_profiling(int on);
/* kernels this library has launched so far in this process (kernel nodes of a replayed CUDA graph count at every replay);
 * bench.py reports the difference across its timed region as "gpu_launches" */
int bp_launch_count(uint64_t* launches);
int bp_msm_stage_ms(float out7[7]);
int bp_msm_accumulate_kernel_ms(float* ms);   /* k_accumulate alone (stage [3] also holds the bucket memset and the fix-ups) */

/* ---- fixed-base tables for repeated generator sets -----------------------------------------------------
 * The commitment / L,R / verifier call sites of a Bulletproofs instance pass the same group elements on every call
 * (src/utils/commitments.py:9-13, src/innerproduct/inner_product_prover.py:98-99, src/rangeproofs/rangeproof_prover.py:
 * 47,57,78-86).  The library recognises a repeated point set by a hash of its bytes and answers from a precomputed
 * table (255 multiples per byte window, 522 KB per point) instead of the bucket method: same canonical result, ~5x
 * lower latency for the 2..4097-term MSMs of a prover.  mode 0 = never, 1 = build at the second use of a set (default),
 * 2 = build at first use.  bp_fb_clear drops every table.  A cache hit is confirmed by comparing the generator bytes. */
int bp_fb_set_mode(int mode);
int bp_fb_stats(uint64_t* tables, uint64_t* bytes, uint64_t* hits, uint64_t* builds);
int bp_fb_clear(void);

/* ---- a + b for two points: fastecdsa Point.__add__ where the reference adds outside a multiexp
 * (src/innerproduct/inner_product_prover.py:33, src/utils/commitments.py:6).  One launch, one inversion. */
int bp_point_add(const uint8_t a64[64], const uint8_t b64[64], uint8_t out64[64]);

/* ---- independent scalar multiplications --------------------------------------------------------
 * out[i] = sc[i] * pts[i]:  hsp = [(y.inv() ** i) * hs[i] ...]
 * src/rangeproofs/rangeproof_prover.py:77, rangeproof_verifier.py:72,
 * rangeproof_aggreg_prover.py:82, rangeproof_aggreg_verifier.py:80; ModP.__mul__(Point) utils.py:43-44 */
int bp_scalar_mul_batch(const uint8_t* pts64, const uint8_t* sc32, size_t n, uint8_t* out64);

/* ---- range-proof prover: polynomial algebra over Z_q on the host (SURVEY 8(f) N1) --------------------------
 * _get_polynomial_coeffs / _final_compute of src/rangeproofs/rangeproof_prover.py:93-112 and
 * rangeproof_aggreg_prover.py:117-146 for m values of n bits (aL_bits: n*m bytes 0/1, value-major; sL, sR: n*m scalars):
 *   poly1 (after y, z):  t1, t2
 *   poly2 (after x):     ls, rs (the vectors handed to the inner-product argument), t_hat = <ls, rs>, yinv[i] = y^-i and
 *                        hsc[i] = z + z^(2 + i/n) 2^(i mod n) y^-i  (the h-generator scalars of the P multiexp, :78-86)
 * Pure host code (4 x 64-bit Montgomery arithmetic), no GPU needed. */
int bp_rp_prover_poly1(const uint8_t* aL_bits, const uint8_t* sL32, const uint8_t* sR32, size_t n, size_t m, const uint8_t y32[32],
                       const uint8_t z32[32], uint8_t t1_out[32], uint8_t t2_out[32]);
int bp_rp_prover_poly2(const uint8_t* aL_bits, const uint8_t* sL32, const uint8_t* sR32, size_t n, size_t m, const uint8_t y32[32],
                       const uint8_t z32[32], const uint8_t x32[32], uint8_t* ls32, uint8_t* rs32, uint8_t* yinv32, uint8_t* hsc32,
                       uint8_t* rsy32 /* optional: rs[i] * y^-i */, uint8_t that_out[32]);
/* verifier side: yinv[i] = y^-i, hsc[i] = z + z^(2 + i/n) 2^(i mod n) y^-i and
 * delta(y, z) = (z - z^2) sum y^i - sum_{j=1..m} z^(j+2) (2^n - 1)   (rangeproof_verifier.py:69-72, aggregated :72-80) */
int bp_rp_verifier_scalars(size_t n, size_t m, const uint8_t y32[32], const uint8_t z32[32], uint8_t* yinv32, uint8_t* hsc32,
                           uint8_t delta_out[32]);

/* ---- batched lift-x / point decompression (SURVEY 8(f) N4) ---------------------------------------
 * y = sqrt(x^3 + 7) for n candidate x coordinates (32-byte LE, must be < p); ok[i] = 1 when x is on the curve, else
 * out[i] = zeros.  want[i]: 0 = even y, 1 = odd y (bytes_to_point, src/utils/utils.py:119-131), 2 = the root
 * mod_sqrt(...)[0] = (x^3+7)^((p+1)/4), 3 = p - that root (elliptic_hash, src/utils/elliptic_curve_hash.py:17-23);
 * want == NULL means 2 for all. */
int bp_lift_x_batch(const uint8_t* xs32, const uint8_t* want, size_t n, uint8_t* out64, uint8_t* ok);

/* ---- inner-product argument ---------------------------------------------------------------------
 * One folding step, for step-wise parity tests:
 *   g'[i] = xinv*g[i] + x*g[i+n/2],  h'[i] = x*h[i] + xinv*h[i+n/2]      (inner_product_prover.py:107-108)
 *   a'[i] = x*a[i] + xinv*a[i+n/2],  b'[i] = xinv*b[i] + x*b[i+n/2] mod q (inner_product_prover.py:109-110)
 * n is the current (even) length; outputs have n/2 entries.  xinv is computed on the device side. */
int bp_ipa_fold_round(const uint8_t* g64, const uint8_t* h64, const uint8_t* a32, const uint8_t* b32, size_t n,
                      const uint8_t x32[32], uint8_t* g_out64, uint8_t* h_out64, uint8_t* a_out32, uint8_t* b_out32);

/* FastNIProver2.prove()                         src/innerproduct/inner_product_prover.py:70-110
 * n = power of two (1 allowed: zero rounds).  `transcript` is the digest so far (the Transcript
 * object's bytes, already including base64(seed) + "&"); the Fiat-Shamir hashing of each round
 * runs on the host inside this call (SHA-256 / base64 / decimal printing restated in C, see
 * csrc/transcript.h).  Outputs: Ls, Rs (log2 n points), xs (log2 n scalars), final a, b, and the
 * full transcript digest (tout_len receives its length; error if tout_cap is too small). */
int bp_ipa_prove(const uint8_t* g64, const uint8_t* h64, const uint8_t u64_[64], const uint8_t* a32, const uint8_t* b32,
                 size_t n, const uint8_t* transcript, size_t transcript_len, uint8_t* Ls64, uint8_t* Rs64, uint8_t* xs32,
                 uint8_t a_out32[32], uint8_t b_out32[32], uint8_t* transcript_out, size_t tout_cap, size_t* tout_len);

/* How the host's Fiat-Shamir step (one SHA-256 per round, inner_product_prover.py:102-106) meets the device work of a proof:
 *   1 (default)  the whole proof is enqueued once; the stream waits on a mapped host word for every challenge and signals
 *                every L, R pair through another one (stream wait-value / write-value operations) while the calling thread
 *                polls: no stream synchronisation, launch or callback thread between two rounds;
 *   2            the same sequence with the host side as host nodes (cudaLaunchHostFunc), captured into ONE CUDA graph per
 *                vector length and replayed: one launch per proof;
 *   0            plain stream launches, one cudaStreamSynchronize per round. */
int bp_ipa_set_graphs(int mode);
/* Table rounds of proofs with n <= 4096 as two launches per round (scalar work of the round in one block reading the mapped
 * parameter block; table MSM whose last block reduces and writes L, R into mapped host memory): on by default, 0 = the
 * four-launch form with copy operations. */
int bp_ipa_set_fast_rounds(int on);

/* Same, with the h generators given as (h, hscale): the effective generators are hscale_i * h_i, which are never
 * materialised (hscale32 = NULL means all ones).  The range-proof prover passes hs with hscale_i = y^-i instead of the
 * list hsp of src/rangeproofs/rangeproof_prover.py:77. */
int bp_ipa_prove_hs(const uint8_t* g64, const uint8_t* h64, const uint8_t* hscale32, const uint8_t u64_[64], const uint8_t* a32,
                    const uint8_t* b32, size_t n, const uint8_t* transcript, size_t transcript_len, uint8_t* Ls64, uint8_t* Rs64,
                    uint8_t* xs32, uint8_t a_out32[32], uint8_t b_out32[32], uint8_t* transcript_out, size_t tout_cap,
                    size_t* tout_len);
int bp_ipa_verify_eq_hs(const uint8_t* g64, const uint8_t* h64, const uint8_t* hscale32, const uint8_t u64_[64], const uint8_t P64[64],
                        size_t n, const uint8_t a32[32], const uint8_t b32[32], const uint8_t* xs32, const uint8_t* Ls64,
                        const uint8_t* Rs64, int* accept);

/* The statement of the argument, P = sum a_i g_i + sum bs_i h_i + c u (NIProver's P + (x c) u, inner_product_prover.py:25-45,
 * without the caller first evaluating P): one multiexp over [u | g | h], served by the same table as bp_ipa_prove_hs. */
int bp_ipa_statement(const uint8_t* g64, const uint8_t* h64, const uint8_t u64_[64], const uint8_t* a32, const uint8_t* bs32,
                     const uint8_t c32[32], size_t n, uint8_t P_out64[64]);

/* Verifier1 + Verifier2 in one device pass (inner_product_verifier.py:44-58 on top of :127-147): additionally checks
 * P_new == P + xc*u and u_new == x*u with xc = x*c, x the Protocol-1 challenge; the Verifier2 equation then uses u_new, P_new */
int bp_ipa_verify1_eq_hs(const uint8_t* g64, const uint8_t* h64, const uint8_t* hscale32, const uint8_t u64_[64], const uint8_t P64[64],
                         const uint8_t xc32[32], const uint8_t x32[32], const uint8_t u_new64[64], const uint8_t P_new64[64], size_t n,
                         const uint8_t a32[32], const uint8_t b32[32], const uint8_t* xs32, const uint8_t* Ls64, const uint8_t* Rs64,
                         int* accept);

/* Verifier2.get_ss + the two multiexps of Verifier2.verify   inner_product_verifier.py:91-102,132-145
 * accept = 1 iff  MSM(g||h||u ; a*s || b*s^-1 || a*b) == P + MSM(Ls||Rs ; x^2 || x^-2).
 * (The transcript re-check, :104-125, is host string work done by the Python/C host layer.) */
int bp_ipa_verify_eq(const uint8_t* g64, const uint8_t* h64, const uint8_t u64_[64], const uint8_t P64[64], size_t n,
                     const uint8_t a32[32], const uint8_t b32[32], const uint8_t* xs32, const uint8_t* Ls64,
                     const uint8_t* Rs64, int* accept);

/* ---- batch verification of independent 64-bit (or n-bit) single-value range proofs ---------------
 * RangeVerifier.verify()                        src/rangeproofs/rangeproof_verifier.py:42-97
 * over `nproofs` proofs that share one generator set (gs, hs: n points each; g, h, u).
 * Packed proof record (little-endian scalars, 64-byte affine points), see INTEGRATION.md:
 *   V, A, S, T1, T2 (5 x 64) | taux, mu, t_hat (3 x 32) | u_new, P_new (2 x 64) | a, b (2 x 32)
 *   | xs (log2 n x 32) | Ls (log2 n x 64) | Rs (log2 n x 64)
 * transcripts: the three byte strings of each proof (range transcript, Protocol-1 transcript,
 * Protocol-2 transcript) concatenated; tr_off has 3*nproofs+1 entries.  start_transcript per proof.
 * accept[i] = 1/0 reproduces the reference's True / Exception("Proof invalid"); accept[i] = 2 marks
 * a non-numeric y/z/x slot (the reference raises ValueError from int(), rangeproof_verifier.py:49-53).
 * Host threads for the transcript checks: all cores, divided by LOCAL_WORLD_SIZE when several ranks share a node.
 * Development switches read from the environment: BP_VERIFY_CHUNK (proofs per chunk), BP_VERIFY_TIMING (host time per
 * chunk on stderr). */
int bp_rp_verify_batch(const uint8_t* gs64, const uint8_t* hs64, const uint8_t g64[64], const uint8_t h64[64],
                       const uint8_t u64_[64], size_t n, const uint8_t* proofs, size_t proof_stride, size_t nproofs,
                       const uint8_t* transcripts, const uint64_t* tr_off, const uint32_t* start_transcript,
                       uint8_t* accept);
size_t bp_rp_proof_stride(size_t n);
/* Proof-sharded form (SURVEY.md 8e, config 5): this rank verifies its block of `nproofs` proofs, then every rank's accept
 * bytes -- padded to `width` >= the largest block -- are all-gathered device to device (one ncclAllGather over NVLink, the
 * single exchange step) and copied out once: accept_all = nranks x width bytes, rank-major.  Needs bp_nccl_init for more
 * than one rank.  Every rank must call it (nproofs may be 0). */
int bp_rp_verify_batch_gather(const uint8_t* gs64, const uint8_t* hs64, const uint8_t g64[64], const uint8_t h64[64],
                              const uint8_t u64_[64], size_t n, const uint8_t* proofs, size_t proof_stride, size_t nproofs,
                              const uint8_t* transcripts, const uint64_t* tr_off, const uint32_t* start_transcript,
                              size_t width, uint8_t* accept_all);
/* Batch verification of AGGREGATED range proofs (m values x n bits each, n*m a power of two <= 2048) over one generator set:
 * the data-parallel form of AggregRangeVerifier(Vs_i, g, h, gs, hs, u, proof_i).verify() for every i
 * (/root/reference/src/rangeproofs/rangeproof_aggreg_verifier.py:42-108), same decisions; m = 1 is RangeVerifier.verify.
 * Record of one proof (little-endian scalars, 64-byte affine points), L = log2(n*m):
 *   V_0..V_{m-1} | A | S | T1 | T2 | taux | mu | t_hat | u_new | P_new | a | b | xs[L] | Ls[L] | Rs[L]      (bp_rp_aggreg_proof_stride bytes)
 * transcripts / tr_off / start_transcript and the accept bytes (1 accept, 0 reject, 2 = replay through the Python classes: the
 * reference would raise) as for bp_rp_verify_batch.  Host: transcript checks and every term scalar (OpenMP, csrc/rp_algebra.h);
 * device: generator terms from the set's byte table (bucket method until the set has one), proof-specific terms through the batched
 * bucket MSM, four exact identity checks per proof (csrc/bp_aggreg.inl). */
size_t bp_rp_aggreg_proof_stride(size_t n, size_t m);
int bp_rp_verify_aggreg_batch(const uint8_t* gs64, const uint8_t* hs64, const uint8_t g64[64], const uint8_t h64[64], const uint8_t u64_[64],
                              size_t n, size_t m, const uint8_t* proofs, size_t proof_stride, size_t nproofs, const uint8_t* transcripts,
                              const uint64_t* tr_off, const uint32_t* start_transcript, uint8_t* accept);
/* Batch verification by ONE random linear combination (csrc/bp_rlc.inl, csrc/rlc.cuh).  Inputs as for bp_rp_verify_aggreg_batch
 * (m = 1: the record of bp_rp_verify_batch, byte for byte).  Proof p's equations E1..E4 are weighted with rho_p^1..rho_p^4,
 * rho_p = SHA-256(seed32 || le64(p)) read little-endian, mod q (1 if that is 0), and summed; the sum is tested once.
 * A proof whose transcript checks give 0 or 2, or with a point off the curve / not canonical (accept byte 0), stays out of the sum.
 *   sum == identity: every proof in it is accepted, *combined = 1 (also for an empty batch or one in which no proof entered);
 *   otherwise:       *combined = 0 and accept holds the bytes of the exact verifier over the whole batch (bp_rp_verify_batch for
 *                    m = 1 and n <= 128, else bp_rp_verify_aggreg_batch).
 * Guarantee: the decisions equal the exact verifier's except with probability <= 4/q, PROVIDED seed32 is unpredictable to whoever
 * made the proofs -- draw it from a CSPRNG for every call.  A fixed or guessable seed lets an adversary craft invalid proofs whose
 * errors cancel in the sum (two proofs off by d and -d rho_0/rho_1 are then both accepted); the parameter exists for
 * reproducibility and tests.  seed32 = NULL is an error; so are a bad n*m, a short proof_stride and nproofs*(m + 6 + 2 log2(n m))
 * >= 2^31.  combined may be NULL. */
int bp_rp_verify_batch_rlc(const uint8_t* gs64, const uint8_t* hs64, const uint8_t g64[64], const uint8_t h64[64], const uint8_t u64_[64],
                           size_t n, size_t m, const uint8_t* proofs, size_t proof_stride, size_t nproofs, const uint8_t* transcripts,
                           const uint64_t* tr_off, const uint32_t* start_transcript, const uint8_t seed32[32],
                           uint8_t* accept, int* combined);
/* One random linear combination over a batch of MIXED shapes (csrc/bp_rlc.inl): proof p has n = ns[p] bits per value and
 * m = ms[p] values, N_p = ns[p]*ms[p] a power of two <= nset, and is checked against the prefixes gs[:N_p], hs[:N_p] of one set of
 * nset <= 2048 generators per side (gs64, hs64: nset points each) -- AggregRangeVerifier(Vs_p, g, h, gs[:N_p], hs[:N_p], u,
 * proof_p).verify(), with m = 1 RangeVerifier.  Records back to back in the caller's order, each bp_rp_aggreg_proof_stride(ns[p],
 * ms[p]) bytes (m = 1: the bp_rp_verify_batch record), proofs_bytes their sum; transcripts / tr_off / start_transcript and the
 * accept bytes as for bp_rp_verify_batch_rlc.  Weights rho_p as there, p the index in the caller's order; one sum over every proof
 * of every shape, tested once (all shapes' generator columns add into the 2 nset + 5 rows of the set, whose byte table is the one
 * bp_rp_verify_aggreg_batch / bp_rp_verify_batch_rlc build for n*m = nset).
 *   sum == identity: every proof in it is accepted, *combined = 1 (also for an empty batch);
 *   otherwise:       *combined = 0 and each shape is decided by the exact verifier over its prefix set (bp_rp_verify_batch for
 *                    m = 1 and n <= 128, else bp_rp_verify_aggreg_batch), the bytes in the caller's order.
 * Guarantee as for bp_rp_verify_batch_rlc: the decisions equal the exact verifier's except with probability <= 4/q, PROVIDED
 * seed32 is unpredictable to whoever made the proofs -- draw it from a CSPRNG for every call.  Errors: seed32 = NULL, nset > 2048,
 * a shape with N_p not a power of two or larger than nset, proofs_bytes not the sum of the record sizes, and
 * sum_p (m_p + 6 + 2 log2 N_p) >= 2^31.  combined may be NULL. */
int bp_rp_verify_mixed_rlc(const uint8_t* gs64, const uint8_t* hs64, const uint8_t g64[64], const uint8_t h64[64], const uint8_t u64_[64],
                           size_t nset, const uint32_t* ns, const uint32_t* ms, const uint8_t* proofs, size_t proofs_bytes,
                           size_t nproofs, const uint8_t* transcripts, const uint64_t* tr_off, const uint32_t* start_transcript,
                           const uint8_t seed32[32], uint8_t* accept, int* combined);
/* The random linear combination of bp_rp_verify_mixed_rlc, and when it fails, the invalid proofs LOCATED by sub-combinations
 * instead of the exact verifier over the whole batch (csrc/bp_rlc.inl, csrc/rlc.cuh).  Arguments as for bp_rp_verify_mixed_rlc
 * (a batch of one shape passes ns[p] = n, ms[p] = m for every p and nset = n*m), plus `leaf`.
 *   sum == identity: the result of bp_rp_verify_mixed_rlc, *combined = 1; no leaf work runs.
 *   otherwise:       *combined = 0.  The batch, in the order it is processed (grouped by shape, cut into chunks of 64 .. 2048
 *                    proofs of one shape), is cut into leaves of `leaf` consecutive proofs of one chunk (the last leaf of a chunk
 *                    may be shorter).  Each leaf's part of the weighted sum is tested on the device; the proofs of failing leaves
 *                    that entered the sum are decided by the exact verifier of their shape (bp_rp_verify_batch for m = 1 and
 *                    n <= 128, else bp_rp_verify_aggreg_batch), the others keep the byte of the combination (1).
 * Proofs settled before the sum (transcript verdict 0 or 2, a point off the curve or not canonical) keep that byte, which is the
 * exact verifier's.  leaf = 0 lets the library pick (the smallest power of two >= sqrt(512 nproofs^2 / sum_p n_p m_p), within
 * 8 .. 256); an explicit leaf places the boundaries for tests and is not a performance switch.
 * Guarantee: a rejection is exact.  When the whole sum fails, at least one leaf fails (the leaf sums add up to it).  The accept
 * bytes equal the exact verifier's except with probability <= 4 (K + 1)/q for K leaves, PROVIDED seed32 is unpredictable to whoever
 * made the proofs (as for bp_rp_verify_batch_rlc).  Errors: those of bp_rp_verify_mixed_rlc, leaf >= 2^32, and a leaf pass larger
 * than its 32-bit offsets (K (2 nset + 5) >= 2^30).  combined may be NULL. */
int bp_rp_verify_rlc_locate(const uint8_t* gs64, const uint8_t* hs64, const uint8_t g64[64], const uint8_t h64[64], const uint8_t u64_[64],
                            size_t nset, const uint32_t* ns, const uint32_t* ms, const uint8_t* proofs, size_t proofs_bytes,
                            size_t nproofs, const uint8_t* transcripts, const uint64_t* tr_off, const uint32_t* start_transcript,
                            const uint8_t seed32[32], size_t leaf, uint8_t* accept, int* combined);
/* the last bp_rp_verify_rlc_locate call: [0] leaf size used, [1] leaves (0: no leaf pass ran), [2] failing leaves, [3] proofs
 * of failing leaves that entered the sum, i.e. decided by the exact step (when every leaf fails, the exact verifier runs over the
 * whole batch as in bp_rp_verify_mixed_rlc; the settled proofs keep the bytes they had) */
int bp_rp_rlc_locate_stats(uint64_t out4[4]);
/* Batch PROVER (csrc/bp_prove.inl): AggregNIRangeProver(vs_p, n, g, h, gs, hs, gammas_p, u, secp256k1, seed_p).prove() for every
 * proof p (NIRangeProver when m = 1), byte for byte.  N = n*m a power of two <= 2048, gs64 / hs64 N points each.
 * values32, gammas32: nproofs*m scalars (32 bytes little-endian), proof-major, taken as the reference takes v.x / gamma.x: the
 * bits are (v >> i) & 1 for i < n (a value >= 2^n gives the same invalid proof as the per-proof prover), gamma is reduced mod q.
 * seeds: the proofs' transcript seeds back to back, proof p's at [seed_off[p], seed_off[p+1]) (nproofs + 1 offsets).  The blinding
 * factors derive from the seed alone, as in the reference: two proofs with the same seed share them.
 * Output = the input of bp_rp_verify_aggreg_batch / bp_rp_verify_batch_rlc:
 *   records: nproofs * bp_rp_aggreg_proof_stride(n, m) bytes, V_j = v_j g + gamma_j h first (m = 1: the bp_rp_verify_batch record);
 *   transcripts / tr_off (3 nproofs + 1 offsets) / start_transcript: each proof's range, Protocol-1 and Protocol-2 transcripts.
 * Errors: a bad n*m, and tr_cap smaller than the transcripts (*tr_len receives the bytes needed; records are complete).
 * nproofs = 0 does no device work.  Measurements through bp_rp_verify_stats. */
int bp_rp_prove_batch(const uint8_t* gs64, const uint8_t* hs64, const uint8_t g64[64], const uint8_t h64[64], const uint8_t u64_[64],
                      size_t n, size_t m, const uint8_t* values32, const uint8_t* gammas32, const uint8_t* seeds,
                      const uint64_t* seed_off, size_t nproofs, uint8_t* records, uint8_t* transcripts, size_t tr_cap,
                      size_t* tr_len, uint64_t* tr_off, uint32_t* start_transcript);
/* measurements of the last batch call, bp_rp_verify_batch or bp_rp_prove_batch: [0] wall ms, [1] host ms (transcript checks /
 * prover host steps, sum over chunks), [2] device span ms (CUDA events on the library stream: first chunk's first kernel .. last
 * kernel), [3] chunks, [4] host threads, [5] table mode (0 bucket method, 1 byte tables, 2 16-bit tables), [6] proofs */
int bp_rp_verify_stats(double out7[7]);

/* ---- host-side Fiat-Shamir helpers (exported for tests; src/utils/utils.py:84-111) -------------- */
int bp_mod_hash(const uint8_t* msg, size_t len, uint8_t out32[32]);            /* mod_hash(msg, q) */
/* out[i] = mod_hash(str(first + i) + suffix, q), i < count: the sL / sR blinding vectors
 * (src/rangeproofs/rangeproof_prover.py:48-55, rangeproof_aggreg_prover.py:53-60); host only */
int bp_mod_hash_indexed(const uint8_t* suffix, size_t len, uint32_t first, uint32_t count, uint8_t* out32);
int bp_sha256(const uint8_t* msg, size_t len, uint8_t out32[32]);              /* hashlib.sha256(msg).digest() */
int bp_sha256_set_portable(int on);   /* 1: force the portable compression function; returns the active one (1 = SHA-NI) */
int bp_point_to_b64(const uint8_t pt64[64], char out[45], size_t* out_len);    /* point_to_b64 */

/* ---- measurement --------------------------------------------------------------------------------
 * Times `iters` back-to-back resident MSMs with CUDA events on the library stream after `warmup`
 * untimed ones; between iterations an L2 flush (write of a 256 MiB buffer) runs outside the
 * timed events when flush_l2 != 0.  ms_each receives per-iteration milliseconds. */
int bp_bench_msm(bp_handle points, bp_handle scalars, size_t n, int warmup, int iters, int flush_l2, float* ms_each,
                 uint8_t out64[64]);
/* IMAD.WIDE.U32 issue-rate microbenchmark: returns measured 32x32+64 multiply-accumulates per
 * second (the roofline denominator of DESIGN.md) and the lane-ops executed. */
int bp_imad_peak(int iters, double* macs_per_s, float* ms);
/* other integer-pipe probes: mode 0 IMAD.WIDE.U32, 1 IMAD (32-bit), 2 carry-chained IMAD.WIDE.U32.X rows as
 * fp_mul issues them, 3 whole field multiplications (ops = fp_mul/s) */
int bp_pipe_probe(int mode, int iters, double* ops_per_s, float* ms);

/* ---- arithmetic self-test hooks (known-answer tests against big-int arithmetic) ------------------
 * fp: op 0 mul, 1 add, 2 sub, 3 inv, 4 neg  (inputs any 256-bit residue, output canonical)
 * ec: op 0 mixed add a+b, 1 full add, 2 double a, 3 negate a; +10 runs them on a re-projected a;
 *     op 4 coop_add(a, b), 5 coop_dbl(a): the 4-lane cooperative forms of csrc/coop4.cuh, one quad per pair (4n lanes, the last
 *     warp padded with identity pairs); +10 re-projects both operands
 * fq: op 0 mul, 1 add, 2 sub, 3 inv, 4 neg; on_device = 0 runs the same code on the host; 5 mul, 6 inv, 7 square through
 *     the device-only standard-form arithmetic of csrc/fqdev.cuh (on_device = 0: the portable forms) */
int bp_test_fp(int op, const uint8_t* a32, const uint8_t* b32, size_t n, uint8_t* out32);
int bp_test_ec(int op, const uint8_t* a64, const uint8_t* b64, size_t n, uint8_t* out64);
int bp_test_fq(int op, int on_device, const uint8_t* a32, const uint8_t* b32, size_t n, uint8_t* out32);
/* host F_p (csrc/fp_host.h): count <= 8 XYZZ points (128 bytes each) -> canonical affine, as the IPA prover's host step finishes L and R */
int bp_test_xyzz_to_affine_host(const uint8_t* xyzz128, size_t count, uint8_t* out64);
/* host sum of canonical affine points (64 zero bytes = identity): the rank partials of a sharded host-result MSM (csrc/fp_host.h) */
int bp_test_affine_sum_host(const uint8_t* pts64, size_t count, uint8_t out64[64]);
/* host Horner over the U window sums (XYZZ, 128 bytes each) of one MSM, as bp_msm finishes a host-result MSM (csrc/fp_host.h: horner_host);
   U = W + dbl, unit U-1 (and U-2 when dbl) the top window */
int bp_test_horner_host(const uint8_t* winsum128, int c, int W, int U, int dbl, uint8_t out64[64]);

/* ---- multi-GPU (one process per GPU) ---------------------------------------------------------------
 * NCCL communicator over the ranks of a torchrun job; `unique_id` is the 128-byte ncclUniqueId
 * produced by bp_nccl_unique_id on rank 0 and shared by the launcher's store. */
int bp_nccl_unique_id(uint8_t out128[128]);
int bp_nccl_init(int rank, int nranks, const uint8_t unique_id[128]);
/* slice [first, first+n) of a resident MSM on this rank, ncclAllGather of the XYZZ partials over
 * NVLink, every rank adds them and returns the same canonical affine point. */
int bp_msm_sharded(bp_handle points, bp_handle scalars, size_t first, size_t n, uint8_t out64[64]);
int bp_allgather_bytes(const uint8_t* send, size_t nbytes, uint8_t* recv);
/* same with this rank's slice in HOST buffers (H2D inside the call): the end-to-end form */
int bp_msm_sharded_host(const uint8_t* pts64, const uint8_t* sc32, size_t n, uint8_t out64[64]);
/* bp_bench_msm for the sharded path: the timed region of each iteration covers the slice MSM, the
 * all-gather and the R-way sum. */
int bp_bench_msm_sharded(bp_handle points, bp_handle scalars, size_t first, size_t n, int warmup, int iters, int flush_l2,
                         float* ms_each, uint8_t out64[64]);

/* ---- pinned host staging memory (cudaHostAlloc) for full-rate host<->device copies ------------------- */
void* bp_host_alloc(size_t bytes);
int bp_host_free(void* p);

#ifdef __cplusplus
}
#endif
#endif /* BP_GPU_H */
