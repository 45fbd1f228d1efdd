// ipa.cuh -- kernels for the inner-product-argument rounds and the scalar-multiplication batch.
//
// Replaces: the body of FastNIProver2.prove's while-loop
// (/root/reference/src/innerproduct/inner_product_prover.py:84-110) and the `hsp` list
// comprehension (/root/reference/src/rangeproofs/rangeproof_prover.py:77 and siblings).
//
// Device layout of one prover instance: points  P = [ u | g_0..g_{m-1} | h_0..h_{m-1} ]
// (affine, 64 B each), scalars a, b (32 B each, standard form, reduced).  Each round reads P, a, b
// of length m = 2k and writes the folded vectors of length k into the ping-pong twins.
#pragma once
#include "ec.cuh"
#include "fq.cuh"

namespace bp {

BP_DI Fq ld_fq(const Fq* p) {
  const uint4* q = reinterpret_cast<const uint4*>(p);
  uint4 a = q[0], b = q[1];
  Fq r; r.v[0] = a.x; r.v[1] = a.y; r.v[2] = a.z; r.v[3] = a.w; r.v[4] = b.x; r.v[5] = b.y; r.v[6] = b.z; r.v[7] = b.w;
  return r;
}
BP_DI void st_fq(Fq* p, const Fq& a) {
  uint4* q = reinterpret_cast<uint4*>(p);
  q[0] = make_uint4(a.v[0], a.v[1], a.v[2], a.v[3]);
  q[1] = make_uint4(a.v[4], a.v[5], a.v[6], a.v[7]);
}

// v[i] <- v[i] mod q  (inputs are ModP.x values that may be unreduced, SURVEY.md A.4)
__global__ void __launch_bounds__(128) k_reduce_scalars(Fq* __restrict__ v, u32 n) {
  u32 i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) st_fq(v + i, fq_reduce(ld_fq(v + i)));
}

// k * p, left-to-right double-and-add on the bits of k (k < q).  Lanes diverge on the add only.
BP_DI XYZZ scalar_mul_affine(const Affine& p, const Fq& k) {
  XYZZ acc = xyzz_identity();
  if (affine_is_identity(p)) return acc;
  for (int i = 255; i >= 0; i--) {
    acc = xyzz_dbl_ni(acc);
    if ((k.v[i >> 5] >> (i & 31)) & 1) xyzz_madd_ni(acc, p);
  }
  return acc;
}

// out[i] = sc[i] * pts[i]
__global__ void __launch_bounds__(64) k_scalar_mul(const Affine* __restrict__ pts, const Fq* __restrict__ sc, u32 n, Affine* __restrict__ out) {
  u32 i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  Fq k = fq_reduce(ld_fq(sc + i));
  Affine p = ld_affine(pts + i);
  st_affine(out + i, xyzz_to_affine(scalar_mul_affine(p, k)));
}

// sum of `count` XYZZ partials -> canonical affine (count is tiny: one per GPU)
__global__ void k_xyzz_sum(const XYZZ* __restrict__ in, u32 count, Affine* __restrict__ out) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  XYZZ acc = xyzz_identity();
  for (u32 i = 0; i < count; i++) { XYZZ v = ld_xyzz(in + i); xyzz_add_ni(acc, v); }
  st_affine(out, xyzz_to_affine(acc, true));
}

// Generator folding with a SHARED pair of scalars (divergence-free Shamir ladder):
//   i <  k : g'[i] = s_inv * g[i] + s * g[k+i]            inner_product_prover.py:107
//   i >= k : h'[j] = s * h[j] + s_inv * h[k+j], j = i-k   inner_product_prover.py:108
// src = [u | g (2k) | h (2k)], dst = [u | g' (k) | h' (k)]  (thread 2k copies u).
__global__ void __launch_bounds__(64) k_fold_points(const Affine* __restrict__ src, Affine* __restrict__ dst, u32 k, Fq s, Fq s_inv) {
  u32 i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i > 2 * k) return;
  if (i == 2 * k) { st_affine(dst, ld_affine(src)); return; }
  const bool is_h = i >= k;
  u32 j = is_h ? i - k : i;
  const Affine* base = src + 1 + (is_h ? 2 * k : 0);
  Affine lo = ld_affine(base + j), hi = ld_affine(base + k + j);
  Fq klo = is_h ? s : s_inv, khi = is_h ? s_inv : s;
  XYZZ acc = xyzz_identity();
  for (int b = 255; b >= 0; b--) {
    acc = xyzz_dbl_ni(acc);
    if ((klo.v[b >> 5] >> (b & 31)) & 1) xyzz_madd_ni(acc, lo);
    if ((khi.v[b >> 5] >> (b & 31)) & 1) xyzz_madd_ni(acc, hi);
  }
  st_affine(dst + 1 + (is_h ? k : 0) + j, xyzz_to_affine(acc));
}

// a'[i] = x*a[i] + xinv*a[k+i] ; b'[i] = xinv*b[i] + x*b[k+i]   (inner_product_prover.py:109-110)
// xm, xim = Montgomery forms of x, x^-1 so that fq_mont(v, xm) = v*x.
__global__ void __launch_bounds__(128) k_fold_scalars(const Fq* __restrict__ a, const Fq* __restrict__ b, u32 k, Fq xm, Fq xim,
                                                      Fq* __restrict__ a2, Fq* __restrict__ b2) {
  u32 i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= k) return;
  st_fq(a2 + i, fq_add(fq_mont(ld_fq(a + i), xm), fq_mont(ld_fq(a + k + i), xim)));
  st_fq(b2 + i, fq_add(fq_mont(ld_fq(b + i), xim), fq_mont(ld_fq(b + k + i), xm)));
}

// Builds the two (2k+1)-term MSMs of one round and their inner products:
//   c_L = <a_lo, b_hi>, c_R = <a_hi, b_lo>                          inner_product_prover.py:96-97
//   L   = MSM(g_hi || h_lo || u ; a_lo || b_hi || c_L)              :98
//   R   = MSM(g_lo || h_hi || u ; a_hi || b_lo || c_R)              :99
// One block of 256 threads.  term index t in [0, 2k+1) for L, + (2k+1) for R.
__global__ void __launch_bounds__(256) k_build_lr(const Fq* __restrict__ a, const Fq* __restrict__ b, u32 k, Fq* __restrict__ tsc,
                                                  u32* __restrict__ tidx) {
  __shared__ Fq sl[256], sr[256];
  const u32 n1 = 2 * k + 1;
  Fq accl = fq_zero(), accr = fq_zero();
  for (u32 i = threadIdx.x; i < k; i += 256) {
    Fq alo = ld_fq(a + i), ahi = ld_fq(a + k + i), blo = ld_fq(b + i), bhi = ld_fq(b + k + i);
    accl = fq_add(accl, fq_mont(alo, bhi));      // carries a factor R^-1, removed below
    accr = fq_add(accr, fq_mont(ahi, blo));
    // points live in [u | g (2k) | h (2k)]
    tsc[i] = alo;            tidx[i] = 1 + k + i;            // g_hi[i]
    tsc[k + i] = bhi;        tidx[k + i] = 1 + 2 * k + i;    // h_lo[i]
    tsc[n1 + i] = ahi;       tidx[n1 + i] = 1 + i;           // g_lo[i]
    tsc[n1 + k + i] = blo;   tidx[n1 + k + i] = 1 + 3 * k + i;   // h_hi[i]
  }
  sl[threadIdx.x] = accl; sr[threadIdx.x] = accr;
  __syncthreads();
  for (int off = 128; off > 0; off >>= 1) {
    if (threadIdx.x < off) {
      sl[threadIdx.x] = fq_add(sl[threadIdx.x], sl[threadIdx.x + off]);
      sr[threadIdx.x] = fq_add(sr[threadIdx.x], sr[threadIdx.x + off]);
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    tsc[2 * k] = fq_to_mont(sl[0]);  tidx[2 * k] = 0;            // (sum * R^-1) * R = sum ; point u
    tsc[n1 + 2 * k] = fq_to_mont(sr[0]);  tidx[n1 + 2 * k] = 0;
  }
}

// ---- prover rounds without materialising the folded generators -----------------------------------------------
// After j rounds the folded generator g^(j)_i is a fixed linear combination of the ORIGINAL generators,
//   g^(j)_i = sum over t = i (mod m) of cg[t] * g_t,   cg[t] = prod_{r<j} x_r^(+1 if t lay in the upper half at round r, else -1)
// (h likewise with inverted exponents, ch[t]), m = n / 2^j.  The round's commitments
//   L = <a_lo, g_hi> + <b_hi, h_lo> + c_L u,   R = <a_hi, g_lo> + <b_lo, h_hi> + c_R u     (inner_product_prover.py:96-99)
// are therefore two (n+1)-term multi-scalar multiplications over the original points with scalars a*cg / b*ch -- the
// same group elements as the reference computes, at the cost of one batched MSM per round and no 256-bit scalar
// multiplication per generator.  cg, ch are kept in Montgomery form; a, b in standard form.
// Point numbering of the terms: g_t -> g0 + t, h_t -> h0 + t, u -> iu.  A single proof's points are [u | g (n) | h (n)]
// = {1, 1 + n, 0}; a batch of range proofs addresses the rows of its generator set instead (bp_prove.inl).
struct IpaRows { u32 g0, h0, iu; };

// a'[t] = x*a[t] + xinv*a[m+t], b'[t] = xinv*b[t] + x*b[m+t] for t < m (inner_product_prover.py:109-110) and the coefficient
// update cg[t] *= (upper ? x : x^-1), ch[t] *= (upper ? x^-1 : x) for the generator fold (:107-108); m = new length, 2m = old.
BP_DI void ipa_fold_elem(Fq* __restrict__ a, Fq* __restrict__ b, Fq* __restrict__ cg, Fq* __restrict__ ch, u32 t, u32 m,
                         const Fq& xm, const Fq& xim) {
  const bool hi = (t % (2 * m)) >= m;
  st_fq(cg + t, fq_mont(ld_fq(cg + t), hi ? xm : xim));
  st_fq(ch + t, fq_mont(ld_fq(ch + t), hi ? xim : xm));
  if (t < m) {
    Fq alo = ld_fq(a + t), ahi = ld_fq(a + m + t), blo = ld_fq(b + t), bhi = ld_fq(b + m + t);
    st_fq(a + t, fq_add(fq_mont(alo, xm), fq_mont(ahi, xim)));
    st_fq(b + t, fq_add(fq_mont(blo, xim), fq_mont(bhi, xm)));
  }
}
// The L and R terms of original generator t (t < n) in a round of length m: slots [0, n/2) g-part, [n/2, n) h-part of
// each MSM, R at offset n + 1
BP_DI void ipa_lr_term(const Fq* __restrict__ a, const Fq* __restrict__ b, const Fq* __restrict__ cg, const Fq* __restrict__ ch,
                       u32 t, u32 n, u32 m, IpaRows rows, Fq* __restrict__ tsc, u32* __restrict__ tidx) {
  const u32 k = m >> 1, n1 = n + 1;
  const u32 i = t % m, blk = t / m;
  const bool hi = i >= k;
  const u32 slot = blk * k + (hi ? i - k : i);                 // position among the n/2 terms of its kind
  const Fq cgt = ld_fq(cg + t), cht = ld_fq(ch + t);
  if (hi) {
    st_fq(tsc + slot, fq_mont(ld_fq(a + i - k), cgt));              tidx[slot] = rows.g0 + t;              // L: a_lo[i-k] * g_t
    st_fq(tsc + n1 + n / 2 + slot, fq_mont(ld_fq(b + i - k), cht)); tidx[n1 + n / 2 + slot] = rows.h0 + t; // R: b_lo[i-k] * h_t
  } else {
    st_fq(tsc + n1 + slot, fq_mont(ld_fq(a + i + k), cgt));         tidx[n1 + slot] = rows.g0 + t;         // R: a_hi[i] * g_t
    st_fq(tsc + n / 2 + slot, fq_mont(ld_fq(b + i + k), cht));      tidx[n / 2 + slot] = rows.h0 + t;      // L: b_hi[i] * h_t
  }
}

// One block of 256 threads.  Points live in [u | g (n) | h (n)].
__global__ void __launch_bounds__(256) k_build_lr_sv(const Fq* __restrict__ a, const Fq* __restrict__ b, const Fq* __restrict__ cg,
                                                     const Fq* __restrict__ ch, u32 n, const u32* __restrict__ m_ptr, Fq* __restrict__ tsc,
                                                     u32* __restrict__ tidx) {
  __shared__ Fq sl[256], sr[256];
  const u32 m = *m_ptr;                                         // IpaRound::m (device resident, set per round)
  const u32 k = m >> 1, n1 = n + 1;
  Fq accl = fq_zero(), accr = fq_zero();
  for (u32 i = threadIdx.x; i < k; i += 256) {                 // c_L = <a_lo, b_hi>, c_R = <a_hi, b_lo>
    accl = fq_add(accl, fq_mont(ld_fq(a + i), ld_fq(b + k + i)));
    accr = fq_add(accr, fq_mont(ld_fq(a + k + i), ld_fq(b + i)));
  }
  for (u32 t = threadIdx.x; t < n; t += 256) ipa_lr_term(a, b, cg, ch, t, n, m, IpaRows{1, 1 + n, 0}, tsc, tidx);
  sl[threadIdx.x] = accl; sr[threadIdx.x] = accr;
  __syncthreads();
  for (int off = 128; off > 0; off >>= 1) {
    if (threadIdx.x < off) {
      sl[threadIdx.x] = fq_add(sl[threadIdx.x], sl[threadIdx.x + off]);
      sr[threadIdx.x] = fq_add(sr[threadIdx.x], sr[threadIdx.x + off]);
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    tsc[n] = fq_to_mont(sl[0]);       tidx[n] = 0;             // (sum * R^-1) * R ; point u
    tsc[n1 + n] = fq_to_mont(sr[0]);  tidx[n1 + n] = 0;
  }
}
// after the challenge: cg[t] *= (upper ? x : x^-1), ch[t] *= (upper ? x^-1 : x)   (xm, xim Montgomery forms)
__global__ void __launch_bounds__(128) k_update_coef(Fq* __restrict__ cg, Fq* __restrict__ ch, u32 n, u32 m, Fq xm, Fq xim) {
  u32 t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n) return;
  const bool hi = (t % m) >= (m >> 1);
  st_fq(cg + t, fq_mont(ld_fq(cg + t), hi ? xm : xim));
  st_fq(ch + t, fq_mont(ld_fq(ch + t), hi ? xim : xm));
}
// ---- graph-friendly forms: per-round values come from a device-resident parameter block, so that ONE captured CUDA
// graph (fold with the previous challenge -> build L/R terms -> batched MSM -> copy L, R out) is replayed every round.
struct IpaRound {
  u32 m;        // vector length of this round (after folding with the previous challenge)
  u32 fold;     // 1: first apply the previous round's challenge (xm, xim); 0: first round
  u32 pad0, pad1;
  Fq xm, xim;   // Montgomery forms of the previous challenge and its inverse
};
// a'[i] = x*a[i] + xinv*a[m+i], b'[i] = xinv*b[i] + x*b[m+i] in place (inner_product_prover.py:109-110) and the
// coefficient update of k_update_coef for the generator fold (:107-108); m = new length, 2m = old length.
__global__ void __launch_bounds__(128) k_round_fold(Fq* __restrict__ a, Fq* __restrict__ b, Fq* __restrict__ cg, Fq* __restrict__ ch, u32 n,
                                                    const IpaRound* __restrict__ rp) {
  if (!rp->fold) return;
  const u32 t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n) return;
  ipa_fold_elem(a, b, cg, ch, t, rp->m, ld_fq(&rp->xm), ld_fq(&rp->xim));
}
// One round's scalar work of one proof in ONE block: the fold with the previous challenge (fold), a block barrier, then the L/R
// terms with c_L, c_R (build = 1) or, after the last challenge, the copy-out of the final a, b (build = 0).  The u terms get
// c * umul R^-2: umul = R^2 gives c itself, x R^2 gives x c (terms over u when the proof's generator is u_new = x u).
BP_DI void ipa_round_block(Fq* __restrict__ a, Fq* __restrict__ b, Fq* __restrict__ cg, Fq* __restrict__ ch, u32 n, u32 m, bool fold,
                           const Fq& xm, const Fq& xim, int build, IpaRows rows, const Fq& umul, Fq* __restrict__ tsc,
                           u32* __restrict__ tidx, Fq* __restrict__ ab_out) {
  __shared__ Fq sl[32], sr[32];
  if (fold) {
    for (u32 t = threadIdx.x; t < n; t += blockDim.x) ipa_fold_elem(a, b, cg, ch, t, m, xm, xim);
    __syncthreads();                                           // the folded a, b, cg, ch are visible to the whole block
  }
  if (!build) {
    if (threadIdx.x == 0) { st_fq(ab_out, ld_fq(a)); st_fq(ab_out + 1, ld_fq(b)); __threadfence_system(); }
    return;
  }
  const u32 k = m >> 1, n1 = n + 1;
  Fq accl = fq_zero(), accr = fq_zero();
  for (u32 i = threadIdx.x; i < k; i += blockDim.x) {
    accl = fq_add(accl, fq_mont(ld_fq(a + i), ld_fq(b + k + i)));
    accr = fq_add(accr, fq_mont(ld_fq(a + k + i), ld_fq(b + i)));
  }
  for (u32 t = threadIdx.x; t < n; t += blockDim.x) ipa_lr_term(a, b, cg, ch, t, n, m, rows, tsc, tidx);
  // inner products: lane sums by shuffles, warp sums through shared memory
  const u32 lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  for (int off = 16; off > 0; off >>= 1) {
    Fq xl, xr;
#pragma unroll
    for (int i = 0; i < 8; i++) { xl.v[i] = __shfl_down_sync(0xFFFFFFFFu, accl.v[i], off); xr.v[i] = __shfl_down_sync(0xFFFFFFFFu, accr.v[i], off); }
    accl = fq_add(accl, xl); accr = fq_add(accr, xr);
  }
  if (lane == 0) { sl[warp] = accl; sr[warp] = accr; }
  __syncthreads();
  if (warp == 0) {
    accl = lane < nw ? sl[lane] : fq_zero(); accr = lane < nw ? sr[lane] : fq_zero();
    for (int off = 16; off > 0; off >>= 1) {
      Fq xl, xr;
#pragma unroll
      for (int i = 0; i < 8; i++) { xl.v[i] = __shfl_down_sync(0xFFFFFFFFu, accl.v[i], off); xr.v[i] = __shfl_down_sync(0xFFFFFFFFu, accr.v[i], off); }
      accl = fq_add(accl, xl); accr = fq_add(accr, xr);
    }
    if (lane == 0) {
      st_fq(tsc + n, fq_mont(accl, umul));       tidx[n] = rows.iu;        // (sum * R^-1) * umul * R^-1 ; point u
      st_fq(tsc + n1 + n, fq_mont(accr, umul));  tidx[n1 + n] = rows.iu;
    }
  }
}
// The latency-bound small proofs (n <= 4096): one round of one proof per launch.  rp and ab_out may live in mapped host
// memory: rp is read once into shared memory.
__global__ void __launch_bounds__(1024) k_ipa_round_prep(Fq* __restrict__ a, Fq* __restrict__ b, Fq* __restrict__ cg, Fq* __restrict__ ch, u32 n,
                                                         const IpaRound* __restrict__ rp, Fq* __restrict__ tsc, u32* __restrict__ tidx,
                                                         int build, Fq* __restrict__ ab_out) {
  __shared__ IpaRound s_rp;
  if (threadIdx.x < sizeof(IpaRound) / 4) ((u32*)&s_rp)[threadIdx.x] = ((const volatile u32*)rp)[threadIdx.x];
  __syncthreads();
  ipa_round_block(a, b, cg, ch, n, s_rp.m, s_rp.fold != 0, s_rp.xm, s_rp.xim, build, IpaRows{1, 1 + n, 0}, fq_const_r2(), tsc, tidx, ab_out);
}
// The same round for a batch of proofs of one length n, one block per proof (bp_rp_prove_batch).  Proof p owns a, b, cg, ch
// at p * n, its L/R terms at p * 2(n + 1), its final a, b at ab_out + 2p, and the Montgomery forms of its own previous
// challenge and inverse at xs[2p], xs[2p + 1].  Terms address the rows [gs | hs | g | h | u | ...] of the generator set, the u
// terms with c * x (umul = x R^2): the proof's u_new = x u is not a row.
__global__ void __launch_bounds__(256) k_ipa_round_batch(Fq* __restrict__ a, Fq* __restrict__ b, Fq* __restrict__ cg, Fq* __restrict__ ch,
                                                         u32 n, u32 m, int fold, const Fq* __restrict__ xs, int build, Fq umul,
                                                         Fq* __restrict__ tsc, u32* __restrict__ tidx, Fq* __restrict__ ab_out) {
  const size_t p = blockIdx.x;
  const Fq xm = fold ? ld_fq(xs + 2 * p) : fq_zero(), xim = fold ? ld_fq(xs + 2 * p + 1) : fq_zero();
  ipa_round_block(a + p * n, b + p * n, cg + p * n, ch + p * n, n, m, fold != 0, xm, xim, build, IpaRows{0, n, 2 * n + 2}, umul,
                  tsc + p * 2 * (n + 1), tidx + p * 2 * (n + 1), ab_out + 2 * p);
}
__global__ void __launch_bounds__(128) k_to_mont(Fq* __restrict__ v, u32 n) {
  u32 t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t < n) st_fq(v + t, fq_to_mont(fq_reduce(ld_fq(v + t))));
}
__global__ void __launch_bounds__(128) k_fill_one_mont(Fq* __restrict__ v, u32 n) {
  u32 t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t < n) st_fq(v + t, fq_const_r());
}

}  // namespace bp
