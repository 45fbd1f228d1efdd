// rlc.cuh -- device side of the batch verifier that checks ONE random linear combination of every proof's four equations
// (bp_rlc.inl).  Proof p's equations E1..E4 (bp_aggreg.inl) are weighted with w_e = rho_p^e and summed over the batch:
//   generator columns   gs_i  sum_p w4 a s_i
//                       hs_i  sum_p y^-i (w2 z^(2+j) 2^(i mod n) + w4 b s_{N-1-i})          j = i / n
//                       g     sum_p w1 (t_hat - delta)     h  sum_p (w1 taux - w2 mu)     u  sum_p x1 (w2 t_hat + w3)
//                       Gsum  sum_p -w2 z                  Hsum  sum_p w2 z
//   proof points        V_j -w1 z^(2+j) | T1 -w1 x | T2 -w1 x^2 | A w2 | S w2 x | P_new -(w2 + w4) | u_new w4 a b - w3
//                       | L_j -w4 x_j^2 | R_j -w4 x_j^-2
// k_rlc_prep (a warp per proof) gathers and curve-checks the proof's points, writes their scalars and a small table per proof;
// k_rlc_fold adds the tables' products into the 2N generator columns (a thread per column pair, proofs of a group from shared
// memory); k_rlc_colsum adds the groups in a fixed order (mod-q sums, no atomics: the result does not depend on scheduling) into
// the 2 nset + 5 columns of the generator set, of which a proof of N <= nset generators per side uses the prefixes gs[:N], hs[:N].
// Standard-form arithmetic of fqdev.cuh throughout.
#pragma once
#include "verify.cuh"
#include "svar.cuh"

namespace bp {

struct RlcShape {
  u32 n, m, N, L, hi, lo;      // N = n m = 2^L; s-vector and y^-i split as A[i >> lo] * B[i & (2^lo - 1)], hi = L - lo
  u32 nsc, npt, ts;            // scalar record (RS_* order of verify.cuh), points per proof, fold table per proof (Fq)
  u32 stride;                  // bytes per proof record on the device
  u32 oV, oA, oS, oT1, oT2, oUnew, oPnew, oLs, oRs;      // point offsets inside a record (bp_aggreg.inl: agg_offsets)
};
// fold table of one proof: [w4 a A : H] [w4 b A : H] [B : Bn] [y^-(k 2^lo) : H] [y^-l : Bn] [w2 z^(2+j) : m] [g, h, u, Gsum, Hsum]
BP_DI u32 rlc_oB(const RlcShape& s) { return 2u << s.hi; }
BP_DI u32 rlc_oAy(const RlcShape& s) { return (2u << s.hi) + (1u << s.lo); }
BP_DI u32 rlc_oBy(const RlcShape& s) { return (3u << s.hi) + (1u << s.lo); }
BP_DI u32 rlc_oGam(const RlcShape& s) { return (3u << s.hi) + (2u << s.lo); }
BP_DI u32 rlc_oCol(const RlcShape& s) { return rlc_oGam(s) + s.m; }

// gathered point t of a proof: V_0..V_{m-1}, T1, T2, A, S, P_new, u_new, L_0..L_{L-1}, R_0..R_{L-1}
BP_DI u32 rlc_point_off(const RlcShape& s, u32 t) {
  if (t < s.m) return s.oV + 64 * t;
  t -= s.m;
  if (t < 6) return t == 0 ? s.oT1 : t == 1 ? s.oT2 : t == 2 ? s.oA : t == 3 ? s.oS : t == 4 ? s.oPnew : s.oUnew;
  t -= 6;
  return t < s.L ? s.oLs + 64 * t : s.oRs + 64 * (t - s.L);
}

// 2^k mod q for k < 2^16: 2^(k mod 256) * (2^256)^(k / 256), 2^256 mod q = fq_const_r()
BP_DI Fq fq_pow2_dev(u32 k) {
  Fq t = fq_zero();
  t.v[(k & 255u) >> 5] = 1u << (k & 31u);
#pragma unroll 1
  for (u32 i = 0; i < (k >> 8); i++) t = fq_mul_ni(t, fq_const_r());
  return t;
}

// b^(lane+1) on every lane (product scan of b across the warp)
BP_DI Fq warp_pow_incl(const Fq& b, u32 lane) {
  Fq incl = b;
#pragma unroll 1
  for (int d = 1; d < 32; d <<= 1) {
    const Fq up = shfl_up_fq(incl, d);
    if ((int)lane >= d) incl = fq_mul_ni(incl, up);
  }
  return incl;
}
BP_DI Fq warp_pow_excl(const Fq& incl, u32 lane) {     // b^lane from warp_pow_incl's result
  const Fq e = shfl_up_fq(incl, 1);
  return lane == 0 ? fq_one() : e;
}
BP_DI Fq warp_sum_fq(Fq a) {                           // every lane gets the sum of all 32 lanes' values
#pragma unroll 1
  for (int off = 16; off > 0; off >>= 1) {
    Fq o;
#pragma unroll
    for (int i = 0; i < 8; i++) o.v[i] = __shfl_xor_sync(0xFFFFFFFFu, a.v[i], off);
    a = fq_add(a, o);
  }
  return a;
}

// One warp per proof.  rho[p] = 0 (the host's transcript checks did not pass) or a point off the curve (bad[p] = 1): the proof
// contributes nothing -- zero scalars, identity points, zero table.
__global__ void __launch_bounds__(128) k_rlc_prep(const uint8_t* __restrict__ rec, RlcShape s, u32 cn, const Fq* __restrict__ psc,
                                                  const Fq* __restrict__ inv, const Fq* __restrict__ rho, Affine* __restrict__ pts,
                                                  Fq* __restrict__ vsc, Fq* __restrict__ tabs, uint8_t* __restrict__ bad) {
  const u32 p = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (p >= cn) return;                                   // whole warps
  const uint8_t* R = rec + (size_t)p * s.stride;        // 32-byte aligned record, points at multiples of 32
  Affine* P = pts + (size_t)p * s.npt;
  Fq* VS = vsc + (size_t)p * s.npt;
  Fq* T = tabs + (size_t)p * s.ts;
  bool ok = true;
  for (u32 t = lane; t < s.npt; t += 32) ok = affine_on_curve(ld_affine(reinterpret_cast<const Affine*>(R + rlc_point_off(s, t)))) && ok;
  ok = __all_sync(0xFFFFFFFFu, ok);
  if (lane == 0) bad[p] = ok ? 0 : 1;
  const Fq r = ok ? ld_fq(rho + p) : fq_zero();
  if (fq_is_zero(r)) {
    Affine zp; zp.x = fp_zero(); zp.y = fp_zero();
    for (u32 t = lane; t < s.npt; t += 32) { st_affine(P + t, zp); st_fq(VS + t, fq_zero()); }
    for (u32 t = lane; t < s.ts; t += 32) st_fq(T + t, fq_zero());
    return;
  }
  for (u32 t = lane; t < s.npt; t += 32) st_affine(P + t, ld_affine(reinterpret_cast<const Affine*>(R + rlc_point_off(s, t))));
  const Fq* S = psc + (size_t)p * s.nsc;
  const Fq* IV = inv + (size_t)p * (s.L + 1);
  const Fq y = ld_fq(S + RS_Y), z = ld_fq(S + RS_Z), yi = ld_fq(IV);
  const Fq w1 = r, w2 = fq_mul_ni(r, r), w3 = fq_mul_ni(w2, r), w4 = fq_mul_ni(w2, w2);
  const u32 H = 1u << s.hi, Bn = 1u << s.lo;
  // z^(2+j): gamma_j = w2 z^(2+j) into the table, -w1 z^(2+j) on V_j; sum_j z^j for delta
  const Fq z2 = fq_mul_ni(z, z);
  Fq zsum = fq_zero();
  {
    const Fq zin = warp_pow_incl(z, lane);
    const Fq z32 = shfl_fq(zin, 31);
    const Fq g2 = fq_mul_ni(w2, z2), v1 = fq_neg(fq_mul_ni(w1, z2));
    Fq zj = warp_pow_excl(zin, lane);
    for (u32 j = lane; j < s.m; j += 32) {
      st_fq(T + rlc_oGam(s) + j, fq_mul_ni(g2, zj));
      st_fq(VS + j, fq_mul_ni(v1, zj));
      zsum = fq_add(zsum, zj);
      zj = fq_mul_ni(zj, z32);
    }
    zsum = warp_sum_fq(zsum);
  }
  // sum_{i<N} y^i = (sum_{k<H} y^(k 2^lo)) (sum_{l<Bn} y^l); the same split of y^-i goes into the table
  Fq sum_y;
  {
    const Fq yin = warp_pow_incl(y, lane);
    const Fq Y = shfl_fq(yin, (int)Bn - 1);                             // y^(2^lo)
    const Fq yl = warp_pow_excl(yin, lane);
    const Fq s1 = warp_sum_fq(lane < Bn ? yl : fq_zero());
    const Fq Yin = warp_pow_incl(Y, lane);
    const Fq Yl = warp_pow_excl(Yin, lane), Y32 = shfl_fq(Yin, 31);
    Fq part = lane < H ? Yl : fq_zero();
    if (lane + 32 < H) part = fq_add(part, fq_mul_ni(Yl, Y32));
    sum_y = fq_mul_ni(s1, warp_sum_fq(part));
    const Fq iin = warp_pow_incl(yi, lane);
    const Fq Yi = shfl_fq(iin, (int)Bn - 1);
    const Fq il = warp_pow_excl(iin, lane);
    if (lane < Bn) st_fq(T + rlc_oBy(s) + lane, il);
    const Fq Iin = warp_pow_incl(Yi, lane);
    const Fq Il = warp_pow_excl(Iin, lane), I32 = shfl_fq(Iin, 31);
    if (lane < H) st_fq(T + rlc_oAy(s) + lane, Il);
    if (lane + 32 < H) st_fq(T + rlc_oAy(s) + lane + 32, fq_mul_ni(Il, I32));
  }
  // s-vector half products (k_rp_expand): A over the top hi challenge bits (scaled by w4 a and by w4 b), B over the low lo bits
  const Fq a = ld_fq(S + RS_A), b = ld_fq(S + RS_B);
  {
    const Fq alpha = fq_mul_ni(w4, a), beta = fq_mul_ni(w4, b);
    for (u32 idx = lane; idx < H; idx += 32) {
      Fq acc = fq_one();
      for (u32 j = 0; j < s.hi; j++) {
        const bool bit = (idx >> (s.hi - 1 - j)) & 1u;
        acc = fq_mul_ni(acc, bit ? ld_fq(S + RS_XS + j) : ld_fq(IV + 1 + j));
      }
      st_fq(T + idx, fq_mul_ni(alpha, acc));
      st_fq(T + H + idx, fq_mul_ni(beta, acc));
    }
    if (lane < Bn) {
      Fq acc = fq_one();
      for (u32 j = 0; j < s.lo; j++) {
        const bool bit = (lane >> (s.lo - 1 - j)) & 1u;
        acc = fq_mul_ni(acc, bit ? ld_fq(S + RS_XS + s.hi + j) : ld_fq(IV + 1 + s.hi + j));
      }
      st_fq(T + rlc_oB(s) + lane, acc);
    }
  }
  if (lane < s.L) {
    const Fq xj = ld_fq(S + RS_XS + lane), xij = ld_fq(IV + 1 + lane);
    st_fq(VS + s.m + 6 + lane, fq_neg(fq_mul_ni(w4, fq_mul_ni(xj, xj))));
    st_fq(VS + s.m + 6 + s.L + lane, fq_neg(fq_mul_ni(w4, fq_mul_ni(xij, xij))));
  }
  if (lane == 0) {
    const Fq x = ld_fq(S + RS_X), x1 = ld_fq(S + RS_X1), that = ld_fq(S + RS_THAT), taux = ld_fq(S + RS_TAUX), mu = ld_fq(S + RS_MU);
    // delta = (z - z^2) sum y^i - z^3 (2^n - 1) sum_{j<m} z^j                                 rangeproof_aggreg_verifier.py:72-79
    const Fq tn1 = fq_sub(fq_pow2_dev(s.n), fq_one());
    const Fq delta = fq_sub(fq_mul_ni(fq_sub(z, z2), sum_y), fq_mul_ni(fq_mul_ni(fq_mul_ni(z2, z), zsum), tn1));
    const Fq w2z = fq_mul_ni(w2, z), w1x = fq_mul_ni(w1, x);
    Fq* C = T + rlc_oCol(s);
    st_fq(C + 0, fq_mul_ni(w1, fq_sub(that, delta)));                                    // g
    st_fq(C + 1, fq_sub(fq_mul_ni(w1, taux), fq_mul_ni(w2, mu)));                        // h
    st_fq(C + 2, fq_mul_ni(x1, fq_add(fq_mul_ni(w2, that), w3)));                        // u
    st_fq(C + 3, fq_neg(w2z));                                                           // Gsum
    st_fq(C + 4, w2z);                                                                   // Hsum
    Fq* V = VS + s.m;
    st_fq(V + 0, fq_neg(w1x));                                                           // T1
    st_fq(V + 1, fq_neg(fq_mul_ni(w1x, x)));                                             // T2
    st_fq(V + 2, w2);                                                                    // A
    st_fq(V + 3, fq_mul_ni(w2, x));                                                      // S
    st_fq(V + 4, fq_neg(fq_add(w2, w4)));                                                // P_new
    st_fq(V + 5, fq_sub(fq_mul_ni(w4, fq_mul_ni(a, b)), w3));                            // u_new
  }
}

// part[grp][0, N) = gs columns, [N, 2N) = hs columns, [2N, 2N+5) = g, h, u, Gsum, Hsum of the G proofs of group grp.  A thread
// owns generator position i (its gs and its hs column): per proof 1 + 4 multiplications, sums in registers.
// spread != 0 (proofs shorter than the set, N < nset): the set's Gsum / Hsum rows sum more generators than the proof uses, so
// each proof's -w2 z and w2 z go into its own N gs / hs columns instead and the Gsum / Hsum entries of part are 0.
__global__ void __launch_bounds__(128) k_rlc_fold(const Fq* __restrict__ tabs, RlcShape s, u32 cn, u32 G, u32 spread, Fq* __restrict__ part) {
  extern __shared__ Fq smt[];
  const u32 grp = blockIdx.y, p0 = grp * G, np = cn - p0 < G ? cn - p0 : G;
  {
    const uint4* src = reinterpret_cast<const uint4*>(tabs + (size_t)p0 * s.ts);
    uint4* dst = reinterpret_cast<uint4*>(smt);
    for (u32 k = threadIdx.x; k < 2 * np * s.ts; k += blockDim.x) dst[k] = src[k];
  }
  __syncthreads();
  const u32 F = 2 * s.N + 5, H = 1u << s.hi, mask = (1u << s.lo) - 1u;
  Fq* out = part + (size_t)grp * F;
  const u32 i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < s.N) {
    const u32 j = i / s.n, c = s.N - 1 - i;
    const Fq t2k = fq_pow2_dev(i - j * s.n);
    const u32 ih = i >> s.lo, il = i & mask, chi = c >> s.lo, clo = c & mask;
    const u32 oB = rlc_oB(s), oAy = rlc_oAy(s), oBy = rlc_oBy(s), oG = rlc_oGam(s) + j;
    Fq accG = fq_zero(), accH = fq_zero();
#pragma unroll 1
    for (u32 q = 0; q < np; q++) {
      const Fq* T = smt + (size_t)q * s.ts;
      accG = fq_add(accG, fq_mul_dev(ld_fq(T + ih), ld_fq(T + oB + il)));                                   // w4 a s_i
      const Fq v = fq_add(fq_mul_dev(ld_fq(T + oG), t2k), fq_mul_dev(ld_fq(T + H + chi), ld_fq(T + oB + clo)));  // w2 z^(2+j) 2^k + w4 b s_{N-1-i}
      accH = fq_add(accH, fq_mul_dev(fq_mul_dev(ld_fq(T + oAy + ih), ld_fq(T + oBy + il)), v));               // times y^-i
      if (spread) {
        accG = fq_add(accG, ld_fq(T + rlc_oCol(s) + 3));                                                   // -w2 z
        accH = fq_add(accH, ld_fq(T + rlc_oCol(s) + 4));                                                   // w2 z
      }
    }
    st_fq(out + i, accG);
    st_fq(out + s.N + i, accH);
  }
  if (blockIdx.x == 0 && threadIdx.x < 5) {
    Fq acc = fq_zero();
    if (!spread || threadIdx.x < 3)
      for (u32 q = 0; q < np; q++) acc = fq_add(acc, ld_fq(smt + (size_t)q * s.ts + rlc_oCol(s) + threadIdx.x));
    st_fq(out + 2 * s.N + threadIdx.x, acc);
  }
}

// col[set column of c] += sum over the groups of part[grp][c], groups in order.  part has the 2N + 5 columns of a proof of N
// generators per side, col the 2 nset + 5 of the set: gs_i stays at i, hs_i goes to nset + i, the five tail columns to 2 nset + k.
__global__ void __launch_bounds__(128) k_rlc_colsum(const Fq* __restrict__ part, u32 ngroups, u32 N, u32 nset, Fq* __restrict__ col) {
  const u32 F = 2 * N + 5, c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= F) return;
  const u32 dst = c < N ? c : c < 2 * N ? nset + (c - N) : 2 * nset + (c - 2 * N);
  Fq acc = ld_fq(col + dst);
  for (u32 k = 0; k < ngroups; k++) acc = fq_add(acc, ld_fq(part + (size_t)k * F + c));
  st_fq(col + dst, acc);
}

// out[0] = 1 if the XYZZ partials (one per chunk, then the generator MSM) add up to the identity
__global__ void k_rlc_final(const XYZZ* __restrict__ parts, u32 nparts, uint8_t* __restrict__ out) {
  if (threadIdx.x != 0) return;
  XYZZ acc = xyzz_identity();
  for (u32 k = 0; k < nparts; k++) { XYZZ v = ld_xyzz(parts + k); xyzz_add_ni(acc, v); }
  out[0] = xyzz_is_identity(acc) ? 1 : 0;
}

// Leaf pass of bp_rp_verify_rlc_locate (bp_rlc.inl): a leaf is a run of consecutive proofs of one chunk made of whole fold groups,
// leaf[k] = {offset of its first group's partials in part, its groups, N of its shape}.  A thread per (leaf k, set column c):
// cols[k F + c] = the leaf's partials of the part column that k_rlc_colsum maps to c, groups in order (fixed order, no atomics);
// offs[k] = k F (the leaves' generator MSMs end to end, F = 2 nset + 5); rows[k F + c] = c (the generator row of every term).
__global__ void __launch_bounds__(128) k_rlc_leaf_cols(const Fq* __restrict__ part, const uint4* __restrict__ leaf, u32 K, u32 nset,
                                                       Fq* __restrict__ cols, u32* __restrict__ offs, u32* __restrict__ rows) {
  const u32 F = 2 * nset + 5;
  const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (size_t)K * F) return;
  const u32 k = (u32)(t / F), c = (u32)(t - (size_t)k * F);
  const uint4 d = leaf[k];
  const u32 N = d.z, FN = 2 * N + 5;
  const u32 pc = c < nset ? (c < N ? c : FN) : c < 2 * nset ? (c - nset < N ? N + (c - nset) : FN) : 2 * N + (c - 2 * nset);
  Fq acc = fq_zero();
  if (pc < FN)
    for (u32 q = 0; q < d.y; q++) acc = fq_add(acc, ld_fq(part + d.x + (size_t)q * FN + pc));
  st_fq(cols + t, acc);
  rows[t] = c;
  if (c == 0) offs[k] = k * F;
  if (t == 0) offs[K] = K * F;
}

// out[k] = 1 if leaf k's generator part and proof-point part add up to the identity
__global__ void __launch_bounds__(128) k_rlc_leaf_test(const XYZZ* __restrict__ gen, const XYZZ* __restrict__ pts, u32 K,
                                                       uint8_t* __restrict__ out) {
  const u32 k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= K) return;
  XYZZ a = ld_xyzz(gen + k);
  const XYZZ b = ld_xyzz(pts + k);
  xyzz_add_ni(a, b);
  out[k] = xyzz_is_identity(a) ? 1 : 0;
}

}  // namespace bp
