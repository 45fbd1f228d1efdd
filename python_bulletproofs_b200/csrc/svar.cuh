// svar.cuh -- the proof-specific ("variable-base") terms of the batch verifier: per proof the 5 + 2 log2(n) points that
// carry a full 256-bit scalar (V, T1, T2 | S | u_new, L_j, R_j) and the unit-scalar terms (A, -P_new, -u_new) of the four
// equations of verify.cuh.
//
// Replaces, per proof, the proof-dependent part of the reference's multiexps: z^2*V + x*T1 + x^2*T2
// (/root/reference/src/rangeproofs/rangeproof_verifier.py:73-76), A + x*S (:78, :88-97), (a*b)*u_new and
// MSM(Ls || Rs ; x_j^2 || x_j^-2) (/root/reference/src/innerproduct/inner_product_verifier.py:134-143).
//
// Round 1 sent these 21 terms per proof through the bucket pipeline (four bucket reductions and four Horner chains per proof,
// 3.07 ms per 4096 proofs against 1.63 ms for the 202 generator terms).  Here they are evaluated window-parallel:
//   k_sv_table  one thread per (proof, point): curve check, 2P..8P (XYZZ), GLV split + signed 4-bit recoding of its scalar
//   k_sv_main   one WARP per proof, lane = 4-bit window position w of the 128-bit GLV halves: for every sub-term one table
//               read + one addition per lane, no doublings:  A_w = sum_i d_{i,w} * P_i   (per equation)
//   k_sv_comb1  one thread per (proof, equation, 8 windows): Horner with 4 doublings per step
//   k_sv_comb2  one thread per (proof, equation): the remaining 96 doublings (Jacobian doubling chains), plus the
//               unit-scalar terms; result = the variable part of "MSM == identity", added to the table part by k_rp_fold
// Work per 64-bit proof: 119 table operations, ~1020 additions, 624 doublings -- 0.6 of the bucket pass's multiplications and
// no latency chain longer than 96 doublings.
#pragma once
#include "ec.cuh"
#include "fq.cuh"
#include "glv.cuh"
#include "coop4.cuh"
#include "verify.cuh"
#include "msm.cuh"

namespace bp {

#define BP_SV_ENT 7                      // table entries per variable point: 2P .. 8P (P itself is read from the point array)
#define BP_SV_NONE 0xFFFFFFFFu

// variable term order: 0 V, 1 T1, 2 T2 (E1) | 3 S (E2) | 4 u_new, 5.. L_j, 5+L.. R_j (E4)
BP_DI u32 sv_slot(u32 v) { return v == 0 ? (u32)RP_V : v == 1 ? (u32)RP_T1 : v == 2 ? (u32)RP_T2 : v == 3 ? (u32)RP_S : v == 4 ? (u32)RP_UNEW : (u32)RP_LS + (v - 5); }
BP_DI u32 sv_term(u32 slot) {
  return slot == RP_V ? 0u : slot == RP_T1 ? 1u : slot == RP_T2 ? 2u : slot == RP_S ? 3u : slot == RP_UNEW ? 4u
       : slot >= RP_LS ? 5u + (slot - RP_LS) : BP_SV_NONE;
}

// on-curve test of a proof-supplied point: the identity (64 zero bytes) is a group element; anything else must be canonical
// (x, y < p) and satisfy y^2 = x^3 + 7.  fastecdsa's Point constructor raises for such coordinates, so a reference verifier
// can never be handed one; the C ABI rejects the proof.
BP_DI bool affine_on_curve(const Affine& P) {
  if (affine_is_identity(P)) return true;
  const Fp xc = fp_canon(P.x), yc = fp_canon(P.y);
  bool ok = true;
#pragma unroll
  for (int i = 0; i < 8; i++) ok = ok && xc.v[i] == P.x.v[i] && yc.v[i] == P.y.v[i];
  Fp seven = fp_zero(); seven.v[0] = 7;
  const Fp rhs = fp_add(fp_mul(fp_sqr(P.x), P.x), seven);
  return ok && fp_is_zero(fp_sub(fp_sqr(P.y), rhs));
}

// bucket-method path of the batch verifier: the curve check on its own
__global__ void __launch_bounds__(128) k_rp_check_points(const Affine* __restrict__ pts, u32 npt, u32 cn, uint8_t* __restrict__ bad) {
  const u32 t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= cn * npt) return;
  if (!affine_on_curve(ld_affine(pts + t))) bad[t / npt] = 1;
}

// Montgomery's trick across a warp: every lane receives the inverse of its own `acc` (all non-zero mod p) -- two shuffle scans
// and ONE binary-GCD inversion by lane 31, which runs on the ALU pipe while the other warps of the SM keep the multiplier busy
BP_DI Fp warp_batch_inverse(const Fp& acc, u32 lane) {
  Fp S = acc, T = acc;                       // inclusive prefix / suffix products over the lanes
#pragma unroll 1
  for (int off = 1; off < 32; off <<= 1) {
    const Fp a = shfl_up_fp(S, off), b = shfl_down_fp(T, off);
    const bool up = lane >= (u32)off;        // S <- S * S[lane - off]   else   T <- T * T[lane + off]: both scans share one multiplier site
    const Fp x = fp_mul(S, a);
    const Fp y = fp_mul(T, b);
    if (up) S = x;
    if (lane + (u32)off < 32u) T = y;
  }
  Fp inv = fp_zero();
  if (lane == 31) inv = fp_inv_gcd(S);       // 1 / (product of all 32)
  inv = shfl_fp(inv, 31);
  Fp Sm = shfl_up_fp(S, 1), Tp = shfl_down_fp(T, 1);
  if (lane == 0) Sm = fp_one();
  if (lane == 31) Tp = fp_one();
  return fp_mul(fp_mul(Sm, Tp), inv);        // 1/acc_l = (acc_0 .. acc_{l-1}) * (acc_{l+1} .. acc_31) / total
}

// One thread per (proof, point slot).  pts = the chunk's proof points (npt per proof), vsc = its variable scalars (nv per proof,
// written by k_rp_expand).  bad[] must be zeroed beforehand.  var_e3[p] receives -u_new (the whole variable part of E3).
// The multiples 2P .. 8P leave the kernel in AFFINE form (T: 64 bytes per entry), so that k_sv_main's ~1300 additions per proof
// are mixed additions (8M + 2S instead of 12M + 2S): the chain is built in XYZZ (parked in `scr`, with the prefix products of the
// ZZZ values in `pre`), the product of a thread's seven ZZZ is inverted together with those of the 31 other lanes
// (warp_batch_inverse above: two shuffle scans, one binary GCD per warp) and the thread walks back through its entries
// (Montgomery's trick).  No thread leaves before the shared inversion; threads without a table contribute 1.
__global__ void __launch_bounds__(128) k_sv_table(const Affine* __restrict__ pts, RpLayout lay, u32 cn, const Fq* __restrict__ vsc,
                                                  Affine* __restrict__ T, XYZZ* scr, Fp* pre, uint4* __restrict__ kd, u32* __restrict__ kflags,
                                                  uint8_t* __restrict__ bad, XYZZ* __restrict__ var_e3) {
  const u32 t = blockIdx.x * blockDim.x + threadIdx.x, lane = threadIdx.x & 31;
  const bool in_range = t < cn * lay.npt;
  const u32 p = in_range ? t / lay.npt : 0u, slot = in_range ? t % lay.npt : 0u, nv = 5 + 2 * lay.L;
  Affine P; P.x = fp_zero(); P.y = fp_zero();
  if (in_range) P = ld_affine(pts + t);
  const bool ok = affine_on_curve(P);
  if (in_range && !ok) bad[p] = 1;
  const bool ident = affine_is_identity(P) || !ok;         // (a rejected proof's garbage never enters the formulas)
  if (in_range && slot == RP_UNEW) {
    XYZZ e = xyzz_identity();
    if (!ident) { e.X = P.x; e.Y = fp_neg(P.y); e.ZZ = fp_one(); e.ZZZ = fp_one(); }
    st_xyzz(var_e3 + p, e);
  }
  const u32 v = in_range ? sv_term(slot) : BP_SV_NONE;
  const bool var = v != BP_SV_NONE;
  const size_t idx = (size_t)p * nv + (var ? v : 0u);
  if (var) {
    // k = k1 + k2*lambda, |k_i| < 2^128; signed 4-bit digits d_w = nibble_w(|k_i| + 0x0888..8) - 8 for w < 31 (in [-8, 7]) and the
    // top window unrecoded, d_31 = (|k_i| + 0x0888..8) >> 124 in [0, 16]
    Fq k = fq_reduce(ld_fq(vsc + idx)), m[2];
    bool neg[2];
    glv_split(k, m[0], neg[0], m[1], neg[1]);
    u32 flags = (neg[0] ? 1u : 0u) | (neg[1] ? 2u : 0u);
#pragma unroll
    for (int h = 0; h < 2; h++) {
      const u32 C[4] = {0x88888888u, 0x88888888u, 0x88888888u, 0x08888888u};
      u32 r[4];
      u64 cy = 0;
#pragma unroll
      for (int i = 0; i < 4; i++) { cy += (u64)m[h].v[i] + C[i]; r[i] = (u32)cy; cy >>= 32; }
      if (cy) flags |= 4u << h;
      kd[2 * idx + h] = make_uint4(r[0], r[1], r[2], r[3]);
    }
    kflags[idx] = flags;
  }
  const bool tab = var && !ident;
  Affine* out = T + idx * BP_SV_ENT;
  XYZZ* sc = scr + idx * BP_SV_ENT;
  Fp* pr = pre + idx * BP_SV_ENT;
  Fp prod = fp_one();
  if (var && ident) {
    Affine z; z.x = fp_zero(); z.y = fp_zero();
    for (int j = 0; j < BP_SV_ENT; j++) st_affine(out + j, z);
  }
  if (tab) {
    XYZZ acc = xyzz_mdbl(P);
#pragma unroll 1
    for (int j = 0; j < BP_SV_ENT; j++) {
      if (j) xyzz_madd_ni(acc, P);
      st_xyzz(sc + j, acc);
      st_fp(pr + j, prod);                                 // ZZZ_0 .. ZZZ_{j-1}
      prod = fp_mul(prod, acc.ZZZ);                        // (never zero: jP, j <= 8, of a point of prime order)
    }
  }
  Fp inv = warp_batch_inverse(prod, lane);                 // 1 / (ZZZ_0 .. ZZZ_6) of this thread
  if (!tab) return;
#pragma unroll 1
  for (int j = BP_SV_ENT - 1; j >= 0; j--) {
    XYZZ e;
    e.X = ld_fp_plain(&sc[j].X); e.Y = ld_fp_plain(&sc[j].Y); e.ZZ = ld_fp_plain(&sc[j].ZZ); e.ZZZ = ld_fp_plain(&sc[j].ZZZ);
    const Fp zi3 = fp_mul(inv, ld_fp_plain(pr + j));       // ZZZ_j^-1
    inv = fp_mul(inv, e.ZZZ);
    const Fp zi2 = fp_mul(fp_sqr(e.ZZ), fp_sqr(zi3));      // ZZ^-1 = ZZ^2 * ZZZ^-2
    Affine a;
    a.x = fp_mul(e.X, zi2); a.y = fp_mul(e.Y, zi3);
    st_affine(out + j, a);
  }
}

// One warp per proof; lane = window.  Aw[(p*3 + e)*32 + w] = sum over the sub-terms of equation e (0: E1, 1: E2, 2: E4) of
// digit_w * (P or phi(P)).
__global__ void __launch_bounds__(128, 4) k_sv_main(const Affine* __restrict__ pts, RpLayout lay, u32 cn, const Affine* __restrict__ T,
                                                    const uint4* __restrict__ kd, const u32* __restrict__ kflags, XYZZ* __restrict__ Aw) {
  const u32 p = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (p >= cn) return;                                    // whole warps
  const u32 nv = 5 + 2 * lay.L;
  const Fp beta = {BP_BETA_LIMBS};
#pragma unroll 1
  for (u32 eq = 0; eq < 3; eq++) {
    const u32 v0 = eq == 0 ? 0u : (eq == 1 ? 3u : 4u), v1 = eq == 0 ? 3u : (eq == 1 ? 4u : nv);
    XYZZ acc = xyzz_identity();
#pragma unroll 1
    for (u32 s = 2 * v0; s < 2 * v1; s++) {                // sub-term (v, half)
      __syncwarp();
      const u32 v = s >> 1, h = s & 1u;
      const size_t idx = (size_t)p * nv + v;
      const uint4 kk = __ldg(kd + 2 * idx + h);
      const u32 fl = __ldg(kflags + idx);
      const u32 limb = lane < 8 ? kk.x : (lane < 16 ? kk.y : (lane < 24 ? kk.z : kk.w));
      const u32 nib = (limb >> (4 * (lane & 7u))) & 15u;
      const int d = lane < 31 ? (int)nib - 8 : (int)(nib + (((fl >> (2 + h)) & 1u) << 4));
      const bool neg = (((fl >> h) & 1u) != 0u) != (d < 0);
      const u32 mag = d < 0 ? (u32)(-d) : (u32)d;
      const u32 m0 = mag > 8u ? 8u : 0u, m1 = mag - m0;    // only the top window can exceed 8: two additions there
      const bool any0 = __any_sync(BP_FULL_MASK, m0 != 0u);
#pragma unroll 1
      for (int rep = any0 ? 0 : 1; rep < 2; rep++) {
        const u32 mm = rep == 0 ? m0 : m1;
        if (mm == 0u) continue;
        Affine e = ld_affine(mm == 1u ? pts + (size_t)p * lay.npt + sv_slot(v) : T + idx * BP_SV_ENT + (mm - 2u));
        if (h) e.x = fp_mul(e.x, beta);                    // phi(x, y) = (beta x, y)
        if (neg) e.y = fp_neg(e.y);
        xyzz_madd(acc, e);
      }
    }
    st_xyzz(Aw + ((size_t)p * 3 + eq) * 32 + lane, acc);
  }
}

// ---- doubling chains in Jacobian coordinates -----------------------------------------------------------------------------
// The tails below are chains of doublings with an occasional addition.  A Jacobian doubling on a = 0 (dbl-2009-l) costs
// 2M + 5S = 369 IMAD.WIDE against 6M + 3S = 567 for the XYZZ doubling, and the change of coordinates is cheap:
//   XYZZ (X, Y, ZZ, ZZZ) -> Jacobian (X*ZZ, Y*ZZZ, ZZ)      [x = X*ZZ/ZZ^2, y = Y*ZZZ/ZZ^3 with ZZ^3 = ZZZ^2]        2M
//   Jacobian (X, Y, Z)   -> XYZZ (X, Y, Z^2, Z^3)                                                                     1M + 1S
struct Jac { Fp X, Y, Z; };
BP_DI Jac jac_from_xyzz(const XYZZ& p) { Jac r; r.X = fp_mul(p.X, p.ZZ); r.Y = fp_mul(p.Y, p.ZZZ); r.Z = p.ZZ; return r; }
BP_DI XYZZ xyzz_from_jac(const Jac& p) { XYZZ r; r.X = p.X; r.Y = p.Y; r.ZZ = fp_sqr(p.Z); r.ZZZ = fp_mul(r.ZZ, p.Z); return r; }
BP_DI Jac jac_dbl(const Jac& p) {          // the identity (Z = 0) stays the identity
  Jac r;
  const Fp A = fp_sqr(p.X), B = fp_sqr(p.Y), C = fp_sqr(B);
  const Fp XB = fp_add(p.X, B);
  const Fp D = fp_dbl(fp_sub(fp_sub(fp_sqr(XB), A), C));
  const Fp E = fp_add(fp_dbl(A), A);
  const Fp F = fp_sqr(E);
  r.X = fp_sub(F, fp_dbl(D));
  r.Y = fp_sub(fp_mul(E, fp_sub(D, r.X)), fp_dbl(fp_dbl(fp_dbl(C))));
  r.Z = fp_dbl(fp_mul(p.Y, p.Z));
  return r;
}
// 2^k * p
__device__ __noinline__ XYZZ xyzz_dbl_k(const XYZZ& p, int k) {
  Jac j = jac_from_xyzz(p);
#pragma unroll 1
  for (int d = 0; d < k; d++) j = jac_dbl(j);
  return xyzz_from_jac(j);
}

// One thread per (proof, equation, group of 8 windows): G = sum_{j<8} 16^j A_{8g+j}
__global__ void __launch_bounds__(128) k_sv_comb1(const XYZZ* __restrict__ Aw, u32 total, XYZZ* __restrict__ G) {
  const u32 t = blockIdx.x * blockDim.x + threadIdx.x;     // (p*3 + e)*4 + g
  if (t >= total) return;
  const XYZZ* A = Aw + (size_t)(t >> 2) * 32 + 8 * (t & 3u);
  XYZZ acc = ld_xyzz(A + 7);
#pragma unroll 1
  for (int j = 6; j >= 0; j--) {
    acc = xyzz_dbl_k(acc, 4);
    XYZZ v = ld_xyzz(A + j);
    xyzz_add_ni(acc, v);
  }
  st_xyzz(G + t, acc);
}

// One thread per (equation kind, proof): sum_g 2^(32g) G_g by Horner (96 doublings), then the unit-scalar terms
// (E2: + A - P_new, E4: - P_new).  Threads are ordered kind-major like the MSM index m = E*cn + p of verify.cuh; the result
// goes to var[m] (E3's slot was written by k_sv_table).  Thread form on purpose: the 4-lane cooperative form has the
// shorter chain but costs ~3x the multiplier-pipe time, and this kernel runs underneath the table lookups of the same chunk.
__global__ void __launch_bounds__(128) k_sv_comb2(const XYZZ* __restrict__ G, const Affine* __restrict__ pts, RpLayout lay, u32 cn,
                                                  XYZZ* __restrict__ var) {
  const u32 q = blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= 3 * cn) return;
  const u32 eq = q / cn, p = q % cn;
  const XYZZ* Gp = G + ((size_t)p * 3 + eq) * 4;
  XYZZ acc = ld_xyzz(Gp + 3);
#pragma unroll 1
  for (int g4 = 2; g4 >= 0; g4--) {
    acc = xyzz_dbl_k(acc, 32);
    XYZZ v = ld_xyzz(Gp + g4);
    xyzz_add_ni(acc, v);
  }
  const Affine* PP = pts + (size_t)p * lay.npt;
  if (eq == 1u) { const Affine A = ld_affine(PP + RP_A); xyzz_madd_ni(acc, A); }
  if (eq >= 1u) { const Affine Pn = affine_neg(ld_affine(PP + RP_PNEW)); xyzz_madd_ni(acc, Pn); }
  st_xyzz(var + (size_t)(eq == 2u ? 3u : eq) * cn + p, acc);
}

// ---- latency form of the last Horner stage for small chunks (<= ~1500 proofs: a rank's share of a sharded batch) ------------------
// With a thousand proofs in flight k_sv_comb2 is a single-thread chain of 96 doublings on 24 blocks (215 us); as 4-lane cooperative
// operations (coop4.cuh) it takes 152 us.  Measured and NOT kept for the other two stages: four warps per proof in k_sv_main
// (286 against 254 us: at 1024 proofs that kernel is already multiplier-bound, 1.1 M full additions) and a 4-lane k_sv_comb1
// (109 against 111 us: 28 doublings + 7 additions whose ~24 KB loop body is fetched cold by too few warps).
// one QUAD per (equation kind, proof): sum_g 2^(32g) G_g by Horner (96 doublings), then the unit-scalar terms
__global__ void __launch_bounds__(128) k_sv_comb2q(const XYZZ* __restrict__ G, const Affine* __restrict__ pts, RpLayout lay, u32 cn,
                                                   XYZZ* __restrict__ var) {
  u32 q = (blockIdx.x * blockDim.x + threadIdx.x) >> 2;
  const int lane = threadIdx.x & 31, role = lane & 3, base = lane & ~3;
  const bool live = q < 3 * cn;
  if (!live) q = 3 * cn - 1;
  const u32 eq = q / cn, p = q % cn;
  const XYZZ* Gp = G + ((size_t)p * 3 + eq) * 4;
  XYZZ acc = ld_xyzz(Gp + 3);
#pragma unroll 1
  for (int g4 = 2; g4 >= 0; g4--) {
#pragma unroll 1
    for (int d = 0; d < 32; d++) acc = coop_dbl(acc, role, base);
    XYZZ v = ld_xyzz(Gp + g4);
    acc = coop_add(acc, v, role, base);
  }
  const Affine* PP = pts + (size_t)p * lay.npt;
  // unit-scalar terms (E1: none, E2: + A - P_new, E4: - P_new); every quad runs both additions, the unused ones add the identity
  XYZZ a1 = eq == 1u ? xyzz_from_affine(ld_affine(PP + RP_A)) : xyzz_identity();
  XYZZ a2 = eq >= 1u ? xyzz_from_affine(affine_neg(ld_affine(PP + RP_PNEW))) : xyzz_identity();
  acc = coop_add(acc, a1, role, base);
  acc = coop_add(acc, a2, role, base);
  if (live && role == 0) st_xyzz(var + (size_t)(eq == 2u ? 3u : eq) * cn + p, acc);
}

}  // namespace bp
