// coop4.cuh -- 4-lane cooperative XYZZ point operations for the latency-bound tails of the MSM
// (bucket reduction, window sums, Horner combine).
//
// In those stages only a few hundred additions are in flight while each one is a chain of 9..14
// dependent field multiplications, so a lone thread per point leaves the SM idle.  Here four
// consecutive lanes (a "quad") hold identical copies of the operands, each lane computes ONE of the
// up-to-four independent products of a formula level, and the products are exchanged with warp
// shuffles: a full XYZZ addition becomes 4 multiplication levels instead of 14 sequential
// multiplications, a doubling 3 levels instead of 9.  All 32 lanes of a warp must call these functions
// together (the shuffles use the full mask); exceptional cases are resolved with selects and a
// warp-uniform vote, never with divergent shuffles.  Results are identical in the four lanes.
#pragma once
#include "ec.cuh"

namespace bp {

#define BP_FULL_MASK 0xFFFFFFFFu

// (Out-of-line variants of these operations were measured: the quad kernels got ~30 % slower from the call/spill
// overhead, so they stay inlined; the thread-per-unit kernels of the batch path do use out-of-line point operations,
// ec.cuh, because there instruction fetch was the top stall reason.)
BP_DI Fp shfl_fp(const Fp& m, int src_lane) {
  Fp r;
#pragma unroll
  for (int i = 0; i < 8; i++) r.v[i] = __shfl_sync(BP_FULL_MASK, m.v[i], src_lane);
  return r;
}
BP_DI Fp shfl_down_fp(const Fp& m, int delta) {
  Fp r;
#pragma unroll
  for (int i = 0; i < 8; i++) r.v[i] = __shfl_down_sync(BP_FULL_MASK, m.v[i], delta);
  return r;
}
BP_DI Fp shfl_up_fp(const Fp& m, int delta) {
  Fp r;
#pragma unroll
  for (int i = 0; i < 8; i++) r.v[i] = __shfl_up_sync(BP_FULL_MASK, m.v[i], delta);
  return r;
}
BP_DI Fp sel_fp(bool c, const Fp& a, const Fp& b) {
  Fp r;
#pragma unroll
  for (int i = 0; i < 8; i++) r.v[i] = c ? a.v[i] : b.v[i];
  return r;
}
BP_DI XYZZ sel_xyzz(bool c, const XYZZ& a, const XYZZ& b) {
  XYZZ r; r.X = sel_fp(c, a.X, b.X); r.Y = sel_fp(c, a.Y, b.Y); r.ZZ = sel_fp(c, a.ZZ, b.ZZ); r.ZZZ = sel_fp(c, a.ZZZ, b.ZZZ);
  return r;
}
// one multiplication level: lane `role` multiplies (x_role, y_role); every lane receives all four products
BP_DI void coop_level(int role, int base, const Fp& x0, const Fp& y0, const Fp& x1, const Fp& y1, const Fp& x2, const Fp& y2,
                      const Fp& x3, const Fp& y3, Fp& p0, Fp& p1, Fp& p2, Fp& p3) {
  Fp x = sel_fp(role == 0, x0, sel_fp(role == 1, x1, sel_fp(role == 2, x2, x3)));
  Fp y = sel_fp(role == 0, y0, sel_fp(role == 1, y1, sel_fp(role == 2, y2, y3)));
  Fp m = fp_mul(x, y);
  p0 = shfl_fp(m, base); p1 = shfl_fp(m, base + 1); p2 = shfl_fp(m, base + 2); p3 = shfl_fp(m, base + 3);
}

// a = 2a   (dbl-2008-s-1, a = 0):  3 levels
BP_DI XYZZ coop_dbl(const XYZZ& a, int role, int base) {
  Fp U = fp_dbl(a.Y);
  Fp V, XX, d0, d1;
  coop_level(role, base, U, U, a.X, a.X, U, U, a.X, a.X, V, XX, d0, d1);                // V = U^2, XX = X^2
  Fp M = fp_add(fp_dbl(XX), XX);
  Fp W, S, MM;
  coop_level(role, base, U, V, a.X, V, M, M, M, M, W, S, MM, d0);                       // W = U*V, S = X*V, MM = M^2
  Fp X3 = fp_sub(MM, fp_dbl(S));
  Fp Ya, Wy, ZZ3, ZZZ3;
  coop_level(role, base, M, fp_sub(S, X3), W, a.Y, V, a.ZZ, W, a.ZZZ, Ya, Wy, ZZ3, ZZZ3);
  XYZZ r; r.X = X3; r.Y = fp_sub(Ya, Wy); r.ZZ = ZZ3; r.ZZZ = ZZZ3;
  return sel_xyzz(xyzz_is_identity(a), a, r);
}

// a + b   (add-2008-s), complete:  4 levels (+ a warp-uniform doubling pass when some quad adds a point to itself)
BP_DI XYZZ coop_add(const XYZZ& a, const XYZZ& b, int role, int base) {
  const bool ida = xyzz_is_identity(a), idb = xyzz_is_identity(b);
  Fp U1, U2, S1, S2;
  coop_level(role, base, a.X, b.ZZ, b.X, a.ZZ, a.Y, b.ZZZ, b.Y, a.ZZZ, U1, U2, S1, S2);
  Fp Pd = fp_sub(U2, U1), R = fp_sub(S2, S1);
  Fp PP, RR, Za, Zb;
  coop_level(role, base, Pd, Pd, R, R, a.ZZ, b.ZZ, a.ZZZ, b.ZZZ, PP, RR, Za, Zb);
  Fp PPP, Q, ZZ3, d0;
  coop_level(role, base, Pd, PP, U1, PP, Za, PP, Pd, PP, PPP, Q, ZZ3, d0);
  Fp X3 = fp_sub(fp_sub(RR, PPP), fp_dbl(Q));
  Fp ZZZ3, T, Ya;
  coop_level(role, base, Zb, PPP, S1, PPP, R, fp_sub(Q, X3), Zb, PPP, ZZZ3, T, Ya, d0);
  XYZZ r; r.X = X3; r.Y = fp_sub(Ya, T); r.ZZ = ZZ3; r.ZZZ = ZZZ3;
  const bool pz = fp_is_zero(Pd), rz = fp_is_zero(R);
  const bool both = !ida && !idb;
  const bool need_dbl = both && pz && rz;                   // same point: double
  if (__any_sync(BP_FULL_MASK, need_dbl)) {                 // (moving this pass out of line miscomputed on sm_100a; it stays inline)
    XYZZ d = coop_dbl(a, role, base);
    r = sel_xyzz(need_dbl, d, r);
  }
  r = sel_xyzz(both && pz && !rz, xyzz_identity(), r);      // opposite points
  r = sel_xyzz(ida, b, r);
  r = sel_xyzz(!ida && idb, a, r);
  return r;
}

}  // namespace bp
