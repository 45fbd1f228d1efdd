// fp.cuh -- secp256k1 base-field arithmetic for sm_100a, 8 x 32-bit limbs held in registers.
//
// Replaces: the F_p arithmetic the reference reaches through fastecdsa/GMP on every
// Point.__add__ (/root/reference/src/pippenger/group.py:31-32).
//
// Representation: little-endian limbs, "lazy" residues in [0, 2^256) (not necessarily < p).
// p = 2^256 - C with C = 2^32 + 977, so 2^256 = C (mod p) and a 512-bit product folds with
// 8 + 1 extra IMAD.WIDE instead of the 64 + 8 a Montgomery REDC needs (see DESIGN.md, "Why
// not Montgomery for F_p").  The 8x8 schoolbook product uses separate even/odd column
// accumulators so that every 32x32->64 partial product is one IMAD.WIDE.U32 whose carry rides
// the predicate chain (IMAD.WIDE.U32.X); checked with cuobjdump -sass, see profiles/.
#pragma once
#include <cstdint>

namespace bp {

typedef uint32_t u32;
typedef uint64_t u64;

struct __align__(16) Fp { u32 v[8]; };

#define BP_DI __device__ __forceinline__
#define BP_HAVE_FP_MUL_WIDE 1

// 2^256 - p
#define BP_PC_LO 977u   // C = 2^32 + 977 : limb0 = 977, limb1 = 1

BP_DI Fp fp_zero() { Fp r;
#pragma unroll
  for (int i = 0; i < 8; i++) r.v[i] = 0; return r; }
BP_DI Fp fp_one() { Fp r = fp_zero(); r.v[0] = 1; return r; }

// ---- multi-limb carry chains (one asm block each so the CC flag never crosses statements) ----
// r = a + b, returns carry
BP_DI u32 add256(u32 r[8], const u32 a[8], const u32 b[8]) {
  u32 c;
  asm("add.cc.u32 %0,%9,%17; addc.cc.u32 %1,%10,%18; addc.cc.u32 %2,%11,%19; addc.cc.u32 %3,%12,%20;"
      "addc.cc.u32 %4,%13,%21; addc.cc.u32 %5,%14,%22; addc.cc.u32 %6,%15,%23; addc.cc.u32 %7,%16,%24;"
      "addc.u32 %8,0,0;"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(c)
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(a[4]), "r"(a[5]), "r"(a[6]), "r"(a[7]),
        "r"(b[0]), "r"(b[1]), "r"(b[2]), "r"(b[3]), "r"(b[4]), "r"(b[5]), "r"(b[6]), "r"(b[7]));
  return c;
}
// r = a - b, returns borrow (1 if a < b)
BP_DI u32 sub256(u32 r[8], const u32 a[8], const u32 b[8]) {
  u32 c;
  asm("sub.cc.u32 %0,%9,%17; subc.cc.u32 %1,%10,%18; subc.cc.u32 %2,%11,%19; subc.cc.u32 %3,%12,%20;"
      "subc.cc.u32 %4,%13,%21; subc.cc.u32 %5,%14,%22; subc.cc.u32 %6,%15,%23; subc.cc.u32 %7,%16,%24;"
      "subc.u32 %8,0,0;"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(c)
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(a[4]), "r"(a[5]), "r"(a[6]), "r"(a[7]),
        "r"(b[0]), "r"(b[1]), "r"(b[2]), "r"(b[3]), "r"(b[4]), "r"(b[5]), "r"(b[6]), "r"(b[7]));
  return c & 1u;   // subc.u32 0,0 yields 0xffffffff on borrow
}
// r += k*C for k in {0,1}; returns carry out
BP_DI u32 add_kc(u32 r[8], u32 k) {
  u32 c;
  asm("mad.lo.cc.u32 %0,%9,977,%0; addc.cc.u32 %1,%1,%9; addc.cc.u32 %2,%2,0; addc.cc.u32 %3,%3,0;"
      "addc.cc.u32 %4,%4,0; addc.cc.u32 %5,%5,0; addc.cc.u32 %6,%6,0; addc.cc.u32 %7,%7,0; addc.u32 %8,0,0;"
      : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]), "=r"(c)
      : "r"(k));
  return c;
}
// r -= k*C for k in {0,1}; returns borrow
BP_DI u32 sub_kc(u32 r[8], u32 k) {
  u32 c, lo = k * BP_PC_LO;
  asm("sub.cc.u32 %0,%0,%9; subc.cc.u32 %1,%1,%10; subc.cc.u32 %2,%2,0; subc.cc.u32 %3,%3,0;"
      "subc.cc.u32 %4,%4,0; subc.cc.u32 %5,%5,0; subc.cc.u32 %6,%6,0; subc.cc.u32 %7,%7,0; subc.u32 %8,0,0;"
      : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]), "=r"(c)
      : "r"(lo), "r"(k));
  return c & 1u;
}

// Speculative forms (BP_SPEC_ADDSUB): the wrapped candidate (s + C resp. d - C) is computed alongside the plain sum /
// difference -- its carry chain trails the first one by one limb instead of waiting for its end -- and a select on the
// carry picks the result: ~11 dependent steps instead of 20 (add) / 26 (sub).  The second wrap (both operands
// non-canonical and near 2^256, or a difference within C of a multiple of 2^256) takes a rare branch.
#ifndef BP_SPEC_ADDSUB
#define BP_SPEC_ADDSUB 0   // measured on B200: 4-lane doubling 2534 -> 2460 cycles, but the accumulation kernel 1.98 -> 2.02 ms (registers); off
#endif
BP_DI Fp fp_add(const Fp& a, const Fp& b) {
  Fp r;
#if BP_SPEC_ADDSUB
  u32 s[8], t[8], k1, k2;
  k1 = add256(s, a.v, b.v);
  asm("add.cc.u32 %0,%9,977; addc.cc.u32 %1,%10,1; addc.cc.u32 %2,%11,0; addc.cc.u32 %3,%12,0;"
      "addc.cc.u32 %4,%13,0; addc.cc.u32 %5,%14,0; addc.cc.u32 %6,%15,0; addc.cc.u32 %7,%16,0; addc.u32 %8,0,0;"
      : "=r"(t[0]), "=r"(t[1]), "=r"(t[2]), "=r"(t[3]), "=r"(t[4]), "=r"(t[5]), "=r"(t[6]), "=r"(t[7]), "=r"(k2)
      : "r"(s[0]), "r"(s[1]), "r"(s[2]), "r"(s[3]), "r"(s[4]), "r"(s[5]), "r"(s[6]), "r"(s[7]));
#pragma unroll
  for (int i = 0; i < 8; i++) r.v[i] = k1 ? t[i] : s[i];
  if (k1 & k2) add_kc(r.v, 1u);        // a + b >= 2^257 - C: the wrapped value is below C, one more + C cannot carry
#else
  u32 k = add256(r.v, a.v, b.v);
  k = add_kc(r.v, k);        // 2^256 = C (mod p)
  // a second wrap needs a + b >= 2^256 + p (both operands non-canonical): rare, still handled
  asm("mad.lo.cc.u32 %0,%3,977,%0; addc.cc.u32 %1,%1,%3; addc.u32 %2,%2,0;" : "+r"(r.v[0]), "+r"(r.v[1]), "+r"(r.v[2]) : "r"(k));
#endif
  return r;
}
BP_DI Fp fp_sub(const Fp& a, const Fp& b) {
  Fp r;
#if BP_SPEC_ADDSUB
  u32 d[8], e[8], k1, k2;
  k1 = sub256(d, a.v, b.v);
  asm("sub.cc.u32 %0,%9,977; subc.cc.u32 %1,%10,1; subc.cc.u32 %2,%11,0; subc.cc.u32 %3,%12,0;"
      "subc.cc.u32 %4,%13,0; subc.cc.u32 %5,%14,0; subc.cc.u32 %6,%15,0; subc.cc.u32 %7,%16,0; subc.u32 %8,0,0;"
      : "=r"(e[0]), "=r"(e[1]), "=r"(e[2]), "=r"(e[3]), "=r"(e[4]), "=r"(e[5]), "=r"(e[6]), "=r"(e[7]), "=r"(k2)
      : "r"(d[0]), "r"(d[1]), "r"(d[2]), "r"(d[3]), "r"(d[4]), "r"(d[5]), "r"(d[6]), "r"(d[7]));
#pragma unroll
  for (int i = 0; i < 8; i++) r.v[i] = k1 ? e[i] : d[i];
  if (k1 & k2 & 1u) sub_kc(r.v, 1u);   // a - b + 2^256 < C: subtract C once more (wraps to just below 2^256, cannot borrow again)
#else
  u32 k = sub256(r.v, a.v, b.v);
  k = sub_kc(r.v, k);        // -2^256 = -C
  sub_kc(r.v, k);            // second borrow only when the first left r < C; cannot borrow again
#endif
  return r;
}
BP_DI Fp fp_dbl(const Fp& a) { return fp_add(a, a); }
BP_DI Fp fp_neg(const Fp& a) { return fp_sub(fp_zero(), a); }

BP_DI bool fp_is_zero(const Fp& a) {   // 0 or p
  u32 o = a.v[0] | a.v[1] | a.v[2] | a.v[3] | a.v[4] | a.v[5] | a.v[6] | a.v[7];
  u32 n = (a.v[0] ^ 0xFFFFFC2Fu) | (a.v[1] ^ 0xFFFFFFFEu) | ~(a.v[2] & a.v[3] & a.v[4] & a.v[5] & a.v[6] & a.v[7]);
  return o == 0 || n == 0;
}
// canonical representative in [0, p)
BP_DI Fp fp_canon(const Fp& a) {
  Fp r = a;
  bool hi = (a.v[2] & a.v[3] & a.v[4] & a.v[5] & a.v[6] & a.v[7]) == 0xFFFFFFFFu;
  bool ge = hi && (a.v[1] == 0xFFFFFFFFu || (a.v[1] == 0xFFFFFFFEu && a.v[0] >= 0xFFFFFC2Fu));
  add_kc(r.v, ge ? 1u : 0u);   // a - p = a + C - 2^256
  return r;
}

// ---- 8x8 limb product, even/odd columns --------------------------------------------------------
BP_DI void mul_row_init(u32* acc, u32 a0, u32 a1, u32 a2, u32 a3, u32 b) {
  asm("mul.lo.u32 %0,%8,%12; mul.hi.u32 %1,%8,%12; mul.lo.u32 %2,%9,%12; mul.hi.u32 %3,%9,%12;"
      "mul.lo.u32 %4,%10,%12; mul.hi.u32 %5,%10,%12; mul.lo.u32 %6,%11,%12; mul.hi.u32 %7,%11,%12;"
      : "=r"(acc[0]), "=r"(acc[1]), "=r"(acc[2]), "=r"(acc[3]), "=r"(acc[4]), "=r"(acc[5]), "=r"(acc[6]), "=r"(acc[7])
      : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b));
}
BP_DI void mul_row_mad(u32* acc, u32 a0, u32 a1, u32 a2, u32 a3, u32 b) {
  asm("mad.lo.cc.u32 %0,%9,%13,%0; madc.hi.cc.u32 %1,%9,%13,%1; madc.lo.cc.u32 %2,%10,%13,%2; madc.hi.cc.u32 %3,%10,%13,%3;"
      "madc.lo.cc.u32 %4,%11,%13,%4; madc.hi.cc.u32 %5,%11,%13,%5; madc.lo.cc.u32 %6,%12,%13,%6; madc.hi.cc.u32 %7,%12,%13,%7;"
      "addc.u32 %8,%8,0;"
      : "+r"(acc[0]), "+r"(acc[1]), "+r"(acc[2]), "+r"(acc[3]), "+r"(acc[4]), "+r"(acc[5]), "+r"(acc[6]), "+r"(acc[7]), "+r"(acc[8])
      : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b));
}
// t[0..15] = a * b
BP_DI void mul_wide(u32 t[16], const u32 a[8], const u32 b[8]) {
  // ev[k] sits at limb position k, od[k] at limb position k+1
  u32 ev[18], od[18];
#pragma unroll
  for (int k = 8; k < 18; k++) { ev[k] = 0; od[k] = 0; }
  mul_row_init(ev, a[0], a[2], a[4], a[6], b[0]);
  mul_row_init(od, a[1], a[3], a[5], a[7], b[0]);
#pragma unroll
  for (int i = 1; i < 8; i++) {
    if (i & 1) {
      mul_row_mad(od + i - 1, a[0], a[2], a[4], a[6], b[i]);
      mul_row_mad(ev + i + 1, a[1], a[3], a[5], a[7], b[i]);
    } else {
      mul_row_mad(ev + i, a[0], a[2], a[4], a[6], b[i]);
      mul_row_mad(od + i, a[1], a[3], a[5], a[7], b[i]);
    }
  }
  t[0] = ev[0];
  asm("add.cc.u32 %0,%15,%30; addc.cc.u32 %1,%16,%31; addc.cc.u32 %2,%17,%32; addc.cc.u32 %3,%18,%33; addc.cc.u32 %4,%19,%34;"
      "addc.cc.u32 %5,%20,%35; addc.cc.u32 %6,%21,%36; addc.cc.u32 %7,%22,%37; addc.cc.u32 %8,%23,%38; addc.cc.u32 %9,%24,%39;"
      "addc.cc.u32 %10,%25,%40; addc.cc.u32 %11,%26,%41; addc.cc.u32 %12,%27,%42; addc.cc.u32 %13,%28,%43; addc.u32 %14,%29,%44;"
      : "=r"(t[1]), "=r"(t[2]), "=r"(t[3]), "=r"(t[4]), "=r"(t[5]), "=r"(t[6]), "=r"(t[7]), "=r"(t[8]), "=r"(t[9]), "=r"(t[10]),
        "=r"(t[11]), "=r"(t[12]), "=r"(t[13]), "=r"(t[14]), "=r"(t[15])
      : "r"(ev[1]), "r"(ev[2]), "r"(ev[3]), "r"(ev[4]), "r"(ev[5]), "r"(ev[6]), "r"(ev[7]), "r"(ev[8]), "r"(ev[9]), "r"(ev[10]),
        "r"(ev[11]), "r"(ev[12]), "r"(ev[13]), "r"(ev[14]), "r"(ev[15]),
        "r"(od[0]), "r"(od[1]), "r"(od[2]), "r"(od[3]), "r"(od[4]), "r"(od[5]), "r"(od[6]), "r"(od[7]), "r"(od[8]), "r"(od[9]),
        "r"(od[10]), "r"(od[11]), "r"(od[12]), "r"(od[13]), "r"(od[14]));
}

// ---- one level of Karatsuba on top of the even/odd 4x4 product: 48 IMAD.WIDE instead of 64 -----------------------
// ncu shows the accumulation kernel bound by the fmaheavy pipe (IMAD.WIDE at half rate, ~80 % busy) with the ALU pipe
// under 50 %, so trading 16 wide multiplies for ~60 adds/logic ops is a net win on B200.
// acc[0..3] += {x0, x1} * b at two consecutive 64-bit slots, carry into acc[4]
BP_DI void mad_chain2(u32* acc, u32 x0, u32 x1, u32 b) {
  asm("mad.lo.cc.u32 %0,%5,%7,%0; madc.hi.cc.u32 %1,%5,%7,%1; madc.lo.cc.u32 %2,%6,%7,%2; madc.hi.cc.u32 %3,%6,%7,%3; addc.u32 %4,%4,0;"
      : "+r"(acc[0]), "+r"(acc[1]), "+r"(acc[2]), "+r"(acc[3]), "+r"(acc[4]) : "r"(x0), "r"(x1), "r"(b));
}
// r[0..7] = a[0..3] * b[0..3]
BP_DI void mul4_wide(u32 r[8], const u32 a[4], const u32 b[4]) {
  u32 ev[10], od[10];
#pragma unroll
  for (int k = 4; k < 10; k++) { ev[k] = 0; od[k] = 0; }
  asm("mul.lo.u32 %0,%4,%6; mul.hi.u32 %1,%4,%6; mul.lo.u32 %2,%5,%6; mul.hi.u32 %3,%5,%6;"
      : "=r"(ev[0]), "=r"(ev[1]), "=r"(ev[2]), "=r"(ev[3]) : "r"(a[0]), "r"(a[2]), "r"(b[0]));
  asm("mul.lo.u32 %0,%4,%6; mul.hi.u32 %1,%4,%6; mul.lo.u32 %2,%5,%6; mul.hi.u32 %3,%5,%6;"
      : "=r"(od[0]), "=r"(od[1]), "=r"(od[2]), "=r"(od[3]) : "r"(a[1]), "r"(a[3]), "r"(b[0]));
  mad_chain2(od + 0, a[0], a[2], b[1]);
  mad_chain2(ev + 2, a[1], a[3], b[1]);
  mad_chain2(ev + 2, a[0], a[2], b[2]);
  mad_chain2(od + 2, a[1], a[3], b[2]);
  mad_chain2(od + 2, a[0], a[2], b[3]);
  mad_chain2(ev + 4, a[1], a[3], b[3]);
  r[0] = ev[0];
  asm("add.cc.u32 %0,%7,%14; addc.cc.u32 %1,%8,%15; addc.cc.u32 %2,%9,%16; addc.cc.u32 %3,%10,%17;"
      "addc.cc.u32 %4,%11,%18; addc.cc.u32 %5,%12,%19; addc.u32 %6,%13,%20;"
      : "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
      : "r"(ev[1]), "r"(ev[2]), "r"(ev[3]), "r"(ev[4]), "r"(ev[5]), "r"(ev[6]), "r"(ev[7]),
        "r"(od[0]), "r"(od[1]), "r"(od[2]), "r"(od[3]), "r"(od[4]), "r"(od[5]), "r"(od[6]));
}
// t[0..15] = a * b
BP_DI void mul_wide_karatsuba(u32 t[16], const u32 a[8], const u32 b[8]) {
  u32 z0[8], z2[8], m[8], sa[4], sb[4], ca, cb;
  mul4_wide(z0, a, b);
  mul4_wide(z2, a + 4, b + 4);
  asm("add.cc.u32 %0,%5,%9; addc.cc.u32 %1,%6,%10; addc.cc.u32 %2,%7,%11; addc.cc.u32 %3,%8,%12; addc.u32 %4,0,0;"
      : "=r"(sa[0]), "=r"(sa[1]), "=r"(sa[2]), "=r"(sa[3]), "=r"(ca)
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(a[4]), "r"(a[5]), "r"(a[6]), "r"(a[7]));
  asm("add.cc.u32 %0,%5,%9; addc.cc.u32 %1,%6,%10; addc.cc.u32 %2,%7,%11; addc.cc.u32 %3,%8,%12; addc.u32 %4,0,0;"
      : "=r"(sb[0]), "=r"(sb[1]), "=r"(sb[2]), "=r"(sb[3]), "=r"(cb)
      : "r"(b[0]), "r"(b[1]), "r"(b[2]), "r"(b[3]), "r"(b[4]), "r"(b[5]), "r"(b[6]), "r"(b[7]));
  mul4_wide(m, sa, sb);
  // mid = (sa + ca*2^128)(sb + cb*2^128) = m + (ca ? sb : 0)*2^128 + (cb ? sa : 0)*2^128 + (ca & cb)*2^256   (9 limbs)
  const u32 ma = 0u - ca, mb = 0u - cb;
  u32 mid[9];
#pragma unroll
  for (int k = 0; k < 4; k++) mid[k] = m[k];
  asm("add.cc.u32 %0,%5,%9; addc.cc.u32 %1,%6,%10; addc.cc.u32 %2,%7,%11; addc.cc.u32 %3,%8,%12; addc.u32 %4,%13,0;"
      : "=r"(mid[4]), "=r"(mid[5]), "=r"(mid[6]), "=r"(mid[7]), "=r"(mid[8])
      : "r"(m[4]), "r"(m[5]), "r"(m[6]), "r"(m[7]), "r"(sb[0] & ma), "r"(sb[1] & ma), "r"(sb[2] & ma), "r"(sb[3] & ma), "r"(ca & cb));
  asm("add.cc.u32 %0,%0,%5; addc.cc.u32 %1,%1,%6; addc.cc.u32 %2,%2,%7; addc.cc.u32 %3,%3,%8; addc.u32 %4,%4,0;"
      : "+r"(mid[4]), "+r"(mid[5]), "+r"(mid[6]), "+r"(mid[7]), "+r"(mid[8])
      : "r"(sa[0] & mb), "r"(sa[1] & mb), "r"(sa[2] & mb), "r"(sa[3] & mb));
  // z1 = mid - z0 - z2   (0 <= z1 < 2^258)
  asm("sub.cc.u32 %0,%0,%9; subc.cc.u32 %1,%1,%10; subc.cc.u32 %2,%2,%11; subc.cc.u32 %3,%3,%12; subc.cc.u32 %4,%4,%13;"
      "subc.cc.u32 %5,%5,%14; subc.cc.u32 %6,%6,%15; subc.cc.u32 %7,%7,%16; subc.u32 %8,%8,0;"
      : "+r"(mid[0]), "+r"(mid[1]), "+r"(mid[2]), "+r"(mid[3]), "+r"(mid[4]), "+r"(mid[5]), "+r"(mid[6]), "+r"(mid[7]), "+r"(mid[8])
      : "r"(z0[0]), "r"(z0[1]), "r"(z0[2]), "r"(z0[3]), "r"(z0[4]), "r"(z0[5]), "r"(z0[6]), "r"(z0[7]));
  asm("sub.cc.u32 %0,%0,%9; subc.cc.u32 %1,%1,%10; subc.cc.u32 %2,%2,%11; subc.cc.u32 %3,%3,%12; subc.cc.u32 %4,%4,%13;"
      "subc.cc.u32 %5,%5,%14; subc.cc.u32 %6,%6,%15; subc.cc.u32 %7,%7,%16; subc.u32 %8,%8,0;"
      : "+r"(mid[0]), "+r"(mid[1]), "+r"(mid[2]), "+r"(mid[3]), "+r"(mid[4]), "+r"(mid[5]), "+r"(mid[6]), "+r"(mid[7]), "+r"(mid[8])
      : "r"(z2[0]), "r"(z2[1]), "r"(z2[2]), "r"(z2[3]), "r"(z2[4]), "r"(z2[5]), "r"(z2[6]), "r"(z2[7]));
  // t = z0 + z1*2^128 + z2*2^256
#pragma unroll
  for (int k = 0; k < 4; k++) t[k] = z0[k];
  asm("add.cc.u32 %0,%12,%24; addc.cc.u32 %1,%13,%25; addc.cc.u32 %2,%14,%26; addc.cc.u32 %3,%15,%27;"
      "addc.cc.u32 %4,%16,%28; addc.cc.u32 %5,%17,%29; addc.cc.u32 %6,%18,%30; addc.cc.u32 %7,%19,%31;"
      "addc.cc.u32 %8,%20,%32; addc.cc.u32 %9,%21,0; addc.cc.u32 %10,%22,0; addc.u32 %11,%23,0;"
      : "=r"(t[4]), "=r"(t[5]), "=r"(t[6]), "=r"(t[7]), "=r"(t[8]), "=r"(t[9]), "=r"(t[10]), "=r"(t[11]), "=r"(t[12]), "=r"(t[13]),
        "=r"(t[14]), "=r"(t[15])
      : "r"(z0[4]), "r"(z0[5]), "r"(z0[6]), "r"(z0[7]), "r"(z2[0]), "r"(z2[1]), "r"(z2[2]), "r"(z2[3]), "r"(z2[4]), "r"(z2[5]),
        "r"(z2[6]), "r"(z2[7]),
        "r"(mid[0]), "r"(mid[1]), "r"(mid[2]), "r"(mid[3]), "r"(mid[4]), "r"(mid[5]), "r"(mid[6]), "r"(mid[7]), "r"(mid[8]));
}

// r = t mod p (lazy), t 512 bits:  t = lo + hi*2^256 = lo + hi*C
BP_DI void fold512(u32 r[8], const u32 t[16]) {
  // hi * 977 as two sets of independent 32x32->64 products: se[2k..2k+1] = t[8+2k]*977 at limb 2k, so[2k..2k+1] =
  // t[9+2k]*977 at limb 2k+1.  Both sets live in aligned register pairs with no addend, so every product is a bare
  // IMAD.WIDE (a mad chain through the odd positions needed pairs that straddle two products: ~16 register moves per
  // fold on the multiplier pipe, the top non-arithmetic cost in the accumulation kernel's SASS).
  // The same products on the FP64 pipe (DFMA on 2^52 + t) were measured slower: k_accumulate 1.79 -> 2.08 ms at 2^20 (DESIGN.md 5).
  u32 se[8], so[8];
  asm("mul.lo.u32 %0,%8,%12; mul.hi.u32 %1,%8,%12; mul.lo.u32 %2,%9,%12; mul.hi.u32 %3,%9,%12;"
      "mul.lo.u32 %4,%10,%12; mul.hi.u32 %5,%10,%12; mul.lo.u32 %6,%11,%12; mul.hi.u32 %7,%11,%12;"
      : "=r"(se[0]), "=r"(se[1]), "=r"(se[2]), "=r"(se[3]), "=r"(se[4]), "=r"(se[5]), "=r"(se[6]), "=r"(se[7])
      : "r"(t[8]), "r"(t[10]), "r"(t[12]), "r"(t[14]), "r"(977u));
  asm("mul.lo.u32 %0,%8,%12; mul.hi.u32 %1,%8,%12; mul.lo.u32 %2,%9,%12; mul.hi.u32 %3,%9,%12;"
      "mul.lo.u32 %4,%10,%12; mul.hi.u32 %5,%10,%12; mul.lo.u32 %6,%11,%12; mul.hi.u32 %7,%11,%12;"
      : "=r"(so[0]), "=r"(so[1]), "=r"(so[2]), "=r"(so[3]), "=r"(so[4]), "=r"(so[5]), "=r"(so[6]), "=r"(so[7])
      : "r"(t[9]), "r"(t[11]), "r"(t[13]), "r"(t[15]), "r"(977u));
  // w = so + hi (both at limb 1), u = lo + se (limb 0): in these two chains ptxas folds each product into an
  // IMAD.WIDE whose 64-bit addend is an aligned pair; the third chain u += w << 32 is plain adds.
  u32 w[8], u[9], top, top2;
  asm("add.cc.u32 %0,%9,%17; addc.cc.u32 %1,%10,%18; addc.cc.u32 %2,%11,%19; addc.cc.u32 %3,%12,%20;"
      "addc.cc.u32 %4,%13,%21; addc.cc.u32 %5,%14,%22; addc.cc.u32 %6,%15,%23; addc.cc.u32 %7,%16,%24; addc.u32 %8,0,0;"
      : "=r"(w[0]), "=r"(w[1]), "=r"(w[2]), "=r"(w[3]), "=r"(w[4]), "=r"(w[5]), "=r"(w[6]), "=r"(w[7]), "=r"(top2)
      : "r"(t[8]), "r"(t[9]), "r"(t[10]), "r"(t[11]), "r"(t[12]), "r"(t[13]), "r"(t[14]), "r"(t[15]),
        "r"(so[0]), "r"(so[1]), "r"(so[2]), "r"(so[3]), "r"(so[4]), "r"(so[5]), "r"(so[6]), "r"(so[7]));
  asm("add.cc.u32 %0,%9,%17; addc.cc.u32 %1,%10,%18; addc.cc.u32 %2,%11,%19; addc.cc.u32 %3,%12,%20;"
      "addc.cc.u32 %4,%13,%21; addc.cc.u32 %5,%14,%22; addc.cc.u32 %6,%15,%23; addc.cc.u32 %7,%16,%24; addc.u32 %8,0,0;"
      : "=r"(u[0]), "=r"(u[1]), "=r"(u[2]), "=r"(u[3]), "=r"(u[4]), "=r"(u[5]), "=r"(u[6]), "=r"(u[7]), "=r"(u[8])
      : "r"(t[0]), "r"(t[1]), "r"(t[2]), "r"(t[3]), "r"(t[4]), "r"(t[5]), "r"(t[6]), "r"(t[7]),
        "r"(se[0]), "r"(se[1]), "r"(se[2]), "r"(se[3]), "r"(se[4]), "r"(se[5]), "r"(se[6]), "r"(se[7]));
  asm("add.cc.u32 %0,%0,%9; addc.cc.u32 %1,%1,%10; addc.cc.u32 %2,%2,%11; addc.cc.u32 %3,%3,%12;"
      "addc.cc.u32 %4,%4,%13; addc.cc.u32 %5,%5,%14; addc.cc.u32 %6,%6,%15; addc.cc.u32 %7,%7,%16; addc.u32 %8,0,0;"
      : "+r"(u[1]), "+r"(u[2]), "+r"(u[3]), "+r"(u[4]), "+r"(u[5]), "+r"(u[6]), "+r"(u[7]), "+r"(u[8]), "=r"(top)
      : "r"(w[0]), "r"(w[1]), "r"(w[2]), "r"(w[3]), "r"(w[4]), "r"(w[5]), "r"(w[6]), "r"(w[7]));
  top += top2;                       // e = u[8] + top*2^32 < 2^34
  // second fold: r = u[0..7] + e*977 + (e << 32)
  u64 m = (u64)u[8] * 977ull + (((u64)(top * 977u)) << 32);   // e*977 < 2^44
  u32 m0 = (u32)m, m1 = (u32)(m >> 32), k, k2;
#pragma unroll
  for (int i = 0; i < 8; i++) r[i] = u[i];
  asm("add.cc.u32 %0,%0,%9; addc.cc.u32 %1,%1,%10; addc.cc.u32 %2,%2,0; addc.cc.u32 %3,%3,0;"
      "addc.cc.u32 %4,%4,0; addc.cc.u32 %5,%5,0; addc.cc.u32 %6,%6,0; addc.cc.u32 %7,%7,0; addc.u32 %8,0,0;"
      : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]), "=r"(k)
      : "r"(m0), "r"(m1));
  asm("add.cc.u32 %0,%0,%8; addc.cc.u32 %1,%1,%9; addc.cc.u32 %2,%2,0; addc.cc.u32 %3,%3,0;"
      "addc.cc.u32 %4,%4,0; addc.cc.u32 %5,%5,0; addc.cc.u32 %6,%6,0; addc.u32 %7,0,0;"
      : "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]), "=r"(k2)
      : "r"(u[8]), "r"(top));
  // at most one of the two adds wrapped (the sum is < 2^256 + 2^67); the wrapped value is tiny
  k += k2;
  asm("mad.lo.cc.u32 %0,%3,977,%0; addc.cc.u32 %1,%1,%3; addc.u32 %2,%2,0;" : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]) : "r"(k));
}

#ifndef BP_KARATSUBA
#define BP_KARATSUBA 0   // measured on B200: 0.098 vs 0.104 T fp_mul/s and a 24 % slower accumulation (ALU pipe + registers); kept for reference
#endif
BP_DI Fp fp_mul(const Fp& a, const Fp& b) {
  u32 t[16];
  if (BP_KARATSUBA) mul_wide_karatsuba(t, a.v, b.v); else mul_wide(t, a.v, b.v);
  Fp r;
  fold512(r.v, t);
  return r;
}
// ---- dedicated squaring: 28 cross products (doubled by a 1-bit shift) + 8 squares = 36 IMAD.WIDE instead of 64 ------
// The cross products a_i*a_j (i < j) are taken by DIAGONALS j - i = d: the products of one diagonal sit at consecutive
// 64-bit slots (limb 2i + d), so each diagonal is one carry chain into the even (d even) or odd (d odd) accumulator,
// followed by a carry ripple to the accumulator's top.  The two longest diagonals start from empty accumulators and
// are bare products.  (A row-wise layout materialised a carry word and a zeroed pair per row: ~25 extra multiplier-
// pipe instructions per squaring in the SASS.)
BP_DI void sqr_diag_5_2(u32* acc, u32 x0, u32 y0, u32 x1, u32 y1, u32 x2, u32 y2, u32 x3, u32 y3, u32 x4, u32 y4) {
  asm("mad.lo.cc.u32 %0,%13,%14,%0; madc.hi.cc.u32 %1,%13,%14,%1; madc.lo.cc.u32 %2,%15,%16,%2;"
      "madc.hi.cc.u32 %3,%15,%16,%3; madc.lo.cc.u32 %4,%17,%18,%4; madc.hi.cc.u32 %5,%17,%18,%5;"
      "madc.lo.cc.u32 %6,%19,%20,%6; madc.hi.cc.u32 %7,%19,%20,%7; madc.lo.cc.u32 %8,%21,%22,%8;"
      "madc.hi.cc.u32 %9,%21,%22,%9; addc.cc.u32 %10,%10,0; addc.cc.u32 %11,%11,0; addc.u32 %12,%12,0;"
      : "+r"(acc[0]), "+r"(acc[1]), "+r"(acc[2]), "+r"(acc[3]), "+r"(acc[4]), "+r"(acc[5]), "+r"(acc[6]), "+r"(acc[7]), "+r"(acc[8]), "+r"(acc[9]), "+r"(acc[10]), "+r"(acc[11]), "+r"(acc[12])
      : "r"(x0), "r"(y0), "r"(x1), "r"(y1), "r"(x2), "r"(y2), "r"(x3), "r"(y3), "r"(x4), "r"(y4));
}
BP_DI void sqr_diag_4_2(u32* acc, u32 x0, u32 y0, u32 x1, u32 y1, u32 x2, u32 y2, u32 x3, u32 y3) {
  asm("mad.lo.cc.u32 %0,%11,%12,%0; madc.hi.cc.u32 %1,%11,%12,%1; madc.lo.cc.u32 %2,%13,%14,%2;"
      "madc.hi.cc.u32 %3,%13,%14,%3; madc.lo.cc.u32 %4,%15,%16,%4; madc.hi.cc.u32 %5,%15,%16,%5;"
      "madc.lo.cc.u32 %6,%17,%18,%6; madc.hi.cc.u32 %7,%17,%18,%7; addc.cc.u32 %8,%8,0; addc.cc.u32 %9,%9,0;"
      "addc.u32 %10,%10,0;"
      : "+r"(acc[0]), "+r"(acc[1]), "+r"(acc[2]), "+r"(acc[3]), "+r"(acc[4]), "+r"(acc[5]), "+r"(acc[6]), "+r"(acc[7]), "+r"(acc[8]), "+r"(acc[9]), "+r"(acc[10])
      : "r"(x0), "r"(y0), "r"(x1), "r"(y1), "r"(x2), "r"(y2), "r"(x3), "r"(y3));
}
BP_DI void sqr_diag_3_4(u32* acc, u32 x0, u32 y0, u32 x1, u32 y1, u32 x2, u32 y2) {
  asm("mad.lo.cc.u32 %0,%11,%12,%0; madc.hi.cc.u32 %1,%11,%12,%1; madc.lo.cc.u32 %2,%13,%14,%2;"
      "madc.hi.cc.u32 %3,%13,%14,%3; madc.lo.cc.u32 %4,%15,%16,%4; madc.hi.cc.u32 %5,%15,%16,%5;"
      "addc.cc.u32 %6,%6,0; addc.cc.u32 %7,%7,0; addc.cc.u32 %8,%8,0; addc.cc.u32 %9,%9,0;"
      "addc.u32 %10,%10,0;"
      : "+r"(acc[0]), "+r"(acc[1]), "+r"(acc[2]), "+r"(acc[3]), "+r"(acc[4]), "+r"(acc[5]), "+r"(acc[6]), "+r"(acc[7]), "+r"(acc[8]), "+r"(acc[9]), "+r"(acc[10])
      : "r"(x0), "r"(y0), "r"(x1), "r"(y1), "r"(x2), "r"(y2));
}
BP_DI void sqr_diag_2_4(u32* acc, u32 x0, u32 y0, u32 x1, u32 y1) {
  asm("mad.lo.cc.u32 %0,%9,%10,%0; madc.hi.cc.u32 %1,%9,%10,%1; madc.lo.cc.u32 %2,%11,%12,%2;"
      "madc.hi.cc.u32 %3,%11,%12,%3; addc.cc.u32 %4,%4,0; addc.cc.u32 %5,%5,0; addc.cc.u32 %6,%6,0;"
      "addc.cc.u32 %7,%7,0; addc.u32 %8,%8,0;"
      : "+r"(acc[0]), "+r"(acc[1]), "+r"(acc[2]), "+r"(acc[3]), "+r"(acc[4]), "+r"(acc[5]), "+r"(acc[6]), "+r"(acc[7]), "+r"(acc[8])
      : "r"(x0), "r"(y0), "r"(x1), "r"(y1));
}
BP_DI void sqr_diag_1_6(u32* acc, u32 x0, u32 y0) {
  asm("mad.lo.cc.u32 %0,%9,%10,%0; madc.hi.cc.u32 %1,%9,%10,%1; addc.cc.u32 %2,%2,0; addc.cc.u32 %3,%3,0;"
      "addc.cc.u32 %4,%4,0; addc.cc.u32 %5,%5,0; addc.cc.u32 %6,%6,0; addc.cc.u32 %7,%7,0; addc.u32 %8,%8,0;"
      : "+r"(acc[0]), "+r"(acc[1]), "+r"(acc[2]), "+r"(acc[3]), "+r"(acc[4]), "+r"(acc[5]), "+r"(acc[6]), "+r"(acc[7]), "+r"(acc[8])
      : "r"(x0), "r"(y0));
}
// t[0..15] = a * a
BP_DI void sqr_wide(u32 t[16], const u32 a[8]) {
  // ev[k] sits at limb k, od[k] at limb k+1
  u32 ev[16], od[16];
  ev[0] = 0; ev[1] = 0; ev[14] = 0; ev[15] = 0; od[14] = 0; od[15] = 0;
  // d = 1: a0a1 a1a2 ... a6a7 at od[0], od[2], ..., od[12];   d = 2: a0a2 ... a5a7 at ev[2], ..., ev[12]
  asm("mul.lo.u32 %0,%14,%15; mul.hi.u32 %1,%14,%15; mul.lo.u32 %2,%15,%16; mul.hi.u32 %3,%15,%16;"
      "mul.lo.u32 %4,%16,%17; mul.hi.u32 %5,%16,%17; mul.lo.u32 %6,%17,%18; mul.hi.u32 %7,%17,%18;"
      "mul.lo.u32 %8,%18,%19; mul.hi.u32 %9,%18,%19; mul.lo.u32 %10,%19,%20; mul.hi.u32 %11,%19,%20;"
      "mul.lo.u32 %12,%20,%21; mul.hi.u32 %13,%20,%21;"
      : "=r"(od[0]), "=r"(od[1]), "=r"(od[2]), "=r"(od[3]), "=r"(od[4]), "=r"(od[5]), "=r"(od[6]), "=r"(od[7]), "=r"(od[8]), "=r"(od[9]),
        "=r"(od[10]), "=r"(od[11]), "=r"(od[12]), "=r"(od[13])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(a[4]), "r"(a[5]), "r"(a[6]), "r"(a[7]));
  asm("mul.lo.u32 %0,%12,%14; mul.hi.u32 %1,%12,%14; mul.lo.u32 %2,%13,%15; mul.hi.u32 %3,%13,%15;"
      "mul.lo.u32 %4,%14,%16; mul.hi.u32 %5,%14,%16; mul.lo.u32 %6,%15,%17; mul.hi.u32 %7,%15,%17;"
      "mul.lo.u32 %8,%16,%18; mul.hi.u32 %9,%16,%18; mul.lo.u32 %10,%17,%19; mul.hi.u32 %11,%17,%19;"
      : "=r"(ev[2]), "=r"(ev[3]), "=r"(ev[4]), "=r"(ev[5]), "=r"(ev[6]), "=r"(ev[7]), "=r"(ev[8]), "=r"(ev[9]), "=r"(ev[10]), "=r"(ev[11]),
        "=r"(ev[12]), "=r"(ev[13])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(a[4]), "r"(a[5]), "r"(a[6]), "r"(a[7]));
  sqr_diag_5_2(od + 2, a[0], a[3], a[1], a[4], a[2], a[5], a[3], a[6], a[4], a[7]);      // d = 3 -> od[2..11], ripple to od[14]
  sqr_diag_4_2(ev + 4, a[0], a[4], a[1], a[5], a[2], a[6], a[3], a[7]);                  // d = 4 -> ev[4..11], ripple to ev[14]
  sqr_diag_3_4(od + 4, a[0], a[5], a[1], a[6], a[2], a[7]);                              // d = 5 -> od[4..9]
  sqr_diag_2_4(ev + 6, a[0], a[6], a[1], a[7]);                                          // d = 6 -> ev[6..9]
  sqr_diag_1_6(od + 6, a[0], a[7]);                                                      // d = 7 -> od[6..7]
  // c = ev + (od << 32)
  u32 c[16];
  c[0] = ev[0];
  asm("add.cc.u32 %0,%15,%30; addc.cc.u32 %1,%16,%31; addc.cc.u32 %2,%17,%32; addc.cc.u32 %3,%18,%33; addc.cc.u32 %4,%19,%34;"
      "addc.cc.u32 %5,%20,%35; addc.cc.u32 %6,%21,%36; addc.cc.u32 %7,%22,%37; addc.cc.u32 %8,%23,%38; addc.cc.u32 %9,%24,%39;"
      "addc.cc.u32 %10,%25,%40; addc.cc.u32 %11,%26,%41; addc.cc.u32 %12,%27,%42; addc.cc.u32 %13,%28,%43; addc.u32 %14,%29,%44;"
      : "=r"(c[1]), "=r"(c[2]), "=r"(c[3]), "=r"(c[4]), "=r"(c[5]), "=r"(c[6]), "=r"(c[7]), "=r"(c[8]), "=r"(c[9]), "=r"(c[10]),
        "=r"(c[11]), "=r"(c[12]), "=r"(c[13]), "=r"(c[14]), "=r"(c[15])
      : "r"(ev[1]), "r"(ev[2]), "r"(ev[3]), "r"(ev[4]), "r"(ev[5]), "r"(ev[6]), "r"(ev[7]), "r"(ev[8]), "r"(ev[9]), "r"(ev[10]),
        "r"(ev[11]), "r"(ev[12]), "r"(ev[13]), "r"(ev[14]), "r"(ev[15]),
        "r"(od[0]), "r"(od[1]), "r"(od[2]), "r"(od[3]), "r"(od[4]), "r"(od[5]), "r"(od[6]), "r"(od[7]), "r"(od[8]), "r"(od[9]),
        "r"(od[10]), "r"(od[11]), "r"(od[12]), "r"(od[13]), "r"(od[14]));
  // double the cross sum (it is < 2^511)
#pragma unroll
  for (int k = 15; k > 0; k--) c[k] = __funnelshift_l(c[k - 1], c[k], 1);
  c[0] <<= 1;
  // + squares a_i^2 at limb 2i: one 16-limb carry chain of 8 IMAD.WIDE
  asm("mad.lo.cc.u32 %0,%8,%8,%0; madc.hi.cc.u32 %1,%8,%8,%1; madc.lo.cc.u32 %2,%9,%9,%2; madc.hi.cc.u32 %3,%9,%9,%3;"
      "madc.lo.cc.u32 %4,%10,%10,%4; madc.hi.cc.u32 %5,%10,%10,%5; madc.lo.cc.u32 %6,%11,%11,%6; madc.hi.cc.u32 %7,%11,%11,%7;"
      : "+r"(c[0]), "+r"(c[1]), "+r"(c[2]), "+r"(c[3]), "+r"(c[4]), "+r"(c[5]), "+r"(c[6]), "+r"(c[7])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]));
  asm("madc.lo.cc.u32 %0,%8,%8,%0; madc.hi.cc.u32 %1,%8,%8,%1; madc.lo.cc.u32 %2,%9,%9,%2; madc.hi.cc.u32 %3,%9,%9,%3;"
      "madc.lo.cc.u32 %4,%10,%10,%4; madc.hi.cc.u32 %5,%10,%10,%5; madc.lo.cc.u32 %6,%11,%11,%6; madc.hi.u32 %7,%11,%11,%7;"
      : "+r"(c[8]), "+r"(c[9]), "+r"(c[10]), "+r"(c[11]), "+r"(c[12]), "+r"(c[13]), "+r"(c[14]), "+r"(c[15])
      : "r"(a[4]), "r"(a[5]), "r"(a[6]), "r"(a[7]));
#pragma unroll
  for (int k = 0; k < 16; k++) t[k] = c[k];
}
BP_DI Fp fp_sqr(const Fp& a) {
  u32 t[16];
  sqr_wide(t, a.v);
  Fp r;
  fold512(r.v, t);
  return r;
}

BP_DI Fp fp_sqr_n(Fp a, int n) {
  for (int i = 0; i < n; i++) a = fp_sqr(a);
  return a;
}
// a^(p-2): 255 squarings + 15 multiplications (addition chain on the run structure of p-2:
// 223 ones, 0, 22 ones, 0000, 1, 0, 11, 0, 1).  Every step is "square n times, multiply by an earlier power", done by
// ONE out-of-line routine with a rolled loop: an inversion is always a single-thread latency chain at the end of a
// kernel, and fully inlined it was 270 KB of straight-line code fetched cold on every call (instruction-cache misses
// cost more than the arithmetic); this form is ~8 KB.
__device__ __noinline__ void fp_sqrn_mul(Fp& x, int n, const Fp& m) {
  Fp t = x;
#pragma unroll 1
  for (int i = 0; i < n; i++) t = fp_sqr(t);
  x = fp_mul(t, m);
}
__device__ __noinline__ Fp fp_inv(const Fp& a) {
  Fp x2 = a; fp_sqrn_mul(x2, 1, a);
  Fp x3 = x2; fp_sqrn_mul(x3, 1, a);
  Fp x6 = x3; fp_sqrn_mul(x6, 3, x3);
  Fp x9 = x6; fp_sqrn_mul(x9, 3, x3);
  Fp x11 = x9; fp_sqrn_mul(x11, 2, x2);
  Fp x22 = x11; fp_sqrn_mul(x22, 11, x11);
  Fp x44 = x22; fp_sqrn_mul(x44, 22, x22);
  Fp x88 = x44; fp_sqrn_mul(x88, 44, x44);
  Fp t = x88; fp_sqrn_mul(t, 88, x88);      // x176
  fp_sqrn_mul(t, 44, x44);                  // x220
  fp_sqrn_mul(t, 3, x3);                    // x223
  fp_sqrn_mul(t, 23, x22);
  fp_sqrn_mul(t, 5, a);
  fp_sqrn_mul(t, 3, x2);
  fp_sqrn_mul(t, 2, a);
  return t;
}

// a^((p+1)/4): the square root of a quadratic residue (p = 3 mod 4); same addition-chain prefix as fp_inv, tail
// x223 -> (23 squarings)*x22 -> (6 squarings)*x2 -> 2 squarings  [(p+1)/4 = 2^254 - 2^30 - 244].  The caller checks
// r^2 == a (non-residues give a root of -a).  Replaces fastecdsa.util.mod_sqrt as used by
// /root/reference/src/utils/elliptic_curve_hash.py:19 and /root/reference/src/utils/utils.py:127.
__device__ __noinline__ Fp fp_sqrt(const Fp& a) {
  Fp x2 = a; fp_sqrn_mul(x2, 1, a);
  Fp x3 = x2; fp_sqrn_mul(x3, 1, a);
  Fp x6 = x3; fp_sqrn_mul(x6, 3, x3);
  Fp x9 = x6; fp_sqrn_mul(x9, 3, x3);
  Fp x11 = x9; fp_sqrn_mul(x11, 2, x2);
  Fp x22 = x11; fp_sqrn_mul(x22, 11, x11);
  Fp x44 = x22; fp_sqrn_mul(x44, 22, x22);
  Fp x88 = x44; fp_sqrn_mul(x88, 44, x44);
  Fp t = x88; fp_sqrn_mul(t, 88, x88);      // x176
  fp_sqrn_mul(t, 44, x44);                  // x220
  fp_sqrn_mul(t, 3, x3);                    // x223
  fp_sqrn_mul(t, 23, x22);
  fp_sqrn_mul(t, 6, x2);
  t = fp_sqr(t);
  return fp_sqr(t);
}

// a^-1 mod p by the binary extended Euclidean algorithm (shifts, adds, subtractions only): for ONE thread finishing an
// MSM this is ~2.4x quicker than the Fermat chain above (~50 k vs 118 k cycles); data-dependent loop counts make it a
// poor fit for warps that invert in lockstep, which keep fp_inv.  Invariants: x1*a = u, x2*a = v (mod p).  0 -> 0.
BP_DI void shr1_256(u32 r[8], u32 top) {      // (top:r) >>= 1
#pragma unroll
  for (int i = 0; i < 7; i++) r[i] = __funnelshift_r(r[i], r[i + 1], 1);
  r[7] = __funnelshift_r(r[7], top, 1);
}
BP_DI void half_mod_p(u32 x[8]) {             // x = x / 2 mod p, x < p
  const u32 P_[8] = {0xFFFFFC2Fu, 0xFFFFFFFEu, 0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu};
  u32 top = 0;
  if (x[0] & 1u) top = add256(x, x, P_);
  shr1_256(x, top);
}
__device__ __noinline__ Fp fp_inv_gcd(const Fp& a_in) {
  const u32 P_[8] = {0xFFFFFC2Fu, 0xFFFFFFFEu, 0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu};
  Fp a = fp_canon(a_in);
  a = fp_canon(a);                              // lazy residues may exceed p by less than 2^33: one pass suffices, two are free
  u32 u[8], v[8], x1[8], x2[8];
#pragma unroll
  for (int i = 0; i < 8; i++) { u[i] = a.v[i]; v[i] = P_[i]; x1[i] = i == 0 ? 1u : 0u; x2[i] = 0u; }
  if (fp_is_zero(a)) return fp_zero();
  for (;;) {
    u32 ou = u[0] ^ 1u, ov = v[0] ^ 1u;
#pragma unroll
    for (int i = 1; i < 8; i++) { ou |= u[i]; ov |= v[i]; }
    if (ou == 0u || ov == 0u) {                 // u == 1 or v == 1
      Fp r;
#pragma unroll
      for (int i = 0; i < 8; i++) r.v[i] = ou == 0u ? x1[i] : x2[i];
      return r;
    }
    while (!(u[0] & 1u)) { shr1_256(u, 0); half_mod_p(x1); }
    while (!(v[0] & 1u)) { shr1_256(v, 0); half_mod_p(x2); }
    u32 d[8];
    if (sub256(d, u, v) == 0u) {                // u >= v
#pragma unroll
      for (int i = 0; i < 8; i++) u[i] = d[i];
      if (sub256(x1, x1, x2)) add256(x1, x1, P_);
    } else {
      sub256(v, v, u);
      if (sub256(x2, x2, x1)) add256(x2, x2, P_);
    }
  }
}

}  // namespace bp
