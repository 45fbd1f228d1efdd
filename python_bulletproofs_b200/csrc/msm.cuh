// msm.cuh -- batched bucket-method multi-scalar multiplication on secp256k1 for sm_100a.
//
// Replaces: Pippenger.multiexp / Pippenger._multiexp_bin
// (/root/reference/src/pippenger/pippenger.py:22-94).  The reference runs Pippenger's subset-table
// method; this is the bucket method (same result: the canonical affine sum of e_i * g_i, scalars
// taken mod q, empty input => identity).
//
// One pipeline serves both shapes on the hot path:
//   * one large MSM (config C3, 2^10..2^20 terms): nmsm = 1, window c up to 16 bits;
//   * many small independent MSMs (L/R of an IPA round, the per-proof verifier equations of
//     config C5): nmsm up to tens of thousands, c = 4..8.
// Stages (all on one stream, no host round trip in between):
//   k_digits      scalars -> sign-normalised signed c-bit digits, bucket histogram (atomics)
//   scan          exclusive prefix sum of the histogram -> bucket_start
//   k_scatter     counting-sort scatter of (term, sign) into bucket order
//   k_accumulate  one thread per bucket: XYZZ += (+/-)affine point, points gathered with 128-bit loads
//   k_reduce_seg  per (msm, window, segment): running-sum trick  sum_i (i+1) * B_i
//   k_window_sum  per (msm, window): tree-sum of the segment results in shared memory
//   k_combine     per msm: Horner over windows (c doublings each), one inversion, canonical affine
#pragma once
#include <cuda_runtime.h>
#include <cstdio>
#include <cstdlib>
#include <cmath>
#include "ec.cuh"
#include "fq.cuh"
#include "glv.cuh"
#include "coop4.cuh"

namespace bp {

#ifndef BP_CHUNK
#define BP_CHUNK 32                // entries per accumulation thread (large problems)
#endif
#define BP_FIXUP_SERIAL_MAX 64     // buckets spanning more chunks than this are summed by a whole block

struct MsmShape {
  int c;          // window bits
  int W;          // windows = ceil(128 / c): the GLV halves are < 2^128 in magnitude
  int U;          // bucket units of H buckets per MSM: W, or W + 1 when c divides 128 -- the top window then takes its
                  // digit unrecoded in [0, 2^c] (it absorbs the signed-digit carry) and owns two consecutive units
  int dbl;        // 1 when the top window owns two units
  u32 H;          // buckets per unit = 2^(c-1)
  u32 chunk;      // entries per accumulation thread (BP_CHUNK, or 8 for small problems where latency rules)
  u32 S;          // buckets per reduce segment
  int seg_plain;  // 1: first reduction level runs one thread per segment (very wide units), 0: one quad per segment
  u32 nseg;       // segments per window
};
#define BP_GLV_BITS 128

// Entries per accumulation thread: small problems want short chains, large ones few partial sums.
inline u32 acc_chunk(double entries) {
  return entries <= 1300000.0 ? 8 : (entries <= 2600000.0 ? 16 : BP_CHUNK);
}

inline MsmShape msm_shape(size_t terms_per_msm, size_t nmsm, int force_c = 0) {
  MsmShape s;
  int best = 1; double bestc = 1e300;
  const double n = (double)terms_per_msm;
  for (int c = 1; c <= 16; c++) {
    double W = (BP_GLV_BITS + c - 1) / c, H = (double)(1u << (c - 1));
    double entries = 2.0 * n * W;                                          // non-zero digits: 2 halves x W windows
    double cost;
    if (nmsm <= 8) {
      // a few MSMs: measured on B200 (profiles/r1_window_sweep.txt).  Windows whose top digit keeps only a few
      // significant bits of the 128-bit halves make hot buckets, so only c = 10, 13, 16 are used: 128 mod c is 8, 11, 0.
      // (n <= 64: c = 5 -- 0.47-0.50 ms against 0.52-0.54 ms at c = 10: the 512-bucket reduction is pure latency there)
      // re-measured after the tail kernels got faster: c = 13 wins from 2^10 (0.534 vs 0.537 ms) to 2^16 (0.758 vs 0.790 at c = 16),
      // c = 16 from 2^17 (0.916 vs 0.977 ms at c = 13)
      int pick = n <= 64.0 ? 5 : (n < 1024.0 ? 10 : (n <= 65536.0 ? 13 : 16));
      cost = c == pick ? 0.0 : 1.0;
    } else {
      // many MSMs: everything is throughput; count field multiplications
      cost = entries * 10 + 2 * W * H * 14 + c * (W - 1) * 9.0 + W * 14;
    }
    if (cost < bestc) { bestc = cost; best = c; }
  }
  s.c = force_c > 0 ? force_c : best;
  s.W = (BP_GLV_BITS + s.c - 1) / s.c;
  s.dbl = (BP_GLV_BITS % s.c) == 0 ? 1 : 0;
  s.U = s.W + s.dbl;
  s.H = 1u << (s.c - 1);
  s.chunk = acc_chunk(2.0 * n * s.W * (double)nmsm);
  // first reduction level: with >= 32768 segments in flight a thread per segment of 4 buckets saturates the SMs
  // (k_reduce_seg_plain); below that the 4-lane cooperative form over 8 buckets has the shorter chain
  s.seg_plain = (nmsm <= 8 && (double)s.U * s.H / 4 >= 32768.0) ? 1 : 0;
  s.S = s.seg_plain ? 4 : (s.H < 8 ? s.H : 8);
  s.nseg = s.H / s.S;
  return s;
}

// ---- scalar -> digits --------------------------------------------------------------------------
BP_DI u32 scalar_bits(const Fq& k, int lo, int n) {   // n <= 16 bits from bit `lo`; bits >= 256 read as 0
  if (lo >= 256) return 0;
  int w = lo >> 5, sh = lo & 31;
  u64 v = k.v[w];
  if (w + 1 < 8) v |= (u64)k.v[w + 1] << 32;
  return (u32)(v >> sh) & ((1u << n) - 1);
}

// msm id of term t given exclusive offsets[0..nmsm]
BP_DI u32 find_msm(const u32* __restrict__ offsets, u32 nmsm, u32 t) {
  u32 lo = 0, hi = nmsm;          // invariant: offsets[lo] <= t < offsets[hi]
  while (hi - lo > 1) { u32 mid = (lo + hi) >> 1; if (__ldg(offsets + mid) <= t) lo = mid; else hi = mid; }
  return lo;
}

// One thread per term: k mod q -> GLV halves (k1, k2) -> sign-normalised magnitudes < 2^128 -> signed c-bit
// digits.  Sub-term 2t carries k1 on P_t, sub-term 2t+1 carries k2 on phi(P_t).  digits is [W][2T].
// skip_idx / skip_below (optional): terms whose point index is below skip_below count as zero scalars -- the caller
// evaluates them elsewhere (fixed-base tables of the batch verifier) and this MSM covers the remaining terms only.
__global__ void __launch_bounds__(256) k_digits(const Fq* __restrict__ scalars, u32 T, const u32* __restrict__ offsets, u32 nmsm,
                                                MsmShape sh, int* __restrict__ digits, u32* __restrict__ bucket_count,
                                                const u32* __restrict__ skip_idx, u32 skip_below) {
  u32 t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= T) return;
  const uint4* sp = reinterpret_cast<const uint4*>(scalars + t);
  uint4 a = __ldg(sp), b = __ldg(sp + 1);
  Fq k; k.v[0] = a.x; k.v[1] = a.y; k.v[2] = a.z; k.v[3] = a.w; k.v[4] = b.x; k.v[5] = b.y; k.v[6] = b.z; k.v[7] = b.w;
  k = fq_reduce(k);                                   // es = [ei % order]   pippenger.py:26
  if (skip_idx && __ldg(skip_idx + t) < skip_below) k = fq_zero();
  Fq half[2];
  bool hneg[2];
  glv_split(k, half[0], hneg[0], half[1], hneg[1]);   // magnitudes < 2^128 and signs
  u32 m = nmsm > 1 ? find_msm(offsets, nmsm, t) : 0;
#pragma unroll
  for (int j = 0; j < 2; j++) {
    const Fq kk = half[j];
    const bool neg = hneg[j];                         // negative half: the digits act on the negated point
    u32 carry = 0;
    for (int w = 0; w < sh.W; w++) {
      u32 d = scalar_bits(kk, w * sh.c, sh.c) + carry;
      int sd;
      // signed recoding below the top window; the top window keeps its digit (<= 2^(c-1) when c does not divide 128,
      // <= 2^c otherwise, where it spills into the second bucket unit) so no further window is needed
      if (w + 1 < sh.W && d > sh.H) { sd = (int)d - (int)(2u * sh.H); carry = 1; } else { sd = (int)d; carry = 0; }
      if (neg) sd = -sd;
      digits[(size_t)w * (2 * (size_t)T) + 2 * t + j] = sd;
      // histogram with warp-aggregated atomics: lanes that hit the same bucket (common for the top window, whose
      // digit has only a few significant bits, and for repeated scalars) issue ONE atomicAdd between them
      u32 mag = sd < 0 ? (u32)(-sd) : (u32)sd;
      u32 bkt = sd != 0 ? (u32)(((size_t)m * sh.U + w) * sh.H + (mag - 1)) : 0xFFFFFFFFu;
      u32 act = __activemask();
      // aggregation only when the warp shows a repeated bucket among neighbouring lanes (hot buckets: repeated scalars,
      // small windows); MATCH.ANY costs more than the atomics it saves when every lane hits its own bucket
      const u32 nb1 = __shfl_xor_sync(act, bkt, 1), nb2 = __shfl_xor_sync(act, bkt, 2);      // (both shuffles before the ||: no lane may skip one)
      const bool rep = __any_sync(act, bkt == nb1 || bkt == nb2);
      if (rep) {
        u32 peers = __match_any_sync(act, bkt);
        if (sd != 0 && (u32)(__ffs(peers) - 1) == (threadIdx.x & 31)) atomicAdd(bucket_count + bkt, (u32)__popc(peers));
      } else if (sd != 0) atomicAdd(bucket_count + bkt, 1u);
    }
  }
}

// one thread per sub-term: entry = {term | phi-flag << 30 | sign << 31, bucket}; cursor[b] starts at bucket_start[b], so the
// atomic hands out absolute slots (one L2 transaction less per entry than offset + separate base load)
__global__ void __launch_bounds__(256) k_scatter(const int* __restrict__ digits, u32 T, const u32* __restrict__ offsets, u32 nmsm,
                                                 MsmShape sh, u32* __restrict__ cursor, uint2* __restrict__ entries, const u32* __restrict__ run_if = nullptr) {
  u32 st = blockIdx.x * blockDim.x + threadIdx.x;
  if (st >= 2 * T) return;
  if (run_if && __ldg(run_if) == 0) return;           // fallback of the slot sort (k_digits_slots): runs only when a bucket overflowed
  u32 t = st >> 1;
  u32 m = nmsm > 1 ? find_msm(offsets, nmsm, t) : 0;
  for (int w = 0; w < sh.W; w++) {
    int sd = digits[(size_t)w * (2 * (size_t)T) + st];
    u32 mag = sd < 0 ? (u32)(-sd) : (u32)sd;
    u32 b = sd != 0 ? (u32)(((size_t)m * sh.U + w) * sh.H + (mag - 1)) : 0xFFFFFFFFu;
    // warp-aggregated cursor: one atomicAdd per distinct bucket per warp, lanes take consecutive slots (here the returning
    // atomics dominate: making the MATCH.ANY conditional as in k_digits measured no gain)
    u32 act = __activemask();
    u32 peers = __match_any_sync(act, b);
    u32 lane = threadIdx.x & 31, leader = (u32)(__ffs(peers) - 1);
    u32 base = 0;
    if (sd != 0 && lane == leader) base = atomicAdd(cursor + b, (u32)__popc(peers));
    base = __shfl_sync(act, base, leader);
    if (sd == 0) continue;
    u32 pos = base + (u32)__popc(peers & ((1u << lane) - 1));     // cursor[] was initialised to bucket_start[]: absolute slot
    entries[pos] = make_uint2(t | ((st & 1u) << 30) | (sd < 0 ? 0x80000000u : 0u), b);
  }
}

// Slot sort of the plain path (one MSM, >= 2^18 terms; see "slot sort" further down): k_digits with the histogram atomic turned
// into the slot hand-out -- digits, one returning atomic and one 4-byte store per entry in a single pass; the digit array is
// still written (coalesced, free) because the gated fallback k_scatter reads it.  Entry = term | phi-flag << 30 | sign << 31.
__global__ void __launch_bounds__(256) k_digits_slots(const Fq* __restrict__ scalars, u32 T, MsmShape sh, int* __restrict__ digits, u32 cap,
                                                      u32* __restrict__ count, u32* __restrict__ slots, u32* __restrict__ overflow) {
  u32 t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= T) return;
  const uint4* sp = reinterpret_cast<const uint4*>(scalars + t);
  uint4 a = __ldg(sp), b = __ldg(sp + 1);
  Fq k; k.v[0] = a.x; k.v[1] = a.y; k.v[2] = a.z; k.v[3] = a.w; k.v[4] = b.x; k.v[5] = b.y; k.v[6] = b.z; k.v[7] = b.w;
  k = fq_reduce(k);
  Fq half[2];
  bool hneg[2];
  glv_split(k, half[0], hneg[0], half[1], hneg[1]);
#pragma unroll
  for (int j = 0; j < 2; j++) {
    const Fq kk = half[j];
    const bool neg = hneg[j];
    u32 carry = 0;
    for (int w = 0; w < sh.W; w++) {
      u32 d = scalar_bits(kk, w * sh.c, sh.c) + carry;
      int sd;
      if (w + 1 < sh.W && d > sh.H) { sd = (int)d - (int)(2u * sh.H); carry = 1; } else { sd = (int)d; carry = 0; }
      if (neg) sd = -sd;
      digits[(size_t)w * (2 * (size_t)T) + 2 * t + j] = sd;
      if (sd == 0) continue;
      const u32 mag = sd < 0 ? (u32)(-sd) : (u32)sd;
      const u32 bkt = (u32)w * sh.H + (mag - 1);
      const u32 r = atomicAdd(count + bkt, 1u);
      if (r < cap) slots[(size_t)bkt * cap + r] = t | ((u32)j << 30) | (sd < 0 ? 0x80000000u : 0u);
      else atomicAdd(overflow, 1u);
    }
  }
}

// phi[t] = (beta * x_t, y_t) for every term (through the optional index list), so that the accumulation
// gathers a ready-made point for the k2 half instead of multiplying by beta once per (sub-term, window).
__global__ void __launch_bounds__(128) k_phi(const Affine* __restrict__ points, const u32* __restrict__ point_idx, u32 T,
                                             Affine* __restrict__ phi) {
  u32 t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= T) return;
  Affine p = ld_affine(points + (point_idx ? __ldg(point_idx + t) : t));
  if (!affine_is_identity(p)) { const Fp beta = {BP_BETA_LIMBS}; p.x = fp_canon(fp_mul(p.x, beta)); }
  st_affine(phi + t, p);
}

// ---- exclusive scan of u32 counts (3 passes; totals < 2^32) ---------------------------------------
#define BP_SCAN_TILE 2048
__global__ void __launch_bounds__(256) k_scan_tiles(const u32* __restrict__ in, u32* __restrict__ out, u32* __restrict__ tile_sum, size_t n) {
  __shared__ u32 sm[256];
  size_t base = (size_t)blockIdx.x * BP_SCAN_TILE + (size_t)threadIdx.x * 8;
  u32 v[8], s = 0;
#pragma unroll
  for (int i = 0; i < 8; i++) { v[i] = base + i < n ? in[base + i] : 0; s += v[i]; }
  sm[threadIdx.x] = s;
  __syncthreads();
  for (int off = 1; off < 256; off <<= 1) {
    u32 x = threadIdx.x >= off ? sm[threadIdx.x - off] : 0;
    __syncthreads();
    sm[threadIdx.x] += x;
    __syncthreads();
  }
  u32 excl = sm[threadIdx.x] - s;
#pragma unroll
  for (int i = 0; i < 8; i++) { if (base + i < n) out[base + i] = excl; excl += v[i]; }
  if (threadIdx.x == 255) tile_sum[blockIdx.x] = sm[255];
}
__global__ void __launch_bounds__(1024) k_scan_sums(u32* __restrict__ tile_sum, size_t ntiles) {   // one block
  __shared__ u32 sm[1024];
  __shared__ u32 carry;
  if (threadIdx.x == 0) carry = 0;
  __syncthreads();
  for (size_t base = 0; base < ntiles; base += 1024) {
    size_t i = base + threadIdx.x;
    u32 s = i < ntiles ? tile_sum[i] : 0;
    sm[threadIdx.x] = s;
    __syncthreads();
    for (int off = 1; off < 1024; off <<= 1) {
      u32 x = threadIdx.x >= off ? sm[threadIdx.x - off] : 0;
      __syncthreads();
      sm[threadIdx.x] += x;
      __syncthreads();
    }
    if (i < ntiles) tile_sum[i] = carry + sm[threadIdx.x] - s;
    __syncthreads();
    if (threadIdx.x == 1023) carry += sm[1023];
    __syncthreads();
  }
}
__global__ void __launch_bounds__(256) k_scan_add(u32* __restrict__ out, const u32* __restrict__ tile_sum, size_t n, u32* __restrict__ total_slot) {
  size_t base = (size_t)blockIdx.x * BP_SCAN_TILE + (size_t)threadIdx.x * 8;
  u32 add = tile_sum[blockIdx.x];
#pragma unroll
  for (int i = 0; i < 8; i++) if (base + i < n) out[base + i] += add;
  (void)total_slot;
}

// ---- bucket accumulation, load-balanced ----------------------------------------------------------
// The bucket-sorted entry list (E entries) is cut into fixed chunks of BP_CHUNK entries, one thread per
// chunk, so every lane performs the same number of mixed additions whatever the bucket-size
// distribution is (uniform scalars, range-proof shaped scalars with thousands of equal digits, windows
// whose top digit has only a few significant bits).  A run of equal bucket ids that lies entirely
// inside a chunk is written straight to buckets[b]; a run cut by a chunk boundary leaves a partial in
// part[2*chunk + 0] (piece starting at the chunk start) or part[2*chunk + 1] (piece starting inside the
// chunk and running past its end); k_fixup adds the pieces of every bucket that spans chunks.
// bucket_start has nb + 1 entries (the last = E).  buckets[] must be zeroed (identity) beforehand.

BP_DI const Affine* entry_point_ptr(const Affine* __restrict__ points, const u32* __restrict__ point_idx,
                                    const Affine* __restrict__ phi, u32 e) {
  u32 t = e & 0x3FFFFFFFu;
  if (e & 0x40000000u) return phi + t;                       // k2 half: phi(P_t), materialised per term
  return points + (point_idx ? __ldg(point_idx + t) : t);
}

#ifndef BP_ACC_MINB
#define BP_ACC_MINB 4
#endif
#ifndef BP_ACC_PIPELINE
#define BP_ACC_PIPELINE 0   // 1: next point loaded into registers under the current addition -- measured slower (2.035 vs 1.984 ms: 128 registers + spill); L2 prefetch only
#endif
__global__ void __launch_bounds__(128, BP_ACC_MINB) k_accumulate(const Affine* __restrict__ points, const u32* __restrict__ point_idx, const Affine* __restrict__ phi,
                                                    const u32* __restrict__ bucket_start, const uint2* __restrict__ entries,
                                                    const u32* __restrict__ gs_ptr, const u32* __restrict__ ge_ptr, u32 CL,
                                                    XYZZ* __restrict__ buckets, XYZZ* __restrict__ part, u32 hb = 0, int into = 0,
                                                    const u32* __restrict__ run_if = nullptr) {
  if (run_if && __ldg(run_if) == 0) return;                              // fallback of the slot sort (k_scatter_slots_pre)
  // hb / into: a host-operand MSM whose points arrive in K parts (msm_run_parts) sorts every part on its own over the same hb
  // bucket ids, and all parts accumulate into ONE set of hb bucket values: from the second part on (into = 1) the first piece of
  // every bucket starts from the stored value instead of the identity.
  // entry range [gs, ge) of this launch: both bounds are bucket_start[] words, read on the device so that no host round trip
  // separates the sort from the accumulation
  u32 chunk = blockIdx.x * blockDim.x + threadIdx.x;
  const u32 gs = __ldg(gs_ptr), E = __ldg(ge_ptr);
  u32 cs = gs + chunk * CL;
  if (cs >= E) return;
  u32 ce = cs + CL < E ? cs + CL : E;
  uint2 ent = __ldg(entries + cs);
  u32 b = ent.y;
  u32 s = __ldg(bucket_start + b), e = __ldg(bucket_start + b + 1);
  bool first = true;
  XYZZ acc = xyzz_identity();
  if (into && s >= cs) acc = ld_xyzz(buckets + b % hb);                  // this chunk holds the first piece of bucket b
#if BP_ACC_PIPELINE
  // software pipeline: the point of entry i+1 is loaded into registers while the mixed addition of entry i runs
  Affine pnext = ld_affine(entry_point_ptr(points, point_idx, phi, ent.x));
#endif
  // ONE flat loop with the same trip count in every lane: the warp stays converged on the mixed add;
  // only the short flush at a bucket boundary diverges.
  for (u32 i = cs; i < ce; i++) {
    if (i == e) {                                                      // previous run is complete
      if (first && s < cs) st_xyzz(part + 2 * (size_t)chunk, acc);     // it began in an earlier chunk
      else st_xyzz(buckets + (hb ? b % hb : b), acc);                  // whole bucket inside this chunk
      first = false;
      b = ent.y;                                                       // next non-empty bucket (ent = entries[i])
      acc = into ? ld_xyzz(buckets + b % hb) : xyzz_identity();
      s = e; e = __ldg(bucket_start + b + 1);
    }
    u32 cur = ent.x;
#if BP_ACC_PIPELINE
    Affine p = pnext;
    if (i + 1 < ce) {
      ent = __ldg(entries + i + 1);
      pnext = ld_affine(entry_point_ptr(points, point_idx, phi, ent.x));
      if (i + 2 < ce) asm volatile("prefetch.global.L2 [%0];" ::"l"(entry_point_ptr(points, point_idx, phi, __ldg(&entries[i + 2].x))));
    }
#else
    if (i + 1 < ce) {
      ent = __ldg(entries + i + 1);
      asm volatile("prefetch.global.L2 [%0];" ::"l"(entry_point_ptr(points, point_idx, phi, ent.x)));
    }
    Affine p = ld_affine(entry_point_ptr(points, point_idx, phi, cur));
#endif
    if (cur >> 31) p.y = fp_neg(p.y);
    xyzz_madd(acc, p);
  }
  if (e > ce) st_xyzz(part + 2 * (size_t)chunk + (first ? 0 : 1), acc);   // run continues in the next chunk
  else if (first && s < cs) st_xyzz(part + 2 * (size_t)chunk, acc);
  else st_xyzz(buckets + (hb ? b % hb : b), acc);
}

// s, c0, c are relative to the launch's first entry gs
BP_DI const XYZZ* bucket_piece(const XYZZ* part, u32 s, u32 c0, u32 c, u32 CL) {
  if (c == c0) return part + 2 * (size_t)c + (s == c0 * CL ? 0 : 1);
  return part + 2 * (size_t)c;
}

// one thread per bucket: buckets spanning up to BP_FIXUP_SERIAL_MAX chunks are summed here, larger ones are queued: up to
// BP_FIXUP_WARP_MAX chunks for k_fixup_mid (one warp each), beyond that for k_fixup_big (one block each).
// queue layout (u32 words): [0] big count, [1] mid count, [2 .. 2+cap) big list, [2+cap .. 2+2cap) mid list
#define BP_FIXUP_WARP_MAX 2048
__global__ void __launch_bounds__(128) k_fixup(const u32* __restrict__ bucket_start, size_t b0, size_t nb, const u32* __restrict__ gs_ptr, u32 CL,
                                               const XYZZ* __restrict__ part, XYZZ* __restrict__ buckets, u32* __restrict__ queue, u32 cap, u32 hb = 0) {
  u32* big_count = queue; u32* mid_count = queue + 1; u32* big_list = queue + 2; u32* mid_list = queue + 2 + cap;
  size_t b = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= nb) return;
  b += b0;
  const u32 gs = __ldg(gs_ptr);
  u32 s = __ldg(bucket_start + b), e = __ldg(bucket_start + b + 1);
  if (e == s) return;
  s -= gs; e -= gs;
  u32 c0 = s / CL, c1 = (e - 1) / CL;
  if (c0 == c1) return;
  if (c1 - c0 >= BP_FIXUP_WARP_MAX) { big_list[atomicAdd(big_count, 1u)] = (u32)b; return; }
  if (c1 - c0 >= BP_FIXUP_SERIAL_MAX) { mid_list[atomicAdd(mid_count, 1u)] = (u32)b; return; }
  XYZZ acc = ld_xyzz(bucket_piece(part, s, c0, c0, CL));
  for (u32 c = c0 + 1; c <= c1; c++) { XYZZ v = ld_xyzz(bucket_piece(part, s, c0, c, CL)); xyzz_add(acc, v); }
  st_xyzz(buckets + (hb ? b % hb : b), acc);
}

// persistent warps over the queue of medium buckets: 32 lanes stride over the pieces, tree in shared memory
__global__ void __launch_bounds__(256) k_fixup_mid(const u32* __restrict__ bucket_start, const u32* __restrict__ gs_ptr, u32 CL,
                                                   const XYZZ* __restrict__ part, XYZZ* __restrict__ buckets, const u32* __restrict__ queue, u32 cap, u32 hb = 0) {
  __shared__ XYZZ sm[8][32];
  const u32 n = queue[1], warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const u32* mid_list = queue + 2 + cap;
  const u32 gs = __ldg(gs_ptr);
  for (u32 q = blockIdx.x * 8 + warp; q < n; q += gridDim.x * 8) {
    const u32 b = mid_list[q];
    const u32 s = __ldg(bucket_start + b) - gs, e = __ldg(bucket_start + b + 1) - gs;
    const u32 c0 = s / CL, c1 = (e - 1) / CL;
    XYZZ acc = xyzz_identity();
    for (u32 c = c0 + lane; c <= c1; c += 32) { XYZZ v = ld_xyzz(bucket_piece(part, s, c0, c, CL)); xyzz_add_ni(acc, v); }
    sm[warp][lane] = acc;
    __syncwarp();
    for (int off = 16; off > 0; off >>= 1) {
      if ((int)lane < off) { XYZZ v = sm[warp][lane + off]; xyzz_add_ni(acc, v); sm[warp][lane] = acc; }
      __syncwarp();
    }
    if (lane == 0) st_xyzz(buckets + (hb ? b % hb : b), acc);
    __syncwarp();
  }
}

// persistent blocks over the queue of giant buckets: 256 threads stride over the pieces, tree in shared memory
__global__ void __launch_bounds__(256) k_fixup_big(const u32* __restrict__ bucket_start, const u32* __restrict__ gs_ptr, u32 CL,
                                                   const XYZZ* __restrict__ part, XYZZ* __restrict__ buckets, const u32* __restrict__ queue, u32 hb = 0) {
  __shared__ XYZZ sm[256];
  const u32* big_list = queue + 2;
  u32 n = queue[0];
  const u32 gs = __ldg(gs_ptr);
  for (u32 q = blockIdx.x; q < n; q += gridDim.x) {
    u32 b = big_list[q];
    u32 s = __ldg(bucket_start + b) - gs, e = __ldg(bucket_start + b + 1) - gs;
    u32 c0 = s / CL, c1 = (e - 1) / CL;
    XYZZ acc = xyzz_identity();
    for (u32 c = c0 + threadIdx.x; c <= c1; c += blockDim.x) { XYZZ v = ld_xyzz(bucket_piece(part, s, c0, c, CL)); xyzz_add_ni(acc, v); }
    sm[threadIdx.x] = acc;
    __syncthreads();
    for (int off = (int)blockDim.x >> 1; off > 0; off >>= 1) {
      if (threadIdx.x < off) { XYZZ v = sm[threadIdx.x + off]; xyzz_add_ni(acc, v); sm[threadIdx.x] = acc; }
      __syncthreads();
    }
    if (threadIdx.x == 0) st_xyzz(buckets + (hb ? b % hb : b), acc);
    __syncthreads();
  }
}

// ---- tails: bucket reduction, window sums, Horner -- 4 lanes per point operation (coop4.cuh) -------------
// Level 1 -- one QUAD per (msm*W + w, seg): plain and weighted sums of the S buckets of a segment by the running-sum
// trick:  run = sum_i B[i],  sum = sum_i (i+1) * B[i].
__global__ void __launch_bounds__(128) k_reduce_seg(const XYZZ* __restrict__ buckets, MsmShape sh, size_t nmw,
                                                    XYZZ* __restrict__ seg_run, XYZZ* __restrict__ seg_sum) {
  const size_t total = nmw * sh.nseg;
  size_t qid = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 2;
  const int lane = threadIdx.x & 31, role = lane & 3, base = lane & ~3;
  const bool active = qid < total;
  if (!active) qid = total - 1;                       // idle quads shadow the last one (shuffles need the whole warp)
  const XYZZ* B = buckets + qid * sh.S;               // segments are contiguous: (mw * nseg + seg) * S
  XYZZ run = xyzz_identity(), sum = xyzz_identity();
  for (int i = (int)sh.S - 1; i >= 0; i--) {
    XYZZ bk = ld_xyzz(B + i);
    run = coop_add(run, bk, role, base);
    sum = coop_add(sum, run, role, base);
  }
  if (active && role == 0) { st_xyzz(seg_run + qid, run); st_xyzz(seg_sum + qid, sum); }
}

// Level 1, throughput form: one THREAD per segment (used when tens of thousands of segments are in flight).
__global__ void __launch_bounds__(128) k_reduce_seg_plain(const XYZZ* __restrict__ buckets, MsmShape sh, size_t nmw,
                                                          XYZZ* __restrict__ seg_run, XYZZ* __restrict__ seg_sum) {
  const size_t total = nmw * sh.nseg;
  size_t q = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= total) return;
  const XYZZ* B = buckets + q * sh.S;
  XYZZ run = xyzz_identity(), sum = xyzz_identity();
  for (int i = (int)sh.S - 1; i >= 0; i--) {
    XYZZ bk = ld_xyzz(B + i);
    xyzz_add_ni(run, bk);
    xyzz_add_ni(sum, run);
  }
  st_xyzz(seg_run + q, run);
  st_xyzz(seg_sum + q, sum);
}

// Level 2 -- one QUAD per group of G consecutive segments of one window (G = 16, or nseg when smaller).  With segment
// j of group u starting at bucket (u*G + j)*S, the group's share of  sum_b (b+1) * B_b  is
//   P + S * T + (u*G*S) * R,   P = sum_j seg_sum_j,  T = sum_j j * seg_run_j,  R = sum_j seg_run_j,
// where the last product is a double-and-add over the bits of u followed by log2(G*S) doublings.
__global__ void __launch_bounds__(128) k_reduce_grp(const XYZZ* __restrict__ seg_run, const XYZZ* __restrict__ seg_sum, MsmShape sh,
                                                    size_t nmw, u32 unit0, u32 G, int lgS, int lgG, int ubits, XYZZ* __restrict__ grpsum) {
  const u32 ngrp = sh.nseg / G;
  const size_t total = nmw * ngrp;
  size_t qid = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 2;
  const int lane = threadIdx.x & 31, role = lane & 3, base = lane & ~3;
  const bool active = qid < total;
  if (!active) qid = total - 1;
  u32 u = (u32)(qid % ngrp);
  if (sh.dbl && (int)((qid / ngrp + unit0) % sh.U) == sh.U - 1) u += ngrp;   // second unit of the top window: weights continue at H
  const XYZZ* Rn = seg_run + qid * G;
  const XYZZ* Sm = seg_sum + qid * G;
  XYZZ run = xyzz_identity(), T = xyzz_identity(), P = xyzz_identity();
  for (int j = (int)G - 1; j >= 0; j--) {
    XYZZ r = ld_xyzz(Rn + j), sj = ld_xyzz(Sm + j);
    run = coop_add(run, r, role, base);
    if (j > 0) T = coop_add(T, run, role, base);                             // weights j = 0..G-1 (uniform branch)
    P = coop_add(P, sj, role, base);
  }
  // S * T, then u * R by double-and-add, then * G * S: one doubling site and one addition site (code size)
  XYZZ acc = xyzz_identity();
  const int nd = ubits > 0 ? ubits + lgS + lgG : 0;
  for (int d = 0; d < lgS + nd; d++) {
    const bool onT = d < lgS;
    XYZZ x = sel_xyzz(onT, T, acc);
    x = coop_dbl(x, role, base);
    if (onT) T = x; else acc = x;
    const int i = ubits - 1 - (d - lgS);                                     // bit of u consumed after this doubling
    if (!onT && i >= 0) {
      XYZZ t = coop_add(acc, run, role, base);
      acc = sel_xyzz((u >> i) & 1, t, acc);
    }
  }
#pragma unroll 1
  for (int k = 0; k < 2; k++) P = coop_add(P, k == 0 ? T : acc, role, base);
  if (active && role == 0) st_xyzz(grpsum + qid, P);
}

// one block (256 threads = 64 quads) per (msm, window): winsum = sum of nseg segment results
__global__ void __launch_bounds__(256) k_window_sum(const XYZZ* __restrict__ segsum, u32 nseg, XYZZ* __restrict__ winsum) {
  __shared__ XYZZ sm[64];
  const size_t mw = blockIdx.x;
  const int lane = threadIdx.x & 31, role = lane & 3, base = lane & ~3;
  const u32 q = threadIdx.x >> 2, nq = blockDim.x >> 2;      // nq quads, a power of two <= 64
  XYZZ acc = xyzz_identity();
  for (u32 i0 = 0; i0 < nseg; i0 += nq) {             // uniform trip count; out-of-range quads add the identity
    u32 i = i0 + q;
    XYZZ v = i < nseg ? ld_xyzz(segsum + mw * nseg + i) : xyzz_identity();
    acc = coop_add(acc, v, role, base);
  }
  if (role == 0) sm[q] = acc;
  __syncthreads();
  for (u32 off = nq >> 1; off > 0; off >>= 1) {
    XYZZ v = (q < off) ? sm[q + off] : xyzz_identity();
    acc = coop_add(acc, v, role, base);
    __syncthreads();
    if (q < off && role == 0) sm[q] = acc;
    __syncthreads();
  }
  if (threadIdx.x == 0) st_xyzz(winsum + mw, acc);
}

// ---- throughput variants of the tails for large batches of small MSMs (one thread per unit / per MSM) -------------
// With tens of thousands of MSMs in flight every lane already has its own independent chain, so the 4-lane
// cooperative forms would only waste lanes.  Used when a unit is a single segment (H <= 16).
__global__ void __launch_bounds__(128) k_reduce_unit_plain(const XYZZ* __restrict__ buckets, MsmShape sh, size_t nmw, XYZZ* __restrict__ unitsum) {
  size_t id = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (id >= nmw) return;
  const XYZZ* B = buckets + id * sh.H;
  XYZZ run = xyzz_identity(), sum = xyzz_identity();
  for (int i = (int)sh.H - 1; i >= 0; i--) {
    XYZZ b = ld_xyzz(B + i);
    xyzz_add_ni(run, b);
    xyzz_add_ni(sum, run);
  }
  if (sh.dbl && (int)(id % sh.U) == sh.U - 1) {        // second unit of the top window: weights H + i + 1
    XYZZ t = run;
    for (int d = 0; d < sh.c - 1; d++) t = xyzz_dbl_ni(t);
    xyzz_add_ni(sum, t);
  }
  st_xyzz(unitsum + id, sum);
}
__global__ void __launch_bounds__(128) k_combine_plain(const XYZZ* __restrict__ winsum, MsmShape sh, size_t nmsm, Affine* __restrict__ out,
                                                       XYZZ* __restrict__ out_xyzz) {
  size_t m = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (m >= nmsm) return;
  const XYZZ* ws = winsum + m * sh.U;
  XYZZ acc = ld_xyzz(ws + sh.U - 1);
  if (sh.dbl) { XYZZ v = ld_xyzz(ws + sh.U - 2); xyzz_add_ni(acc, v); }
  for (int w = sh.W - 2; w >= 0; w--) {
    for (int d = 0; d < sh.c; d++) acc = xyzz_dbl_ni(acc);
    XYZZ v = ld_xyzz(ws + w);
    xyzz_add_ni(acc, v);
  }
  if (out_xyzz) st_xyzz(out_xyzz + m, acc);
  if (out) st_affine(out + m, xyzz_to_affine(acc));
}

// one QUAD per msm: Horner over windows (c doublings each), then canonical affine (optionally XYZZ partials for sharding)
__global__ void __launch_bounds__(128) k_combine(const XYZZ* __restrict__ winsum, MsmShape sh, size_t nmsm, Affine* __restrict__ out,
                                                 XYZZ* __restrict__ out_xyzz) {
  size_t m = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 2;
  const int lane = threadIdx.x & 31, role = lane & 3, base = lane & ~3;
  const bool active = m < nmsm;
  if (!active) m = nmsm - 1;
  const XYZZ* ws = winsum + m * sh.U;
  XYZZ acc = ld_xyzz(ws + sh.U - 1);
  if (sh.dbl) { XYZZ v = ld_xyzz(ws + sh.U - 2); acc = coop_add(acc, v, role, base); }     // both units of the top window
  for (int w = sh.W - 2; w >= 0; w--) {
    for (int d = 0; d < sh.c; d++) acc = coop_dbl(acc, role, base);
    XYZZ v = ld_xyzz(ws + w);
    acc = coop_add(acc, v, role, base);
  }
  if (!active || role != 0) return;
  if (out_xyzz) st_xyzz(out_xyzz + m, acc);
  if (out) st_affine(out + m, xyzz_to_affine(acc, nmsm <= 2));
}

// ---- resident point vectors with precomputed window multiples ("pre" path) ---------------------------------------------------
// For a point vector that stays in HBM across many MSMs (bp_points_precompute: the generator vectors of a commitment scheme, the
// resident operand of the C3 benchmark) the multiples 2^(c*w) * P_i, w = 0 .. W-1, are stored once (W * 64 bytes per point:
// 0.94 GB for 2^20 points at c = 19 -- HBM3e capacity spent to delete work).  Every signed c-bit digit of a 256-bit scalar then
// addresses a ready-made point, so ALL windows share ONE unit of 2^(c-1) buckets:
//   * no Horner chain over windows (the 112 dependent doublings of k_combine), one bucket reduction instead of U of them;
//   * the bucket unit no longer multiplies with the window count, so the window can widen (c = 19: 14 mixed additions per
//     point instead of 16) while the reduction stays at 2^18 buckets;
//   * no endomorphism split: a 256-bit scalar over W windows costs the same additions as two 128-bit halves over W/2, and the
//     digit kernel loses its two 256x256-bit products per scalar, k_phi disappears.
// Same sort / accumulate / fix-up / reduce kernels as the plain path: an entry's point index is w * stride + first + t.
// The 257 bits a signed recoding of k < q needs are dealt out EVENLY over the W = ceil(257/c) windows (widths c or c-1): a top
// window of only a few bits would put its whole share of the entries into a handful of buckets (hot atomics in the sort,
// buckets cut into hundreds of chunks).
#define BP_PRE_MAXW 33
struct PreShape { int c, W; u32 H; unsigned short off[BP_PRE_MAXW + 1]; };   // window w covers scalar bits [off[w], off[w+1])
inline PreShape pre_shape(int c) {
  PreShape p; p.c = c; p.W = (257 + c - 1) / c; p.H = 1u << (c - 1);
  const int base = 257 / p.W, extra = 257 % p.W;           // `extra` windows of base + 1 bits (the low ones), the rest base bits
  int o = 0;
  for (int w = 0; w <= BP_PRE_MAXW; w++) { p.off[w] = (unsigned short)o; if (w < p.W) o += base + (w < extra ? 1 : 0); }
  return p;
}
inline int pre_pick_window(size_t n) {     // measured on B200 (profiles/r2_pre_window_sweep.txt): best window per vector length
  return n < ((size_t)1 << 13) ? 13 : (n < ((size_t)1 << 15) ? 15 : (n < ((size_t)1 << 19) ? 17 : 18));
}

// One thread per point: out[w * n + i] = 2^off[w] * P_i (canonical affine), one inversion per point (Montgomery's trick over the
// W Z coordinates), doublings in Jacobian coordinates (2M + 5S).
__global__ void __launch_bounds__(128) k_pre_build(const Affine* __restrict__ pts, u32 n, PreShape ps, Affine* __restrict__ out) {
  const u32 i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const Affine P = ld_affine(pts + i);
  st_affine(out + i, P);
  if (affine_is_identity(P)) {
    for (int w = 1; w < ps.W; w++) st_affine(out + (size_t)w * n + i, P);
    return;
  }
  // Jacobian chain: J_w = 2^(c*w) P; X, Y parked in the output slots, Z products kept in local memory
  Fp X = P.x, Y = P.y, Z = fp_one();
  Fp zs[BP_PRE_MAXW], pre[BP_PRE_MAXW];
  Fp acc = fp_one();
  for (int w = 1; w < ps.W; w++) {
#pragma unroll 1
    for (int d = ps.off[w - 1]; d < ps.off[w]; d++) {
      const Fp A = fp_sqr(X), B = fp_sqr(Y), C = fp_sqr(B);
      const Fp D = fp_dbl(fp_sub(fp_sub(fp_sqr(fp_add(X, B)), A), C));
      const Fp E = fp_add(fp_dbl(A), A);
      const Fp X3 = fp_sub(fp_sqr(E), fp_dbl(D));
      const Fp Z3 = fp_dbl(fp_mul(Y, Z));
      Y = fp_sub(fp_mul(E, fp_sub(D, X3)), fp_dbl(fp_dbl(fp_dbl(C))));
      X = X3; Z = Z3;
    }
    Affine t; t.x = X; t.y = Y;
    st_affine(out + (size_t)w * n + i, t);          // Jacobian X, Y for now
    zs[w] = Z;
    acc = fp_mul(acc, Z);
    pre[w] = acc;                                   // Z_1 ... Z_w  (never zero: P has prime order)
  }
  Fp inv = fp_inv(acc);
  for (int w = ps.W - 1; w >= 1; w--) {
    const Fp zi = w > 1 ? fp_mul(inv, pre[w - 1]) : inv;      // Z_w^-1
    inv = fp_mul(inv, zs[w]);
    const Fp zi2 = fp_sqr(zi), zi3 = fp_mul(zi2, zi);
    Affine* slot = out + (size_t)w * n + i;
    Affine t;
    t.x = fp_canon(fp_mul(ld_fp_plain(&slot->x), zi2));
    t.y = fp_canon(fp_mul(ld_fp_plain(&slot->y), zi3));
    st_affine(slot, t);
  }
}

// signed digit of window w of the reduced scalar k (carry = the recoding carry out of window w-1, updated)
BP_DI int pre_digit(const Fq& k, const PreShape& ps, int w, u32& carry) {
  // window w covers bits [off, off + width): the `extra` low windows are one bit wider (pre_shape) -- computed, not read from
  // ps.off[]: a dynamically indexed kernel parameter is copied to local memory, 2 more LSU requests per digit in kernels that
  // are bound by exactly those
  const int base = 257 / ps.W, extra = 257 % ps.W;
  const int width = base + (w < extra ? 1 : 0), off = w * base + (w < extra ? w : extra);
  const u32 half = 1u << (width - 1);
  const u32 d = scalar_bits(k, off, width) + carry;
  // (the top window holds bit 256, which is clear: its digit stays <= half without recoding)
  if (w + 1 < ps.W && d > half) { carry = 1; return (int)d - (int)(2u * half); }
  carry = 0;
  return (int)d;
}
BP_DI Fq pre_load_scalar(const Fq* __restrict__ scalars, u32 t) {
  const uint4* sp = reinterpret_cast<const uint4*>(scalars + t);
  uint4 a = __ldg(sp), b = __ldg(sp + 1);
  Fq k; k.v[0] = a.x; k.v[1] = a.y; k.v[2] = a.z; k.v[3] = a.w; k.v[4] = b.x; k.v[5] = b.y; k.v[6] = b.z; k.v[7] = b.w;
  return fq_reduce(k);                                  // es = [ei % order]   pippenger.py:26
}
// One thread per term: k mod q -> W signed digits of the windows of `ps`, histogram over the single bucket unit.  No digit array:
// the scatter pass derives the digits again from the scalar (32 bytes read instead of 4 W written and read back).
__global__ void __launch_bounds__(256) k_digits_pre(const Fq* __restrict__ scalars, u32 T, PreShape ps, u32* __restrict__ bucket_count) {
  const u32 t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= T) return;
  const Fq k = pre_load_scalar(scalars, t);
  u32 carry = 0;
  for (int w = 0; w < ps.W; w++) {
    const int sd = pre_digit(k, ps, w, carry);
    if (sd != 0) atomicAdd(bucket_count + ((sd < 0 ? (u32)(-sd) : (u32)sd) - 1u), 1u);
  }
}

// counting-sort scatter: entry = {point index | sign << 31, bucket}, point index = w * stride + first + t
__global__ void __launch_bounds__(256) k_scatter_pre(const Fq* __restrict__ scalars, u32 T, PreShape ps, u32 stride, u32 first,
                                                     u32* __restrict__ cursor, uint2* __restrict__ entries, const u32* __restrict__ run_if = nullptr) {
  const u32 t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= T) return;
  if (run_if && __ldg(run_if) == 0) return;             // fallback of the slot sort: runs only when a bucket overflowed its slots
  const Fq k = pre_load_scalar(scalars, t);
  u32 carry = 0;
  for (int w = 0; w < ps.W; w++) {
    const int sd = pre_digit(k, ps, w, carry);
    if (sd == 0) continue;
    const u32 bkt = (sd < 0 ? (u32)(-sd) : (u32)sd) - 1u;
    const u32 pos = atomicAdd(cursor + bkt, 1u);        // cursor[] starts at bucket_start[]: absolute slot
    entries[pos] = make_uint2(((u32)w * stride + first + t) | (sd < 0 ? 0x80000000u : 0u), bkt);
  }
}

// ---- slot sort: ONE scattered pass instead of histogram + scatter -------------------------------------------------------------
// Both passes of the counting sort run at the same ~0.47 scattered L2 requests per clock and SM (15.7 M RED in 111 us, 15.7 M ATOM +
// 15.7 M 8-byte stores in 232 us at 2^20; profiles/r2_sort_ncu.txt) -- what counts is the NUMBER of scattered requests per entry:
// three.  For scalars whose digits spread evenly the histogram can be skipped: bucket b owns a fixed range of `cap` 4-byte slots
// (cap = mean + 9.5 sigma of the fullest buckets' Poisson load), one returning atomic on count[b] hands out the slot, the entry is
// stored there: two requests per entry, and the atomics leave count[] exactly as the histogram pass would.  The exclusive scan
// of count[] still runs: k_accumulate_slots cuts the COMPACT index space [0, E) into equal chunks (same load balance, same
// partial sums, same fix-up kernels) and maps index i of bucket b to slots[b * cap + (i - start[b])].  An entry that finds its
// bucket full bumps *overflow; then this path's accumulation returns at once and the exact counting sort + k_accumulate, queued
// behind it and gated on the same word, do the work (scalars with thousands of equal digits: range-proof vectors).
// B = windows handled together: the B returning atomics of a group are issued back to back, then the B stores (B = 1 / 4 / 8:
// 2.280 / 2.275 / 2.283 ms per 2^20-term MSM -- the pass is bound by the request rate, not by the latency of one atomic)
template <int B>
__global__ void __launch_bounds__(256) k_scatter_slots_pre(const Fq* __restrict__ scalars, u32 T, PreShape ps, u32 stride, u32 first, u32 cap,
                                                           u32* __restrict__ count, u32* __restrict__ slots, u32* __restrict__ overflow) {
  const u32 t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= T) return;
  const Fq k = pre_load_scalar(scalars, t);
  u32 carry = 0;
  for (int w0 = 0; w0 < ps.W; w0 += B) {
    int sd[B]; u32 r[B];
#pragma unroll
    for (int j = 0; j < B; j++) sd[j] = w0 + j < ps.W ? pre_digit(k, ps, w0 + j, carry) : 0;
#pragma unroll
    for (int j = 0; j < B; j++)
      if (sd[j] != 0) r[j] = atomicAdd(count + ((sd[j] < 0 ? (u32)(-sd[j]) : (u32)sd[j]) - 1u), 1u);
#pragma unroll
    for (int j = 0; j < B; j++) {
      if (sd[j] == 0) continue;
      const u32 bkt = (sd[j] < 0 ? (u32)(-sd[j]) : (u32)sd[j]) - 1u;
      if (r[j] < cap) slots[(size_t)bkt * cap + r[j]] = ((u32)(w0 + j) * stride + first + t) | (sd[j] < 0 ? 0x80000000u : 0u);
      else atomicAdd(overflow, 1u);
    }
  }
}
// k_accumulate over the slot layout (precomputed path: direct point indices, no phi, no parts).  bucket_start[0 .. nb] is the
// exclusive scan of the bucket counts; chunk boundaries, part[] and buckets[] are exactly those of k_accumulate.
// PHI: entries carry the phi flag of the plain path (bit 30: the point is phi[t], materialised per term by k_phi)
template <bool PHI>
BP_DI const Affine* slot_point_ptr(const Affine* __restrict__ points, const Affine* __restrict__ phi, u32 e) {
  if (PHI) return ((e & 0x40000000u) ? phi : points) + (e & 0x3FFFFFFFu);
  return points + (e & 0x7FFFFFFFu);
}
template <bool PHI>
__global__ void __launch_bounds__(128, BP_ACC_MINB) k_accumulate_slots(const Affine* __restrict__ points, const Affine* __restrict__ phi,
                                                                       const u32* __restrict__ bucket_start, u32 nb,
                                                                       const u32* __restrict__ slots, u32 cap, const u32* __restrict__ overflow, u32 CL,
                                                                       XYZZ* __restrict__ buckets, XYZZ* __restrict__ part) {
  if (__ldg(overflow) != 0) return;
  const u32 chunk = blockIdx.x * blockDim.x + threadIdx.x;
  const u32 E = __ldg(bucket_start + nb);
  const u32 cs = chunk * CL;
  if (cs >= E) return;
  const u32 ce = cs + CL < E ? cs + CL : E;
  u32 b = 0;
  {   // the bucket that holds compact index cs: the largest b with bucket_start[b] <= cs (empty buckets share their successor's start)
    u32 hi = nb;
    while (hi - b > 1) { const u32 mid = (b + hi) >> 1; if (__ldg(bucket_start + mid) <= cs) b = mid; else hi = mid; }
  }
  u32 s = __ldg(bucket_start + b), e = __ldg(bucket_start + b + 1);
  const u32* sp = slots + (size_t)b * cap - s;                            // entry i of bucket b
  bool first = true;
  XYZZ acc = xyzz_identity();
  u32 ent = __ldg(sp + cs);
  for (u32 i = cs; i < ce; i++) {
    if (i == e) {                                                        // previous run is complete
      if (first && s < cs) st_xyzz(part + 2 * (size_t)chunk, acc);       // it began in an earlier chunk
      else st_xyzz(buckets + b, acc);                                    // whole bucket inside this chunk
      first = false;
      do { b++; s = e; e = __ldg(bucket_start + b + 1); } while (e == s);      // next non-empty bucket (i < E: there is one)
      acc = xyzz_identity();
      sp = slots + (size_t)b * cap - s;
      ent = __ldg(sp + i);
    }
    const u32 cur = ent;
    if (i + 1 < ce && i + 1 < e) {                                       // (across a bucket boundary the entry is fetched after the flush)
      ent = __ldg(sp + i + 1);
      asm volatile("prefetch.global.L2 [%0];" ::"l"(slot_point_ptr<PHI>(points, phi, ent)));
    }
    Affine p = ld_affine(slot_point_ptr<PHI>(points, phi, cur));
    if (cur >> 31) p.y = fp_neg(p.y);
    xyzz_madd(acc, p);
  }
  if (e > ce) st_xyzz(part + 2 * (size_t)chunk + (first ? 0 : 1), acc);   // run continues in the next chunk
  else if (first && s < cs) st_xyzz(part + 2 * (size_t)chunk, acc);
  else st_xyzz(buckets + b, acc);
}

// ---- reduction of ONE large bucket unit (H = R x C buckets, b = hi*C + lo) -----------------------------------------------------
//   sum_b (b+1) B_b  =  sum_lo (lo+1) * Col_lo  +  C * sum_hi hi * Row_hi,     Col_lo = sum_hi B[hi][lo],  Row_hi = sum_lo B[hi][lo]
// The 2H additions of the marginal sums are plain sums (trees of independent thread-level additions, throughput bound); only
// the R + C marginals enter a weighted stage, each with a <= 10-bit weight (double-and-add per element, then a tree).  The
// running-sum form of the plain path (k_reduce_seg / k_reduce_grp) carries a dependent chain through every level instead.
// One launch reduces rows and columns by a factor K each (blockIdx.y = 0: rows, contiguous; 1: columns, strided):
//   rows: out[i] = sum_{k<K} in[i*K + k]           (i < nrow_out)
//   cols: out[g*C + lo] = sum_{k<K} in[(g*K + k)*C + lo]   (g < ncol_groups, lo < C)
__global__ void __launch_bounds__(128) k_pre_marginals(const XYZZ* __restrict__ row_in, XYZZ* __restrict__ row_out, u32 nrow_out, u32 Krow,
                                                       const XYZZ* __restrict__ col_in, XYZZ* __restrict__ col_out, u32 ncol_groups, u32 C, u32 Kcol) {
  const u32 i = blockIdx.x * blockDim.x + threadIdx.x;
  if (blockIdx.y == 0) {
    if (i >= nrow_out || Krow == 0) return;
    const XYZZ* src = row_in + (size_t)i * Krow;
    XYZZ acc = ld_xyzz(src);
#pragma unroll 1
    for (u32 k = 1; k < Krow; k++) { XYZZ v = ld_xyzz(src + k); xyzz_add_ni(acc, v); }
    st_xyzz(row_out + i, acc);
  } else {
    if (i >= ncol_groups * C || Kcol == 0) return;
    const u32 gq = i / C, lo = i % C;
    const XYZZ* src = col_in + (size_t)gq * Kcol * C + lo;
    XYZZ acc = ld_xyzz(src);
#pragma unroll 1
    for (u32 k = 1; k < Kcol; k++) { XYZZ v = ld_xyzz(src + (size_t)k * C); xyzz_add_ni(acc, v); }
    st_xyzz(col_out + i, acc);
  }
}
// Second level + weights: one block of 64 threads = 16 quads per marginal (blocks 0 .. C-1: column lo, weight lo + 1; blocks
// C .. C+R-1: row hi, weight hi).  4-lane cooperative operations throughout (coop4.cuh: ~2 us per addition against ~4-8 us for
// a lone thread's out-of-line call): the quads add the marginal's np partial sums (np <= 128, a power of two), a shared-memory
// tree joins them, the first quad multiplies by the <= 11-bit weight (double-and-add) and stores wsum[block].
__global__ void __launch_bounds__(64) k_pre_rowcol(const XYZZ* __restrict__ rowpart, u32 np_r, const XYZZ* __restrict__ colpart, u32 np_c,
                                                   u32 C, u32 R, XYZZ* __restrict__ wsum) {
  __shared__ XYZZ sm[16];
  const u32 bq = blockIdx.x, t = threadIdx.x, q = t >> 2;
  const int lane = t & 31, role = lane & 3, base = lane & ~3;
  const bool is_col = bq < C;
  const u32 j = is_col ? bq : bq - C, np = is_col ? np_c : np_r;
  XYZZ acc = xyzz_identity();
  for (u32 e0 = 0; e0 < np; e0 += 16) {                  // uniform trip count; quads past the end add the identity
    const u32 e = e0 + q;
    XYZZ v = e < np ? ld_xyzz(is_col ? colpart + (size_t)e * C + j : rowpart + (size_t)j * np_r + e) : xyzz_identity();
    acc = coop_add(acc, v, role, base);
  }
  if (role == 0) sm[q] = acc;
  __syncthreads();
  for (u32 off = 8; off > 0; off >>= 1) {
    XYZZ v = q < off ? sm[q + off] : xyzz_identity();
    acc = coop_add(acc, v, role, base);
    __syncthreads();
    if (q < off && role == 0) sm[q] = acc;
    __syncthreads();
  }
  if (t >= 32) return;                                   // the first warp (quad 0 holds the sum; its other quads shadow it)
  acc = sm[0];
  const u32 wgt = is_col ? j + 1 : j;
  XYZZ r = xyzz_identity();
  for (int bit = 31 - __clz(wgt | 1u); bit >= 0; bit--) {
    r = coop_dbl(r, role, base);
    XYZZ s2 = coop_add(r, acc, role, base);
    r = sel_xyzz((wgt >> bit) & 1u, s2, r);
  }
  if (t == 0) st_xyzz(wsum + bq, r);
}
// sums[side] = sum of wsum[side == 0 ? 0 .. C : C .. C+R): one block of 256 threads = 64 quads per side
__global__ void __launch_bounds__(256) k_pre_total(const XYZZ* __restrict__ wsum, u32 C, u32 R, XYZZ* __restrict__ sums) {
  __shared__ XYZZ sm[64];
  const u32 side = blockIdx.x, t = threadIdx.x, q = t >> 2, n = side == 0 ? C : R;
  const int lane = t & 31, role = lane & 3, base = lane & ~3;
  const XYZZ* src = wsum + (side == 0 ? 0u : C);
  XYZZ acc = xyzz_identity();
  for (u32 e0 = 0; e0 < n; e0 += 64) {
    const u32 e = e0 + q;
    XYZZ v = e < n ? ld_xyzz(src + e) : xyzz_identity();
    acc = coop_add(acc, v, role, base);
  }
  if (role == 0) sm[q] = acc;
  __syncthreads();
  for (u32 off = 32; off > 0; off >>= 1) {
    XYZZ v = q < off ? sm[q + off] : xyzz_identity();
    acc = coop_add(acc, v, role, base);
    __syncthreads();
    if (q < off && role == 0) sm[q] = acc;
    __syncthreads();
  }
  if (t == 0) st_xyzz(sums + side, acc);
}
// result = sums[0] + 2^lgC * sums[1]  (sums[0] = weighted columns, sums[1] = weighted rows); one quad
__global__ void __launch_bounds__(32) k_pre_finish(const XYZZ* __restrict__ sums, int lgC, Affine* __restrict__ out, XYZZ* __restrict__ out_xyzz) {
  const int lane = threadIdx.x & 31, role = lane & 3, base = lane & ~3;
  XYZZ acc = ld_xyzz(sums + 1);
  for (int d = 0; d < lgC; d++) acc = coop_dbl(acc, role, base);
  XYZZ v = ld_xyzz(sums);
  acc = coop_add(acc, v, role, base);
  if (threadIdx.x != 0) return;
  if (out_xyzz) st_xyzz(out_xyzz, acc);
  if (out) st_affine(out, xyzz_to_affine(acc, true));
}

}  // namespace bp
