// bp_gpu.cu -- C-ABI entry points of libbpgpu.so (see include/bp_gpu.h) and the host drivers
// that sequence the kernels of msm.cuh / ipa.cuh on one CUDA stream.
#include <cuda_runtime.h>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <cstdlib>
#include <map>
#include <mutex>
#include <string>
#include <vector>
#include <algorithm>

#include "../../include/bp_gpu.h"
#include "ctx.h"
#include "msm.cuh"
#include "ipa.cuh"
#include "transcript.h"
#include "verify.cuh"
#include "svar.cuh"
#include "fixedbase.cuh"
#include "ipa_round.cuh"
#include "rlc.cuh"
#include "rp_algebra.h"
#include <nccl.h>
#include <thread>

#include "fp_host.h"
namespace bp {

thread_local std::string g_err;
Ctx g;

int fail(const char* fmt, ...) {
  char buf[512];
  va_list ap; va_start(ap, fmt); vsnprintf(buf, sizeof buf, fmt, ap); va_end(ap);
  g_err = buf;
  return 1;
}

// ---- bucket reduction + window combination (the "tails") of nmsm MSMs whose nmsm * sh.U bucket units are complete ----------
static int msm_tails(const XYZZ* buckets, const MsmShape& sh, u32 nmsm, Affine* out_affine, XYZZ* out_xyzz, bool prof, cudaStream_t st) {
  const size_t nmw = (size_t)nmsm * sh.U;
  const bool plain_tails = nmsm >= 2048 && sh.H <= 512;     // big batch of small MSMs: throughput forms
  XYZZ* segsum = (XYZZ*)g.ws_segsum.ensure(nmw * sh.nseg * sizeof(XYZZ));
  XYZZ* winsum = (XYZZ*)g.ws_winsum.ensure(nmw * sizeof(XYZZ));
  if (!segsum || !winsum) return fail("workspace allocation failed");
  size_t nsegs = nmw * sh.nseg;
  const XYZZ* ws;
  if (plain_tails) {
    ++g.nlaunch, k_reduce_unit_plain<<<(unsigned)((nmw + 127) / 128), 128, 0, st>>>(buckets, sh, nmw, segsum);
    ws = segsum;
    if (prof) cudaEventRecord(g.ev[5], st);
    // Horner + output: one thread per MSM saturates the machine only for very many MSMs; below that the chain of
    // ~126 doublings is pure latency and the 4-lane form (2.3 -> 1.3 us per doubling) wins
    if (nmsm <= 12288 && !out_affine) ++g.nlaunch, k_combine<<<(unsigned)((4 * (size_t)nmsm + 127) / 128), 128, 0, st>>>(ws, sh, nmsm, out_affine, out_xyzz);
    else ++g.nlaunch, k_combine_plain<<<(unsigned)((nmsm + 127) / 128), 128, 0, st>>>(ws, sh, nmsm, out_affine, out_xyzz);
  } else {
    XYZZ* seg_run = (XYZZ*)g.ws_segrun.ensure(nsegs * sizeof(XYZZ));
    if (!seg_run) return fail("workspace allocation failed");
    if (sh.seg_plain) ++g.nlaunch, k_reduce_seg_plain<<<(unsigned)((nsegs + 127) / 128), 128, 0, st>>>(buckets, sh, nmw, seg_run, segsum);
    else ++g.nlaunch, k_reduce_seg<<<(unsigned)((4 * nsegs + 127) / 128), 128, 0, st>>>(buckets, sh, nmw, seg_run, segsum);
    // level 2: groups of G = 8 segments (measured at 2^20, c = 16 after the thread-per-segment first level:
    // G = 4 / 8 / 16 / 32 -> reduce stage 0.390 / 0.296 / 0.335 / 0.423 ms; the quad form pays ~2.4x the multiplications'
    // issue cost in glue, so many small groups turn it throughput bound)
    // (quad first level, S = 8, c = 13: G = 2 / 4 / 8 / 16 -> reduce stage 0.148 / 0.157 / 0.179 / 0.235 ms at 2^16)
    const u32 Gmax = sh.seg_plain ? 8 : 2;
    u32 G = sh.nseg < Gmax ? sh.nseg : Gmax, ngrp = sh.nseg / G;
    int lgS = 0, lgG = 0, ubits = 0;
    while ((1u << lgS) < sh.S) lgS++;
    while ((1u << lgG) < G) lgG++;
    while ((1u << ubits) < ngrp * (1u + sh.dbl)) ubits++;
    XYZZ* grpsum = (XYZZ*)g.ws_grpsum.ensure(nmw * ngrp * sizeof(XYZZ));
    if (!grpsum) return fail("workspace allocation failed");
    ++g.nlaunch, k_reduce_grp<<<(unsigned)((4 * nmw * ngrp + 127) / 128), 128, 0, st>>>(seg_run, segsum, sh, nmw, 0, G, lgS, lgG, ubits, grpsum);
    ws = grpsum;
    if (ngrp >= 1024) {
      // level 3 in two steps: 64 quads per block sum 256 groups each, then one small block per unit adds the partials
      const u32 split = ngrp / 256;   // ngrp is a power of two
      XYZZ* partial = (XYZZ*)g.ws_winpart.ensure(nmw * split * sizeof(XYZZ));
      if (!partial) return fail("workspace allocation failed");
      ++g.nlaunch, k_window_sum<<<(unsigned)(nmw * split), 256, 0, st>>>(grpsum, 256, partial);
      ++g.nlaunch, k_window_sum<<<(unsigned)nmw, split < 8 ? 32 : 4 * split, 0, st>>>(partial, split, winsum);
      ws = winsum;
    } else if (ngrp > 1) { ++g.nlaunch, k_window_sum<<<(unsigned)nmw, 256, 0, st>>>(grpsum, ngrp, winsum); ws = winsum; }
    if (prof) cudaEventRecord(g.ev[5], st);
    if (g.hf_want && nmsm == 1 && out_affine && !out_xyzz) {      // the caller finishes the Horner chain on the host (msm_finish_to_host)
      g.hf.ws = ws; g.hf.c = sh.c; g.hf.W = sh.W; g.hf.U = sh.U; g.hf.dbl = sh.dbl; g.hf.pending = true;
      return 0;
    }
    ++g.nlaunch, k_combine<<<(unsigned)((4 * (size_t)nmsm + 127) / 128), 128, 0, st>>>(ws, sh, nmsm, out_affine, out_xyzz);
  }
  return 0;
}

// ---- the MSM pipeline on device-resident operands ----------------------------------------------
// points/point_idx/scalars/offsets are device pointers; out_affine/out_xyzz device (either may be null)
// Per-call options of msm_run (passed by value: nothing a failed call could leave behind for the next one).
//   skip_below  terms whose point index is below this count as zero scalars (the caller evaluates them elsewhere, see k_digits)
//   pts_ready   event the points are complete at (host-operand MSM whose points upload on the copy stream)
//   parts       0, or the operands arrive in that many parts, each its scalars (g.ev_part_sc[k]) followed by its points
//               (g.ev_half[k]; upload_operands): sorted and accumulated part by part (msm_run_parts)
//   host_finish the result goes to the host: leave the window sums for horner_host instead of running k_combine (g.hf)
struct MsmOpts { u32 skip_below = 0; cudaEvent_t pts_ready = nullptr; int parts = 0; bool host_finish = false; };
// Host-operand MSM whose operands arrive in K parts, each part = its scalars followed by its points (upload_operands): every part
// is sorted on its own as soon as its scalars are in (digits, scan, scatter over T/K terms) and accumulated as soon as its points
// are in, all parts adding into ONE bucket set (k_accumulate's `into`); reduction and combination are those of a single MSM.
// Against one sort over all scalars (the part as the major sort key) the chain no longer starts with the upload of ALL scalars
// plus a full-size sort: the first quarter's sort runs while the second quarter is on the wire.
static int msm_run_parts(const Affine* points, const Fq* scalars, u32 T, u32 K, Affine* out_affine, XYZZ* out_xyzz) {
  cudaStream_t st = g.stream;
  if (g.ensure_aux()) return 1;
  cudaStream_t ss = g.aux_stream;                           // the sorts: atomics / memory bound, they run under the previous part's accumulation
  const u32 Tp = (T + K - 1) / K + 1;                       // terms of the largest part (bound)
  MsmShape sh = msm_shape(Tp, 1, g.force_c);
  g.last_c = sh.c;
  const size_t nb = (size_t)sh.U * sh.H;
  g.last_nb = nb;
  const bool prof = g.profiling;
  if (prof) for (int i = 0; i < 7; i++) cudaEventRecord(g.ev[i], st), (void)0;
  const size_t emax = (size_t)sh.W * 2 * Tp, nchunks = (emax + sh.chunk - 1) / sh.chunk;
  const size_t ntiles = (nb + 1 + BP_SCAN_TILE - 1) / BP_SCAN_TILE;
  // sort buffers twice (parity of the part): part k+1 is sorted while part k is accumulated
  int* digits2 = (int*)g.ws_digits.ensure(2 * emax * sizeof(int));
  uint2* entries2 = (uint2*)g.ws_entries.ensure(2 * emax * sizeof(uint2));
  u32* count2 = (u32*)g.ws_count.ensure(2 * (nb + 1) * sizeof(u32));
  u32* start2 = (u32*)g.ws_start.ensure(2 * (nb + 1) * sizeof(u32));
  u32* cursor2 = (u32*)g.ws_cursor.ensure(2 * (nb + 1) * sizeof(u32));
  u32* tiles2 = (u32*)g.ws_tiles.ensure(2 * ntiles * sizeof(u32));
  Affine* phi = (Affine*)g.ws_phi.ensure((size_t)Tp * sizeof(Affine));
  XYZZ* buckets = (XYZZ*)g.ws_buckets.ensure(nb * sizeof(XYZZ));
  XYZZ* part = (XYZZ*)g.ws_part.ensure(2 * nchunks * sizeof(XYZZ));
  const u32 big_cap = (u32)(emax / ((size_t)sh.chunk * (BP_FIXUP_SERIAL_MAX - 1)) + 16);
  u32* big = (u32*)g.ws_big.ensure((2 * (size_t)big_cap + 4) * sizeof(u32));
  if (!digits2 || !entries2 || !phi || !count2 || !start2 || !cursor2 || !tiles2 || !buckets || !part || !big) return fail("workspace allocation failed");
  u32* zero_word = big + 2 * (size_t)big_cap + 3;
  BP_CUDA(cudaMemsetAsync(buckets, 0, nb * sizeof(XYZZ), st));
  BP_CUDA(cudaMemsetAsync(zero_word, 0, sizeof(u32), st));
  BP_CUDA(cudaEventRecord(g.aux_free[0], st)); BP_CUDA(cudaEventRecord(g.aux_free[1], st));      // earlier work on the sort buffers is done
  for (u32 k = 0; k < K; k++) {
    const u32 t0 = (u32)((unsigned long long)T * k / K), tn = (u32)((unsigned long long)T * (k + 1) / K) - t0;
    if (tn == 0) continue;
    const u32 par = k & 1u;
    int* digits = digits2 + (size_t)par * emax; uint2* entries = entries2 + (size_t)par * emax;
    u32* count = count2 + (size_t)par * (nb + 1); u32* start = start2 + (size_t)par * (nb + 1); u32* cursor = cursor2 + (size_t)par * (nb + 1);
    u32* tiles = tiles2 + (size_t)par * ntiles;
    // ---- sort stream: this part's scalars -> digits, histogram, scan, scatter
    BP_CUDA(cudaStreamWaitEvent(ss, g.ev_part_sc[k], 0));   // its scalars have landed
    BP_CUDA(cudaStreamWaitEvent(ss, g.aux_free[par], 0));   // the accumulation of part k-2 has released these buffers
    if (k == 0) g.dbg_rec(4, ss);
    BP_CUDA(cudaMemsetAsync(count, 0, (nb + 1) * sizeof(u32), ss));
    ++g.nlaunch, k_digits<<<(tn + 255) / 256, 256, 0, ss>>>(scalars + t0, tn, nullptr, 1, sh, digits, count, nullptr, 0);
    ++g.nlaunch, k_scan_tiles<<<(unsigned)ntiles, 256, 0, ss>>>(count, start, tiles, nb + 1);
    ++g.nlaunch, k_scan_sums<<<1, 1024, 0, ss>>>(tiles, ntiles);
    ++g.nlaunch, k_scan_add<<<(unsigned)ntiles, 256, 0, ss>>>(start, tiles, nb + 1, nullptr);
    BP_CUDA(cudaMemcpyAsync(cursor, start, (nb + 1) * sizeof(u32), cudaMemcpyDeviceToDevice, ss));
    ++g.nlaunch, k_scatter<<<(2 * tn + 255) / 256, 256, 0, ss>>>(digits, tn, nullptr, 1, sh, cursor, entries);
    if (k == 0) g.dbg_rec(5, ss);
    BP_CUDA(cudaEventRecord(g.aux_ready[par], ss));
    // ---- main stream: accumulate into the shared buckets
    BP_CUDA(cudaStreamWaitEvent(st, g.aux_ready[par], 0));
    BP_CUDA(cudaStreamWaitEvent(st, g.ev_half[k], 0));      // ... and its points
    BP_CUDA(cudaMemsetAsync(big, 0, 2 * sizeof(u32), st));
    ++g.nlaunch, k_phi<<<(tn + 127) / 128, 128, 0, st>>>(points + t0, nullptr, tn, phi);
    if (prof && k == 0) cudaEventRecord(g.ev_k0, st);
    ++g.nlaunch, k_accumulate<<<(unsigned)((nchunks + 127) / 128), 128, 0, st>>>(points + t0, nullptr, phi, start, entries, zero_word, start + nb, sh.chunk, buckets, part, (u32)nb, k ? 1 : 0);
    if (prof && k == K - 1) cudaEventRecord(g.ev_k1, st);
    ++g.nlaunch, k_fixup<<<(unsigned)((nb + 127) / 128), 128, 0, st>>>(start, 0, nb, zero_word, sh.chunk, part, buckets, big, big_cap, (u32)nb);
    ++g.nlaunch, k_fixup_mid<<<2 * g.sm_count, 256, 0, st>>>(start, zero_word, sh.chunk, part, buckets, big, big_cap, (u32)nb);
    ++g.nlaunch, k_fixup_big<<<g.sm_count, 256, 0, st>>>(start, zero_word, sh.chunk, part, buckets, big, (u32)nb);
    BP_CUDA(cudaEventRecord(g.aux_free[par], st));
    g.dbg_rec(6 + (k == K - 1 ? 1 : 0), st);
  }
  if (prof) for (int i = 0; i <= 4; i++) cudaEventRecord(g.ev[i], st), (void)0;
  if (msm_tails(buckets, sh, 1, out_affine, out_xyzz, prof, st)) return 1;
  if (prof) cudaEventRecord(g.ev[6], st);
  BP_CUDA(cudaGetLastError());
  return 0;
}

struct HfScope { HfScope(bool want) { g.hf_want = want && g.hf_enabled; g.hf.pending = false; } ~HfScope() { g.hf_want = false; } };
int msm_run(const Affine* points, const u32* point_idx, const Fq* scalars, u32 T, const u32* d_offsets, u32 nmsm,
            size_t terms_per_msm, Affine* out_affine, XYZZ* out_xyzz, MsmOpts opt = MsmOpts()) {
  HfScope hf_scope(opt.host_finish && nmsm == 1 && !g.profiling);
  if (opt.parts) {
    if (nmsm != 1 || point_idx || d_offsets || T < 64 || opt.parts < 2 || opt.parts > 8)
      return fail("msm: operands in %d parts need one MSM of >= 64 terms without index or offset lists", opt.parts);
    return msm_run_parts(points, scalars, T, (u32)opt.parts, out_affine, out_xyzz);
  }
  cudaStream_t st = g.stream;
  MsmShape sh = msm_shape(terms_per_msm, nmsm, g.force_c);
  g.last_c = sh.c;
  size_t nmw = (size_t)nmsm * sh.U, nb = nmw * sh.H;
  g.last_nb = nb;
  bool prof = g.profiling;
  if (prof) for (int i = 0; i < 7; i++) cudaEventRecord(g.ev[i], st), (void)0;
  if (T == 0) {   // all identities
    if (opt.pts_ready) cudaStreamWaitEvent(st, opt.pts_ready, 0);
    BP_CUDA(cudaMemsetAsync(out_affine ? (void*)out_affine : (void*)out_xyzz, 0, out_affine ? nmsm * sizeof(Affine) : nmsm * sizeof(XYZZ), st));
    if (out_affine && out_xyzz) BP_CUDA(cudaMemsetAsync(out_xyzz, 0, nmsm * sizeof(XYZZ), st));
    return 0;
  }
  if (T >= (1u << 30) || (unsigned long long)sh.W * 2ull * T >= 0xFFFFFFF0ull) return fail("msm: too many terms for 32-bit entry indices");
  int* digits = (int*)g.ws_digits.ensure((size_t)sh.W * 2 * T * sizeof(int));
  uint2* entries = (uint2*)g.ws_entries.ensure((size_t)sh.W * 2 * T * sizeof(uint2));
  Affine* phi = (Affine*)g.ws_phi.ensure((size_t)T * sizeof(Affine));
  u32* count = (u32*)g.ws_count.ensure((nb + 1) * sizeof(u32));
  u32* start = (u32*)g.ws_start.ensure((nb + 1) * sizeof(u32));
  u32* cursor = (u32*)g.ws_cursor.ensure((nb + 1) * sizeof(u32));
  size_t ntiles = (nb + 1 + BP_SCAN_TILE - 1) / BP_SCAN_TILE;
  u32* tiles = (u32*)g.ws_tiles.ensure(ntiles * sizeof(u32));
  XYZZ* buckets = (XYZZ*)g.ws_buckets.ensure(nb * sizeof(XYZZ));
  XYZZ* segsum = (XYZZ*)g.ws_segsum.ensure(nmw * sh.nseg * sizeof(XYZZ));
  XYZZ* winsum = (XYZZ*)g.ws_winsum.ensure(nmw * sizeof(XYZZ));
  // every (term, window) pair is at most one entry, so E <= W*T: size the chunk structures for the bound
  size_t emax = (size_t)sh.W * 2 * T, nchunks = (emax + sh.chunk - 1) / sh.chunk;
  XYZZ* part = (XYZZ*)g.ws_part.ensure(2 * nchunks * sizeof(XYZZ));
  const u32 big_cap = (u32)(emax / ((size_t)sh.chunk * (BP_FIXUP_SERIAL_MAX - 1)) + 16);      // buckets that can span that many chunks
  u32* big = (u32*)g.ws_big.ensure((2 * (size_t)big_cap + 4) * sizeof(u32));
  u32* zero_word = big + 2 * (size_t)big_cap + 3;
  if (!digits || !entries || !count || !start || !cursor || !tiles || !buckets || !segsum || !winsum || !part || !big || !phi)
    return fail("workspace allocation failed");

  // slot sort (msm.cuh): one scattered pass for one large MSM; the exact counting sort stays queued behind it, gated on the overflow word
  // (only where a bucket holds >= 48 entries: at a bucket boundary k_accumulate_slots fetches the next entry AFTER the flush, an
  //  exposed load per boundary -- 2^18 terms, 16 entries per bucket: accumulate 0.567 -> 0.624 ms, the whole MSM 1.19 -> 1.23 ms;
  //  2^20 terms, 64 per bucket: 2.870 -> 2.798 ms.  Mode 2, the test hook, takes every size.)
  const bool use_slots = g.pre_slots > 0 && nmsm == 1 && !d_offsets && !point_idx && !opt.skip_below && T >= g.pre_slots_min &&
                         (g.pre_slots == 2 || 2.0 * (double)T / (double)sh.H >= 48.0 || g.pre_slots_any);
  u32 cap = 0; u32* slots = nullptr; u32* overflow = nullptr;
  if (use_slots) {
    const double lam = 2.0 * (double)T / (double)sh.H;                   // every unit takes 2T sub-terms over H buckets
    cap = g.pre_slots == 2 ? 8u : (u32)(lam + 9.5 * sqrt(lam) + 8.0);
    cap = (cap + 7u) & ~7u;
    slots = (u32*)g.ws_slots.ensure(nb * (size_t)cap * sizeof(u32));
    overflow = (u32*)g.ws_slots_ovf.ensure(64);
    if (!slots || !overflow) return fail("workspace allocation failed");
    BP_CUDA(cudaMemsetAsync(overflow, 0, sizeof(u32), st));
  }
  BP_CUDA(cudaMemsetAsync(count, 0, (nb + 1) * sizeof(u32), st));
  if (prof) cudaEventRecord(g.ev[0], st);
  g.dbg_rec(4, st);
  if (use_slots) ++g.nlaunch, k_digits_slots<<<(T + 255) / 256, 256, 0, st>>>(scalars, T, sh, digits, cap, count, slots, overflow);
  else ++g.nlaunch, k_digits<<<(T + 255) / 256, 256, 0, st>>>(scalars, T, d_offsets, nmsm, sh, digits, count, opt.skip_below ? point_idx : nullptr, opt.skip_below);
  if (prof) cudaEventRecord(g.ev[1], st);
  ++g.nlaunch, k_scan_tiles<<<(unsigned)ntiles, 256, 0, st>>>(count, start, tiles, nb + 1);
  ++g.nlaunch, k_scan_sums<<<1, 1024, 0, st>>>(tiles, ntiles);
  ++g.nlaunch, k_scan_add<<<(unsigned)ntiles, 256, 0, st>>>(start, tiles, nb + 1, nullptr);
  if (prof) cudaEventRecord(g.ev[2], st);
  BP_CUDA(cudaMemcpyAsync(cursor, start, (nb + 1) * sizeof(u32), cudaMemcpyDeviceToDevice, st));   // cursors start at the bucket offsets
  ++g.nlaunch, k_scatter<<<(2 * T + 255) / 256, 256, 0, st>>>(digits, T, d_offsets, nmsm, sh, cursor, entries, overflow);
  if (prof) cudaEventRecord(g.ev[3], st);
  g.dbg_rec(5, st);
  BP_CUDA(cudaMemsetAsync(buckets, 0, nb * sizeof(XYZZ), st));          // empty buckets = identity (ZZ = 0)
  BP_CUDA(cudaMemsetAsync(zero_word, 0, sizeof(u32), st));
  BP_CUDA(cudaMemsetAsync(big, 0, 2 * sizeof(u32), st));   // [0] = queue length, kept zero word for gs = 0 lives at big[big_cap + 1]
  if (opt.pts_ready) BP_CUDA(cudaStreamWaitEvent(st, opt.pts_ready, 0));   // points may still be uploading
  ++g.nlaunch, k_phi<<<(T + 127) / 128, 128, 0, st>>>(points, point_idx, T, phi);
  // E (= start[nb]) stays on the device: launch for the upper bound W*T, threads past E exit at once
  if (prof) cudaEventRecord(g.ev_k0, st);
  if (use_slots) ++g.nlaunch, k_accumulate_slots<true><<<(unsigned)((nchunks + 127) / 128), 128, 0, st>>>(points, phi, start, (u32)nb, slots, cap, overflow, sh.chunk, buckets, part);
  ++g.nlaunch, k_accumulate<<<(unsigned)((nchunks + 127) / 128), 128, 0, st>>>(points, point_idx, phi, start, entries, zero_word, start + nb, sh.chunk, buckets, part, 0, 0, overflow);
  if (prof) cudaEventRecord(g.ev_k1, st);
  ++g.nlaunch, k_fixup<<<(unsigned)((nb + 127) / 128), 128, 0, st>>>(start, 0, nb, zero_word, sh.chunk, part, buckets, big, big_cap);
  ++g.nlaunch, k_fixup_mid<<<2 * g.sm_count, 256, 0, st>>>(start, zero_word, sh.chunk, part, buckets, big, big_cap);
  ++g.nlaunch, k_fixup_big<<<g.sm_count, 256, 0, st>>>(start, zero_word, sh.chunk, part, buckets, big);
  if (prof) cudaEventRecord(g.ev[4], st);
  if (msm_tails(buckets, sh, nmsm, out_affine, out_xyzz, prof, st)) return 1;
  if (prof) cudaEventRecord(g.ev[6], st);
  BP_CUDA(cudaGetLastError());
  return 0;
}

// ---- single MSM over a resident point vector with precomputed window multiples (msm.cuh, "pre" path) -----------------------
// pre = [W][stride] affine multiples 2^(c*w) * P_i; the MSM covers points first .. first+T-1 of the vector.
static int msm_run_pre(const Affine* pre, u32 stride, u32 first, int c, const Fq* scalars, u32 T, Affine* out_affine, XYZZ* out_xyzz) {
  cudaStream_t st = g.stream;
  const PreShape ps = pre_shape(c);
  MsmShape sh;                                         // shape of the tails: ONE unit of H buckets, nothing to combine
  sh.c = c; sh.W = 1; sh.U = 1; sh.dbl = 0; sh.H = ps.H;
  const double ent_bound = (double)ps.W * (double)T;
  sh.chunk = acc_chunk(ent_bound);
  sh.seg_plain = (double)sh.H / 4 >= 32768.0 ? 1 : 0;
  sh.S = sh.seg_plain ? 4 : (sh.H < 8 ? sh.H : 8);
  sh.nseg = sh.H / sh.S;
  g.last_c = c; g.last_nb = sh.H;
  const bool prof = g.profiling;
  if (prof) for (int i = 0; i < 7; i++) cudaEventRecord(g.ev[i], st), (void)0;
  if (T == 0) {
    BP_CUDA(cudaMemsetAsync(out_affine ? (void*)out_affine : (void*)out_xyzz, 0, out_affine ? sizeof(Affine) : sizeof(XYZZ), st));
    if (out_affine && out_xyzz) BP_CUDA(cudaMemsetAsync(out_xyzz, 0, sizeof(XYZZ), st));
    return 0;
  }
  if ((unsigned long long)ps.W * stride >= (1ull << 30)) return fail("msm: too many terms for 30-bit point indices");
  const size_t nb = sh.H, emax = (size_t)ps.W * T;
  if (emax >= 0xFFFFFFF0ull) return fail("msm: too many entries");
  const size_t nchunks = (emax + sh.chunk - 1) / sh.chunk;
  uint2* entries = (uint2*)g.ws_entries.ensure(emax * sizeof(uint2));
  u32* count = (u32*)g.ws_count.ensure((nb + 1) * sizeof(u32));
  u32* start = (u32*)g.ws_start.ensure((nb + 1) * sizeof(u32));
  u32* cursor = (u32*)g.ws_cursor.ensure((nb + 1) * sizeof(u32));
  const size_t ntiles = (nb + 1 + BP_SCAN_TILE - 1) / BP_SCAN_TILE;
  u32* tiles = (u32*)g.ws_tiles.ensure(ntiles * sizeof(u32));
  XYZZ* buckets = (XYZZ*)g.ws_buckets.ensure(nb * sizeof(XYZZ));
  XYZZ* part = (XYZZ*)g.ws_part.ensure(2 * nchunks * sizeof(XYZZ));
  const u32 big_cap = (u32)(emax / ((size_t)sh.chunk * (BP_FIXUP_SERIAL_MAX - 1)) + 16);
  u32* big = (u32*)g.ws_big.ensure((2 * (size_t)big_cap + 4) * sizeof(u32));
  if (!entries || !count || !start || !cursor || !tiles || !buckets || !part || !big) return fail("workspace allocation failed");
  u32* zero_word = big + 2 * (size_t)big_cap + 3;
  // slot sort (msm.cuh): one scattered pass instead of histogram + scatter for large MSMs; the exact counting sort stays queued
  // behind it as the fallback, gated on the overflow word
  const bool use_slots = g.pre_slots > 0 && T >= g.pre_slots_min;
  u32 cap = 0; u32* slots = nullptr; u32* overflow = nullptr;
  if (use_slots) {
    double lam = 0;                                                      // mean load of the fullest buckets: the low ones, which every window reaches
    for (int w = 0; w < ps.W; w++) lam += (double)T / (double)(1u << (ps.off[w + 1] - ps.off[w] - 1));
    cap = g.pre_slots == 2 ? 8u : (u32)(lam + 9.5 * sqrt(lam) + 8.0);    // (mode 2: a test hook that makes every large bucket overflow)
    cap = (cap + 7u) & ~7u;
    slots = (u32*)g.ws_slots.ensure(nb * (size_t)cap * sizeof(u32));
    overflow = (u32*)g.ws_slots_ovf.ensure(64);
    if (!slots || !overflow) return fail("workspace allocation failed");
    BP_CUDA(cudaMemsetAsync(overflow, 0, sizeof(u32), st));
  }
  BP_CUDA(cudaMemsetAsync(count, 0, (nb + 1) * sizeof(u32), st));
  if (prof) cudaEventRecord(g.ev[0], st);
  if (use_slots) ++g.nlaunch, k_scatter_slots_pre<4><<<(T + 255) / 256, 256, 0, st>>>(scalars, T, ps, stride, first, cap, count, slots, overflow);
  else ++g.nlaunch, k_digits_pre<<<(T + 255) / 256, 256, 0, st>>>(scalars, T, ps, count);
  if (prof) cudaEventRecord(g.ev[1], st);
  ++g.nlaunch, k_scan_tiles<<<(unsigned)ntiles, 256, 0, st>>>(count, start, tiles, nb + 1);
  ++g.nlaunch, k_scan_sums<<<1, 1024, 0, st>>>(tiles, ntiles);
  ++g.nlaunch, k_scan_add<<<(unsigned)ntiles, 256, 0, st>>>(start, tiles, nb + 1, nullptr);
  if (prof) cudaEventRecord(g.ev[2], st);
  BP_CUDA(cudaMemcpyAsync(cursor, start, (nb + 1) * sizeof(u32), cudaMemcpyDeviceToDevice, st));
  ++g.nlaunch, k_scatter_pre<<<(T + 255) / 256, 256, 0, st>>>(scalars, T, ps, stride, first, cursor, entries, overflow);
  if (prof) cudaEventRecord(g.ev[3], st);
  BP_CUDA(cudaMemsetAsync(buckets, 0, nb * sizeof(XYZZ), st));
  BP_CUDA(cudaMemsetAsync(zero_word, 0, sizeof(u32), st));
  BP_CUDA(cudaMemsetAsync(big, 0, 2 * sizeof(u32), st));
  if (prof) cudaEventRecord(g.ev_k0, st);
  if (use_slots) ++g.nlaunch, k_accumulate_slots<false><<<(unsigned)((nchunks + 127) / 128), 128, 0, st>>>(pre, nullptr, start, (u32)nb, slots, cap, overflow, sh.chunk, buckets, part);
  ++g.nlaunch, k_accumulate<<<(unsigned)((nchunks + 127) / 128), 128, 0, st>>>(pre, nullptr, nullptr, start, entries, zero_word, start + nb, sh.chunk, buckets, part, 0, 0, overflow);
  if (prof) cudaEventRecord(g.ev_k1, st);
  ++g.nlaunch, k_fixup<<<(unsigned)((nb + 127) / 128), 128, 0, st>>>(start, 0, nb, zero_word, sh.chunk, part, buckets, big, big_cap);
  ++g.nlaunch, k_fixup_mid<<<2 * g.sm_count, 256, 0, st>>>(start, zero_word, sh.chunk, part, buckets, big, big_cap);
  ++g.nlaunch, k_fixup_big<<<g.sm_count, 256, 0, st>>>(start, zero_word, sh.chunk, part, buckets, big);
  if (prof) cudaEventRecord(g.ev[4], st);
  if (sh.H < 4096) {                                   // small unit: the running-sum tails of the plain path
    if (msm_tails(buckets, sh, 1, out_affine, out_xyzz, prof, st)) return 1;
  } else {
    // H = R x C buckets: marginal sums by factors of 8 (rows contiguous, columns strided), weighted stage on R + C points
    int lgH = c - 1, lgC = (lgH + 1) / 2, lgR = lgH - lgC;
    const u32 C = 1u << lgC, R = 1u << lgR;
    // level 1: factors of K (rows contiguous, columns strided) in one launch
    // K = 8 for the 2^17-bucket unit of large MSMs, 4 below (gpurun_out/prek.log: 2^16 terms, c = 17: K = 8 / 4 / 2 -> 0.432 / 0.416 /
    // 0.414 ms, the first level is a latency chain of K - 1 lone-thread additions there; 2^20 terms, c = 18: 2.268 / 2.284 / 2.303 ms,
    // twice the partial sums cost the weighted stage more than the shorter first level saves)
    const u32 Kpre = sh.H >= (1u << 17) ? 8u : 4u;
    const u32 Kr = C >= Kpre ? Kpre : C, Kc = R >= Kpre ? Kpre : R;
    const u32 np_r = C / Kr, np_c = R / Kc;              // partial sums per row / per column
    XYZZ* ping = (XYZZ*)g.ws_segsum.ensure(((size_t)nb / Kr + (size_t)nb / Kc + 8192) * sizeof(XYZZ));
    XYZZ* wsum = (XYZZ*)g.ws_winsum.ensure((size_t)(C + R + 2) * sizeof(XYZZ));
    if (!ping || !wsum) return fail("workspace allocation failed");
    XYZZ* rpart = ping; XYZZ* cpart = ping + ((size_t)nb / Kr + 4096);
    const u32 nrow_out = R * np_r, ncol_out = np_c * C;
    ++g.nlaunch, k_pre_marginals<<<dim3(((nrow_out > ncol_out ? nrow_out : ncol_out) + 127) / 128, 2), 128, 0, st>>>(buckets, rpart, nrow_out, Kr, buckets, cpart, np_c, C, Kc);
    if (prof) cudaEventRecord(g.ev[5], st);
    ++g.nlaunch, k_pre_rowcol<<<C + R, 64, 0, st>>>(rpart, np_r, cpart, np_c, C, R, wsum);
    XYZZ* two = wsum + C + R;
    ++g.nlaunch, k_pre_total<<<2, 256, 0, st>>>(wsum, C, R, two);
    ++g.nlaunch, k_pre_finish<<<1, 32, 0, st>>>(two, lgC, out_affine, out_xyzz);
  }
  if (prof) cudaEventRecord(g.ev[6], st);
  BP_CUDA(cudaGetLastError());
  return 0;
}

#include "bp_fixed.inl"

// Host operands -> device: scalars first on the compute stream (the digit/sort stages only need them), points on a
// second stream so that their (twice as large) upload overlaps those stages; msm_run waits for the points right
// before the first kernel that reads them.
// Large host -> device copies go down in pieces: on the B200 hosts measured here one cudaMemcpyAsync of 32-96 MiB from pinned
// memory runs at 18-38 GB/s, the same bytes as <= 8 MiB copies back to back at 52 GB/s (tools/h2d_probe.py, profiles/r2_h2d_probe.txt).
static size_t h2d_piece() {
  static const size_t v = [] { const char* e = getenv("BP_H2D_PIECE_MIB"); long m = e ? atol(e) : 6; return (size_t)(m > 0 ? m : 6) << 20; }();
  return v;
}
static cudaError_t h2d_chunked(void* dst, const void* src, size_t bytes, cudaStream_t st) {
  const size_t piece = h2d_piece();
  for (size_t off = 0; off < bytes; off += piece) {
    const size_t len = bytes - off < piece ? bytes - off : piece;
    cudaError_t e = cudaMemcpyAsync((char*)dst + off, (const char*)src + off, len, cudaMemcpyHostToDevice, st);
    if (e != cudaSuccess) return e;
  }
  return cudaSuccess;
}
static int upload_operands(Affine* d_pts, const uint8_t* pts64, Fq* d_sc, const uint8_t* sc32, size_t n, MsmOpts* opt) {
  *opt = MsmOpts();
  BP_CUDA(cudaEventRecord(g.ev_copy_gate, g.stream));                     // earlier work may still read d_pts
  BP_CUDA(cudaStreamWaitEvent(g.copy_stream, g.ev_copy_gate, 0));
  if (n >= ((size_t)1 << 17) && g.force_c == 0 && !g.profiling) {
    // big MSM: everything on the copy stream in the order it is needed -- per part its scalars, then its points -- and
    // msm_run_parts sorts each part as soon as its scalars are in and accumulates it into one set of buckets as soon as its
    // points are.  K = 4: the accumulation of a quarter (0.49 ms) roughly matches its upload (0.44 ms at the 36-38 GB/s this host
    // sustains), so the GPU neither waits for the last part nor starts late (profiles/r2_e2e_timeline.txt)
    static const int parts = [] { const char* e = getenv("BP_E2E_PARTS"); int v = e ? atoi(e) : 4; return v >= 2 && v <= 8 ? v : 4; }();
    opt->parts = parts;
    g.dbg_rec(0, g.copy_stream);
    for (int k = 0; k < parts; k++) {                      // part k = terms [n*k/K, n*(k+1)/K)  (the same cut as msm_run_parts')
      const size_t lo = (size_t)((unsigned long long)n * k / parts), hi = (size_t)((unsigned long long)n * (k + 1) / parts);
      BP_CUDA(h2d_chunked(d_sc + lo, sc32 + lo * 32, (hi - lo) * 32, g.copy_stream));
      BP_CUDA(cudaEventRecord(g.ev_part_sc[k], g.copy_stream));
      if (k == 0) g.dbg_rec(1, g.copy_stream);
      BP_CUDA(h2d_chunked(d_pts + lo, pts64 + lo * 64, (hi - lo) * 64, g.copy_stream));
      BP_CUDA(cudaEventRecord(g.ev_half[k], g.copy_stream));
      if (k == 0) g.dbg_rec(2, g.copy_stream);
      if (k == parts - 1) g.dbg_rec(3, g.copy_stream);
    }
    return 0;
  }
  BP_CUDA(h2d_chunked(d_sc, sc32, n * 32, g.stream));
  BP_CUDA(h2d_chunked(d_pts, pts64, n * 64, g.copy_stream));
  BP_CUDA(cudaEventRecord(g.ev_pts, g.copy_stream));
  opt->pts_ready = g.ev_pts;
  return 0;
}

// Result of the MSM just enqueued on g.stream -> host: either the affine point k_combine wrote to d_out, or -- host-finished
// Horner -- the window sums, combined here (fp_host.h)
static int msm_finish_to_host(const Affine* d_out, uint8_t* out64) {
  if (g.hf.pending) {
    g.hf.pending = false;
    uint8_t ws[132 * 128];                        // c = 1: 128 windows + the second unit of the top one
    if (g.hf.U > 132) return fail("host finish: too many window sums");
    BP_CUDA(cudaMemcpyAsync(ws, g.hf.ws, (size_t)g.hf.U * 128, cudaMemcpyDeviceToHost, g.stream));
    BP_CUDA(cudaStreamSynchronize(g.stream));
    horner_host(ws, g.hf.c, g.hf.W, g.hf.U, g.hf.dbl, out64);
    return 0;
  }
  BP_CUDA(cudaMemcpyAsync(out64, d_out, 64, cudaMemcpyDeviceToHost, g.stream));
  BP_CUDA(cudaStreamSynchronize(g.stream));
  return 0;
}
static int msm_to_host(const Affine* d_pts, const Fq* d_sc, size_t n, uint8_t* out64, MsmOpts opt = MsmOpts()) {
  Affine* d_out = (Affine*)g.ws_out.ensure(sizeof(Affine));
  if (!d_out) { cudaStreamSynchronize(g.copy_stream); return fail("workspace allocation failed"); }
  opt.host_finish = true;
  if (msm_run(d_pts, nullptr, d_sc, (u32)n, nullptr, 1, n, d_out, nullptr, opt)) { cudaStreamSynchronize(g.copy_stream); return 1; }
  return msm_finish_to_host(d_out, out64);
}

// kind 0 = points, 1 = scalars; pre/pre_c: precomputed window multiples of a point vector (bp_points_precompute)
struct HandleRec { void* p; size_t n; int kind; Affine* pre = nullptr; int pre_c = 0; };
static std::map<bp_handle, HandleRec> g_handles;
static bp_handle g_next_handle = 1;
static std::mutex g_mu;

static int get_handle(bp_handle h, int kind, HandleRec* out) {
  auto it = g_handles.find(h);
  if (it == g_handles.end() || it->second.kind != kind) return fail("bad handle %llu", (unsigned long long)h);
  *out = it->second;
  return 0;
}

// ---- integer-pipe microbenchmarks (the measured roofline denominators) ---------------------------
// Every probe keeps its operands data dependent so that ptxas can neither hoist the products nor turn the
// multiply-accumulate into adds (it does both for loop-invariant operands); the SASS of each mode is
// checked with cuobjdump (profiles/r1_pipe_probe.txt lists the opcode mix).
// mode 0: IMAD.WIDE.U32 Rd, Ra, Rb, RZ  -- 32x32->64 product, both halves consumed as the next operands
// mode 1: IMAD (32-bit mad.lo with accumulate)
// mode 2: IMAD.WIDE.U32(.X) carry-chained rows (mad.lo.cc / madc.hi.cc pairs), as fp_mul issues them
// mode 3: whole fp_mul (field multiplications per second; 72 IMAD.WIDE(.X) each)
// mode 4: IADD3 (32-bit adds; ptxas spreads them over the ALU and the FMA pipe as IADD3 / IMAD.IADD)
// mode 5: whole fp_sqr
template <int MODE>
__global__ void __launch_bounds__(256) k_pipe_probe(u32* out, u32 seed, int iters) {
  u32 a = seed + threadIdx.x, b = seed * 3 + blockIdx.x;
  if (MODE == 0) {
    u64 p[16];
#pragma unroll
    for (int i = 0; i < 16; i++) p[i] = ((u64)(a + i) << 32) | (b + 7 * i);
    for (int it = 0; it < iters; it++) {
#pragma unroll
      for (int r = 0; r < 2; r++)
#pragma unroll
        for (int i = 0; i < 16; i++) asm volatile("mul.wide.u32 %0, %1, %2;" : "=l"(p[i]) : "r"((u32)p[i]), "r"((u32)(p[i] >> 32)));
    }
    u64 s = 0;
#pragma unroll
    for (int i = 0; i < 16; i++) s ^= p[i];
    if (s == 0x1234567u) out[0] = (u32)s;
  } else if (MODE == 1) {
    u32 p[16];
#pragma unroll
    for (int i = 0; i < 16; i++) p[i] = a + i;
    for (int it = 0; it < iters; it++) {
#pragma unroll
      for (int r = 0; r < 2; r++)
#pragma unroll
        for (int i = 0; i < 16; i++) asm volatile("mad.lo.u32 %0, %1, %2, %0;" : "+r"(p[i]) : "r"(p[(i + 5) & 15]), "r"(b));
    }
    u32 s = 0;
#pragma unroll
    for (int i = 0; i < 16; i++) s ^= p[i];
    if (s == 0x1234567u) out[0] = s;
  } else if (MODE == 2) {
    u32 acc[4][9];
#pragma unroll
    for (int j = 0; j < 4; j++)
#pragma unroll
      for (int i = 0; i < 9; i++) acc[j][i] = a + i + j;
    for (int it = 0; it < iters; it++) {
#pragma unroll
      for (int r = 0; r < 2; r++)
#pragma unroll
        for (int j = 0; j < 4; j++) mul_row_mad(acc[j], a, b, a ^ b, a + b, acc[(j + 1) & 3][0]);   // 4 IMAD.WIDE(.X) + 1 IADD3.X
    }
    u32 s = 0;
#pragma unroll
    for (int j = 0; j < 4; j++)
#pragma unroll
      for (int i = 0; i < 9; i++) s ^= acc[j][i];
    if (s == 0x1234567u) out[0] = s;
  } else if (MODE == 10 || MODE == 11) {
    // 10: DFMA alone (fp64 pipe); 11: the same 32 DFMA per iteration interleaved with 32 IMAD.WIDE (fmaheavy pipe): do the two issue
    // side by side?  (next-step question of DESIGN.md 5: 52-bit limbs on the FP64 pipe next to / instead of 32-bit limbs on IMAD.WIDE)
    double f[16];
    u64 p[16];
#pragma unroll
    for (int i = 0; i < 16; i++) { f[i] = (double)(a + i) * 1.0000001; p[i] = ((u64)(a + i) << 32) | (b + 7 * i); }
    const double m = 1.0 + (double)(b & 7) * 1e-9;
    for (int it = 0; it < iters; it++) {
#pragma unroll
      for (int r = 0; r < 2; r++)
#pragma unroll
        for (int i = 0; i < 16; i++) {
          asm volatile("fma.rz.f64 %0, %0, %1, %2;" : "+d"(f[i]) : "d"(m), "d"(f[(i + 5) & 15]));
          if (MODE == 11) asm volatile("mul.wide.u32 %0, %1, %2;" : "=l"(p[i]) : "r"((u32)p[i]), "r"((u32)(p[i] >> 32)));
        }
    }
    double sd = 0; u64 s = 0;
#pragma unroll
    for (int i = 0; i < 16; i++) { sd += f[i]; s ^= p[i]; }
    if (sd == 1.2345 || s == 0x1234567u) out[0] = (u32)s;
  } else if (MODE == 4) {
    u32 p[16];
#pragma unroll
    for (int i = 0; i < 16; i++) p[i] = a + i;
    for (int it = 0; it < iters; it++) {
#pragma unroll
      for (int r = 0; r < 2; r++)
#pragma unroll
        for (int i = 0; i < 16; i++) asm volatile("add.u32 %0, %0, %1;" : "+r"(p[i]) : "r"(p[(i + 5) & 15]));
    }
    u32 s = 0;
#pragma unroll
    for (int i = 0; i < 16; i++) s ^= p[i];
    if (s == 0x1234567u) out[0] = s;
  } else if (MODE >= 6) {
    // latency probes (launched as ONE warp): dependent chains of the operations the MSM tails are made of
    Fp x, y;
#pragma unroll
    for (int i = 0; i < 8; i++) { x.v[i] = a * (i + 1); y.v[i] = b + i; }
    XYZZ P; P.X = x; P.Y = y; P.ZZ = fp_sqr(y); P.ZZZ = fp_mul(P.ZZ, y);
    XYZZ Q; Q.X = y; Q.Y = x; Q.ZZ = fp_sqr(x); Q.ZZZ = fp_mul(Q.ZZ, x);
    const int role = threadIdx.x & 3, base = threadIdx.x & ~3;
    if (MODE == 6) { for (int it = 0; it < iters; it++) x = fp_mul(x, y); P.X = x; }
    else if (MODE == 7) { for (int it = 0; it < iters; it++) P = coop_dbl(P, role, base); }
    else if (MODE == 8) { for (int it = 0; it < iters; it++) P = xyzz_dbl(P); }
    else { for (int it = 0; it < iters; it++) P = coop_add(P, Q, role, base); }
    u32 s = 0;
#pragma unroll
    for (int i = 0; i < 8; i++) s ^= P.X.v[i] ^ P.Y.v[i] ^ P.ZZ.v[i] ^ P.ZZZ.v[i];
    if (s == 0x1234567u) out[0] = s;
  } else {
    Fp x, y;
#pragma unroll
    for (int i = 0; i < 8; i++) { x.v[i] = a * (i + 1); y.v[i] = b + i; }
    if (MODE == 3) { for (int it = 0; it < iters; it++) { x = fp_mul(x, y); y = fp_mul(y, x); } }
    else { for (int it = 0; it < iters; it++) { x = fp_sqr(x); y = fp_sqr(y); } }
    u32 s = 0;
#pragma unroll
    for (int i = 0; i < 8; i++) s ^= x.v[i] ^ y.v[i];
    if (s == 0x1234567u) out[0] = s;
  }
}

}  // namespace bp

using namespace bp;

#define BP_NEED_INIT() do { if (!g.inited) { if (bp_init(-1)) return 1; } } while (0)

extern "C" {

const char* bp_last_error(void) { return g_err.c_str(); }

int bp_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
  return n;
}

int bp_init(int device) {
  std::lock_guard<std::mutex> lk(g_mu);
  if (g.inited && (device < 0 || device == g.device)) return 0;
  if (g.inited) return fail("bp_init: already bound to device %d", g.device);
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n == 0) { cudaGetLastError(); return fail("no CUDA device available (%s): libbpgpu has no CPU fallback", cudaGetErrorString(e)); }
  if (device < 0) {   // lazy initialisation (first library call without bp_init): one process per GPU under torchrun => LOCAL_RANK
    const char* lr = getenv("LOCAL_RANK");
    device = lr && *lr ? atoi(lr) % n : 0;
  }
  if (device >= n) return fail("bp_init: device %d out of range (%d devices)", device, n);
  BP_CUDA(cudaSetDevice(device));
  cudaDeviceProp prop;
  BP_CUDA(cudaGetDeviceProperties(&prop, device));
  if (prop.major < 10) return fail("bp_init: device %s is sm_%d%d; this library is built for sm_100a only", prop.name, prop.major, prop.minor);
  g.device = device; g.sm_count = prop.multiProcessorCount;
  BP_CUDA(cudaStreamCreateWithFlags(&g.stream, cudaStreamNonBlocking));
  for (int i = 0; i < 8; i++) BP_CUDA(cudaEventCreate(&g.ev[i]));
  BP_CUDA(cudaEventCreate(&g.ev_a)); BP_CUDA(cudaEventCreate(&g.ev_b));
  BP_CUDA(cudaEventCreate(&g.ev_k0)); BP_CUDA(cudaEventCreate(&g.ev_k1));
  BP_CUDA(cudaStreamCreateWithFlags(&g.copy_stream, cudaStreamNonBlocking));
  BP_CUDA(cudaEventCreateWithFlags(&g.ev_pts, cudaEventDisableTiming)); BP_CUDA(cudaEventCreateWithFlags(&g.ev_copy_gate, cudaEventDisableTiming));
  for (int i = 0; i < 8; i++) BP_CUDA(cudaEventCreateWithFlags(&g.ev_half[i], cudaEventDisableTiming));
  for (int i = 0; i < 8; i++) BP_CUDA(cudaEventCreateWithFlags(&g.ev_part_sc[i], cudaEventDisableTiming));
  g.inited = true;
  return 0;
}

static void pre_graphs_clear();
int bp_shutdown(void) {
  std::lock_guard<std::mutex> lk(g_mu);
  if (!g.inited) return 0;
  cudaStreamSynchronize(g.stream);
  pre_graphs_clear();
  for (auto& kv : g_handles) { cudaFree(kv.second.p); if (kv.second.pre) cudaFree(kv.second.pre); }
  g_handles.clear();
  fb_release_all();
  g.free_all();
  for (auto& kv : g.ipa_graphs) cudaGraphExecDestroy(kv.second.exec);
  g.ipa_graphs.clear();
  nccl_shutdown();
  cudaStreamDestroy(g.stream);
  g.inited = false;
  return 0;
}

int bp_device_info(char* name, size_t cap, int* sm_count, int* cc_major, int* cc_minor) {
  BP_NEED_INIT();
  cudaDeviceProp prop;
  BP_CUDA(cudaGetDeviceProperties(&prop, g.device));
  if (name && cap) { strncpy(name, prop.name, cap - 1); name[cap - 1] = 0; }
  if (sm_count) *sm_count = prop.multiProcessorCount;
  if (cc_major) *cc_major = prop.major;
  if (cc_minor) *cc_minor = prop.minor;
  return 0;
}

int bp_msm_set_window(int c) { if (c < 0 || c > 16) return fail("window must be 0..16"); g.force_c = c; return 0; }
int bp_msm_last_window(void) { return g.last_c; }
int bp_msm_accumulate_kernel_ms(float* ms) {      // CUDA-event duration of k_accumulate alone in the last profiled MSM
  BP_NEED_INIT();
  BP_CUDA(cudaStreamSynchronize(g.stream));
  if (cudaEventElapsedTime(ms, g.ev_k0, g.ev_k1) != cudaSuccess) { cudaGetLastError(); *ms = -1.f; }
  return 0;
}
int bp_msm_last_entries(uint64_t* entries) {      // non-zero digits = mixed additions of the last MSM's accumulation
  BP_NEED_INIT();
  if (!g.ws_start.p) return fail("no MSM has run yet");
  uint32_t e = 0;
  BP_CUDA(cudaStreamSynchronize(g.stream));
  BP_CUDA(cudaMemcpy(&e, (const uint32_t*)g.ws_start.p + g.last_nb, 4, cudaMemcpyDeviceToHost));
  *entries = e;
  return 0;
}
int bp_launch_count(uint64_t* launches) { *launches = g.nlaunch; return 0; }
int bp_msm_set_pre_slots(int mode, size_t min_terms) {   /* 0 = exact counting sort only, 1 = slot sort for MSMs of >= min_terms terms (0 = keep), 2 = same with 8 slots per bucket (test hook: forces the fallback) */
  if (g.inited) cudaStreamSynchronize(g.stream);
  g.pre_slots = mode; if (min_terms) g.pre_slots_min = (unsigned)min_terms;
  g.pre_slots_any = min_terms != 0 && min_terms < (1u << 18);      // a lowered threshold (tests) also lifts the plain path's bucket-load condition
  pre_graphs_clear();
  return 0;
}
int bp_msm_set_host_finish(int on) { g.hf_enabled = on != 0; return 0; }   /* 1 (default): host-result MSMs of the plain path finish their Horner chain on the host */
int bp_msm_set_profiling(int on) { g.profiling = on != 0; return 0; }
int bp_msm_stage_ms(float out7[7]) {
  BP_NEED_INIT();
  BP_CUDA(cudaStreamSynchronize(g.stream));
  for (int i = 0; i < 6; i++) { if (cudaEventElapsedTime(&out7[i], g.ev[i], g.ev[i + 1]) != cudaSuccess) { cudaGetLastError(); out7[i] = -1.f; } }
  if (cudaEventElapsedTime(&out7[6], g.ev[0], g.ev[6]) != cudaSuccess) { cudaGetLastError(); out7[6] = -1.f; }
  return 0;
}

int bp_msm(const uint8_t* pts64, const uint8_t* sc32, size_t n, uint8_t out64[64]) {
  BP_NEED_INIT();
  if (n == 0) { memset(out64, 0, 64); return 0; }       // pippenger.py:28-29
  if (n >= (1u << 31)) return fail("bp_msm: n too large");
  Affine* d_pts = (Affine*)g.ws_pts.ensure(n * sizeof(Affine));
  Fq* d_sc = (Fq*)g.ws_sc.ensure(n * sizeof(Fq));
  if (!d_pts || !d_sc) return fail("device allocation failed");
  if (fb_enabled() && n <= fb.max_points) {
    // repeated generator set (a commitment call site of a prover/verifier): table lookups instead of buckets
    const FbSrc src = {{pts64}, {n * 64}, 1};
    const uint64_t key = src.hash(0x6D736D31ull);
    auto hit = fb.tabs.find(key ^ ((uint64_t)n * 0xD6E8FEB86659FD93ull));
    if (hit == fb.tabs.end()) BP_CUDA(cudaMemcpyAsync(d_pts, pts64, n * 64, cudaMemcpyHostToDevice, g.stream));   // needed to build
    const Affine* tab = fb_get(key, src, d_pts, n);
    if (tab) {
      Affine* d_out = (Affine*)g.ws_out.ensure(sizeof(Affine));
      if (!d_out) return fail("workspace allocation failed");
      BP_CUDA(cudaMemcpyAsync(d_sc, sc32, n * 32, cudaMemcpyHostToDevice, g.stream));
      return fb_msm_run_host(tab, nullptr, d_sc, nullptr, 1, n, (u32)n, out64);
    }
  }
  MsmOpts opt;
  if (upload_operands(d_pts, pts64, d_sc, sc32, n, &opt)) return 1;
  return msm_to_host(d_pts, d_sc, n, out64, opt);
}

int bp_fb_set_mode(int mode) {
  if (mode < 0 || mode > 2) return fail("bp_fb_set_mode: 0 = off, 1 = build at the second use, 2 = build at first use");
  fb.mode = mode;
  return 0;
}
int bp_fb_stats(uint64_t* tables, uint64_t* bytes, uint64_t* hits, uint64_t* builds) {
  if (tables) *tables = fb.tabs.size();
  if (bytes) *bytes = fb.bytes;
  if (hits) *hits = fb.hits;
  if (builds) *builds = fb.builds;
  return 0;
}
int bp_fb_clear(void) {
  if (g.inited) cudaStreamSynchronize(g.stream);
  fb_release_all();
  alloc_generation()++;
  return 0;
}

static int upload(const uint8_t* src, size_t n, size_t elt, int kind, bp_handle* h) {
  BP_NEED_INIT();
  void* p = nullptr;
  BP_CUDA(cudaMalloc(&p, n ? n * elt : elt));
  if (n) BP_CUDA(cudaMemcpy(p, src, n * elt, cudaMemcpyHostToDevice));
  std::lock_guard<std::mutex> lk(g_mu);
  *h = g_next_handle++;
  HandleRec rec; rec.p = p; rec.n = n; rec.kind = kind;
  g_handles[*h] = rec;
  return 0;
}
int bp_points_upload(const uint8_t* pts64, size_t n, bp_handle* h) { return upload(pts64, n, 64, 0, h); }
int bp_scalars_upload(const uint8_t* sc32, size_t n, bp_handle* h) { return upload(sc32, n, 32, 1, h); }
int bp_handle_free(bp_handle h) {
  std::lock_guard<std::mutex> lk(g_mu);
  auto it = g_handles.find(h);
  if (it == g_handles.end()) return fail("bad handle");
  cudaStreamSynchronize(g.stream);
  cudaFree(it->second.p);
  if (it->second.pre) cudaFree(it->second.pre);
  g_handles.erase(it);
  return 0;
}

// Small MSMs over a resident vector (<= 2^17 terms) are ~18 short stream operations: as a CUDA graph, captured the second time the
// same (vector, slice, scalars, output) combination is seen and replayed while no workspace has moved, the gaps between them
// shrink from a launch each to a graph-node hand-over (bp_msm_set_small_graphs(0) turns it off; profiling runs eagerly).
struct PreGraph { const void* pre; u32 stride, first; int c; const void* sc; u32 T; void* oa; void* ox; unsigned long long gen, stamp; cudaGraphExec_t exec; unsigned nk; int seen; };
static std::vector<PreGraph> g_pre_graphs;
static unsigned long long g_pre_graph_clock = 0;
static bool g_small_graphs = true;
static void pre_graphs_clear() { for (auto& e : g_pre_graphs) if (e.exec) cudaGraphExecDestroy(e.exec); g_pre_graphs.clear(); }
static int msm_run_pre_small(const Affine* pre, u32 stride, u32 first, int c, const Fq* scalars, u32 T, Affine* out_affine, XYZZ* out_xyzz) {
  if (!g_small_graphs || T == 0 || T > (1u << 17) || g.profiling)
    return msm_run_pre(pre, stride, first, c, scalars, T, out_affine, out_xyzz);
  PreGraph* hit = nullptr;
  for (auto& e : g_pre_graphs)
    if (e.pre == pre && e.stride == stride && e.first == first && e.c == c && e.sc == scalars && e.T == T && e.oa == out_affine && e.ox == out_xyzz) { hit = &e; break; }
  if (hit && hit->exec && hit->gen == alloc_generation()) {
    hit->stamp = ++g_pre_graph_clock;
    BP_CUDA(cudaGraphLaunch(hit->exec, g.stream));
    g.nlaunch += hit->nk;
    const PreShape ps = pre_shape(c);
    g.last_c = c; g.last_nb = ps.H;
    return 0;
  }
  if (!hit) {                                             // first sighting: run eagerly (this also sizes every workspace)
    if (g_pre_graphs.size() >= 32) {                      // drop the least recently used
      size_t v = 0;
      for (size_t i = 1; i < g_pre_graphs.size(); i++) if (g_pre_graphs[i].stamp < g_pre_graphs[v].stamp) v = i;
      if (g_pre_graphs[v].exec) cudaGraphExecDestroy(g_pre_graphs[v].exec);
      g_pre_graphs.erase(g_pre_graphs.begin() + (long)v);
    }
    g_pre_graphs.push_back(PreGraph{pre, stride, first, c, scalars, T, out_affine, out_xyzz, 0, ++g_pre_graph_clock, nullptr, 0, 1});
    return msm_run_pre(pre, stride, first, c, scalars, T, out_affine, out_xyzz);
  }
  // seen before (or its graph went stale with a workspace move): capture, instantiate, launch
  if (hit->exec) { cudaGraphExecDestroy(hit->exec); hit->exec = nullptr; }
  cudaGraph_t graph = nullptr;
  const unsigned long long l0 = g.nlaunch, gen0 = alloc_generation();
  BP_CUDA(cudaStreamBeginCapture(g.stream, cudaStreamCaptureModeRelaxed));
  const int rc = msm_run_pre(pre, stride, first, c, scalars, T, out_affine, out_xyzz);
  const cudaError_t ce = cudaStreamEndCapture(g.stream, &graph);
  const unsigned nk = (unsigned)(g.nlaunch - l0);
  g.nlaunch = l0;
  if (rc || ce != cudaSuccess || !graph || gen0 != alloc_generation()) {      // (a workspace grew during the capture: eager this time)
    cudaGetLastError();
    if (graph) cudaGraphDestroy(graph);
    return msm_run_pre(pre, stride, first, c, scalars, T, out_affine, out_xyzz);
  }
  cudaGraphExec_t exec = nullptr;
  const cudaError_t ci = cudaGraphInstantiate(&exec, graph, 0);
  cudaGraphDestroy(graph);
  if (ci != cudaSuccess || !exec) { cudaGetLastError(); return msm_run_pre(pre, stride, first, c, scalars, T, out_affine, out_xyzz); }
  hit->exec = exec; hit->nk = nk; hit->gen = gen0; hit->stamp = ++g_pre_graph_clock;
  BP_CUDA(cudaGraphLaunch(exec, g.stream));
  g.nlaunch += nk;
  return 0;
}

// MSM over points [first, first + n) of a resident vector: through its precomputed window multiples when it has them
static int handle_msm(const HandleRec& P, size_t first, const Fq* d_sc, size_t n, Affine* out_affine, XYZZ* out_xyzz) {
  if (P.pre && g.force_c == 0) return msm_run_pre_small(P.pre, (u32)P.n, (u32)first, P.pre_c, d_sc, (u32)n, out_affine, out_xyzz);
  return msm_run((const Affine*)P.p + first, nullptr, d_sc, (u32)n, nullptr, 1, n, out_affine, out_xyzz);
}

extern "C" int bp_msm_set_small_graphs(int on) { g_small_graphs = on != 0; if (!on) { if (g.inited) cudaStreamSynchronize(g.stream); pre_graphs_clear(); } return 0; }

static int handle_msm_to_host(const HandleRec& P, size_t first, const Fq* d_sc, size_t n, uint8_t* out64) {
  Affine* d_out = (Affine*)g.ws_out.ensure(sizeof(Affine));
  if (!d_out) return fail("workspace allocation failed");
  if (handle_msm(P, first, d_sc, n, d_out, nullptr)) return 1;
  BP_CUDA(cudaMemcpyAsync(out64, d_out, 64, cudaMemcpyDeviceToHost, g.stream));
  BP_CUDA(cudaStreamSynchronize(g.stream));
  return 0;
}

int bp_points_precompute(bp_handle points, int window_bits) {
  BP_NEED_INIT();
  std::lock_guard<std::mutex> lk(g_mu);
  auto it = g_handles.find(points);
  if (it == g_handles.end() || it->second.kind != 0) return fail("bad handle %llu", (unsigned long long)points);
  HandleRec& P = it->second;
  if (window_bits < 0 || (window_bits > 0 && window_bits < 8) || window_bits > 20) return fail("bp_points_precompute: window_bits 0 (automatic) or 8..20");
  const int c = window_bits ? window_bits : pre_pick_window(P.n);
  if (P.pre && P.pre_c == c) return 0;
  const PreShape ps = pre_shape(c);
  if (P.n == 0) return 0;
  if ((unsigned long long)ps.W * P.n >= (1ull << 30)) return fail("bp_points_precompute: vector too long for 30-bit point indices");
  cudaStreamSynchronize(g.stream);
  if (P.pre) { cudaFree(P.pre); P.pre = nullptr; P.pre_c = 0; }
  Affine* pre = nullptr;
  if (cudaMalloc((void**)&pre, (size_t)ps.W * P.n * sizeof(Affine)) != cudaSuccess) { cudaGetLastError(); return fail("bp_points_precompute: out of device memory (%zu bytes)", (size_t)ps.W * P.n * sizeof(Affine)); }
  ++g.nlaunch, k_pre_build<<<(unsigned)((P.n + 127) / 128), 128, 0, g.stream>>>((const Affine*)P.p, (u32)P.n, ps, pre);
  cudaError_t e = cudaStreamSynchronize(g.stream);
  if (e != cudaSuccess) { cudaGetLastError(); cudaFree(pre); return fail("k_pre_build failed: %s", cudaGetErrorString(e)); }
  P.pre = pre; P.pre_c = c;
  return 0;
}
int bp_points_pre_info(bp_handle points, int* window_bits, int* windows, uint64_t* bytes) {
  HandleRec P;
  if (get_handle(points, 0, &P)) return 1;
  const PreShape ps = pre_shape(P.pre_c ? P.pre_c : 8);
  if (window_bits) *window_bits = P.pre ? P.pre_c : 0;
  if (windows) *windows = P.pre ? ps.W : 0;
  if (bytes) *bytes = P.pre ? (uint64_t)ps.W * P.n * sizeof(Affine) : 0;
  return 0;
}

int bp_msm_h(bp_handle points, const uint8_t* sc32, size_t n, uint8_t out64[64]) {
  BP_NEED_INIT();
  HandleRec P;
  if (get_handle(points, 0, &P)) return 1;
  if (n > P.n) return fail("bp_msm_h: n exceeds the uploaded vector");
  if (n == 0) { memset(out64, 0, 64); return 0; }
  Fq* d_sc = (Fq*)g.ws_sc.ensure(n * sizeof(Fq));
  if (!d_sc) return fail("device allocation failed");
  BP_CUDA(cudaMemcpyAsync(d_sc, sc32, n * 32, cudaMemcpyHostToDevice, g.stream));
  return handle_msm_to_host(P, 0, d_sc, n, out64);
}

int bp_msm_hh(bp_handle points, bp_handle scalars, size_t n, uint8_t out64[64]) {
  BP_NEED_INIT();
  HandleRec P, S;
  if (get_handle(points, 0, &P) || get_handle(scalars, 1, &S)) return 1;
  if (n > P.n || n > S.n) return fail("bp_msm_hh: n exceeds the uploaded vectors");
  if (n == 0) { memset(out64, 0, 64); return 0; }
  return handle_msm_to_host(P, 0, (const Fq*)S.p, n, out64);
}

int bp_msm_hh_partial(bp_handle points, bp_handle scalars, size_t first, size_t n, uint8_t out128[128]) {
  BP_NEED_INIT();
  HandleRec P, S;
  if (get_handle(points, 0, &P) || get_handle(scalars, 1, &S)) return 1;
  if (first + n > P.n || first + n > S.n) return fail("bp_msm_hh_partial: slice exceeds the uploaded vectors");
  if (n == 0) { memset(out128, 0, 128); return 0; }
  XYZZ* d_out = (XYZZ*)g.ws_out.ensure(sizeof(XYZZ));
  if (handle_msm(P, first, (const Fq*)S.p + first, n, nullptr, d_out)) return 1;
  BP_CUDA(cudaMemcpyAsync(out128, d_out, 128, cudaMemcpyDeviceToHost, g.stream));
  BP_CUDA(cudaStreamSynchronize(g.stream));
  return 0;
}

int bp_xyzz_sum(const uint8_t* partials128, size_t count, uint8_t out64[64]) {
  BP_NEED_INIT();
  if (count == 0) { memset(out64, 0, 64); return 0; }
  XYZZ* d_in = (XYZZ*)g.ws_misc.ensure(count * sizeof(XYZZ));
  Affine* d_out = (Affine*)g.ws_out.ensure(sizeof(Affine));
  BP_CUDA(cudaMemcpyAsync(d_in, partials128, count * 128, cudaMemcpyHostToDevice, g.stream));
  ++g.nlaunch, k_xyzz_sum<<<1, 32, 0, g.stream>>>(d_in, (u32)count, d_out);
  BP_CUDA(cudaMemcpyAsync(out64, d_out, 64, cudaMemcpyDeviceToHost, g.stream));
  BP_CUDA(cudaStreamSynchronize(g.stream));
  return 0;
}

int bp_msm_batch(const uint8_t* pts64, const uint8_t* sc32, const uint32_t* offsets, size_t nmsm, uint8_t* out64) {
  BP_NEED_INIT();
  if (nmsm == 0) return 0;
  size_t T = offsets[nmsm];
  size_t maxlen = 0;
  for (size_t j = 0; j < nmsm; j++) { if (offsets[j + 1] < offsets[j]) return fail("bp_msm_batch: offsets not monotone"); size_t l = offsets[j + 1] - offsets[j]; if (l > maxlen) maxlen = l; }
  if (T == 0) { memset(out64, 0, nmsm * 64); return 0; }
  Affine* d_pts = (Affine*)g.ws_pts.ensure(T * sizeof(Affine));
  Fq* d_sc = (Fq*)g.ws_sc.ensure(T * sizeof(Fq));
  u32* d_off = (u32*)g.ws_off.ensure((nmsm + 1) * sizeof(u32));
  Affine* d_out = (Affine*)g.ws_out.ensure(nmsm * sizeof(Affine));
  if (!d_pts || !d_sc || !d_off || !d_out) return fail("device allocation failed");
  BP_CUDA(cudaMemcpyAsync(d_sc, sc32, T * 32, cudaMemcpyHostToDevice, g.stream));
  BP_CUDA(cudaMemcpyAsync(d_off, offsets, (nmsm + 1) * sizeof(u32), cudaMemcpyHostToDevice, g.stream));
  if (fb_enabled() && maxlen <= fb.max_points && nmsm <= 65535 && T == nmsm * maxlen) {
    // every MSM of the batch over the SAME point list (A and S of a range proof, T1 and T2): one table serves all
    bool same = true;
    for (size_t j = 1; j < nmsm && same; j++) same = memcmp(pts64, pts64 + (size_t)offsets[j] * 64, maxlen * 64) == 0;
    if (same) {
      const FbSrc src = {{pts64}, {maxlen * 64}, 1};
      const uint64_t key = src.hash(0x6D736D31ull);
      BP_CUDA(cudaMemcpyAsync(d_pts, pts64, maxlen * 64, cudaMemcpyHostToDevice, g.stream));
      const Affine* tab = fb_get(key, src, d_pts, maxlen);
      if (tab) {
        if (nmsm <= 64) return fb_msm_run_host(tab, nullptr, d_sc, d_off, (u32)nmsm, maxlen, 0, out64);
        if (fb_msm_run(tab, nullptr, d_sc, d_off, (u32)nmsm, maxlen, 0, d_out, nullptr)) return 1;
        BP_CUDA(cudaMemcpyAsync(out64, d_out, nmsm * 64, cudaMemcpyDeviceToHost, g.stream));
        BP_CUDA(cudaStreamSynchronize(g.stream));
        return 0;
      }
    }
  }
  BP_CUDA(cudaMemcpyAsync(d_pts, pts64, T * 64, cudaMemcpyHostToDevice, g.stream));
  size_t avg = (T + nmsm - 1) / nmsm;
  if (msm_run(d_pts, nullptr, d_sc, (u32)T, d_off, (u32)nmsm, avg, d_out, nullptr)) return 1;
  BP_CUDA(cudaMemcpyAsync(out64, d_out, nmsm * 64, cudaMemcpyDeviceToHost, g.stream));
  BP_CUDA(cudaStreamSynchronize(g.stream));
  return 0;
}

int bp_scalar_mul_batch(const uint8_t* pts64, const uint8_t* sc32, size_t n, uint8_t* out64) {
  BP_NEED_INIT();
  if (n == 0) return 0;
  Affine* d_pts = (Affine*)g.ws_pts.ensure(n * sizeof(Affine));
  Fq* d_sc = (Fq*)g.ws_sc.ensure(n * sizeof(Fq));
  Affine* d_out = (Affine*)g.ws_out.ensure(n * sizeof(Affine));
  if (!d_pts || !d_sc || !d_out) return fail("device allocation failed");
  BP_CUDA(cudaMemcpyAsync(d_pts, pts64, n * 64, cudaMemcpyHostToDevice, g.stream));
  BP_CUDA(cudaMemcpyAsync(d_sc, sc32, n * 32, cudaMemcpyHostToDevice, g.stream));
  ++g.nlaunch, k_scalar_mul<<<(unsigned)((n + 63) / 64), 64, 0, g.stream>>>(d_pts, d_sc, (u32)n, d_out);
  BP_CUDA(cudaMemcpyAsync(out64, d_out, n * 64, cudaMemcpyDeviceToHost, g.stream));
  BP_CUDA(cudaStreamSynchronize(g.stream));
  return 0;
}

int bp_bench_msm(bp_handle points, bp_handle scalars, size_t n, int warmup, int iters, int flush_l2, float* ms_each, uint8_t out64[64]) {
  BP_NEED_INIT();
  HandleRec P, S;
  if (get_handle(points, 0, &P) || get_handle(scalars, 1, &S)) return 1;
  if (n > P.n || n > S.n || n == 0) return fail("bp_bench_msm: bad n");
  Affine* d_out = (Affine*)g.ws_out.ensure(sizeof(Affine));
  const size_t flush_bytes = 256u << 20;
  void* d_flush = flush_l2 ? g.ws_flush.ensure(flush_bytes) : nullptr;
  for (int it = 0; it < warmup + iters; it++) {
    if (d_flush) BP_CUDA(cudaMemsetAsync(d_flush, it & 0xff, flush_bytes, g.stream));
    BP_CUDA(cudaEventRecord(g.ev_a, g.stream));
    if (handle_msm(P, 0, (const Fq*)S.p, n, d_out, nullptr)) return 1;
    BP_CUDA(cudaEventRecord(g.ev_b, g.stream));
    BP_CUDA(cudaEventSynchronize(g.ev_b));
    float ms = 0;
    BP_CUDA(cudaEventElapsedTime(&ms, g.ev_a, g.ev_b));
    if (it >= warmup) ms_each[it - warmup] = ms;
  }
  BP_CUDA(cudaMemcpy(out64, d_out, 64, cudaMemcpyDeviceToHost));
  return 0;
}

// ops per launch-thread-iteration for each probe mode
static int pipe_probe(int mode, int iters, double* ops_per_s, float* ms_out) {
  u32* d = (u32*)g.ws_misc.ensure(256);
  int blocks = g.sm_count * 8;
  double per_iter = (mode == 3 || mode == 5) ? 2.0 : 32.0;
  for (int pass = 0; pass < 2; pass++) {      // pass 0 = warm-up (clocks, I-cache), pass 1 timed
    int n = pass == 0 ? (iters / 8 > 0 ? iters / 8 : 1) : iters;
    BP_CUDA(cudaEventRecord(g.ev_a, g.stream));
    switch (mode) {
      case 0: ++g.nlaunch, k_pipe_probe<0><<<blocks, 256, 0, g.stream>>>(d, 12345u, n); break;
      case 1: ++g.nlaunch, k_pipe_probe<1><<<blocks, 256, 0, g.stream>>>(d, 12345u, n); break;
      case 2: ++g.nlaunch, k_pipe_probe<2><<<blocks, 256, 0, g.stream>>>(d, 12345u, n); break;
      case 3: ++g.nlaunch, k_pipe_probe<3><<<blocks, 256, 0, g.stream>>>(d, 12345u, n); break;
      case 4: ++g.nlaunch, k_pipe_probe<4><<<blocks, 256, 0, g.stream>>>(d, 12345u, n); break;
      case 5: ++g.nlaunch, k_pipe_probe<5><<<blocks, 256, 0, g.stream>>>(d, 12345u, n); break;
      case 6: ++g.nlaunch, k_pipe_probe<6><<<1, 32, 0, g.stream>>>(d, 12345u, n); break;
      case 7: ++g.nlaunch, k_pipe_probe<7><<<1, 32, 0, g.stream>>>(d, 12345u, n); break;
      case 8: ++g.nlaunch, k_pipe_probe<8><<<1, 32, 0, g.stream>>>(d, 12345u, n); break;
      case 9: ++g.nlaunch, k_pipe_probe<9><<<1, 32, 0, g.stream>>>(d, 12345u, n); break;
      case 10: ++g.nlaunch, k_pipe_probe<10><<<blocks, 256, 0, g.stream>>>(d, 12345u, n); break;
      case 11: ++g.nlaunch, k_pipe_probe<11><<<blocks, 256, 0, g.stream>>>(d, 12345u, n); break;
      default: return fail("bp_pipe_probe: mode 0..11");
    }
    BP_CUDA(cudaEventRecord(g.ev_b, g.stream));
    BP_CUDA(cudaEventSynchronize(g.ev_b));
  }
  float ms = 0;
  BP_CUDA(cudaEventElapsedTime(&ms, g.ev_a, g.ev_b));
  if (ops_per_s) *ops_per_s = (double)blocks * 256.0 * (double)iters * per_iter / (ms * 1e-3);
  if (ms_out) *ms_out = ms;
  return 0;
}
int bp_pipe_probe(int mode, int iters, double* ops_per_s, float* ms_out) { BP_NEED_INIT(); return pipe_probe(mode, iters, ops_per_s, ms_out); }
int bp_imad_peak(int iters, double* macs_per_s, float* ms_out) { BP_NEED_INIT(); return pipe_probe(0, iters, macs_per_s, ms_out); }

}  // extern "C"
#include "bp_proto.inl"
#include "bp_aggreg.inl"
#include "bp_rlc.inl"
#include "bp_prove.inl"
