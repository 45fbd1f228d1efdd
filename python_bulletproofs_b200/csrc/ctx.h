// ctx.h -- per-process device context of libbpgpu: one GPU, one stream, grow-only workspaces.
#pragma once
#include <cuda_runtime.h>
#include <cuda.h>
#include <cstddef>
#include <cstdlib>
#include <map>
#include <string>
#include <vector>

namespace bp {

int fail(const char* fmt, ...);
void nccl_shutdown();

#define BP_CUDA(call)                                                                              \
  do {                                                                                             \
    cudaError_t e__ = (call);                                                                      \
    if (e__ != cudaSuccess) { cudaGetLastError(); return ::bp::fail("%s failed: %s (%s:%d)", #call, cudaGetErrorString(e__), __FILE__, __LINE__); } \
  } while (0)

inline unsigned long long& alloc_generation() { static unsigned long long gen = 0; return gen; }   // bumps when any workspace moves

struct DevBuf {
  void* p = nullptr;
  size_t cap = 0;
  void* ensure(size_t bytes) {
    if (bytes <= cap && p) return p;
    alloc_generation()++;
    if (p) { cudaFree(p); p = nullptr; cap = 0; }
    size_t want = bytes + bytes / 4 + 256;
    if (cudaMalloc(&p, want) != cudaSuccess) { cudaGetLastError(); p = nullptr; return nullptr; }
    cap = want;
    return p;
  }
  void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
};

struct Ctx {
  bool inited = false;
  int device = -1;
  int sm_count = 0;
  cudaStream_t stream = nullptr;
  cudaEvent_t ev[8];
  cudaEvent_t ev_a, ev_b, ev_k0, ev_k1;
  cudaStream_t copy_stream = nullptr;           // uploads of points overlap the scalar-only stages
  cudaEvent_t ev_pts = nullptr, ev_copy_gate = nullptr;
  // large host-operand MSMs: the operands arrive in K parts (upload_operands), part k's scalars at ev_part_sc[k] and its points
  // at ev_half[k]; msm_run_parts sorts each part as its scalars land and accumulates it as its points land
  cudaEvent_t ev_half[8] = {nullptr}, ev_part_sc[8] = {nullptr};
  cudaEvent_t dbg_ev[12] = {nullptr}; bool dbg_e2e = false;      // BP_E2E_TIMING: timeline of a host-operand MSM (development aid)
  void dbg_rec(int i, cudaStream_t st) { if (!dbg_e2e) return; if (!dbg_ev[i]) cudaEventCreate(&dbg_ev[i]); cudaEventRecord(dbg_ev[i], st); }
  bool profiling = false;
  int force_c = 0, last_c = 0;
  // host-finished Horner (fp_host.h: horner_host): a host-result MSM on the plain path leaves its U window sums where `ws` points
  // instead of launching k_combine; the caller copies them out and finishes on a host core
  struct HostFinish { const void* ws = nullptr; int c = 0, W = 0, U = 0, dbl = 0; bool pending = false; } hf;
  bool hf_want = false, hf_enabled = true;
  int pre_slots = 1; unsigned pre_slots_min = 1u << 18; bool pre_slots_any = false;   // slot sort of the precomputed path (bp_msm_set_pre_slots)
  DevBuf ws_slots, ws_slots_ovf;
  unsigned long long nlaunch = 0;               // kernels launched by this library so far (bp_launch_count)
  size_t last_nb = 0;
  // MSM workspaces
  DevBuf ws_pts, ws_sc, ws_off, ws_out, ws_digits, ws_entries, ws_count, ws_start, ws_cursor, ws_tiles, ws_buckets, ws_segsum,
      ws_winsum, ws_misc, ws_flush, ws_entry_bucket, ws_part, ws_big, ws_phi, ws_segrun, ws_grpsum, ws_winpart, ws_fb_lanes, ws_fb_var;
  // IPA / verifier workspaces
  DevBuf ws_g, ws_h, ws_a, ws_b, ws_g2, ws_h2, ws_a2, ws_b2, ws_idx, ws_lr, ws_terms_sc, ws_small;
  DevBuf ws_sv_tab, ws_sv_acc, ws_sv_sc, ws_rp_sums;      // batch verifier: variable-point tables / window sums / split scalars; Gsum, Hsum
  DevBuf ws_prove;                                        // batch prover: generator rows, two chunks' state, term patterns
  std::vector<unsigned char> rp_sums_src; unsigned long long rp_sums_gen = 0;   // generator bytes the kept sums belong to
  cudaStream_t var_stream[2] = {nullptr, nullptr};        // batch verifier: proof-specific terms, concurrent with the table lookups (one per chunk parity,
                                                          // so that the doubling chains of consecutive chunks overlap)
  cudaEvent_t var_done[2] = {nullptr, nullptr}, ev_rp0 = nullptr, ev_rp1 = nullptr;
  int ensure_var_stream() {
    for (int i = 0; i < 2; i++) {
      if (var_stream[i]) continue;
      int lo = 0, hi = 0;
      cudaDeviceGetStreamPriorityRange(&lo, &hi);
      if (cudaStreamCreateWithPriority(&var_stream[i], cudaStreamNonBlocking, hi) != cudaSuccess) return fail("stream creation failed");
    }
    for (int i = 0; i < 2; i++)
      if (!var_done[i] && cudaEventCreateWithFlags(&var_done[i], cudaEventDisableTiming) != cudaSuccess) return fail("event creation failed");
    return 0;
  }
  // pinned staging for the chunked batch verifier
  unsigned char* stage_p = nullptr; size_t stage_cap = 0;
  cudaEvent_t stage_ev[2] = {nullptr, nullptr};
  unsigned char* pinned_stage(size_t bytes) {
    if (bytes <= stage_cap) return stage_p;
    if (stage_p) cudaFreeHost(stage_p);
    stage_p = nullptr; stage_cap = 0;
    if (cudaHostAlloc((void**)&stage_p, bytes, cudaHostAllocDefault) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    stage_cap = bytes;
    return stage_p;
  }
  // side stream of the batch verifier: per-chunk upload / inversion / expansion under the previous chunk's MSM work
  cudaStream_t aux_stream = nullptr;
  cudaEvent_t aux_ready[2] = {nullptr, nullptr}, aux_free[2] = {nullptr, nullptr};
  int ensure_aux() {
    if (ensure_stage_events()) return 1;
    if (!aux_stream) {   // high priority: its kernels are short latency chains that should slip in between the blocks of the main stream
      int lo = 0, hi = 0;
      cudaDeviceGetStreamPriorityRange(&lo, &hi);
      if (cudaStreamCreateWithPriority(&aux_stream, cudaStreamNonBlocking, hi) != cudaSuccess) return fail("stream creation failed");
    }
    for (int i = 0; i < 2; i++) {
      if (!aux_ready[i] && cudaEventCreateWithFlags(&aux_ready[i], cudaEventDisableTiming) != cudaSuccess) return fail("event creation failed");
      if (!aux_free[i] && cudaEventCreateWithFlags(&aux_free[i], cudaEventDisableTiming) != cudaSuccess) return fail("event creation failed");
    }
    return 0;
  }
  int ensure_stage_events() {
    if (!ev_rp0 && (cudaEventCreate(&ev_rp0) != cudaSuccess || cudaEventCreate(&ev_rp1) != cudaSuccess)) return fail("event creation failed");
    for (int i = 0; i < 2; i++)
      if (!stage_ev[i] && cudaEventCreateWithFlags(&stage_ev[i], cudaEventDisableTiming) != cudaSuccess) return fail("event creation failed");
    return 0;
  }
  // IPA prover: how the host's Fiat-Shamir step meets the stream (bp_ipa_set_graphs; see bp_ipa_prove_hs)
  // Default 1, except under a CUDA tool (ncu, compute-sanitizer: they inject through CUDA_INJECTION64_PATH and run each launch
  // to completion inside the launch call, which can never happen behind a stream wait that the same thread has yet to release)
  // where it is 0; BP_IPA_MODE overrides both.
  static int default_ipa_mode() {
    if (const char* e = getenv("BP_IPA_MODE")) { int m = atoi(e); if (m >= 0 && m <= 2) return m; }
    if (getenv("CUDA_INJECTION64_PATH") || getenv("NV_COMPUTE_PROFILER_PERFWORKS_DIR")) return 0;
    return 1;
  }
  int ipa_mode = default_ipa_mode();
  bool ipa_fast = true;        // two-launch table rounds for n <= 4096 (bp_ipa_set_fast_rounds)
  DevBuf ws_ipa_ticket;
  // stream memory operations, resolved through the runtime (no link-time dependency on libcuda)
  CUresult (*cuWaitValue32)(CUstream, CUdeviceptr, cuuint32_t, unsigned int) = nullptr;
  CUresult (*cuWriteValue32)(CUstream, CUdeviceptr, cuuint32_t, unsigned int) = nullptr;
  int memops_state = 0;        // 0 = not probed, 1 = available, -1 = not available
  bool memops_ready() {
    if (memops_state == 0) {
      cudaDriverEntryPointQueryResult q1, q2;
      void *f1 = nullptr, *f2 = nullptr;
      const bool ok = cudaGetDriverEntryPoint("cuStreamWaitValue32", &f1, cudaEnableDefault, &q1) == cudaSuccess && q1 == cudaDriverEntryPointSuccess && f1 &&
                      cudaGetDriverEntryPoint("cuStreamWriteValue32", &f2, cudaEnableDefault, &q2) == cudaSuccess && q2 == cudaDriverEntryPointSuccess && f2;
      if (!ok) cudaGetLastError();
      cuWaitValue32 = (decltype(cuWaitValue32))f1; cuWriteValue32 = (decltype(cuWriteValue32))f2;
      memops_state = ok ? 1 : -1;
    }
    return memops_state == 1;
  }
  // IPA proof graphs (mode 2): one instantiated graph per vector length, valid while no workspace has been reallocated
  DevBuf ws_ipa_rp;
  struct GraphRec { cudaGraphExec_t exec; unsigned long long gen; const void* tab; unsigned nk; };   // nk = kernel nodes
  std::map<size_t, GraphRec> ipa_graphs;
  // `tab` = the fixed-base table the captured round reads (nullptr: bucket-method round); part of the key
  // (n, table) pairs whose eager proof has sized every workspace, with the allocation generation at that moment
  std::map<size_t, unsigned long long> ipa_sized;
  void ipa_mark_sized(size_t n, const void* tab) { ipa_sized[2 * n + (tab ? 1 : 0)] = alloc_generation(); }
  bool ipa_sized_ok(size_t n, const void* tab) { auto it = ipa_sized.find(2 * n + (tab ? 1 : 0)); return it != ipa_sized.end() && it->second == alloc_generation(); }
  unsigned ipa_graph_kernels(size_t n, const void* tab) { auto it = ipa_graphs.find(2 * n + (tab ? 1 : 0)); return it == ipa_graphs.end() ? 0u : it->second.nk; }
  cudaGraphExec_t ipa_graph_lookup(size_t n, const void* tab) {
    auto it = ipa_graphs.find(2 * n + (tab ? 1 : 0));
    if (it == ipa_graphs.end()) return nullptr;
    if (it->second.gen != alloc_generation() || it->second.tab != tab) { cudaGraphExecDestroy(it->second.exec); ipa_graphs.erase(it); return nullptr; }
    return it->second.exec;
  }
  void ipa_graph_store(size_t n, const void* tab, cudaGraphExec_t e, unsigned nk) {
    auto it = ipa_graphs.find(2 * n + (tab ? 1 : 0));
    if (it != ipa_graphs.end()) cudaGraphExecDestroy(it->second.exec);
    ipa_graphs[2 * n + (tab ? 1 : 0)] = GraphRec{e, alloc_generation(), tab, nk};
  }
  unsigned char* pin_bytes_p = nullptr; size_t pin_bytes_cap = 0;
  unsigned char* pinned_bytes(size_t bytes) {
    if (bytes <= pin_bytes_cap) return pin_bytes_p;
    if (pin_bytes_p) cudaFreeHost(pin_bytes_p);
    pin_bytes_p = nullptr; pin_bytes_cap = 0;
    if (cudaHostAlloc((void**)&pin_bytes_p, bytes, cudaHostAllocDefault) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    pin_bytes_cap = bytes;
    return pin_bytes_p;
  }
  // second pinned block: XYZZ results of small table MSMs that the host finishes (fb_msm_run_host)
  unsigned char* pin2_p = nullptr; size_t pin2_cap = 0;
  unsigned char* pinned2(size_t bytes) {
    if (bytes <= pin2_cap) return pin2_p;
    if (pin2_p) cudaFreeHost(pin2_p);
    pin2_p = nullptr; pin2_cap = 0;
    if (cudaHostAlloc((void**)&pin2_p, bytes, cudaHostAllocDefault) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    pin2_cap = bytes;
    return pin2_p;
  }
  unsigned* h_pin = nullptr;
  unsigned* pinned_u32() { if (!h_pin && cudaHostAlloc((void**)&h_pin, 64, cudaHostAllocDefault) != cudaSuccess) { cudaGetLastError(); h_pin = nullptr; } return h_pin; }
  void free_all() {
    DevBuf* all[] = {&ws_pts, &ws_sc, &ws_off, &ws_out, &ws_digits, &ws_entries, &ws_count, &ws_start, &ws_cursor, &ws_tiles,
                     &ws_buckets, &ws_segsum, &ws_winsum, &ws_misc, &ws_flush, &ws_g, &ws_h, &ws_a, &ws_b, &ws_g2, &ws_h2,
                     &ws_a2, &ws_b2, &ws_idx, &ws_lr, &ws_terms_sc, &ws_small, &ws_entry_bucket, &ws_part, &ws_big, &ws_phi, &ws_segrun, &ws_grpsum, &ws_winpart, &ws_fb_lanes, &ws_fb_var, &ws_sv_tab, &ws_sv_acc, &ws_sv_sc, &ws_rp_sums,
                     &ws_ipa_rp, &ws_ipa_ticket, &ws_slots, &ws_slots_ovf, &ws_prove};
    rp_sums_src.clear();
    for (DevBuf* b : all) b->release();
  }
};

extern Ctx g;

}  // namespace bp
