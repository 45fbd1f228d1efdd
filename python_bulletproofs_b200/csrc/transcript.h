// transcript.h -- host-side Fiat-Shamir helpers, restated in C++ so the sequential challenge
// derivation can run inside the library between kernel launches (no Python in the round loop).
//
// Replaces (bit-exactly): mod_hash, point_to_bytes, point_to_b64
// (/root/reference/src/utils/utils.py:84-111) and Transcript.add_point / add_number / get_modp
// (/root/reference/src/utils/transcript.py:16-33).  hashlib's SHA-256 is restated from FIPS 180-4.
#pragma once
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <string>
#include "fq.cuh"

namespace bp {

// ---- SHA-256 (FIPS 180-4); the compression function lives in sha256_host.cc (portable / SHA-NI) -------------
void sha256_blocks(uint32_t h[8], const uint8_t* p, size_t nblocks);
void sha256_force_portable(int on);
int sha256_impl();

struct Sha256 {          // trivially copyable: a running context can be cloned and finalised
  uint32_t h[8];
  uint8_t buf[64];
  uint64_t len = 0;
  size_t fill = 0;
  Sha256() {
    static const uint32_t iv[8] = {0x6a09e667, 0xbb67ae85, 0x3c6ef372, 0xa54ff53a, 0x510e527f, 0x9b05688c, 0x1f83d9ab, 0x5be0cd19};
    memcpy(h, iv, sizeof h);
  }
  void update(const uint8_t* p, size_t n) {
    len += n;
    if (fill) {
      size_t k = 64 - fill < n ? 64 - fill : n;
      memcpy(buf + fill, p, k); fill += k; p += k; n -= k;
      if (fill == 64) { sha256_blocks(h, buf, 1); fill = 0; }
    }
    if (n >= 64) { size_t nb = n / 64; sha256_blocks(h, p, nb); p += 64 * nb; n -= 64 * nb; }
    if (n) { memcpy(buf, p, n); fill = n; }
  }
  void final(uint8_t out[32]) {
    uint64_t bits = len * 8;
    uint8_t pad[72];
    size_t padlen = (fill < 56 ? 56 : 120) - fill;
    memset(pad, 0, sizeof pad);
    pad[0] = 0x80;
    for (int i = 0; i < 8; i++) pad[padlen + i] = (uint8_t)(bits >> (56 - 8 * i));
    update(pad, padlen + 8);
    for (int i = 0; i < 8; i++) { out[4 * i] = h[i] >> 24; out[4 * i + 1] = h[i] >> 16; out[4 * i + 2] = h[i] >> 8; out[4 * i + 3] = h[i]; }
  }
};

inline bool digest_to_scalar(const uint8_t d[32], Fq* x) {   // big-endian digest -> candidate; false if rejected (>= q or 0)
  for (int i = 0; i < 8; i++)
    x->v[i] = (uint32_t)d[31 - 4 * i] | (uint32_t)d[30 - 4 * i] << 8 | (uint32_t)d[29 - 4 * i] << 16 | (uint32_t)d[28 - 4 * i] << 24;
  return !fq_geq(*x, fq_const_q()) && !fq_is_zero(*x);
}

// mod_hash(msg, q): utils.py:84-97.  q is 256 bits so the `% 2**bit_length` mask is a no-op.
inline Fq mod_hash_q(const uint8_t* msg, size_t len) {
  for (unsigned long ctr = 1;; ctr++) {
    char pre[24];
    int pl = snprintf(pre, sizeof pre, "%lu", ctr);
    Sha256 s;
    s.update((const uint8_t*)pre, (size_t)pl);
    s.update(msg, len);
    uint8_t d[32];
    s.final(d);
    Fq x;
    if (digest_to_scalar(d, &x)) return x;       // else x >= q or x == 0: next counter
  }
}

// The transcript only ever grows, and the accepted counter is "1" except with probability ~2^-128, so the SHA-256
// state of "1" || transcript-so-far is kept and cloned for each challenge instead of re-hashing the whole prefix
// (the reference re-hashes: O(rounds * length)).  Falls back to mod_hash_q when counter 1 is rejected.
struct RunningModHash {
  Sha256 ctx;
  size_t absorbed = 0;
  RunningModHash() { const uint8_t one = '1'; ctx.update(&one, 1); }
  // challenge for the message base[0..upto); base must extend the bytes absorbed so far
  Fq challenge(const uint8_t* base, size_t upto) {
    ctx.update(base + absorbed, upto - absorbed);
    absorbed = upto;
    Sha256 c = ctx;
    uint8_t d[32];
    c.final(d);
    Fq x;
    if (digest_to_scalar(d, &x)) return x;
    return mod_hash_q(base, upto);
  }
};

// str(x): decimal of a 256-bit integer (transcript.py:29-31 via ModP.__str__, utils.py:77-78)
inline std::string fq_to_decimal(const Fq& a) {
  uint32_t w[8];
  memcpy(w, a.v, sizeof w);
  char tmp[80];
  int n = 0;
  bool nz = true;
  while (nz) {
    uint64_t rem = 0;
    nz = false;
    for (int i = 7; i >= 0; i--) {
      uint64_t cur = (rem << 32) | w[i];
      w[i] = (uint32_t)(cur / 1000000000u);
      rem = cur % 1000000000u;
      if (w[i]) nz = true;
    }
    for (int k = 0; k < 9; k++) { tmp[n++] = (char)('0' + rem % 10); rem /= 10; }
  }
  while (n > 1 && tmp[n - 1] == '0') n--;
  std::string s(n, '0');
  for (int i = 0; i < n; i++) s[i] = tmp[n - 1 - i];
  return s;
}

// int(slot) for a plain run of ASCII digits (any length), reduced mod q.  Returns false when the
// slot is empty or contains anything else: Python's int() has more accepting syntax (sign,
// underscores, surrounding whitespace), so the caller must then defer to it.
inline bool decimal_to_fq(const uint8_t* s, size_t n, Fq* out) {
  if (n == 0) return false;
  static const uint32_t P10[10] = {1u, 10u, 100u, 1000u, 10000u, 100000u, 1000000u, 10000000u, 100000000u, 1000000000u};
  Fq acc = fq_zero();
  for (size_t i = 0; i < n;) {                     // nine digits at a time: acc = acc * 10^k + chunk  (mod q)
    size_t k = n - i < 9 ? n - i : 9;
    uint32_t chunk = 0;
    for (size_t j = 0; j < k; j++) {
      if (s[i + j] < '0' || s[i + j] > '9') return false;
      chunk = chunk * 10 + (uint32_t)(s[i + j] - '0');
    }
    acc = fq_add(fq_mul(acc, fq_from_u64(P10[k])), fq_from_u64(chunk));
    i += k;
  }
  *out = acc;
  return true;
}

// base64.b64encode (RFC 4648, with padding): the transcript's seed slot and its points
inline std::string b64_encode(const uint8_t* raw, size_t n) {
  static const char* A = "ABCDEFGHIJKLMNOPQRSTUVWXYZabcdefghijklmnopqrstuvwxyz0123456789+/";
  std::string o;
  o.reserve((n + 2) / 3 * 4);
  for (size_t i = 0; i < n; i += 3) {
    uint32_t v = (uint32_t)raw[i] << 16 | (i + 1 < n ? (uint32_t)raw[i + 1] << 8 : 0) | (i + 2 < n ? raw[i + 2] : 0);
    o += A[(v >> 18) & 63];
    o += A[(v >> 12) & 63];
    o += i + 1 < n ? A[(v >> 6) & 63] : '=';
    o += i + 2 < n ? A[v & 63] : '=';
  }
  return o;
}

// point_to_b64: utils.py:100-111.  pt = 64-byte little-endian affine, identity = zeros.
inline std::string point_to_b64(const uint8_t pt[64]) {
  uint8_t raw[33];
  size_t n;
  bool ident = true;
  for (int i = 0; i < 64; i++) if (pt[i]) { ident = false; break; }
  if (ident) { raw[0] = 0; n = 1; }
  else {
    raw[0] = (pt[32] & 1) ? 3 : 2;                         // parity of y (little-endian byte 0)
    for (int i = 0; i < 32; i++) raw[1 + i] = pt[31 - i];  // x big-endian
    n = 33;
  }
  return b64_encode(raw, n);
}

// ---- allocation-free forms for the batch verifier's per-proof transcript checks ------------------------------
// point_to_b64(pt) == slot, without building a std::string
inline bool b64_point_eq(const uint8_t* slot, size_t len, const uint8_t pt[64]) {
  static const char* A = "ABCDEFGHIJKLMNOPQRSTUVWXYZabcdefghijklmnopqrstuvwxyz0123456789+/";
  bool ident = true;
  for (int i = 0; i < 64; i++) if (pt[i]) { ident = false; break; }
  if (ident) return len == 4 && memcmp(slot, "AA==", 4) == 0;          // base64(b"\x00")
  if (len != 44) return false;
  uint8_t raw[33];
  raw[0] = (pt[32] & 1) ? 3 : 2;
  for (int i = 0; i < 32; i++) raw[1 + i] = pt[31 - i];
  char o[44];
  for (int i = 0, k = 0; i < 33; i += 3, k += 4) {
    uint32_t v = (uint32_t)raw[i] << 16 | (uint32_t)raw[i + 1] << 8 | raw[i + 2];
    o[k] = A[(v >> 18) & 63]; o[k + 1] = A[(v >> 12) & 63]; o[k + 2] = A[(v >> 6) & 63]; o[k + 3] = A[v & 63];
  }
  return memcmp(slot, o, 44) == 0;
}

// Plain 256-bit value of a run of ASCII digits (no reduction).  Returns 0 = not a plain digit run / empty, 1 = value in *out,
// 2 = digits only but the value does not fit 256 bits.  *canonical = no superfluous leading zero (the form str(int) prints).
inline int decimal_to_u256(const uint8_t* s, size_t n, Fq* out, bool* canonical) {
  if (n == 0) return 0;
  *canonical = !(n > 1 && s[0] == '0');
  static const uint64_t P10[20] = {1ull, 10ull, 100ull, 1000ull, 10000ull, 100000ull, 1000000ull, 10000000ull, 100000000ull, 1000000000ull,
                                   10000000000ull, 100000000000ull, 1000000000000ull, 10000000000000ull, 100000000000000ull,
                                   1000000000000000ull, 10000000000000000ull, 100000000000000000ull, 1000000000000000000ull,
                                   10000000000000000000ull};
  uint64_t w[4] = {0, 0, 0, 0};
  bool overflow = false;
  for (size_t i = 0; i < n;) {                     // nineteen digits at a time: w = w * 10^k + chunk
    size_t k = n - i < 19 ? n - i : 19;
    uint64_t chunk = 0;
    for (size_t j = 0; j < k; j++) {
      unsigned d = (unsigned)s[i + j] - '0';
      if (d > 9) return 0;
      chunk = chunk * 10 + d;
    }
    unsigned __int128 cy = chunk;
    for (int l = 0; l < 4; l++) { cy += (unsigned __int128)w[l] * P10[k]; w[l] = (uint64_t)cy; cy >>= 64; }
    if (cy) overflow = true;
    i += k;
  }
  if (overflow) return 2;
  for (int l = 0; l < 4; l++) { out->v[2 * l] = (uint32_t)w[l]; out->v[2 * l + 1] = (uint32_t)(w[l] >> 32); }
  return 1;
}
// slot == str(x) for a reduced scalar x: the slot must be the canonical decimal of exactly that integer
inline bool decimal_slot_eq(const uint8_t* s, size_t n, const Fq& x) {
  Fq v; bool canon;
  return decimal_to_u256(s, n, &v, &canon) == 1 && canon && fq_eq(v, x);
}
// int(slot) mod q for a plain run of digits; fast path for values below 2^256, decimal_to_fq otherwise
inline bool decimal_to_fq_fast(const uint8_t* s, size_t n, Fq* out) {
  Fq v; bool canon;
  int rc = decimal_to_u256(s, n, &v, &canon);
  if (rc == 1) { *out = fq_reduce(v); return true; }
  if (rc == 0) return false;
  return decimal_to_fq(s, n, out);
}

inline void fq_from_le(Fq* r, const uint8_t* b) { memcpy(r->v, b, 32); }
inline void fq_to_le(uint8_t* b, const Fq& a) { memcpy(b, a.v, 32); }

}  // namespace bp
