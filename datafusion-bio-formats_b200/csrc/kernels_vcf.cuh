// kernels_vcf.cuh -- BGZF-VCF on the BAM scan engine: the eight fixed columns and the typed INFO fields.  sm_100a.
//
// Inflate, chunking, the newline scan, the carry of the incomplete tail line, Arrow layout and export are the engine's (engine.cu);
// a record is a line, framed as a SAM line is (sam_frame_kernel: the lines that start in [own_lo, own_hi)).  Per decode slice:
//
//   fields   vcf_fields_kernel<G>: a group of G lanes per line (8; 32 when the previous chunk's lines averaged above 2 KiB).  Each
//            lane tests 16 bytes per step, so a step covers 16 * G bytes of the line.  The group finds the first eight tabs (by the
//            running count of the lanes' tab masks) and then the INFO ';' separators; every INFO token is handed to the lane that
//            holds its terminating ';' (the token's start is the last ';' of the lanes in front, a max-scan), which looks its key
//            up in an open-addressing table of the projected INFO IDs plus END (built on the host, staged in shared memory) and
//            records the value's (offset, length) for that column.  A per-line claim bit per key catches a key given twice.
//   rows     vcf_rows_kernel: a thread per line.  Validates the fixed fields, parses POS / QUAL / END, and per projected column
//            writes the Utf8 byte count or list element count (List<Utf8>: also the bytes of its elements), the Int32 / Float32
//            value, and the validity / Flag words by __ballot_sync, 32 rows per word.  Values of projected INFO columns are checked
//            here against their declared type.
//   offsets  launch_offsets_scan (engine.cu) over every count column.
//   write    vcf_write_kernel<G>: the group copies the Utf8 bytes with grp_map4 (which also flags bytes of 0x80 and above); list
//            elements are parsed by one lane each (Int32 / Float32) or copied by the group (Utf8) with their child offsets and
//            child validity bits.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

#include "f32_parse.h"
#include "kernels_decode.cuh"

namespace bamscan {
namespace vcf {

// error codes of the decode error word (engine.cu::decode_error_to_rc): the first three classes are BAMSCAN_ERR_FORMAT, VALUE is
// BAMSCAN_ERR_SCHEMA, POS0 and LONG are BAMSCAN_ERR_UNSUPPORTED
enum VcfErr : uint32_t {
  VCF_ERR_FIELDS = 40 /* fewer than 8 fields */, VCF_ERR_HASH = 41 /* a '#' line or an empty line */, VCF_ERR_POS = 42,
  VCF_ERR_CHROM = 43 /* empty CHROM */, VCF_ERR_REF = 44 /* empty REF */, VCF_ERR_END = 45 /* END below POS */, VCF_ERR_DUP = 46,
  VCF_ERR_UTF8 = 47, VCF_ERR_QUAL = 48, VCF_ERR_VALUE = 49, VCF_ERR_POS0 = 50, VCF_ERR_LONG = 51,
  // FORMAT columns (kernels_vcf_format.cuh): the first three are BAMSCAN_ERR_FORMAT, FMT_VALUE is BAMSCAN_ERR_SCHEMA
  VCF_ERR_FMT_FIELDS = 52 /* not 9 + samples fields */, VCF_ERR_FMT_DUP = 53 /* a projected FORMAT key given twice */,
  VCF_ERR_FMT_MANY = 54 /* a sample with more values than keys */, VCF_ERR_FMT_VALUE = 55
};

constexpr int32_t K_Boolean = 6, K_ListUtf8 = 17;   // (bamscan_internal.h: HK_Boolean, HK_ListUtf8)
constexpr int MAX_INFO = 112;            // projected INFO columns (the count and byte columns fit the totals page of engine.cu)
constexpr int KEY_SLOTS = 256;
constexpr int KEY_BLOB = 4096;
constexpr uint32_t NOEQ = 0xffffffffu;   // Tok::len of a key without '='
constexpr uint32_t MAX_LINE = 16u << 20;

struct Row { uint32_t f[9]; uint32_t ntab; };   // f[k]: start of field k (k < 8); f[8]: end of INFO + 1; ntab: tabs found (<= 8)

struct InfoCol {
  uint2* tok;          // per row: {1 + offset of the value in U (0: the key is absent), value bytes (NOEQ: no '=')}
  uint32_t* valid;     // row validity words (null for Boolean)
  uint32_t* values;    // Int32 / Float32 values; Boolean: value words
  int32_t* lens;       // Utf8: bytes; list: elements -> offsets
  int32_t* blens;      // List<Utf8>: bytes of the row's elements -> the row's first byte in data
  uint32_t* cvalid;    // list: child validity words
  int32_t* coffs;      // List<Utf8>: child offsets
  uint8_t* data;       // Utf8 bytes; list child values; List<Utf8> child bytes
  int32_t kind;
  uint32_t pad;
};

// The keys looked up per token: the projected INFO IDs (key k is column k), then END when it is not one of them.
struct Keys {
  uint16_t slot[KEY_SLOTS];                // 1 + key, 0 = empty; linear probing from hash & (KEY_SLOTS - 1)
  uint16_t off[MAX_INFO + 2];              // key k = blob[off[k], off[k + 1])
  uint8_t blob[KEY_BLOB];
  int32_t n_keys, end_key;
};

struct Params {
  const uint8_t* U;
  const uint32_t* lines;      // line starts of the slice: row r = [lines[r], lines[r + 1] - 1)
  uint32_t n;
  int32_t zero_based, n_info;
  Row* rows;
  int32_t *l_chrom, *l_id, *l_ref, *l_alt, *l_filter;      // null when not projected
  uint32_t *v_id, *v_alt, *v_qual, *v_filter;
  uint32_t *start, *end, *qual;
  uint8_t *d_chrom, *d_id, *d_ref, *d_alt, *d_filter;
  uint32_t* err;
  Keys keys;
  InfoCol cols[MAX_INFO + 1];   // [end_key] is END's slot when END is not projected
};

__host__ __device__ inline uint32_t key_hash(const uint8_t* s, uint32_t n) {
  uint32_t h = 2166136261u;
  for (uint32_t i = 0; i < n; i++) h = (h ^ s[i]) * 16777619u;
  return h;
}

__device__ __forceinline__ void line_bounds(const Params& P, uint32_t r, uint32_t* b, uint32_t* e) {
  const uint32_t s = P.lines[r];
  uint32_t t = P.lines[r + 1] - 1u;           // the '\n' (or the virtual one behind an unterminated last line)
  if (t > s && P.U[t - 1] == '\r') t--;
  *b = s; *e = t;
}

// field k of a row: [*s, *t)
__device__ __forceinline__ void field(const Row& R, int k, uint32_t* s, uint32_t* t) {
  *s = R.f[k];
  *t = max(R.f[k + 1] - 1u, R.f[k]);
}

__device__ __forceinline__ bool is_dot(const uint8_t* v, uint32_t n) { return n == 1 && v[0] == '.'; }

// [+-]digits in the i32 range
__device__ __forceinline__ bool parse_i32(const uint8_t* s, uint32_t n, int32_t* out) {
  uint32_t k = 0; bool neg = false;
  if (k < n && (s[k] == '+' || s[k] == '-')) { neg = s[k] == '-'; k++; }
  if (k >= n) return false;
  long long x = 0;
  for (; k < n; k++) { if (s[k] < '0' || s[k] > '9') return false; x = x * 10 + (s[k] - '0'); if (x > (1ll << 32)) x = 1ll << 32; }
  x = neg ? -x : x;
  if (x < -2147483648ll || x > 2147483647ll) return false;
  *out = (int32_t)x;
  return true;
}

// One INFO token [a, z) of row r, by one lane: key lookup, duplicate claim, the value's position for the key's column
__device__ __forceinline__ void info_token(const Params& P, const Keys& K, uint32_t* seen, uint32_t r, uint32_t a, uint32_t z) {
  if (z <= a) return;
  uint32_t q = a;
  while (q < z && P.U[q] != '=') q++;
  const uint32_t kl = q - a;
  const uint32_t h = key_hash(P.U + a, kl);
  int key = -1;
  for (int i = 0; i < KEY_SLOTS; i++) {
    const uint32_t sl = K.slot[(h + i) & (KEY_SLOTS - 1)];
    if (!sl) return;                               // not a looked-up key: skipped
    const int k = (int)sl - 1;
    const uint32_t o = K.off[k];
    if (K.off[k + 1] - o != kl) continue;
    uint32_t j = 0;
    while (j < kl && K.blob[o + j] == P.U[a + j]) j++;
    if (j == kl) { key = k; break; }
  }
  if (key < 0) return;
  const uint32_t bit = 1u << (key & 31);
  if (atomicOr(&seen[key >> 5], bit) & bit) { set_err(P.err, VCF_ERR_DUP, r); return; }
  P.cols[key].tok[r] = q < z ? make_uint2(q + 2u, z - q - 1u) : make_uint2(z + 1u, NOEQ);
}

template <int G>
__global__ void __launch_bounds__(256)
vcf_fields_kernel(const Params P) {
  constexpr int NG = 256 / G, SEEN = (MAX_INFO + 1 + 31) / 32;
  __shared__ Keys sk;
  __shared__ uint32_t s_tab[NG][8];
  __shared__ uint32_t s_seen[NG][SEEN];
  for (uint32_t i = threadIdx.x; i < sizeof(Keys) / 4; i += blockDim.x) reinterpret_cast<uint32_t*>(&sk)[i] = reinterpret_cast<const uint32_t*>(&P.keys)[i];
  __syncthreads();
  const int lane = threadIdx.x & 31, gl = lane & (G - 1), grp = threadIdx.x / G;
  const unsigned gmask = G == 32 ? 0xffffffffu : (((1u << G) - 1u) << (lane & ~(G - 1)));
  const uint32_t r = (blockIdx.x * blockDim.x + threadIdx.x) / G;
  if (r >= P.n) return;                            // (whole groups)
  uint32_t b, e;
  line_bounds(P, r, &b, &e);
  // the first eight tabs
  uint32_t found = 0;
  for (uint32_t w = b; w < e && found < 8u; w += G * 16) {
    const uint32_t o = w + gl * 16;
    uint32_t m = 0;
    #pragma unroll
    for (int k = 0; k < 16; k++) if (o + k < e && P.U[o + k] == '\t') m |= 1u << k;
    const uint32_t c = __popc(m);
    uint32_t incl = c;
    #pragma unroll
    for (int s = 1; s < G; s <<= 1) { const uint32_t y = __shfl_up_sync(gmask, incl, s, G); if (gl >= s) incl += y; }
    uint32_t idx = found + incl - c;
    while (m && idx < 8u) { const int k = __ffs((int)m) - 1; m &= m - 1u; s_tab[grp][idx++] = o + k; }
    found += __shfl_sync(gmask, incl, G - 1, G);
  }
  if (gl < SEEN) s_seen[grp][gl] = 0;
  __syncwarp(gmask);
  Row R;
  R.ntab = min(found, 8u);
  R.f[0] = b;
  #pragma unroll
  for (int k = 1; k < 9; k++) R.f[k] = (uint32_t)k <= R.ntab ? s_tab[grp][k - 1] + 1u : e + 1u;
  if (gl == 0) P.rows[r] = R;
  if (R.ntab < 7u) return;
  // INFO = [i0, i1): '.' or ';'-separated tokens
  const uint32_t i0 = R.f[7], i1 = R.f[8] - 1u;
  if (i1 <= i0 || is_dot(P.U + i0, i1 - i0)) return;
  uint32_t tok = i0;                               // start of the token still open (group-uniform)
  for (uint32_t w = i0; w < i1; w += G * 16) {
    const uint32_t o = w + gl * 16;
    uint32_t m = 0;
    #pragma unroll
    for (int k = 0; k < 16; k++) if (o + k < i1 && P.U[o + k] == ';') m |= 1u << k;
    const uint32_t last = m ? o + (31u - __clz(m)) + 1u : 0u;    // 1 + the lane's last ';'
    uint32_t incl = last;
    #pragma unroll
    for (int s = 1; s < G; s <<= 1) { const uint32_t y = __shfl_up_sync(gmask, incl, s, G); if (gl >= s) incl = max(incl, y); }
    uint32_t prev = __shfl_up_sync(gmask, incl, 1, G);
    uint32_t a = (gl > 0 && prev) ? prev : tok;
    while (m) {
      const int k = __ffs((int)m) - 1; m &= m - 1u;
      info_token(P, sk, s_seen[grp], r, a, o + k);
      a = o + k + 1u;
    }
    const uint32_t wl = __shfl_sync(gmask, incl, G - 1, G);
    if (wl) tok = wl;
  }
  if (gl == 0) info_token(P, sk, s_seen[grp], r, tok, i1);
}

// The elements of a list value v[0, n): calls fn(i, begin, len) per element in order
template <typename Fn>
__device__ __forceinline__ uint32_t for_elements(const uint8_t* v, uint32_t n, Fn fn) {
  uint32_t i = 0, a = 0;
  for (uint32_t k = 0; k <= n; k++) {
    if (k == n || v[k] == ',') { fn(i, a, k - a); i++; a = k + 1; }
  }
  return i;
}

__global__ void __launch_bounds__(256)
vcf_rows_kernel(const Params P) {
  const uint32_t r = blockIdx.x * blockDim.x + threadIdx.x;
  const bool on = r < P.n;
  bool id_ok = false, alt_ok = false, qual_ok = false, filter_ok = false;
  Row R{};
  if (on) {
    uint32_t b, e, s, t;
    line_bounds(P, r, &b, &e);
    R = P.rows[r];
    const uint8_t* U = P.U;
    if (P.lines[r + 1] - P.lines[r] > MAX_LINE) set_err(P.err, VCF_ERR_LONG, r);
    if (e == b || U[b] == '#') set_err(P.err, VCF_ERR_HASH, r);
    else if (R.ntab < 7u) set_err(P.err, VCF_ERR_FIELDS, r);
    field(R, 0, &s, &t);
    if (t == s) set_err(P.err, VCF_ERR_CHROM, r);
    if (P.l_chrom) P.l_chrom[r] = (int32_t)(t - s);
    // POS: digits, 1 ..= 2^31 - 1
    field(R, 1, &s, &t);
    uint64_t pos = 0;
    bool pos_ok = t > s && t - s <= 10;
    for (uint32_t k = s; k < t && pos_ok; k++) { if (U[k] < '0' || U[k] > '9') pos_ok = false; else pos = pos * 10 + (U[k] - '0'); }
    if (!pos_ok || pos > 2147483647ull) set_err(P.err, VCF_ERR_POS, r);
    else if (pos == 0) set_err(P.err, VCF_ERR_POS0, r);
    field(R, 2, &s, &t);
    id_ok = !is_dot(U + s, t - s);
    if (P.l_id) P.l_id[r] = id_ok ? (int32_t)(t - s) : 0;
    field(R, 3, &s, &t);
    const uint32_t ref_len = t - s;
    if (ref_len == 0 && R.ntab >= 7u) set_err(P.err, VCF_ERR_REF, r);
    if (P.l_ref) P.l_ref[r] = (int32_t)ref_len;
    field(R, 4, &s, &t);
    alt_ok = !is_dot(U + s, t - s);
    if (P.l_alt) P.l_alt[r] = alt_ok ? (int32_t)(t - s) : 0;
    field(R, 5, &s, &t);
    qual_ok = !is_dot(U + s, t - s);
    uint32_t qbits = 0;
    if (qual_ok && !f32_parse(reinterpret_cast<const char*>(U + s), t - s, &qbits)) { set_err(P.err, VCF_ERR_QUAL, r); qual_ok = false; }
    if (P.qual) P.qual[r] = qual_ok ? qbits : 0u;
    field(R, 6, &s, &t);
    filter_ok = !is_dot(U + s, t - s);
    if (P.l_filter) P.l_filter[r] = filter_ok ? (int32_t)(t - s) : 0;
    // END (always read: `end` depends on it)
    uint64_t end = pos + ref_len - (ref_len ? 1u : 0u);
    const uint2 et = P.cols[P.keys.end_key].tok[r];
    if (et.x) {
      int32_t ev;
      if (et.y == NOEQ) set_err(P.err, VCF_ERR_VALUE, r);
      else if (!is_dot(U + et.x - 1u, et.y)) {
        if (!parse_i32(U + et.x - 1u, et.y, &ev)) set_err(P.err, VCF_ERR_VALUE, r);
        else if ((int64_t)ev < (int64_t)pos) set_err(P.err, VCF_ERR_END, r);
        else end = (uint64_t)ev;
      }
    }
    if (P.start) P.start[r] = (uint32_t)(P.zero_based ? pos - 1u : pos);
    if (P.end) P.end[r] = (uint32_t)end;
  }
  const int lane = threadIdx.x & 31;
  const bool word = lane == 0 && r < ((P.n + 31u) & ~31u);
  #define VCF_BALLOT(dst, pred) do { const uint32_t m_ = __ballot_sync(0xffffffffu, (pred)); if ((dst) && word) (dst)[r >> 5] = m_; } while (0)
  VCF_BALLOT(P.v_id, id_ok); VCF_BALLOT(P.v_alt, alt_ok); VCF_BALLOT(P.v_qual, qual_ok); VCF_BALLOT(P.v_filter, filter_ok);
  for (int c = 0; c < P.n_info; c++) {
    const InfoCol& C = P.cols[c];
    bool valid = false, bit = false;
    if (on) {
      const uint2 t = C.tok[r];
      int32_t len = 0, bytes = 0;
      uint32_t val = 0;
      const uint8_t* v = P.U + t.x - 1u;
      if (C.kind == K_Boolean) {
        if (t.x) { bit = true; if (t.y != NOEQ) set_err(P.err, VCF_ERR_VALUE, r); }
      } else if (t.x && t.y == NOEQ) {
        set_err(P.err, VCF_ERR_VALUE, r);
      } else if (t.x && !is_dot(v, t.y)) {
        const uint32_t vn = t.y;
        bool ok = true;
        switch (C.kind) {
          case K_Int32: ok = parse_i32(v, vn, reinterpret_cast<int32_t*>(&val)); break;
          case K_Float32: ok = f32_parse(reinterpret_cast<const char*>(v), vn, &val); break;
          case K_Utf8: for (uint32_t k = 0; k < vn; k++) if (v[k] == ',') ok = false; len = (int32_t)vn; break;
          default:
            len = (int32_t)for_elements(v, vn, [&](uint32_t, uint32_t a, uint32_t l) {
              if (is_dot(v + a, l)) return;
              if (C.kind == K_ListUtf8) bytes += (int32_t)l;
              else if (C.kind == K_ListInt32) { int32_t x; if (!parse_i32(v + a, l, &x)) ok = false; }
              else { uint32_t x; if (!f32_parse(reinterpret_cast<const char*>(v + a), l, &x)) ok = false; }
            });
        }
        if (!ok) { set_err(P.err, VCF_ERR_VALUE, r); len = 0; bytes = 0; val = 0; }
        valid = ok;
      }
      if (C.lens) C.lens[r] = len;
      if (C.blens) C.blens[r] = bytes;
      if (C.kind == K_Int32 || C.kind == K_Float32) C.values[r] = val;
    }
    VCF_BALLOT(C.valid, valid);
    if (C.kind == K_Boolean) VCF_BALLOT(C.values, bit);
  }
  #undef VCF_BALLOT
}

template <int G>
__global__ void __launch_bounds__(256)
vcf_write_kernel(const Params P) {
  const int lane = threadIdx.x & 31, gl = lane & (G - 1);
  const uint32_t r = (blockIdx.x * blockDim.x + threadIdx.x) / G;
  if (r >= P.n) return;
  const Row R = P.rows[r];
  uint32_t bad = 0, s, t;
  auto copy = [&](uint8_t* d, const int32_t* offs, int k) {
    if (!d) return;
    const uint32_t n = (uint32_t)(offs[r + 1] - offs[r]);
    field(R, k, &s, &t);
    if (n) bad |= grp_map4<G>(d + offs[r], P.U + s, n, gl, 0u);
  };
  copy(P.d_chrom, P.l_chrom, 0); copy(P.d_id, P.l_id, 2); copy(P.d_ref, P.l_ref, 3); copy(P.d_alt, P.l_alt, 4); copy(P.d_filter, P.l_filter, 6);
  for (int c = 0; c < P.n_info; c++) {
    const InfoCol& C = P.cols[c];
    if (C.kind == K_Boolean || C.kind == K_Int32 || C.kind == K_Float32) continue;
    if (C.kind == K_ListUtf8 && r + 1u == P.n && gl == 0) C.coffs[C.lens[P.n]] = C.blens[P.n];   // the child offsets' last entry
    const int32_t o0 = C.lens[r], cnt = C.lens[r + 1] - o0;
    if (cnt == 0) continue;
    const uint2 tk = C.tok[r];
    const uint8_t* v = P.U + tk.x - 1u;
    if (C.kind == K_Utf8) { bad |= grp_map4<G>(C.data + o0, v, (uint32_t)cnt, gl, 0u); continue; }
    if (C.kind == K_ListUtf8) {
      int32_t at = C.blens[r];
      for_elements(v, tk.y, [&](uint32_t i, uint32_t a, uint32_t l) {
        const uint32_t j = (uint32_t)o0 + i;
        const bool null = is_dot(v + a, l);
        if (gl == 0) { C.coffs[j] = at; if (!null) atomicOr(&C.cvalid[j >> 5], 1u << (j & 31)); }
        if (!null) { bad |= grp_map4<G>(C.data + at, v + a, l, gl, 0u); at += (int32_t)l; }
      });
      continue;
    }
    if (gl != 0) continue;
    uint32_t* out = reinterpret_cast<uint32_t*>(C.data);
    for_elements(v, tk.y, [&](uint32_t i, uint32_t a, uint32_t l) {
      const uint32_t j = (uint32_t)o0 + i;
      uint32_t x = 0;
      if (!is_dot(v + a, l)) {
        if (C.kind == K_ListInt32) parse_i32(v + a, l, reinterpret_cast<int32_t*>(&x));
        else f32_parse(reinterpret_cast<const char*>(v + a), l, &x);
        atomicOr(&C.cvalid[j >> 5], 1u << (j & 31));
      }
      out[j] = x;
    });
  }
  if (bad) set_err(P.err, VCF_ERR_UTF8, r);
}

}  // namespace vcf
}  // namespace bamscan
