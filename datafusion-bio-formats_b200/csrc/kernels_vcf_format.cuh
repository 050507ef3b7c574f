// kernels_vcf_format.cuh -- VCF FORMAT columns: the selected FORMAT fields as per-sample list columns.  sm_100a.
//
// Launched behind vcf_fields_kernel / vcf_rows_kernel (kernels_vcf.cuh) only when a FORMAT column is projected; they read the
// FORMAT field's start from vcf::Row::f[8].  Every row has exactly S elements (one per sample), so element e = r * S + j of row r,
// sample j, and every element-level buffer is sized on the host from n * S.  Per decode slice:
//
//   samples  vcf_samples_kernel<G>: a group of G lanes per line walks the tabs behind f[8] (the running tab count of
//            vcf_fields_kernel) and writes each sample's start to samp[e]; the field count must be 9 + S.  Lane 0 parses the
//            FORMAT key list into the line's FmtRow: per projected column the index of its key (a claim bit per column catches
//            a projected key given twice), and writes the outer list offsets r * S.
//   values   vcf_values_kernel: a thread per element walks the sample's ':' values once.  Number=1 Int32 / Float32 values go
//            straight to the child values at e; Utf8 values give their byte count and nested values their leaf count at e (the
//            count columns the engine scans into offsets).  Element validity by __ballot_sync: elements are warp-contiguous.
//            Values are checked against their type here, and Utf8 bytes for 0x80 and above.
//   offsets  launch_offsets_scan (engine.cu) over the count columns, n * S + 1 entries each.
//   write    vcf_fmt_write_kernel: a thread per element copies its Utf8 bytes, or parses its nested leaves into the leaf values
//            with leaf validity.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

#include "f32_parse.h"
#include "kernels_vcf.cuh"

namespace bamscan {
namespace vcf {

constexpr int MAX_FORMAT = 16;             // selected FORMAT IDs (host_schema.cpp refuses more)
constexpr int FMT_BLOB = 1024;
constexpr uint8_t NO_KEY = 0xff;           // FmtRow::k of a column whose key the line does not list
constexpr int32_t K_ListListInt32 = 18, K_ListListFloat32 = 19;   // (bamscan_internal.h: HK_ListListInt32, HK_ListListFloat32)

struct FmtRow { uint32_t nkeys, end; uint8_t k[MAX_FORMAT]; };   // keys in the line's FORMAT field; end of the line; key index per column

struct FmtCol {
  int32_t kind;        // K_ListInt32 / K_ListFloat32 / K_ListUtf8 (Number=1), K_ListListInt32 / K_ListListFloat32
  int32_t* offs;       // outer offsets: r * S
  uint32_t* valid;     // element validity words (n * S bits)
  uint32_t* values;    // Number=1 Int32 / Float32: the element values
  int32_t* counts;     // Utf8: element bytes, nested: element leaves (n * S + 1) -> offsets
  uint32_t* lvalid;    // nested: leaf validity words
  uint8_t* data;       // Utf8 bytes; nested: leaf values
};

struct FormatParams {
  const uint8_t* U;
  const uint32_t* lines;      // line starts of the slice (as vcf::Params::lines)
  const Row* rows;            // vcf_fields_kernel's field starts
  uint32_t n, S;              // rows, samples
  int32_t nf;                 // projected FORMAT columns
  uint32_t* samp;             // [n * S] sample starts
  FmtRow* frow;               // [n]
  uint32_t* err;
  uint16_t off[MAX_FORMAT + 1];   // key c = blob[off[c], off[c + 1])
  uint8_t blob[FMT_BLOB];
  FmtCol cols[MAX_FORMAT];
};

template <int G>
__global__ void __launch_bounds__(256)
vcf_samples_kernel(const FormatParams F) {
  const int lane = threadIdx.x & 31, gl = lane & (G - 1);
  const unsigned gmask = G == 32 ? 0xffffffffu : (((1u << G) - 1u) << (lane & ~(G - 1)));
  const uint32_t r = (blockIdx.x * blockDim.x + threadIdx.x) / G;
  if (r >= F.n) return;                            // (whole groups)
  const uint32_t s = F.lines[r];
  uint32_t e = F.lines[r + 1] - 1u;
  if (e > s && F.U[e - 1] == '\r') e--;
  const Row R = F.rows[r];
  const uint64_t e0 = (uint64_t)r * F.S;
  uint32_t* samp = F.samp + e0;
  // the tabs behind FORMAT: sample j starts behind the (j + 1)-th
  uint32_t found = 0;
  const uint32_t b = R.ntab >= 8u ? R.f[8] : e;
  for (uint32_t w = b; w < e; w += G * 16) {
    const uint32_t o = w + gl * 16;
    uint32_t m = 0;
    #pragma unroll
    for (int k = 0; k < 16; k++) if (o + k < e && F.U[o + k] == '\t') m |= 1u << k;
    const uint32_t c = __popc(m);
    uint32_t incl = c;
    #pragma unroll
    for (int d = 1; d < G; d <<= 1) { const uint32_t y = __shfl_up_sync(gmask, incl, d, G); if (gl >= d) incl += y; }
    uint32_t idx = found + incl - c;
    while (m && idx < F.S) { const int k = __ffs((int)m) - 1; m &= m - 1u; samp[idx++] = o + k + 1u; }
    found += __shfl_sync(gmask, incl, G - 1, G);
  }
  // a line with too few fields gets empty samples at its end, so that the values kernel reads inside the line
  for (uint32_t j = found + gl; j < F.S; j += G) samp[j] = e;
  __syncwarp(gmask);                               // lane 0 reads samp[0] below
  if (gl != 0) return;
  if (R.ntab < 8u || found != F.S) set_err(F.err, VCF_ERR_FMT_FIELDS, r);
  // FORMAT keys ('.' or empty: none)
  FmtRow out;
  out.end = e;
  #pragma unroll
  for (int c = 0; c < MAX_FORMAT; c++) out.k[c] = NO_KEY;
  uint32_t nkeys = 0, claimed = 0;
  const uint32_t fe = found ? samp[0] - 1u : e;
  if (R.ntab >= 8u && fe > b && !is_dot(F.U + b, fe - b)) {
    for (uint32_t a = b;; nkeys++) {
      uint32_t z = a;
      while (z < fe && F.U[z] != ':') z++;
      for (int c = 0; c < F.nf; c++) {
        const uint32_t o = F.off[c], kl = F.off[c + 1] - o;
        if (kl != z - a) continue;
        uint32_t j = 0;
        while (j < kl && F.blob[o + j] == F.U[a + j]) j++;
        if (j != kl) continue;
        if (claimed & (1u << c)) set_err(F.err, VCF_ERR_FMT_DUP, r);
        claimed |= 1u << c;
        out.k[c] = (uint8_t)min(nkeys, 254u);
      }
      if (z >= fe) { nkeys++; break; }
      a = z + 1u;
    }
  }
  out.nkeys = nkeys;
  F.frow[r] = out;
  for (int c = 0; c < F.nf; c++) {
    F.cols[c].offs[r] = (int32_t)e0;
    if (r + 1u == F.n) F.cols[c].offs[F.n] = (int32_t)(e0 + F.S);
  }
}

// the sample of element el: [*a, *z)
__device__ __forceinline__ void sample_bounds(const FormatParams& F, uint64_t el, uint32_t j, uint32_t end, uint32_t* a, uint32_t* z) {
  *a = F.samp[el];
  const uint32_t t = j + 1u < F.S ? F.samp[el + 1] - 1u : end;
  *z = max(t, *a);
}

__global__ void __launch_bounds__(256)
vcf_values_kernel(const FormatParams F) {
  const uint64_t nel = (uint64_t)F.n * F.S;
  const uint64_t el = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const bool on = el < nel;
  uint32_t valid = 0;
  if (on) {
    const uint32_t r = (uint32_t)el / F.S, j = (uint32_t)el - r * F.S;      // (n * S < 2^31: engine.cu cuts the slices so)
    const FmtRow R = F.frow[r];
    uint32_t a, z;
    sample_bounds(F, el, j, R.end, &a, &z);
    const uint8_t* U = F.U;
    uint32_t done = 0;
    // a lone '.' has no values; otherwise value k is the k-th ':'-separated piece
    if (!is_dot(U + a, z - a)) {
      uint32_t k = 0;
      for (uint32_t p = a;; k++) {
        uint32_t q = p;
        while (q < z && U[q] != ':') q++;
        if (k >= R.nkeys) { set_err(F.err, VCF_ERR_FMT_MANY, r); break; }
        for (int c = 0; c < F.nf; c++) {
          if (R.k[c] != k) continue;
          const FmtCol& C = F.cols[c];
          done |= 1u << c;
          const uint8_t* v = U + p;
          const uint32_t vn = q - p;
          if (is_dot(v, vn)) {                                    // '.': NULL
            if (C.kind == K_ListInt32 || C.kind == K_ListFloat32) C.values[el] = 0u; else C.counts[el] = 0;
            continue;
          }
          bool ok = true;
          if (C.kind == K_ListInt32) { int32_t x = 0; ok = parse_i32(v, vn, &x); C.values[el] = ok ? (uint32_t)x : 0u; }
          else if (C.kind == K_ListFloat32) { uint32_t x = 0; ok = f32_parse(reinterpret_cast<const char*>(v), vn, &x); C.values[el] = ok ? x : 0u; }
          else if (C.kind == K_ListUtf8) {
            uint32_t hi = 0;
            for (uint32_t i = 0; i < vn; i++) { if (v[i] == ',') ok = false; hi |= v[i] & 0x80u; }
            if (hi) set_err(F.err, VCF_ERR_UTF8, r);
            C.counts[el] = ok ? (int32_t)vn : 0;
          } else {
            const uint32_t leaves = for_elements(v, vn, [&](uint32_t, uint32_t la, uint32_t ll) {
              if (is_dot(v + la, ll)) return;
              if (C.kind == K_ListListInt32) { int32_t x; if (!parse_i32(v + la, ll, &x)) ok = false; }
              else { uint32_t x; if (!f32_parse(reinterpret_cast<const char*>(v + la), ll, &x)) ok = false; }
            });
            C.counts[el] = ok ? (int32_t)leaves : 0;
          }
          if (!ok) set_err(F.err, VCF_ERR_FMT_VALUE, r);
          else valid |= 1u << c;
        }
        if (q >= z) break;
        p = q + 1u;
      }
    }
    for (int c = 0; c < F.nf; c++) {                 // keys the line does not list, values the sample does not give: NULL
      if (done & (1u << c)) continue;
      const FmtCol& C = F.cols[c];
      if (C.kind == K_ListInt32 || C.kind == K_ListFloat32) C.values[el] = 0u; else C.counts[el] = 0;
    }
  }
  const bool word = (threadIdx.x & 31) == 0 && el < ((nel + 31u) & ~31ull);
  for (int c = 0; c < F.nf; c++) {
    const uint32_t m = __ballot_sync(0xffffffffu, (valid >> c) & 1u);
    if (word) F.cols[c].valid[el >> 5] = m;
  }
}

// Utf8 bytes and nested leaves of the element, behind the scan
__global__ void __launch_bounds__(256)
vcf_fmt_write_kernel(const FormatParams F) {
  const uint64_t nel = (uint64_t)F.n * F.S;
  const uint64_t el = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (el >= nel) return;
  const uint32_t r = (uint32_t)el / F.S, j = (uint32_t)el - r * F.S;
  const FmtRow R = F.frow[r];
  uint32_t todo = 0;
  for (int c = 0; c < F.nf; c++) {
    const FmtCol& C = F.cols[c];
    if ((C.kind == K_ListUtf8 || C.kind == K_ListListInt32 || C.kind == K_ListListFloat32) && C.counts[el + 1] != C.counts[el]) todo |= 1u << c;
  }
  if (!todo) return;
  uint32_t a, z;
  sample_bounds(F, el, j, R.end, &a, &z);
  const uint8_t* U = F.U;
  for (uint32_t p = a, k = 0;; k++) {
    uint32_t q = p;
    while (q < z && U[q] != ':') q++;
    for (int c = 0; c < F.nf; c++) {
      if (!((todo >> c) & 1u) || R.k[c] != k) continue;
      const FmtCol& C = F.cols[c];
      const uint8_t* v = U + p;
      const int32_t o0 = C.counts[el];
      if (C.kind == K_ListUtf8) { for (uint32_t i = 0; i < q - p; i++) C.data[o0 + i] = v[i]; continue; }
      uint32_t* out = reinterpret_cast<uint32_t*>(C.data);
      for_elements(v, q - p, [&](uint32_t i, uint32_t la, uint32_t ll) {
        const uint32_t lj = (uint32_t)o0 + i;
        uint32_t x = 0;
        if (!is_dot(v + la, ll)) {
          if (C.kind == K_ListListInt32) parse_i32(v + la, ll, reinterpret_cast<int32_t*>(&x));
          else f32_parse(reinterpret_cast<const char*>(v + la), ll, &x);
          atomicOr(&C.lvalid[lj >> 5], 1u << (lj & 31));
        }
        out[lj] = x;
      });
    }
    if (q >= z) break;
    p = q + 1u;
  }
}

}  // namespace vcf
}  // namespace bamscan
