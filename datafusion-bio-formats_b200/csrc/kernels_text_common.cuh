// kernels_text_common.cuh -- device helpers shared by the two places that turn text into BAM records: the write path
// (kernels_encode.cuh: Arrow columns -> BAM) and the SAM scan (kernels_sam.cuh: SAM lines -> BAM).  sm_100a.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

namespace bamscan {
namespace enc {

constexpr uint32_t FULLMASK = 0xffffffffu;

__device__ __forceinline__ void report(uint32_t* err, uint32_t code, uint32_t row) { if (atomicCAS(err, 0u, code) == 0u) err[1] = row; }   // err[0] = first code, err[1] = its row

// reference id of the name s[0 .. n): binary search over the names sorted bytewise (blob + offsets [n_ref + 1]) -> ids; -1 if absent
__device__ __forceinline__ int32_t lookup_ref(const uint8_t* blob, const int32_t* off, const int32_t* ids, int32_t n_ref, const uint8_t* s, uint32_t n) {
  int lo = 0, hi = n_ref - 1;
  while (lo <= hi) {
    const int mid = (lo + hi) >> 1;
    const uint8_t* m = blob + off[mid];
    const uint32_t mn = (uint32_t)(off[mid + 1] - off[mid]);
    int c = 0;
    for (uint32_t k = 0; k < min(n, mn) && c == 0; k++) c = (int)s[k] - (int)m[k];
    if (c == 0) c = (n > mn) - (n < mn);
    if (c == 0) return ids[mid];
    if (c < 0) hi = mid - 1; else lo = mid + 1;
  }
  return -1;
}

__device__ __forceinline__ uint32_t elem_size(uint8_t st) { return (st == 'c' || st == 'C') ? 1u : (st == 's' || st == 'S') ? 2u : 4u; }

__device__ __forceinline__ bool int_fits(long long v, uint8_t t) {
  switch (t) {
    case 'c': return v >= -128 && v <= 127;
    case 'C': return v >= 0 && v <= 255;
    case 's': return v >= -32768 && v <= 32767;
    case 'S': return v >= 0 && v <= 65535;
    case 'i': return v >= -2147483648ll && v <= 2147483647ll;
    default: return v >= 0 && v <= 4294967295ll;     // 'I'
  }
}

__device__ __forceinline__ int op_code(uint8_t c) {
  switch (c) { case 'M': return 0; case 'I': return 1; case 'D': return 2; case 'N': return 3; case 'S': return 4; case 'H': return 5; case 'P': return 6; case '=': return 7; case 'X': return 8; default: return -1; }
}

// unaligned 32-bit little-endian load from global memory: two aligned loads + funnel shift (reads up to 3 bytes before / behind)
__device__ __forceinline__ uint32_t ldw(const uint8_t* p) {
  const uintptr_t a = reinterpret_cast<uintptr_t>(p);
  const uint32_t* w = reinterpret_cast<const uint32_t*>(a & ~uintptr_t(3));
  const uint32_t sh = (uint32_t)(a & 3u) * 8u;
  return sh ? __funnelshift_r(w[0], w[1], sh) : w[0];
}

// The decimal number made of the run of digits that ends in front of s[k] (at most 12 digits are looked at; more than that is
// >= 2^28 anyway).  The 12 bytes come with three independent loads: a digit-by-digit backward walk is a chain of dependent
// global loads (one memory round trip per digit, 600+ steps per long-read CIGAR).
__device__ __forceinline__ unsigned long long digits_before(const uint8_t* s, uint32_t k) {
  const uint32_t w0 = ldw(s + (long long)k - 4), w1 = ldw(s + (long long)k - 8), w2 = ldw(s + (long long)k - 12);
  unsigned long long len = 0, mul = 1;
  #pragma unroll
  for (uint32_t j = 0; j < 12; j++) {
    const uint32_t w = j < 4 ? w0 : j < 8 ? w1 : w2;
    const uint32_t d = (w >> (8u * (3u - (j & 3u)))) & 0xffu;
    if (j >= k || d < '0' || d > '9') break;
    len += (unsigned long long)(d - '0') * mul; mul *= 10;
  }
  return len;
}

__device__ __forceinline__ void st_u32(uint8_t* p, uint32_t v) { p[0] = (uint8_t)v; p[1] = (uint8_t)(v >> 8); p[2] = (uint8_t)(v >> 16); p[3] = (uint8_t)(v >> 24); }

__device__ __forceinline__ void st_u16(uint8_t* p, uint32_t v) { p[0] = (uint8_t)v; p[1] = (uint8_t)(v >> 8); }

// dst[i] = op(src[i]) for i < n by a group of G lanes, with destination-aligned 32-bit stores (head / tail bytes singly); `op`
// maps four bytes at a time.  Records are byte packed, so a plain byte loop costs one store instruction and one 32-byte
// sector write per byte (ncu: 9.5 x store-sector amplification in the first version of this kernel).
// grp_xform4_ref takes the op by reference, so an op can also accumulate state over the words it sees (a byte check fused
// into the copy); the single head / tail bytes reach it as words whose upper three bytes are zero.
template <int G, class OP>
__device__ __forceinline__ void grp_xform4_ref(uint8_t* dst, const uint8_t* src, uint32_t n, int gl, OP& op) {
  const uint32_t head = min(n, (uint32_t)((4u - (reinterpret_cast<uintptr_t>(dst) & 3u)) & 3u));
  if ((uint32_t)gl < head) dst[gl] = (uint8_t)op((uint32_t)src[gl]);
  const uint32_t nw = (n - head) >> 2;
  uint32_t* dw = reinterpret_cast<uint32_t*>(dst + head);
  const uint8_t* s = src + head;
  for (uint32_t j = gl; j < nw; j += G) dw[j] = op(ldw(s + 4u * j));
  const uint32_t t0 = head + (nw << 2);
  if (t0 + (uint32_t)gl < n) dst[t0 + gl] = (uint8_t)op((uint32_t)src[t0 + gl]);
}
template <int G, class OP>
__device__ __forceinline__ void grp_xform4(uint8_t* dst, const uint8_t* src, uint32_t n, int gl, OP op) { grp_xform4_ref<G>(dst, src, n, gl, op); }
struct OpCopy { __device__ __forceinline__ uint32_t operator()(uint32_t v) const { return v; } };
struct OpQual { __device__ __forceinline__ uint32_t operator()(uint32_t v) const { return __vsubus4(v, 0x21212121u); } };   // byte-wise saturating - 33

}  // namespace enc
}  // namespace bamscan
