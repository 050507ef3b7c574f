// kernels_scan.cuh -- device prefix sums.  Every stage turns counts into offsets with an exclusive scan; this file is the only one
// that implements one (the warp scans inside the inflate, decode_var, SAM-encode and deflate kernels work on their own lane
// groups and stay there).
//
//   warp_inclusive_scan   32 lanes, shuffles
//   block_sum             NT threads -> thread 0
//   block_exclusive_scan  NT threads
//   cta_exclusive_scan    one CTA of 1024 threads over any n: 1024 elements per step, a carry between steps
//   cta_scan_kernel       cta_exclusive_scan as a kernel, one CTA per column
//
// The block and CTA helpers contain __syncthreads(): every thread of the block has to call them.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

namespace bamscan {

template <typename T>
__device__ __forceinline__ T warp_inclusive_scan(T x) {
  const int lane = threadIdx.x & 31;
  #pragma unroll
  for (int s = 1; s < 32; s <<= 1) { const T y = __shfl_up_sync(0xffffffffu, x, s); if (lane >= s) x += y; }
  return x;
}

// sum of v over the NT threads of the block, valid in thread 0 only.  ws: NT / 32 elements of shared memory.
template <int NT, typename T>
__device__ __forceinline__ T block_sum(T v, T* ws) {
  #pragma unroll
  for (int s = 16; s; s >>= 1) v += __shfl_xor_sync(0xffffffffu, v, s);
  if ((threadIdx.x & 31) == 0) ws[threadIdx.x >> 5] = v;
  __syncthreads();
  T t = 0;
  if (threadIdx.x == 0) { for (int w = 0; w < NT / 32; w++) t += ws[w]; }
  return t;
}

// exclusive scan of v over the NT threads of the block.  ws: NT / 32 elements of shared memory, read after the call's only barrier:
// a second scan in the same kernel takes its own ws.
template <int NT, typename T>
__device__ __forceinline__ T block_exclusive_scan(T v, T* ws) {
  const int warp = threadIdx.x >> 5;
  const T x = warp_inclusive_scan(v);
  if ((threadIdx.x & 31) == 31) ws[warp] = x;
  __syncthreads();
  T base = 0;
  for (int w = 0; w < warp; w++) base += ws[w];
  return base + x - v;
}

constexpr int CTA_SCAN_THREADS = 1024;

// Exclusive scan of n elements by one CTA of CTA_SCAN_THREADS threads, one element per thread and step.  Every thread calls
// load(i) in every step, for i >= n too, where load returns 0 (so load may do warp-wide side work); store(i, excl, v) is called
// for i < n.  Returns the total to every thread.
template <typename T, typename Load, typename Store>
__device__ __forceinline__ T cta_exclusive_scan(uint32_t n, Load load, Store store) {
  __shared__ T ws[32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  T carry = 0;
  for (uint32_t base = 0; base < n; base += CTA_SCAN_THREADS) {
    const uint32_t i = base + threadIdx.x;
    const T v = load(i);
    const T x = warp_inclusive_scan(v);
    if (lane == 31) ws[warp] = x;
    __syncthreads();
    if (warp == 0) ws[lane] = warp_inclusive_scan(ws[lane]);
    __syncthreads();
    if (i < n) store(i, carry + (warp ? ws[warp - 1] : T(0)) + x - v, v);
    carry += ws[31];
    __syncthreads();                                  // ws is rewritten by the next step
  }
  return carry;
}

// One CTA per column: column c is in[c * n, (c + 1) * n), scanned into the same range of out; its total -> totals[c].  in and out
// may be the same array (the offsets scans run in place), so neither is __restrict__.
template <typename In, typename T>
__global__ void __launch_bounds__(CTA_SCAN_THREADS)
cta_scan_kernel(const In* in, T* out, uint32_t n, T* totals) {
  const size_t c = (size_t)blockIdx.x * n;
  const T total = cta_exclusive_scan<T>(n, [&](uint32_t i) { return i < n ? T(in[c + i]) : T(0); },
                                        [&](uint32_t i, T excl, T) { out[c + i] = excl; });
  if (threadIdx.x == 0) totals[blockIdx.x] = total;
}

}  // namespace bamscan
