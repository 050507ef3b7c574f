// kernels_filter.cuh -- row rules of the indexed scan, evaluated on the device and compacted into rec_off[].
//
// Replaces (reference, datafusion/bio-format-bam/src/physical_exec.rs):
//   :1275-1314  mapped region: skip records without alignment_start; keep start(1-based) in [region.start, region.end]
//   :1131-1258  per-reference unmapped tail: from the seek position keep refID == ref && pos == -1, stop at the first
//               record of another reference once the reference has been seen
//   :1038-1129  "*" partition: keep refID == -1 && pos == -1
//   :1333-1344  residual filters (bio-format-core/src/record_filter.rs:57-283) over {chrom, start, end, mapping_quality, flags};
//               a NULL accessor value or a non-accessor column makes the filter pass
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

#include "kernels_boundary.cuh"
#include "kernels_scan.cuh"

namespace bamscan {

constexpr int MAX_DEV_FILTERS = 8, MAX_FILTER_VALUES = 8;

struct DevFilter {
  int32_t column, op, n, is_str;     // is_str: literals are strings (chrom: resolved to reference ids)
  double nums[MAX_FILTER_VALUES];
  int32_t refs[MAX_FILTER_VALUES];   // reference ids of the string literals (-2 = name not in the header)
};

struct RowRule {
  int32_t mode, ref;                 // 1 mapped region, 2 per-reference unmapped tail, 3 "*" unplaced
  uint32_t start1, end1;             // 1-based closed bounds, 0 = open
  int32_t zero_based, n_filters, seen_before, needs_end;
  DevFilter f[MAX_DEV_FILTERS];
};

// flags: [5] first index with refID == rule.ref, [6] stop index (mode 2), [7] kept rows
__global__ void __launch_bounds__(256)
rule_first_target_kernel(const uint8_t* __restrict__ U, const uint32_t* __restrict__ rec_off, uint32_t n, int32_t ref, uint32_t* __restrict__ flags) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  if ((int32_t)ld_u32(U, rec_off[i] + 4) == ref) atomicMin(&flags[5], i);
}

__device__ __forceinline__ bool eval_filter(const DevFilter& F, int32_t ref, bool has_start, double start, bool has_end, double end, double mapq, double flag, bool chrom_null) {
  const bool neg = F.op == 1 || F.op == 7 || F.op == 9;
  if (F.column == 1) {                        // chrom: only = != IN NOT IN on strings are evaluated
    if (chrom_null || !F.is_str) return true;
    if (F.op != 0 && F.op != 1 && F.op != 8 && F.op != 9) return true;
    bool any = false;
    for (int k = 0; k < F.n; k++) any |= F.refs[k] == ref;
    return neg ? !any : any;
  }
  double v; bool has = true;
  switch (F.column) {
    case 2: has = has_start; v = start; break;
    case 3: has = has_end; v = end; break;
    case 6: v = mapq; break;
    case 4: v = flag; break;
    default: return true;                     // not an accessor field: passes (DataFusion re-applies the filter above the scan)
  }
  if (!has) return true;
  if (F.is_str) return (F.op == 8 || F.op == 9) ? false : true;   // numeric field vs string literals: IN sees only UNKNOWNs, the rest pass
  switch (F.op) {
    case 0: return v == F.nums[0];
    case 1: return v != F.nums[0];
    case 2: return v < F.nums[0];
    case 3: return v <= F.nums[0];
    case 4: return v > F.nums[0];
    case 5: return v >= F.nums[0];
    case 6: return v >= F.nums[0] && v <= F.nums[1];
    case 7: return !(v >= F.nums[0] && v <= F.nums[1]);
    case 8: case 9: { bool any = false; for (int k = 0; k < F.n; k++) any |= v == F.nums[k]; return F.op == 8 ? any : !any; }
  }
  return true;
}

__global__ void __launch_bounds__(256)
rule_keep_kernel(const uint8_t* __restrict__ U, const uint32_t* __restrict__ rec_off, uint32_t n, const RowRule R, uint32_t* __restrict__ keep, uint32_t* __restrict__ flags) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint32_t o = rec_off[i];
  const int32_t ref = (int32_t)ld_u32(U, o + 4), pos = (int32_t)ld_u32(U, o + 8);
  bool k;
  if (R.mode == 1) {
    const uint32_t start1 = (uint32_t)pos + 1u;
    k = ref == R.ref && pos >= 0 && (R.start1 == 0 || start1 >= R.start1) && (R.end1 == 0 || start1 <= R.end1);
  } else if (R.mode == 2) {
    const bool target = ref == R.ref;
    if (!target && (R.seen_before || i > flags[5])) atomicMin(&flags[6], i);
    k = target && pos < 0;
  } else {
    k = ref == -1 && pos < 0;
  }
  if (k && R.n_filters) {
    uint32_t w = ld_u32(U, o + 12); const uint32_t l_name = w & 0xffu, mapq = (w >> 8) & 0xffu;
    w = ld_u32(U, o + 16); const uint32_t n_cig = w & 0xffffu, flag = w >> 16;
    uint32_t span = 0;
    if (R.needs_end) for (uint32_t c = 0; c < n_cig; c++) { uint32_t cw = ld_u32(U, o + 36 + l_name + 4u * c); if ((0x18Du >> (cw & 15u)) & 1u) span += cw >> 4; }
    const bool has_start = pos >= 0, has_end = has_start && span > 0;
    const double start = (double)((uint32_t)pos + (R.zero_based ? 0u : 1u)), end = (double)((uint32_t)pos + span);
    const bool chrom_null = R.mode == 3 || ref < 0;
    for (int f = 0; f < R.n_filters && k; f++) k = eval_filter(R.f[f], ref, has_start, start, has_end, end, (double)mapq, (double)flag, chrom_null);
  }
  keep[i] = k ? 1u : 0u;
}

// single CTA: exclusive scan of keep[i] (cut at the stop index) -> pos[i]; total -> flags[7]
__global__ void __launch_bounds__(1024)
rule_scan_kernel(const uint32_t* __restrict__ keep, uint32_t* __restrict__ pos, uint32_t n, uint32_t* __restrict__ flags) {
  const uint32_t stop = flags[6];
  const uint32_t total = cta_exclusive_scan<uint32_t>(n, [&](uint32_t i) { return (i < n && i < stop) ? keep[i] : 0u; },
                                                      [&](uint32_t i, uint32_t excl, uint32_t v) { pos[i] = v ? excl : 0xffffffffu; });
  if (threadIdx.x == 0) flags[7] = total;
}

__global__ void __launch_bounds__(256)
rule_compact_kernel(const uint32_t* __restrict__ rec_off, const uint32_t* __restrict__ pos, uint32_t n, uint32_t* __restrict__ out) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  uint32_t p = pos[i];
  if (p != 0xffffffffu) out[p] = rec_off[i];
}

}  // namespace bamscan
