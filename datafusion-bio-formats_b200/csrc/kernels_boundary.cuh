// kernels_boundary.cuh -- BAM record-boundary resolution over the concatenated inflated stream.
//
// Replaces the serial `reader.read_record(&mut record)` chain of the reference
// (datafusion/bio-format-bam/src/physical_exec.rs:409; noodles-bam io::Reader::read_record):
// next record offset = current + 4 + block_size, records straddle BGZF block seams.
//
// Scheme (exact, not probabilistic):
//   1. the inflated chunk is cut into fixed SEGMENTS (default 16 KiB).  Segment 0 starts at a known
//      record start (end of header, or the carried-over tail of the previous chunk).
//   2. seg_candidates_kernel: one warp per segment tests 32 byte offsets at a time with a strong
//      record-header predicate + 2-record chain confirmation and keeps the first hit.
//   3. seg_walk_kernel: one thread per segment follows the block_size chain from its start to the
//      segment end, counting records and recording the exit offset.
//   4. seg_check_kernel: the exit of every segment must equal the chosen start of the next segment that
//      has one (and no start may lie in between).  Since segment 0 is exact, agreement of all seams
//      proves, by induction, that every start lies on the true chain.  Any disagreement (a false
//      candidate, or a true start the predicate rejected) triggers seg_repair_kernel, a sequential
//      re-chaining from the first start that reuses the per-segment walks that do agree.
//   5. counts are scanned to global record indices and a second walk emits rec_off[].
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

#include "kernels_scan.cuh"

namespace bamscan {

constexpr uint32_t SEG_NONE = 0xffffffffu;

struct BoundaryParams {
  const uint8_t* U;          // chunk buffer base (offsets below are relative to U)
  uint32_t data_lo;          // first valid byte (start of carried tail, or first record)
  uint32_t data_hi;          // one past the last valid byte
  uint32_t own_hi;           // records starting at or after this offset belong to someone else (next shard / region end)
  uint32_t seg0;             // offset where segment 0 begins (start of this chunk's own inflated bytes)
  uint32_t seg_bytes;        // segment size
  uint32_t n_seg;
  uint32_t first_start;      // exact record start feeding segment 0 (SEG_NONE: speculate, shard without known start)
  int32_t n_ref;
  const int32_t* ref_len;    // device array [n_ref]
  uint32_t max_block_size;   // sanity cap for block_size
};

__device__ __forceinline__ uint32_t ld_u32(const uint8_t* U, uint32_t o) {   // unaligned little-endian load
  uintptr_t a = reinterpret_cast<uintptr_t>(U + o);
  const uint32_t* w = reinterpret_cast<const uint32_t*>(a & ~uintptr_t(3));
  uint32_t sh = uint32_t(a & 3) * 8;
  uint32_t lo = w[0];
  if (sh == 0) return lo;
  return __funnelshift_r(lo, w[1], sh);
}
__device__ __forceinline__ uint32_t ld_u16(const uint8_t* U, uint32_t o) { return uint32_t(U[o]) | (uint32_t(U[o + 1]) << 8); }

// Record-header plausibility at offset o.  Every check is skipped when its bytes lie past data_hi.
__device__ __forceinline__ bool header_plausible(const BoundaryParams& P, uint32_t o, uint32_t* next) {
  if (o + 4 > P.data_hi) return false;
  uint32_t bs = ld_u32(P.U, o);
  if (bs < 32 || bs > P.max_block_size) return false;
  *next = o + 4 + bs;
  if (o + 36 > P.data_hi) return true;             // truncated header at the very end of the chunk
  int32_t ref = (int32_t)ld_u32(P.U, o + 4), pos = (int32_t)ld_u32(P.U, o + 8);
  if (ref < -1 || ref >= P.n_ref || pos < -1) return false;
  if (ref >= 0 && pos > P.ref_len[ref]) return false;
  uint32_t l_name = P.U[o + 12];
  if (l_name == 0) return false;
  uint32_t n_cig = ld_u16(P.U, o + 16);
  int32_t l_seq = (int32_t)ld_u32(P.U, o + 20);
  if (l_seq < 0) return false;
  int32_t nref = (int32_t)ld_u32(P.U, o + 24), npos = (int32_t)ld_u32(P.U, o + 28);
  if (nref < -1 || nref >= P.n_ref || npos < -1) return false;
  if (nref >= 0 && npos > P.ref_len[nref]) return false;
  uint64_t need = 32ull + l_name + 4ull * n_cig + ((uint64_t)l_seq + 1) / 2 + (uint64_t)l_seq;
  if (need > bs) return false;
  return true;
}

__device__ __forceinline__ bool record_plausible(const BoundaryParams& P, uint32_t o, uint32_t* next) {
  if (!header_plausible(P, o, next)) return false;
  if (o + 36 > P.data_hi) return true;
  uint32_t l_name = P.U[o + 12];
  uint32_t name_end = o + 36 + l_name;             // one past the NUL
  if (name_end <= P.data_hi) {
    if (P.U[name_end - 1] != 0) return false;
    for (uint32_t k = o + 36; k + 1 < name_end; k++) { uint8_t c = P.U[k]; if (c < 0x21 || c > 0x7e) return false; }
  }
  uint32_t n_cig = ld_u16(P.U, o + 16);
  uint32_t chk = n_cig < 64 ? n_cig : 64;
  for (uint32_t k = 0; k < chk; k++) {
    uint32_t co = name_end + 4 * k;
    if (co + 4 > P.data_hi) break;
    if ((P.U[co] & 15u) > 8u) return false;
  }
  return true;
}

// one warp per segment
__global__ void __launch_bounds__(256)
seg_candidates_kernel(BoundaryParams P, uint32_t* __restrict__ seg_start, int poison) {
  const uint32_t s = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (s >= P.n_seg) return;
  if (P.first_start != SEG_NONE) {
    // the exact first record start may lie several segments into the chunk (an indexed range starts anywhere inside its
    // first BGZF member): the segments before it hold no owned record, the one containing it starts there
    const uint32_t k = P.first_start > P.seg0 ? min((P.first_start - P.seg0) / P.seg_bytes, P.n_seg - 1u) : 0u;
    if (s <= k) { if (lane == 0) seg_start[s] = s == k ? P.first_start : SEG_NONE; return; }
  }
  uint32_t lo = P.seg0 + s * P.seg_bytes;
  uint32_t hi = min(min(lo + P.seg_bytes, P.data_hi), P.own_hi);
  uint32_t found = SEG_NONE;
  for (uint32_t b = lo; b < hi && found == SEG_NONE; b += 32) {
    uint32_t o = b + lane;
    bool ok = false;
    if (o < hi) {
      uint32_t n1, n2, n3;
      ok = record_plausible(P, o, &n1);
      // chain confirmation: the next two records (when inside the chunk) must look like headers too
      if (ok && n1 < P.data_hi) ok = header_plausible(P, n1, &n2);
      else n2 = P.data_hi;
      if (ok && n1 < P.data_hi && n2 < P.data_hi) ok = header_plausible(P, n2, &n3);
    }
    uint32_t m = __ballot_sync(0xffffffffu, ok);
    if (m) found = b + (__ffs(m) - 1);
  }
  if (poison && found != SEG_NONE && (s % 3u) == 1u) found += 1;   // test hook: a deliberately wrong start (repair path)
  if (lane == 0) seg_start[s] = found;
}

struct WalkOut {
  uint32_t* seg_start;   // in/out: chosen record start of the segment (SEG_NONE = no record starts here)
  uint32_t* seg_exit;    // chain position after the segment's last record
  uint32_t* seg_count;   // records starting in the segment
  uint8_t* seg_tail;     // 1: the walk stopped at an incomplete record / end of data
  uint32_t* flags;       // [0] seams that disagree, [1] corrupt block_size (offset|1), [2] tail offset, [3] total records, [4] repairs,
                         // [10] copy of [0] for the stats, [11] first disagreeing segment
};

struct WalkResult { uint32_t n, exit; uint8_t tail; };   // tail: 0 ran past the segment, 1 incomplete record / end of data, 2 corrupt block_size

__device__ __forceinline__ WalkResult walk_segment(const BoundaryParams& P, uint32_t s, uint32_t o) {
  uint32_t hi = (s + 1 == P.n_seg) ? 0xfffffff0u : P.seg0 + (s + 1) * P.seg_bytes;   // records STARTING before hi belong to s
  WalkResult r{0, o, 0};
  while (o < hi) {
    if (o >= P.own_hi) { r.tail = 1; break; }           // ownership ends here: treated like the end of data
    if (o + 4 > P.data_hi) { r.tail = 1; break; }
    uint32_t bs = ld_u32(P.U, o);
    if (bs < 32 || bs > P.max_block_size) { r.tail = 2; break; }
    if ((uint64_t)o + 4 + bs > P.data_hi) { r.tail = 1; break; }    // incomplete record (continues in the next chunk)
    o += 4 + bs; r.n++;
  }
  r.exit = o;
  return r;
}

// one thread per segment
__global__ void __launch_bounds__(128)
seg_walk_kernel(BoundaryParams P, WalkOut W) {
  uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= P.n_seg) return;
  uint32_t o = W.seg_start[s];
  if (o == SEG_NONE) { W.seg_count[s] = 0; W.seg_exit[s] = SEG_NONE; W.seg_tail[s] = 0; return; }
  WalkResult r = walk_segment(P, s, o);
  W.seg_count[s] = r.n; W.seg_exit[s] = r.exit; W.seg_tail[s] = r.tail;
}

// one thread per segment: the next segment that has a start must be the one this segment's chain lands in,
// at exactly that offset.  All seams agreeing <=> the starts form one chain from the first one.
__global__ void __launch_bounds__(128)
seg_check_kernel(BoundaryParams P, WalkOut W) {
  uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= P.n_seg || W.seg_start[s] == SEG_NONE) return;
  uint32_t e = W.seg_exit[s];
  bool bad = false;
  if (W.seg_tail[s]) {
    for (uint32_t u = s + 1; u < P.n_seg; u++) if (W.seg_start[u] != SEG_NONE) { bad = true; break; }
    atomicMin(&W.flags[2], e);
  } else {
    uint32_t t = (e - P.seg0) / P.seg_bytes;
    if (t >= P.n_seg) t = P.n_seg - 1;
    for (uint32_t u = s + 1; u < t; u++) if (W.seg_start[u] != SEG_NONE) { bad = true; break; }
    if (W.seg_start[t] != e) bad = true;
  }
  if (bad) { atomicAdd(&W.flags[0], 1u); atomicMin(&W.flags[11], s); }   // [11] = first segment whose seam disagrees
}

// Parallel repair rounds (in front of the sequential one).  One thread per segment whose seam disagrees -- and whose own walk ran
// past its segment -- re-anchors the segment its chain lands in: the starts in between are dropped, the landing segment is
// re-walked from the landing offset.  This is only right when the fixing segment itself lies on the true chain, which a thread
// cannot know; but segment 0 is exact, so after round r the first r links of the chain are final, a wrong "fix" made by a
// false start is undone in a later round by the true predecessor, and independent errors (the common case in long-read files,
// where a 10 kb record covers whole segments and a false candidate shows up every few thousand segments) are all gone after
// two or three rounds.  Exactness does not rest on these rounds: seg_check runs again behind them and seg_repair_kernel
// re-chains sequentially whatever still disagrees.
__global__ void __launch_bounds__(128)
seg_fix_kernel(BoundaryParams P, WalkOut W, int round) {
  if (W.flags[0] == 0) return;
  uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s == 0 && round == 0) W.flags[10] = W.flags[0];   // seams the first check rejected (stats)
  if (s >= P.n_seg || W.seg_start[s] == SEG_NONE || W.seg_tail[s]) return;
  const uint32_t e = W.seg_exit[s];
  uint32_t t = (e - P.seg0) / P.seg_bytes;
  if (t >= P.n_seg) t = P.n_seg - 1;
  if (t <= s) return;
  for (uint32_t u = s + 1; u < t; u++)
    if (W.seg_start[u] != SEG_NONE) { W.seg_start[u] = SEG_NONE; W.seg_count[u] = 0; W.seg_exit[u] = SEG_NONE; W.seg_tail[u] = 0; }
  if (W.seg_start[t] != e) {
    atomicAdd(&W.flags[4], 1u);
    W.seg_start[t] = e;
    WalkResult r = walk_segment(P, t, e);
    W.seg_count[t] = r.n; W.seg_exit[t] = r.exit; W.seg_tail[t] = r.tail;
  }
}
__global__ void seg_reset_kernel(WalkOut W) {
  if (W.flags[0] == 0) return;
  W.flags[0] = 0; W.flags[2] = 0xffffffffu; W.flags[11] = 0xffffffffu;
}

// Sequential repair (rare): follows the chain from the first start, reusing per-segment walks whose start
// agrees and re-walking those that do not.  Launched with one thread; returns at once when every seam agreed.
__global__ void seg_repair_kernel(BoundaryParams P, WalkOut W) {
  if (W.flags[0] == 0) return;
  if (W.flags[10] == 0) W.flags[10] = W.flags[0];   // reported in the stats (the parallel rounds record the first check's count)
  // every seam before the first disagreeing one was verified, so that segment's own start is on the true chain
  uint32_t s = W.flags[11] < P.n_seg ? W.flags[11] : 0;
  while (s < P.n_seg && W.seg_start[s] == SEG_NONE) s++;
  uint32_t tail_off = P.data_hi;
  while (s < P.n_seg) {
    uint32_t e = W.seg_exit[s];
    bool tail = W.seg_tail[s] != 0;
    uint32_t t = P.n_seg;
    if (tail) tail_off = e;
    else { t = (e - P.seg0) / P.seg_bytes; if (t >= P.n_seg) t = P.n_seg - 1; }
    for (uint32_t u = s + 1; u < t && u < P.n_seg; u++) { W.seg_start[u] = SEG_NONE; W.seg_count[u] = 0; W.seg_exit[u] = SEG_NONE; W.seg_tail[u] = 0; }
    if (tail) break;
    if (W.seg_start[t] != e) {
      W.flags[4]++;
      W.seg_start[t] = e;
      WalkResult r = walk_segment(P, t, e);
      W.seg_count[t] = r.n; W.seg_exit[t] = r.exit; W.seg_tail[t] = r.tail;
    }
    s = t;
  }
  W.flags[2] = tail_off;
  W.flags[0] = 0;
}

// single-CTA exclusive scan of seg_count -> seg_base ; total -> flags[3] ; first owned record -> flags[13] (preset to 0xffffffff)
__global__ void __launch_bounds__(1024)
seg_scan_kernel(const uint32_t* __restrict__ seg_count, const uint32_t* __restrict__ seg_start, const uint32_t* __restrict__ seg_exit,
                const uint8_t* __restrict__ seg_tail, uint32_t* __restrict__ seg_base, uint32_t n_seg, uint32_t* __restrict__ flags) {
  const uint32_t total = cta_exclusive_scan<uint32_t>(n_seg, [&](uint32_t i) {
    const uint32_t v = i < n_seg ? seg_count[i] : 0u;
    {
      // offset of the first owned record of the chunk: one atomic per warp that holds one (a 1.5 GB chunk has 90 k segments with
      // records; one same-address atomic each made this kernel the slowest of the stage)
      const uint32_t mine = v ? seg_start[i] : 0xffffffffu;
      const uint32_t wmin = __reduce_min_sync(0xffffffffu, mine);
      if ((threadIdx.x & 31) == 0 && wmin != 0xffffffffu && wmin < flags[13]) atomicMin(&flags[13], wmin);
    }
    if (i < n_seg && seg_start[i] != SEG_NONE && seg_tail[i] == 2) atomicExch(&flags[1], seg_exit[i] | 1u);   // corrupt block_size on the live chain
    return v;
  }, [&](uint32_t i, uint32_t excl, uint32_t) { seg_base[i] = excl; });
  if (threadIdx.x == 0) flags[3] = total;
}

// one thread per segment: emit record offsets
__global__ void __launch_bounds__(128)
seg_emit_kernel(BoundaryParams P, const uint32_t* __restrict__ seg_start, const uint32_t* __restrict__ seg_count,
                const uint32_t* __restrict__ seg_base, uint32_t* __restrict__ rec_off, uint32_t n_total, uint32_t tail_off) {
  uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s == 0 && blockIdx.x == 0) rec_off[n_total] = tail_off;
  if (s >= P.n_seg) return;
  uint32_t o = seg_start[s], n = seg_count[s], base = seg_base[s];
  for (uint32_t i = 0; i < n; i++) {
    rec_off[base + i] = o;
    o += 4 + ld_u32(P.U, o);
  }
}

}  // namespace bamscan
