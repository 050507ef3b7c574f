// kernels_fastq.cuh -- BGZF-FASTQ on the BAM scan engine: record framing by newline scan, then the four Utf8 columns.
//
// Replaces (SURVEY §8 f3): the per-record loop of datafusion/bio-format-fastq/src/physical_exec.rs:393-468
// (`fastq::io::Reader::read_record` of noodles-fastq 0.23.0 + four StringBuilders) and, for block-range partitions, the record
// synchronisation of physical_exec.rs:184-219 (`synchronize_bgzf_reader`: an '@' line whose line + 2 starts with '+').
// Inflate, chunking, carry of the incomplete tail record, slicing into batches, arena layout and Arrow export are the BAM
// engine's (engine.cu); only the two places that look INSIDE the inflated bytes differ:
//
//   framing   fq_count -> cta_scan_kernel -> fq_lines: the offset of every line start of the chunk, in order (lines[0] = first record
//             start).  A FASTQ record is four lines (noodles-fastq reads exactly four: name, sequence, '+' line, qualities), so
//             record r is lines[4r .. 4r + 4) and the "record offsets" the decode stage is given are that array itself.
//             fq_frame (one warp) turns the line count into rows / tail offset / first record exactly as kernels_boundary.cuh
//             reports them (flags[3], [2], [13]), honours the ownership bound of a block-range partition, and for a partition
//             without a known start picks the first line that starts with '@' whose line + 2 starts with '+' and, when there
//             is one, whose line + 4 starts with '@' again.
//   columns   fq_lengths (thread per record): validates the record ('@' / '+' prefixes), splits the definition line at its
//             first space or tab into name and description (empty description -> NULL, physical_exec.rs:430-434), strips one
//             trailing '\r' per line, writes the per-row byte counts that multi_scan_* turn into Arrow offsets;
//             fq_copy (8 lanes per record): the bytes.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

#include "kernels_decode.cuh"
#include "kernels_scan.cuh"

namespace bamscan {

constexpr int FQ_TILE = 4096;          // bytes per CTA of the newline scan (256 threads x 16 bytes)
enum FastqErr : uint32_t { FQ_ERR_NAME_PREFIX = 20 /* a record does not start with '@' */, FQ_ERR_PLUS = 21 /* third line does not start with '+' */, FQ_ERR_UTF8 = 22 /* non-ASCII byte */ };

__device__ __forceinline__ uint32_t fq_newline_mask16(const uint8_t* U, uint32_t o, uint32_t lo, uint32_t hi) {
  // bit k set: U[o + k] == '\n' and lo <= o + k < hi
  uint32_t m = 0;
  #pragma unroll
  for (int k = 0; k < 16; k++) { const uint32_t p = o + k; if (p >= lo && p < hi && U[p] == '\n') m |= 1u << k; }
  return m;
}

// tile_count[t] = newlines in [data_lo + t * FQ_TILE, ...) clipped to data_hi
__global__ void __launch_bounds__(256)
fq_count_kernel(const uint8_t* __restrict__ U, uint32_t data_lo, uint32_t data_hi, uint32_t* __restrict__ tile_count) {
  __shared__ uint32_t ws[8];
  const uint32_t o = data_lo + blockIdx.x * FQ_TILE + threadIdx.x * 16;
  const uint32_t t = block_sum<256>((uint32_t)__popc(fq_newline_mask16(U, o, data_lo, data_hi)), ws);
  if (threadIdx.x == 0) tile_count[blockIdx.x] = t;
}

// lines[0] = data_lo; lines[k + 1] = offset behind the k-th newline
__global__ void __launch_bounds__(256)
fq_lines_kernel(const uint8_t* __restrict__ U, uint32_t data_lo, uint32_t data_hi, const uint32_t* __restrict__ tile_base, uint32_t* __restrict__ lines, uint32_t cap) {
  __shared__ uint32_t ws[8];
  const uint32_t o = data_lo + blockIdx.x * FQ_TILE + threadIdx.x * 16;
  uint32_t m = fq_newline_mask16(U, o, data_lo, data_hi);
  uint32_t k = tile_base[blockIdx.x] + block_exclusive_scan<256>((uint32_t)__popc(m), ws);
  if (blockIdx.x == 0 && threadIdx.x == 0) lines[0] = data_lo;
  while (m) { const uint32_t b = (uint32_t)__ffs((int)m) - 1u; m &= m - 1u; if (++k < cap) lines[k] = o + b + 1u; }     // (fq_frame reports the overflow)
}

struct FastqFrame {
  const uint8_t* U;
  uint32_t data_lo, data_hi, own_hi;
  uint32_t speculate;      // 1: the first record start is not known (block-range partition > 0)
  uint32_t at_eof;         // 1: data_hi is the end of the FILE: an unterminated last line is a line
  uint32_t cap;            // entries lines[] can hold
};

// One warp.  In: *n_newlines, lines[0 .. n_newlines].  Out (kernels_boundary.cuh convention): flags[3] rows, flags[2] offset of
// the first record that is not emitted (incomplete, or not owned), flags[13] offset of the first emitted record, flags[14] index
// in lines[] of the first record's line (the decode stage reads lines + flags[14]), flags[1] error.
__global__ void fq_frame_kernel(const FastqFrame P, const uint32_t* __restrict__ n_newlines, uint32_t* __restrict__ lines, uint32_t* __restrict__ flags) {
  if (threadIdx.x != 0) return;
  uint32_t L = *n_newlines;                          // complete (newline-terminated) lines: line i = [lines[i], lines[i + 1] - 1)
  if (L + 4u > P.cap) { flags[1] = 0x80000001u; flags[3] = 0; flags[2] = 0xffffffffu; return; }     // more lines than the buffer was sized for
  if (P.at_eof && lines[L] < P.data_hi) { lines[L + 1] = P.data_hi + 1u; L++; }     // unterminated last line of the file
  uint32_t j0 = 0;
  if (P.speculate) {
    // first line j >= 0 with '@' ... line j + 2 with '+' ... (line j + 4 with '@' when it exists).  Line 0 may be the tail of a
    // line that began in the previous partition: it is taken only when it passes the same test (its first byte is the
    // partition's first byte: a record that starts exactly there is this partition's).
    bool found = false;
    for (uint32_t j = 0; j + 2 < L + 1 && j + 2 <= L; j++) {
      if (lines[j] >= P.own_hi) break;
      if (lines[j] < P.data_hi && P.U[lines[j]] == '@' && lines[j + 2] < P.data_hi && P.U[lines[j + 2]] == '+' &&
          (j + 4 > L || lines[j + 4] >= P.data_hi || P.U[lines[j + 4]] == '@')) { j0 = j; found = true; break; }
    }
    if (!found) {                                     // no confirmed record start yet: keep the last lines for the next chunk
      const uint32_t keep = lines[L >= 4u ? L - 4u : 0u];
      flags[3] = 0; flags[14] = 0; flags[2] = (keep >= P.data_hi || keep >= P.own_hi) ? 0xffffffffu : keep;
      return;
    }
  }
  const uint32_t n_complete = (L - j0) / 4u;
  // owned: record r (line j0 + 4r) starts below own_hi
  uint32_t lo = 0, hi = n_complete;
  while (lo < hi) { const uint32_t mid = (lo + hi) >> 1; if (lines[j0 + 4u * mid] < P.own_hi) lo = mid + 1u; else hi = mid; }
  const uint32_t n_rec = lo;
  flags[3] = n_rec;
  flags[14] = j0;
  const uint32_t tail = lines[j0 + 4u * n_rec];
  flags[2] = tail >= P.data_hi ? 0xffffffffu : tail;
  if (n_rec) flags[13] = lines[j0];
}

struct FastqCols {
  const uint8_t* U;
  const uint32_t* lines;      // 4 entries per record (+ the start of the following line)
  uint32_t n;
  int32_t *l_name, *l_desc, *l_seq, *l_qual;      // per-row byte counts (-> offsets), null when not projected
  uint32_t* v_desc;                                // validity words of description
  uint8_t *d_name, *d_desc, *d_seq, *d_qual;
  uint32_t* err;
};

// line i of record r without its '\n' and without one trailing '\r'
__device__ __forceinline__ void fq_line(const FastqCols& P, uint32_t r, int i, uint32_t* b, uint32_t* e) {
  const uint32_t s = P.lines[4u * r + i];
  uint32_t t = P.lines[4u * r + i + 1] - 1u;        // the newline (or the virtual one at the end of the file)
  if (t > s && P.U[t - 1] == '\r') t--;
  *b = s; *e = t;
}
__device__ __forceinline__ void fq_definition(const FastqCols& P, uint32_t r, uint32_t* nb, uint32_t* ne, uint32_t* db, uint32_t* de) {
  uint32_t b, e;
  fq_line(P, r, 0, &b, &e);
  b = min(b + 1u, e);                                 // behind the '@'
  uint32_t k = b;
  while (k < e && P.U[k] != ' ' && P.U[k] != '\t') k++;
  *nb = b; *ne = k; *db = min(k + 1u, e); *de = e;
}

__global__ void __launch_bounds__(256)
fq_lengths_kernel(const FastqCols P) {
  const uint32_t r = blockIdx.x * blockDim.x + threadIdx.x;
  const bool on = r < P.n;
  uint32_t has_desc = 0;
  if (on) {
    uint32_t b, e, nb, ne, db, de;
    fq_line(P, r, 0, &b, &e);
    if (e <= b || P.U[b] != '@') set_err(P.err, FQ_ERR_NAME_PREFIX, r);
    fq_definition(P, r, &nb, &ne, &db, &de);
    has_desc = de > db;
    if (P.l_name) P.l_name[r] = (int32_t)(ne - nb);
    if (P.l_desc) P.l_desc[r] = (int32_t)(de - db);
    fq_line(P, r, 1, &b, &e);
    if (P.l_seq) P.l_seq[r] = (int32_t)(e - b);
    fq_line(P, r, 2, &b, &e);
    if (e <= b || P.U[b] != '+') set_err(P.err, FQ_ERR_PLUS, r);
    fq_line(P, r, 3, &b, &e);
    if (P.l_qual) P.l_qual[r] = (int32_t)(e - b);
  }
  if (P.v_desc) {
    const uint32_t m = __ballot_sync(0xffffffffu, has_desc != 0);
    if ((threadIdx.x & 31) == 0 && r < ((P.n + 31u) & ~31u)) P.v_desc[r >> 5] = m;
  }
}

template <int G>
__global__ void __launch_bounds__(256)
fq_copy_kernel(const FastqCols P) {
  const int lane = threadIdx.x & 31, gl = lane & (G - 1);
  const uint32_t r = (blockIdx.x * blockDim.x + threadIdx.x) / G;
  if (r >= P.n) return;
  uint32_t b, e, nb, ne, db, de;
  uint32_t bad = 0;
  fq_definition(P, r, &nb, &ne, &db, &de);
  if (P.d_name) bad |= grp_map4<G>(P.d_name + P.l_name[r], P.U + nb, ne - nb, gl, 0u);
  if (P.d_desc && de > db) bad |= grp_map4<G>(P.d_desc + P.l_desc[r], P.U + db, de - db, gl, 0u);
  if (P.d_seq) { fq_line(P, r, 1, &b, &e); bad |= grp_map4<G>(P.d_seq + P.l_seq[r], P.U + b, e - b, gl, 0u); }
  if (P.d_qual) { fq_line(P, r, 3, &b, &e); bad |= grp_map4<G>(P.d_qual + P.l_qual[r], P.U + b, e - b, gl, 0u); }
  if (bad) set_err(P.err, FQ_ERR_UTF8, r);          // (std::str::from_utf8(..).unwrap() of the reference panics on invalid UTF-8; non-ASCII is refused here)
}

}  // namespace bamscan
