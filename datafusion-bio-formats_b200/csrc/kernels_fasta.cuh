// kernels_fasta.cuh -- BGZF-FASTA on the BAM scan engine: record framing by '>' line starts, then name / description / sequence.
//
// Inflate, chunking, carry of the incomplete tail record, Arrow layout and export are the engine's (engine.cu), as for FASTQ.
// A FASTA record is a '>' definition line followed by any number of sequence lines, joined with their line breaks removed:
//
//   framing   fq_count -> cta_scan_kernel -> fq_lines (kernels_fastq.cuh): the offset of every line start of the chunk.
//             fa_count -> cta_scan_kernel -> fa_starts: the line index of every line starting with '>' (a record start), in order.
//             fa_frame (one thread) turns them into rows / tail offset / first record as fq_frame reports them, owns the records
//             whose '>' lies in [own_lo, own_hi), and cuts the owned records into decode slices of about SLICE bytes of text.
//   lengths   fa_lines_kernel: per line its content bytes (without '\n' and one trailing '\r'; 0 for a definition line), which
//             one offsets scan (multi_scan_reduce -> cta_scan_kernel -> multi_scan_apply) turns into each line's destination in
//             the chunk's compacted sequence text.
//             fa_lengths_kernel (thread per record): name / description split of the definition line (fq_definition's rule),
//             sequence length = the difference of that scan at the record's two boundary lines.
//   copy      fa_copy_kernel (8 lanes per record): name and description, as fq_copy does.
//             fa_seq_kernel (CTA per FQ_TILE of input text): the sequence column is a compaction of the text.  Each thread finds
//             the line of its 16 bytes from the tile's line base, keeps the content bytes of sequence lines, compacts the tile
//             into shared memory and the CTA writes destination-aligned words.  Line lengths range from 60 bytes to one 250 MB
//             line, so the work is split over the input bytes, not over records or lines.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

#include "kernels_fastq.cuh"
#include "kernels_scan.cuh"

namespace bamscan {

enum FastaErr : uint32_t { FA_ERR_NAME = 30 /* empty name */, FA_ERR_UTF8 = 31 /* byte >= 0x80 */, FA_ERR_TOO_LONG = 32 /* record > 1 GiB */ };
constexpr uint64_t FA_MAX_RECORD = 1ull << 30;     // bytes of text of one record (definition line and line breaks included)
constexpr int FA_MAX_SLICES = 15;

// flag words of a FASTA chunk (d_flags, device; [16, 64) are published to the host page at FA_HFLAGS)
enum : int { FA_F_NEWLINES = 16, FA_F_STARTS = 17, FA_F_LINES = 18, FA_F_LAST_NL = 19, FA_F_LEADING = 20, FA_F_SLICES = 21,
             FA_F_SLICE_REC = 32, FA_F_SLICE_BYTE = 48 };

__device__ __forceinline__ bool fa_is_space(uint8_t c) { return c == ' ' || c == '\t' || c == '\n' || c == '\r' || c == '\f'; }

// bit k: a record starts at o + k + 1 (U[o + k] == '\n', the next byte is '>' and lies in [own_lo, data_hi))
__device__ __forceinline__ uint32_t fa_start_mask16(const uint8_t* U, uint32_t o, uint32_t lo, uint32_t hi, uint32_t own_lo) {
  uint32_t m = 0;
  #pragma unroll
  for (int k = 0; k < 16; k++) {
    const uint32_t p = o + k;
    if (p >= lo && p + 1u < hi && p + 1u >= own_lo && U[p] == '\n' && U[p + 1] == '>') m |= 1u << k;
  }
  return m;
}

struct FastaFrame {
  const uint8_t* U;
  uint32_t data_lo, data_hi, own_lo, own_hi;
  uint32_t lead_ok;        // 1: data_lo starts a line (file start, or a carried record)
  uint32_t at_eof;         // 1: data_hi is the end of the file: an unterminated last line is a line
  uint32_t cap;           // entries lines[] and starts[] can hold
  uint32_t slice_bytes;
};

__device__ __forceinline__ uint32_t fa_lead_start(const FastaFrame& P) {
  return P.lead_ok && P.data_lo >= P.own_lo && P.data_lo < P.data_hi && P.U[P.data_lo] == '>' ? 1u : 0u;
}

// tile_count[t] = record starts whose line break lies in tile t (+ a start at data_lo, counted in tile 0)
__global__ void __launch_bounds__(256)
fa_count_kernel(const FastaFrame P, uint32_t* __restrict__ tile_count) {
  __shared__ uint32_t ws[8];
  const uint32_t o = P.data_lo + blockIdx.x * FQ_TILE + threadIdx.x * 16;
  uint32_t c = __popc(fa_start_mask16(P.U, o, P.data_lo, P.data_hi, P.own_lo));
  if (blockIdx.x == 0 && threadIdx.x == 0) c += fa_lead_start(P);
  const uint32_t t = block_sum<256>(c, ws);
  if (threadIdx.x == 0) tile_count[blockIdx.x] = t;
}

// starts[j] = line index of the j-th record start
__global__ void __launch_bounds__(256)
fa_starts_kernel(const FastaFrame P, const uint32_t* __restrict__ nl_base, const uint32_t* __restrict__ st_base, uint32_t* __restrict__ starts) {
  __shared__ uint32_t ws[2][8];
  const uint32_t o = P.data_lo + blockIdx.x * FQ_TILE + threadIdx.x * 16;
  const uint32_t nm = fq_newline_mask16(P.U, o, P.data_lo, P.data_hi);
  uint32_t sm = fa_start_mask16(P.U, o, P.data_lo, P.data_hi, P.own_lo);
  const uint32_t lead = (blockIdx.x == 0 && threadIdx.x == 0) ? fa_lead_start(P) : 0u;
  const uint32_t nl_ex = block_exclusive_scan<256>((uint32_t)__popc(nm), ws[0]);
  uint32_t k = st_base[blockIdx.x] + block_exclusive_scan<256>(__popc(sm) + lead, ws[1]);
  if (lead && k < P.cap) starts[k++] = 0;
  const uint32_t line0 = nl_base[blockIdx.x] + nl_ex;
  while (sm) {
    const uint32_t b = (uint32_t)__ffs((int)sm) - 1u; sm &= sm - 1u;
    const uint32_t line = line0 + __popc(nm & ((2u << b) - 1u));       // the line behind the newline at o + b
    if (k < P.cap) starts[k] = line;
    k++;
  }
}

// One thread.  In: flags[FA_F_NEWLINES], flags[FA_F_STARTS], lines[], starts[].  Out (fq_frame's convention): flags[3] rows,
// flags[2] offset of the first record not emitted (incomplete, or not owned), flags[13] offset of the first owned record, flags[1]
// buffer overflow; FASTA words: [FA_F_LINES] lines (after the unterminated last line), [FA_F_LAST_NL] the chunk ends with '\n',
// [FA_F_SLICES] + [FA_F_SLICE_REC],
// [FA_F_SLICE_BYTE]: decode slices (first record, first byte; one entry more than slices).  starts[rows] is the line behind the last
// owned record.
__global__ void fa_frame_kernel(const FastaFrame P, uint32_t* __restrict__ lines, uint32_t* __restrict__ starts, uint32_t* __restrict__ flags) {
  if (threadIdx.x != 0) return;
  uint32_t L = flags[FA_F_NEWLINES];
  const uint32_t S = flags[FA_F_STARTS];
  flags[FA_F_SLICES] = 0;
  if (L + 4u > P.cap || S + 2u > P.cap) { flags[1] = 0x80000001u; flags[3] = 0; flags[2] = 0xffffffffu; return; }
  if (P.at_eof && lines[L] < P.data_hi) { lines[L + 1] = P.data_hi + 1u; L++; }     // unterminated last line of the file
  flags[FA_F_LINES] = L;
  flags[FA_F_LAST_NL] = P.data_hi > P.data_lo && P.U[P.data_hi - 1] == '\n' ? 1u : 0u;
  uint32_t lo = 0, hi = S;                                                           // owned: the '>' lies below own_hi
  while (lo < hi) { const uint32_t mid = (lo + hi) >> 1; if (lines[starts[mid]] < P.own_hi) lo = mid + 1u; else hi = mid; }
  const uint32_t owned = lo;
  const uint32_t n_rec = (owned < S || P.at_eof) ? owned : (owned ? owned - 1u : 0u);   // complete: another start follows, or the file ends
  if (n_rec == S) starts[S] = L;                                                     // (at the end of the file)
  flags[3] = n_rec;
  flags[2] = n_rec < S ? lines[starts[n_rec]] : 0xffffffffu;
  if (owned) flags[13] = lines[starts[0]];
  // slices: a record opens a new slice when it starts slice_bytes or more behind the start of the slice's first record
  uint32_t k = 0, a = 0;
  while (a < n_rec && k < (uint32_t)FA_MAX_SLICES) {
    flags[FA_F_SLICE_REC + k] = a; flags[FA_F_SLICE_BYTE + k] = lines[starts[a]];
    const uint64_t lim = (uint64_t)lines[starts[a]] + P.slice_bytes;
    uint32_t l2 = a + 1u, h2 = n_rec;
    while (l2 < h2) { const uint32_t mid = (l2 + h2) >> 1; if ((uint64_t)lines[starts[mid]] < lim) l2 = mid + 1u; else h2 = mid; }
    a = (k + 1u == (uint32_t)FA_MAX_SLICES) ? n_rec : l2;
    k++;
  }
  flags[FA_F_SLICE_REC + k] = n_rec; flags[FA_F_SLICE_BYTE + k] = min(lines[starts[n_rec]], P.data_hi);
  flags[FA_F_SLICES] = k;
}

// The bytes in front of the first '>' of the file must be whitespace: only the first chunks of the range that owns the file's first
// byte run this, and it reads no further than the first record start.
__global__ void __launch_bounds__(256)
fa_leading_kernel(const FastaFrame P, const uint32_t* __restrict__ lines, const uint32_t* __restrict__ starts, uint32_t* __restrict__ flags) {
  const uint32_t lim = flags[FA_F_STARTS] ? lines[starts[0]] : P.data_hi;
  const uint32_t o = P.data_lo + blockIdx.x * FQ_TILE + threadIdx.x * 16;
  if (o >= lim) return;
  uint32_t bad = 0;
  #pragma unroll
  for (int k = 0; k < 16; k++) { const uint32_t p = o + k; if (p >= P.own_lo && p < lim && !fa_is_space(P.U[p])) bad = 1; }
  if (bad) flags[FA_F_LEADING] = 1;
}

// content[i] = bytes of line i without its '\n' and one trailing '\r'; 0 for a definition line ('>' first) -- scanned in place
// into each line's destination in the chunk's sequence text (chunk offsets stay below 4 GiB, so 32 bits hold them exactly)
__global__ void __launch_bounds__(256)
fa_lines_kernel(const uint8_t* __restrict__ U, const uint32_t* __restrict__ lines, uint32_t n_lines, uint32_t* __restrict__ content) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_lines) return;
  const uint32_t s = lines[i];
  uint32_t e = lines[i + 1] - 1u;
  if (e > s && U[e - 1] == '\r') e--;
  content[i] = (e > s && U[s] != '>') ? e - s : 0u;
}

struct FastaCols {
  const uint8_t* U;
  const uint32_t* lines;
  const uint32_t* rec;        // line index of each record's definition line (+ the line behind the last record)
  const uint32_t* seqpos;     // per line: destination of its content in the chunk's sequence text
  uint32_t n;
  int32_t *l_name, *l_desc, *l_seq;
  uint32_t* v_desc;
  uint8_t *d_name, *d_desc;
  uint32_t* err;
};

// the definition line of record r: name and description, fq_definition's rule (behind the '>', split at the first space or tab)
__device__ __forceinline__ void fa_definition(const FastaCols& P, uint32_t r, uint32_t* nb, uint32_t* ne, uint32_t* db, uint32_t* de) {
  const uint32_t li = P.rec[r];
  uint32_t b = P.lines[li], e = P.lines[li + 1] - 1u;
  if (e > b && P.U[e - 1] == '\r') e--;
  b = min(b + 1u, e);
  uint32_t k = b;
  while (k < e && P.U[k] != ' ' && P.U[k] != '\t') k++;
  *nb = b; *ne = k; *db = min(k + 1u, e); *de = e;
}

__global__ void __launch_bounds__(256)
fa_lengths_kernel(const FastaCols P) {
  const uint32_t r = blockIdx.x * blockDim.x + threadIdx.x;
  const bool on = r < P.n;
  uint32_t has_desc = 0;
  if (on) {
    uint32_t nb, ne, db, de;
    fa_definition(P, r, &nb, &ne, &db, &de);
    if (ne == nb) set_err(P.err, FA_ERR_NAME, r);
    if ((uint64_t)(P.lines[P.rec[r + 1]] - P.lines[P.rec[r]]) > FA_MAX_RECORD) set_err(P.err, FA_ERR_TOO_LONG, r);
    has_desc = de > db;
    if (P.l_name) P.l_name[r] = (int32_t)(ne - nb);
    if (P.l_desc) P.l_desc[r] = (int32_t)(de - db);
    if (P.l_seq) P.l_seq[r] = (int32_t)(P.seqpos[P.rec[r + 1]] - P.seqpos[P.rec[r]]);
  }
  if (P.v_desc) {
    const uint32_t m = __ballot_sync(0xffffffffu, has_desc != 0);
    if ((threadIdx.x & 31) == 0 && r < ((P.n + 31u) & ~31u)) P.v_desc[r >> 5] = m;
  }
}

template <int G>
__global__ void __launch_bounds__(256)
fa_copy_kernel(const FastaCols P) {
  const int lane = threadIdx.x & 31, gl = lane & (G - 1);
  const uint32_t r = (blockIdx.x * blockDim.x + threadIdx.x) / G;
  if (r >= P.n) return;
  uint32_t nb, ne, db, de, bad = 0;
  fa_definition(P, r, &nb, &ne, &db, &de);
  if (P.d_name) bad |= grp_map4<G>(P.d_name + P.l_name[r], P.U + nb, ne - nb, gl, 0u);
  if (P.d_desc && de > db) bad |= grp_map4<G>(P.d_desc + P.l_desc[r], P.U + db, de - db, gl, 0u);
  if (bad) set_err(P.err, FA_ERR_UTF8, r);
}

struct FastaSeq {
  const uint8_t* U;
  const uint32_t* lines;
  const uint32_t* seqpos;
  const uint32_t* tile_base;  // newlines in front of each FQ_TILE of [data_lo, data_hi) (the newline scan)
  const uint32_t* rec;        // the slice's records: rec[0 .. n]
  uint32_t n, data_lo, data_hi, t0;
  uint8_t* dst;               // the slice's sequence column data
  uint32_t* err;
};

// CTA per input tile t0 + blockIdx.x.  A byte is kept when it lies on a sequence line of the slice, in front of the line's
// terminator; its destination is seqpos[line] + (offset in the line) - seqpos[first line of the slice].  The kept bytes of a tile
// are one contiguous destination range, so they are compacted in shared memory and stored as aligned words (bytes at the two ends,
// whose words other tiles share).
__global__ void __launch_bounds__(256)
fa_seq_kernel(const FastaSeq P) {
  __shared__ uint4 s_in[FQ_TILE / 16 + 1];
  __shared__ __align__(16) uint8_t s_out[FQ_TILE];
  __shared__ uint32_t ws[8], s_dlo, s_cnt, s_bad_line;
  const uint32_t t = P.t0 + blockIdx.x;
  const uint32_t tlo = P.data_lo + t * FQ_TILE;
  const uint32_t line_a = P.rec[0], line_b = P.rec[P.n];
  const uint32_t base = P.seqpos[line_a];
  const uint32_t ab = tlo & ~15u;
  for (uint32_t i = threadIdx.x; i < FQ_TILE / 16 + 1; i += blockDim.x) s_in[i] = reinterpret_cast<const uint4*>(P.U + ab)[i];
  if (threadIdx.x == 0) {
    s_cnt = 0; s_bad_line = 0xffffffffu;
    const uint32_t l0 = P.tile_base[t];                                   // line of the tile's first byte
    uint32_t d = 0;
    if (l0 >= line_a && l0 < line_b) d = P.seqpos[l0] - base + min(tlo - P.lines[l0], P.seqpos[l0 + 1] - P.seqpos[l0]);
    s_dlo = d;
  }
  __syncthreads();
  const uint8_t* in = reinterpret_cast<const uint8_t*>(s_in) + (tlo - ab) + threadIdx.x * 16;
  const uint32_t o = tlo + threadIdx.x * 16;
  uint32_t nm = 0;
  #pragma unroll
  for (int k = 0; k < 16; k++) if (o + k < P.data_hi && in[k] == '\n') nm |= 1u << k;
  uint32_t li = P.tile_base[t] + block_exclusive_scan<256>((uint32_t)__popc(nm), ws);
  const uint32_t dlo = s_dlo;
  uint32_t cur = 0xffffffffu, ls = 0, len = 0, d = 0, kept = 0, bad = 0;
  #pragma unroll
  for (int k = 0; k < 16; k++) {
    const uint32_t p = o + k;
    if (p >= P.data_hi) break;
    if (li != cur) {
      cur = li; len = 0;
      if (li > line_a && li < line_b) { ls = P.lines[li]; const uint32_t s0 = P.seqpos[li]; len = P.seqpos[li + 1] - s0; d = s0 - base - dlo; }
    }
    if ((nm >> k) & 1u) { li++; continue; }
    const uint32_t off = p - ls;
    if (off < len) {
      const uint8_t c = in[k];
      s_out[d + off] = c;
      kept++;
      if ((c & 0x80u) && !bad) { bad = 1; atomicMin(&s_bad_line, li); }
    }
  }
  if (kept) atomicAdd(&s_cnt, kept);
  __syncthreads();
  const uint32_t cnt = s_cnt;
  if (cnt) {
    uint8_t* g = P.dst + dlo;
    const uint32_t head = min(cnt, (uint32_t)((4u - (reinterpret_cast<uintptr_t>(g) & 3u)) & 3u));
    if (threadIdx.x < head) g[threadIdx.x] = s_out[threadIdx.x];
    const uint32_t nw = (cnt - head) >> 2;
    uint32_t* gw = reinterpret_cast<uint32_t*>(g + head);
    for (uint32_t w = threadIdx.x; w < nw; w += blockDim.x) {
      const uint8_t* q = s_out + head + 4u * w;
      gw[w] = (uint32_t)q[0] | ((uint32_t)q[1] << 8) | ((uint32_t)q[2] << 16) | ((uint32_t)q[3] << 24);
    }
    for (uint32_t i = head + 4u * nw + threadIdx.x; i < cnt; i += blockDim.x) g[i] = s_out[i];
  }
  if (threadIdx.x == 0 && s_bad_line != 0xffffffffu) {
    uint32_t lo = 0, hi = P.n;                                            // the record holding that line
    while (lo < hi) { const uint32_t mid = (lo + hi + 1u) >> 1; if (P.rec[mid] <= s_bad_line) lo = mid; else hi = mid - 1u; }
    set_err(P.err, FA_ERR_UTF8, lo);
  }
}

}  // namespace bamscan
