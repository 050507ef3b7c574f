// kernels_sam.cuh -- plain SAM text on the BAM scan engine: each line is transcoded into a BAM record on the device, then the
// unchanged BAM decode stage (kernels_decode.cuh) makes the columns.  sm_100a.
//
// Replaces: the SAM loop of BamTableProvider (reference physical_exec.rs, `is_sam` in get_stream: noodles-sam's reader filling a
// RecordBuf per line).  Column rules, tag coercions, binary CIGAR, the f32 -> text rendering, arenas and the Arrow export are
// the BAM path's; only the text parsing is here:
//
//   framing    fq_count -> fq_scan -> fq_lines (kernels_fastq.cuh: every line start of the chunk), then sam_frame_kernel: one
//              record per line, rows / tail offset / first record / ownership bound reported as the seg_* kernels report them.
//   size       sam_size_kernel: a thread per line.  Splits the 11 mandatory fields, parses and range-checks every one of them,
//              resolves RNAME / RNEXT against the header's reference names, counts and validates the CIGAR, checks SEQ / QUAL,
//              sizes every aux field.  Out: the BAM record size, a SamLine with the parsed values, the "QUAL is *" flag.  The
//              first error (code + row) goes to err[0..1] (enc::report).
//   offsets    multi_scan_* over the sizes (kernels_decode.cuh): the record offsets in the chunk's BAM buffer.
//   write      sam_records_kernel<G>: a group of G lanes per line writes the record: block_size, the fixed 32 bytes, name + NUL,
//              CIGAR ops (group-parallel text parse, as the write path's enc_records_kernel), packed bases, qualities - 33 (0xFF
//              when QUAL is *), aux fields.  Nothing is validated here: the size pass has.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

#include "f32_parse.h"
#include "kernels_text_common.cuh"
#include "kernels_fastq.cuh"

namespace bamscan {
namespace sam {

enum SamErr : uint32_t {
  SAM_OK = 0, SAM_ERR_FIELDS = 1 /* fewer than 11 fields */, SAM_ERR_NAME = 2, SAM_ERR_FLAG = 3, SAM_ERR_RNAME = 4, SAM_ERR_POS = 5,
  SAM_ERR_MAPQ = 6, SAM_ERR_CIGAR = 7, SAM_ERR_CIGAR_OPS = 8 /* > 65535 ops: unsupported */, SAM_ERR_RNEXT = 9, SAM_ERR_PNEXT = 10,
  SAM_ERR_TLEN = 11, SAM_ERR_SEQ = 12, SAM_ERR_QUAL = 13, SAM_ERR_QUAL_LEN = 14, SAM_ERR_TAG = 15, SAM_ERR_TAG_DUP = 16, SAM_ERR_TAG_RANGE = 17
};

struct SamRefs { const uint8_t* blob; const int32_t* off; const int32_t* ids; int32_t n_ref; };   // names sorted bytewise -> ids

// what the size pass learnt about a line, for the write pass
struct SamLine {
  uint32_t f[12];          // f[k]: offset in U of field k (k < 11); f[11]: of the aux fields (line end + 1 when there are none).
                           // Field k ends at f[k + 1] - 1.
  uint32_t end;            // end of the line: its '\n' (or one trailing '\r', or the end of the file)
  int32_t ref, mref, pos0, mpos0, tlen;
  uint32_t flag, mapq, n_ops, l_seq, l_name;
};

// One thread.  In: *n_newlines and lines[0 .. n_newlines] from fq_lines_kernel.  Records are lines; the first one is the first
// line starting at or after first_start; a record is emitted when it is complete and starts below own_hi.  Out, as the seg_*
// kernels: flags[3] rows, flags[2] offset of the first record not emitted (incomplete or not owned), flags[13] first emitted
// record, flags[14] index in lines[] of the first record, flags[1] error.
__global__ void sam_frame_kernel(const FastqFrame P, uint32_t first_start, const uint32_t* __restrict__ n_newlines, uint32_t* __restrict__ lines,
                                 uint32_t* __restrict__ flags) {
  if (threadIdx.x != 0) return;
  uint32_t L = *n_newlines;                          // complete lines: line i = [lines[i], lines[i + 1] - 1)
  if (L + 4u > P.cap) { flags[1] = 0x80000001u; flags[3] = 0; flags[2] = 0xffffffffu; return; }
  if (P.at_eof && lines[L] < P.data_hi) { lines[L + 1] = P.data_hi + 1u; L++; }     // an unterminated last line of the file is a line
  uint32_t lo = 0, hi = L + 1;
  while (lo < hi) { const uint32_t mid = (lo + hi) >> 1; if (lines[mid] < first_start) lo = mid + 1; else hi = mid; }
  const uint32_t j0 = lo;
  if (j0 >= L) {                                     // no complete line starts in front of the data end
    const uint32_t keep = j0 <= L ? lines[j0] : P.data_hi;
    flags[3] = 0; flags[14] = 0; flags[2] = (keep >= P.data_hi || keep >= P.own_hi) ? 0xffffffffu : keep;
    return;
  }
  lo = j0; hi = L;
  while (lo < hi) { const uint32_t mid = (lo + hi) >> 1; if (lines[mid] < P.own_hi) lo = mid + 1; else hi = mid; }
  const uint32_t n_rec = lo - j0;
  flags[3] = n_rec;
  flags[14] = j0;
  const uint32_t tail = lines[j0 + n_rec];
  flags[2] = tail >= P.data_hi ? 0xffffffffu : tail;
  if (n_rec) flags[13] = lines[j0];
}

__device__ __forceinline__ bool is_digit(uint8_t c) { return c >= '0' && c <= '9'; }

// [+]digits (unsigned) or [+-]digits (signed) -> *v, saturated far outside every SAM range
__device__ __forceinline__ bool parse_int(const uint8_t* s, uint32_t n, bool allow_neg, long long* v) {
  uint32_t k = 0; bool neg = false;
  if (k < n && (s[k] == '+' || (allow_neg && s[k] == '-'))) { neg = s[k] == '-'; k++; }
  if (k >= n) return false;
  unsigned long long x = 0;
  for (; k < n; k++) { if (!is_digit(s[k])) return false; x = x * 10u + (s[k] - '0'); if (x > (1ull << 40)) x = 1ull << 40; }
  *v = neg ? -(long long)x : (long long)x;
  return true;
}
// narrowest BAM integer type of a SAM `i` value: C / S / I when non-negative, c / s / i when negative (0 = out of range)
__device__ __forceinline__ uint8_t int_type(long long v) {
  if (v >= 0) return v <= 255 ? 'C' : v <= 65535 ? 'S' : v <= 4294967295ll ? 'I' : 0;
  return v >= -128 ? 'c' : v >= -32768 ? 's' : v >= -2147483648ll ? 'i' : 0;
}
__device__ __forceinline__ bool is_tag_char(uint8_t c, bool first) { return (c >= 'A' && c <= 'Z') || (c >= 'a' && c <= 'z') || (!first && is_digit(c)); }

// One aux field s[0 .. n) ("TG:T:value"): BAM bytes (tag + type + value), 0 when malformed / out of range (*e set)
__device__ __forceinline__ uint32_t aux_bytes(const uint8_t* s, uint32_t n, uint32_t* e) {
  if (n < 5 || s[2] != ':' || s[4] != ':' || !is_tag_char(s[0], true) || !is_tag_char(s[1], false)) { *e = SAM_ERR_TAG; return 0; }
  const uint8_t ty = s[3];
  const uint8_t* v = s + 5;
  const uint32_t vn = n - 5;
  switch (ty) {
    case 'A': if (vn != 1 || v[0] < '!' || v[0] > '~') { *e = SAM_ERR_TAG; return 0; } return 4;
    case 'i': {
      long long x;
      if (!parse_int(v, vn, true, &x)) { *e = SAM_ERR_TAG; return 0; }
      const uint8_t t = int_type(x);
      if (!t) { *e = SAM_ERR_TAG_RANGE; return 0; }
      return 3u + enc::elem_size(t);
    }
    case 'f': { uint32_t b; if (!f32_parse(reinterpret_cast<const char*>(v), vn, &b)) { *e = SAM_ERR_TAG; return 0; } return 7; }
    case 'Z': for (uint32_t k = 0; k < vn; k++) if (v[k] < ' ' || v[k] > '~') { *e = SAM_ERR_TAG; return 0; } return 3u + vn + 1u;
    case 'H':
      if (vn & 1u) { *e = SAM_ERR_TAG; return 0; }
      for (uint32_t k = 0; k < vn; k++) { const uint8_t c = v[k]; if (!(is_digit(c) || (c >= 'A' && c <= 'F') || (c >= 'a' && c <= 'f'))) { *e = SAM_ERR_TAG; return 0; } }
      return 3u + vn + 1u;
    case 'B': {
      if (vn < 1) { *e = SAM_ERR_TAG; return 0; }
      const uint8_t st = v[0];
      if (!(st == 'c' || st == 'C' || st == 's' || st == 'S' || st == 'i' || st == 'I' || st == 'f')) { *e = SAM_ERR_TAG; return 0; }
      uint32_t cnt = 0, k = 1;
      while (k < vn) {
        if (v[k] != ',') { *e = SAM_ERR_TAG; return 0; }
        uint32_t j = k + 1;
        while (j < vn && v[j] != ',') j++;
        if (st == 'f') { uint32_t b; if (!f32_parse(reinterpret_cast<const char*>(v + k + 1), j - k - 1, &b)) { *e = SAM_ERR_TAG; return 0; } }
        else {
          long long x;
          if (!parse_int(v + k + 1, j - k - 1, true, &x)) { *e = SAM_ERR_TAG; return 0; }
          if (!enc::int_fits(x, st)) { *e = SAM_ERR_TAG_RANGE; return 0; }
        }
        cnt++; k = j;
      }
      return 3u + 1u + 4u + cnt * enc::elem_size(st);
    }
    default: *e = SAM_ERR_TAG; return 0;
  }
}

// position field: 0 = none (-1 in BAM), else <= 2^31 (the BAM i32 of position - 1)
__device__ __forceinline__ bool parse_pos(const uint8_t* s, uint32_t n, int32_t* pos0) {
  long long v;
  if (!parse_int(s, n, false, &v) || v > 2147483648ll) return false;
  *pos0 = (int32_t)(v - 1);
  return true;
}

struct SamSizeArgs {
  const uint8_t* U;
  const uint32_t* lines;     // line starts: record i is [lines[i], lines[i + 1] - 1)
  uint32_t n;
  SamRefs R;
  SamLine* out;
  uint32_t* sizes;           // [n + 1]: BAM bytes of record i (the scan turns them into offsets)
  uint8_t* qual_absent;      // [n]: 1 when QUAL is '*' and SEQ is not
  uint32_t* err;
};

__global__ void __launch_bounds__(256)
sam_size_kernel(const SamSizeArgs a) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= a.n) return;
  const uint8_t* U = a.U;
  const uint32_t b = a.lines[i];
  uint32_t end = a.lines[i + 1] - 1u;
  if (end > b && U[end - 1] == '\r') end--;
  SamLine L;
  uint32_t e = SAM_OK;
  // ---- the 11 mandatory fields
  L.f[0] = b;
  {
    uint32_t k = b, fld = 1;
    for (; k < end && fld <= 11; k++) if (U[k] == '\t') L.f[fld++] = k + 1u;
    if (fld < 11) { e = SAM_ERR_FIELDS; for (; fld < 12; fld++) L.f[fld] = end + 1u; }
    else if (fld == 11) L.f[11] = end + 1u;
  }
  L.end = end;
  auto fs = [&](int k) { return U + L.f[k]; };
  auto fn = [&](int k) { return L.f[k + 1] - 1u - L.f[k]; };
  L.ref = L.mref = -1; L.pos0 = L.mpos0 = -1; L.tlen = 0; L.flag = L.mapq = L.n_ops = L.l_seq = 0; L.l_name = 1;
  uint32_t total = 36;
  if (!e) {
    // QNAME: [!-?A-~]{1,254}; '*' is a missing name, written as "*" like the BAM encoder does
    const uint32_t nn = fn(0);
    if (nn == 0 || nn > 254) e = SAM_ERR_NAME;
    for (uint32_t k = 0; k < nn && !e; k++) { const uint8_t c = fs(0)[k]; if (c < '!' || c > '~' || c == '@') e = SAM_ERR_NAME; }
    L.l_name = nn;
    long long v;
    if (!e && (!parse_int(fs(1), fn(1), false, &v) || v > 65535)) e = SAM_ERR_FLAG;
    L.flag = (uint32_t)v;
    if (!e && !(fn(2) == 1 && fs(2)[0] == '*')) { L.ref = enc::lookup_ref(a.R.blob, a.R.off, a.R.ids, a.R.n_ref, fs(2), fn(2)); if (L.ref < 0) e = SAM_ERR_RNAME; }
    if (!e && !parse_pos(fs(3), fn(3), &L.pos0)) e = SAM_ERR_POS;
    if (!e && (!parse_int(fs(4), fn(4), false, &v) || v > 255)) e = SAM_ERR_MAPQ;
    L.mapq = (uint32_t)v;
    // CIGAR: '*' or (digits op)+ with op lengths < 2^28
    if (!e && !(fn(5) == 1 && fs(5)[0] == '*')) {
      const uint8_t* s = fs(5); const uint32_t n = fn(5);
      unsigned long long len = 0; uint32_t nd = 0, ops = 0;
      for (uint32_t k = 0; k < n && !e; k++) {
        if (is_digit(s[k])) { len = len * 10u + (s[k] - '0'); if (len >= (1ull << 28)) e = SAM_ERR_CIGAR; nd++; continue; }
        if (nd == 0 || enc::op_code(s[k]) < 0) e = SAM_ERR_CIGAR;
        ops++; len = 0; nd = 0;
      }
      if (n == 0 || nd) e = SAM_ERR_CIGAR;
      if (!e && ops > 65535u) e = SAM_ERR_CIGAR_OPS;
      L.n_ops = ops;
    }
    if (!e) {
      const uint8_t* s = fs(6); const uint32_t n = fn(6);
      if (n == 1 && s[0] == '=') L.mref = L.ref;
      else if (!(n == 1 && s[0] == '*')) { L.mref = enc::lookup_ref(a.R.blob, a.R.off, a.R.ids, a.R.n_ref, s, n); if (L.mref < 0) e = SAM_ERR_RNEXT; }
    }
    if (!e && !parse_pos(fs(7), fn(7), &L.mpos0)) e = SAM_ERR_PNEXT;
    if (!e && (!parse_int(fs(8), fn(8), true, &v) || v < -2147483648ll || v > 2147483647ll)) e = SAM_ERR_TLEN;
    L.tlen = (int32_t)v;
    // SEQ: '*' or [A-Za-z=.]+
    if (!e && !(fn(9) == 1 && fs(9)[0] == '*')) {
      const uint8_t* s = fs(9); const uint32_t n = fn(9);
      if (n == 0) e = SAM_ERR_SEQ;
      for (uint32_t k = 0; k < n && !e; k++) { const uint8_t c = s[k] | 0x20; if (!((c >= 'a' && c <= 'z') || s[k] == '=' || s[k] == '.')) e = SAM_ERR_SEQ; }
      L.l_seq = n;
    }
    // QUAL: '*' or one of [!-~] per base
    bool q_absent = false;
    if (!e) {
      const uint8_t* s = fs(10); const uint32_t n = fn(10);
      q_absent = n == 1 && s[0] == '*';
      if (!q_absent) {
        if (n != L.l_seq) e = SAM_ERR_QUAL_LEN;
        for (uint32_t k = 0; k < n && !e; k++) if (s[k] < '!' || s[k] > '~') e = SAM_ERR_QUAL;
      }
    }
    a.qual_absent[i] = (q_absent && L.l_seq > 0) ? 1 : 0;
    total = 36u + L.l_name + 1u + 4u * L.n_ops + (L.l_seq + 1u) / 2u + L.l_seq;
    // aux fields, tab separated; a tag may appear once
    uint32_t k = L.f[11];
    uint32_t n_aux = 0;
    while (!e && k <= end) {
      uint32_t j = k;
      while (j < end && U[j] != '\t') j++;
      total += aux_bytes(U + k, j - k, &e);
      if (!e) {
        const uint8_t t0 = U[k], t1 = U[k + 1];
        for (uint32_t p = L.f[11], c = 0; c < n_aux && !e; c++) {      // earlier fields (a line has a handful; a linear check is fine)
          if (U[p] == t0 && U[p + 1] == t1) e = SAM_ERR_TAG_DUP;
          while (U[p] != '\t') p++;
          p++;
        }
      }
      n_aux++;
      k = j + 1u;
    }
  }
  if (e) { enc::report(a.err, e, i); total = 36; }
  a.sizes[i] = total;
  a.out[i] = L;
}

struct SamWriteArgs {
  const uint8_t* U;
  const SamLine* lines;
  const uint32_t* rec_off;   // [n + 1]
  uint32_t n;
  uint8_t* out;
};

template <int G>
__global__ void __launch_bounds__(256)
sam_records_kernel(const SamWriteArgs a) {
  __shared__ uint8_t base_code[256];
  for (int i = threadIdx.x; i < 256; i += blockDim.x) {
    const char* B = "=ACMGRSVTWYHKDBN";
    uint8_t c = 15;
    #pragma unroll
    for (int k = 0; k < 16; k++) if (i == B[k] || (i >= 'a' && i <= 'z' && i - 32 == B[k])) c = (uint8_t)k;
    base_code[i] = c;
  }
  __syncthreads();
  constexpr int RPW = 32 / G;
  const int lane = threadIdx.x & 31, gl = lane % G, gbase = lane - gl;
  const uint32_t gmask = G == 32 ? enc::FULLMASK : (((1u << G) - 1u) << gbase);
  const uint32_t i = ((blockIdx.x * blockDim.x + threadIdx.x) >> 5) * RPW + (uint32_t)(lane / G);
  const bool live = i < a.n;
  const uint8_t* U = a.U;
  const SamLine& L = a.lines[live ? i : 0u];
  uint8_t* const rec = a.out + (live ? a.rec_off[i] : 0u);
  const uint32_t l_name = L.l_name, n_ops = L.n_ops, l_seq = L.l_seq;
  if (live) {
    // 36 fixed bytes.  `bin` is written as 4680 (the unplaced bin) for every record: nothing downstream reads it -- the decode
    // stage and the Arrow columns take positions from pos and the CIGAR.
    uint32_t w[9];
    w[0] = a.rec_off[i + 1] - a.rec_off[i] - 4u;
    w[1] = (uint32_t)L.ref; w[2] = (uint32_t)L.pos0;
    w[3] = (l_name + 1u) | (L.mapq << 8) | (4680u << 16);
    w[4] = n_ops | (L.flag << 16);
    w[5] = l_seq; w[6] = (uint32_t)L.mref; w[7] = (uint32_t)L.mpos0; w[8] = (uint32_t)L.tlen;
    #pragma unroll
    for (int j = 0; j < 9; j++) if (j % G == gl) enc::st_u32(rec + 4 * j, w[j]);
    enc::grp_xform4<G>(rec + 36, U + L.f[0], l_name, gl, enc::OpCopy());
    if (gl == 0) rec[36 + l_name] = 0;
  }
  uint8_t* const cp = rec + 36 + l_name + 1;
  {
    // CIGAR text, G characters per step: an op character's index is the number of op characters in front of it
    const uint8_t* cig_p = U + L.f[5];
    const uint32_t cig_n = (live && n_ops) ? L.f[6] - 1u - L.f[5] : 0u;
    uint32_t steps = (cig_n + G - 1) / G;
    #pragma unroll
    for (int o = 16; o; o >>= 1) steps = max(steps, __shfl_xor_sync(enc::FULLMASK, steps, o));     // warp-uniform trip count (ballots below)
    uint32_t ops_before = 0;
    for (uint32_t s = 0; s < steps; s++) {
      const uint32_t k = s * G + gl;
      const uint8_t c = (live && k < cig_n) ? cig_p[k] : (uint8_t)'0';
      const bool is_op = !is_digit(c);
      const uint32_t bal = (__ballot_sync(enc::FULLMASK, is_op) & gmask) >> gbase;
      if (is_op) {
        const uint32_t len = (uint32_t)enc::digits_before(cig_p, k);
        const uint32_t idx = ops_before + __popc(bal & ((1u << gl) - 1u));
        if (idx < n_ops) enc::st_u32(cp + 4 * idx, (len << 4) | (uint32_t)max(enc::op_code(c), 0));
      }
      ops_before += __popc(bal);
    }
  }
  if (!live) return;
  // ---- bases (two per byte, high nibble first) + qualities
  uint8_t* const sp = cp + 4 * n_ops;
  const uint8_t* seq_p = U + L.f[9];
  const uint32_t nb = (l_seq + 1u) >> 1;
  {
    auto pack1 = [&](uint32_t k) { const uint32_t hi = base_code[seq_p[2 * k]], lo = (2 * k + 1 < l_seq) ? base_code[seq_p[2 * k + 1]] : 0u; return (uint8_t)((hi << 4) | lo); };
    const uint32_t full = l_seq >> 1;
    const uint32_t head = min(full, (uint32_t)((4u - (reinterpret_cast<uintptr_t>(sp) & 3u)) & 3u));
    if ((uint32_t)gl < head) sp[gl] = pack1(gl);
    const uint32_t nw = (full - head) >> 2;
    uint32_t* dw = reinterpret_cast<uint32_t*>(sp + head);
    const uint8_t* s8 = seq_p + 2u * head;
    for (uint32_t j = gl; j < nw; j += G) {
      const uint32_t x = enc::ldw(s8 + 8u * j), y = enc::ldw(s8 + 8u * j + 4u);
      const uint32_t b0 = (base_code[x & 0xffu] << 4) | base_code[(x >> 8) & 0xffu], b1 = (base_code[(x >> 16) & 0xffu] << 4) | base_code[x >> 24];
      const uint32_t b2 = (base_code[y & 0xffu] << 4) | base_code[(y >> 8) & 0xffu], b3 = (base_code[(y >> 16) & 0xffu] << 4) | base_code[y >> 24];
      dw[j] = b0 | (b1 << 8) | (b2 << 16) | (b3 << 24);
    }
    const uint32_t t0 = head + (nw << 2);
    if (t0 + (uint32_t)gl < nb) sp[t0 + gl] = pack1(t0 + gl);
  }
  uint8_t* const qp = sp + nb;
  const bool q_absent = L.f[11] - 1u - L.f[10] == 1u && U[L.f[10]] == '*';
  if (!q_absent) enc::grp_xform4<G>(qp, U + L.f[10], l_seq, gl, enc::OpQual());
  else { for (uint32_t k = gl; k < l_seq; k += G) qp[k] = 0xff; }
  // ---- aux fields, in line order; every lane of the group walks the field boundaries, strings are copied by the group
  uint8_t* ap = qp + l_seq;
  for (uint32_t k = L.f[11]; k <= L.end;) {
    uint32_t j = k;
    while (j < L.end && U[j] != '\t') j++;
    const uint8_t ty = U[k + 3];
    const uint8_t* v = U + k + 5;
    const uint32_t vn = j - k - 5u;
    if (gl == 0) { ap[0] = U[k]; ap[1] = U[k + 1]; }
    if (ty == 'Z' || ty == 'H') {
      if (gl == 0) { ap[2] = ty; ap[3 + vn] = 0; }
      enc::grp_xform4<G>(ap + 3, v, vn, gl, enc::OpCopy());
      ap += 3u + vn + 1u;
    } else if (ty == 'A') {
      if (gl == 0) { ap[2] = 'A'; ap[3] = v[0]; }
      ap += 4;
    } else if (ty == 'i') {
      long long x = 0; parse_int(v, vn, true, &x);
      const uint8_t t = int_type(x);
      const uint32_t es = enc::elem_size(t);
      if (gl == 0) { ap[2] = t; const uint32_t u = (uint32_t)x; ap[3] = (uint8_t)u; if (es > 1) ap[4] = (uint8_t)(u >> 8); if (es > 2) { ap[5] = (uint8_t)(u >> 16); ap[6] = (uint8_t)(u >> 24); } }
      ap += 3u + es;
    } else if (ty == 'f') {
      if (gl == 0) { uint32_t bits = 0; f32_parse(reinterpret_cast<const char*>(v), vn, &bits); ap[2] = 'f'; enc::st_u32(ap + 3, bits); }
      ap += 7;
    } else {   // 'B'
      const uint8_t st = v[0];
      const uint32_t es = enc::elem_size(st);
      uint32_t cnt = 0;
      for (uint32_t p = 1; p < vn; p++) cnt += v[p] == ',';
      if (gl == 0) {
        ap[2] = 'B'; ap[3] = st; enc::st_u32(ap + 4, cnt);
        uint8_t* ep = ap + 8;
        for (uint32_t p = 1; p < vn;) {
          uint32_t q = p + 1;
          while (q < vn && v[q] != ',') q++;
          uint32_t raw = 0;
          if (st == 'f') f32_parse(reinterpret_cast<const char*>(v + p + 1), q - p - 1, &raw);
          else { long long x = 0; parse_int(v + p + 1, q - p - 1, true, &x); raw = (uint32_t)x; }
          if (es == 1) ep[0] = (uint8_t)raw; else if (es == 2) enc::st_u16(ep, raw); else enc::st_u32(ep, raw);
          ep += es; p = q;
        }
      }
      ap += 8u + cnt * es;
    }
    k = j + 1u;
  }
}

}  // namespace sam
}  // namespace bamscan
