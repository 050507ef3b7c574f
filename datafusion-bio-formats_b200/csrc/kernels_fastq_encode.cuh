// kernels_fastq_encode.cuh -- Arrow columns -> FASTQ text on the device (the FASTQ write path), sm_100a.
//
// A row is written as '@' name [' ' description] '\n' sequence '\n' '+' '\n' quality '\n' -- the layout of the reference's
// FASTQ fixtures (bare '+' line, one space in front of the description, LF line ends).  The description and its separator are
// left out when the description is NULL or empty; the scan reads such a record back with a NULL description.
//
//   fq_enc_size_kernel     one THREAD per row: the NULL rules and the record length (offsets only: no byte is read, so long
//                          reads cost the same as short ones).
//   (exclusive scan of the lengths: dfl::len_tile_sums_kernel / len_offsets_kernel, writer.cu)
//   fq_enc_records_kernel  a GROUP of G lanes per row (G = 8: four rows per warp; 32 for long reads): the four fields go through
//                          grp_xform4_ref with destination-aligned word stores; the checks that keep the file readable as the
//                          same rows (no '\n' / '\r' in any field, no space / tab in the name) run on the words the copy loads.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

#include "kernels_encode.cuh"

namespace bamscan {
namespace fqenc {

using enc::Utf8Col;

enum FqErr : uint32_t {
  FQ_OK = 0, FQ_ERR_NULL_NAME = 1, FQ_ERR_NULL_SEQ = 2, FQ_ERR_NULL_QUAL = 3, FQ_ERR_EOL_NAME = 4, FQ_ERR_WS_NAME = 5,
  FQ_ERR_EOL_DESC = 6, FQ_ERR_EOL_SEQ = 7, FQ_ERR_EOL_QUAL = 8, FQ_ERR_REC_LEN = 9
};

struct FqArgs {
  Utf8Col name, desc, seq, qual;
  int32_t has_desc;            // 0: the input has no description column
  uint32_t row0, n_rows;       // this launch covers rows [row0, row0 + n_rows) of the batch
};

__device__ __forceinline__ uint32_t field_len(const Utf8Col& c, int64_t r) { return (uint32_t)(c.off[r + 1] - c.off[r]); }

__global__ void __launch_bounds__(256)
fq_enc_size_kernel(const FqArgs a, uint32_t* __restrict__ rec_len, uint32_t* __restrict__ err) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= a.n_rows) return;
  const uint32_t row = a.row0 + i;
  uint32_t e = FQ_OK;
  const int64_t rn = a.name.base + row, rs = a.seq.base + row, rq = a.qual.base + row;
  if (!enc::is_valid(a.name.valid, rn)) e = FQ_ERR_NULL_NAME;
  else if (!enc::is_valid(a.seq.valid, rs)) e = FQ_ERR_NULL_SEQ;
  else if (!enc::is_valid(a.qual.valid, rq)) e = FQ_ERR_NULL_QUAL;
  unsigned long long total = 6ull + field_len(a.name, rn) + field_len(a.seq, rs) + field_len(a.qual, rq);   // '@' '\n' "\n+\n" '\n'
  if (a.has_desc) {
    const int64_t rd = a.desc.base + row;
    const uint32_t dn = enc::is_valid(a.desc.valid, rd) ? field_len(a.desc, rd) : 0u;
    if (dn) total += 1ull + dn;
  }
  if (total > 0x7fffffffull && !e) e = FQ_ERR_REC_LEN;
  rec_len[i] = e ? 0u : (uint32_t)total;
  if (e) enc::report(err, e, row);
}

// Copies four bytes at a time and remembers whether any of them is a line break ('\n', '\r') or, for the name, a space or tab.
template <bool NAME>
struct OpCheckCopy {
  uint32_t eol = 0, ws = 0;
  __device__ __forceinline__ uint32_t operator()(uint32_t v) {
    eol |= __vcmpeq4(v, 0x0a0a0a0au) | __vcmpeq4(v, 0x0d0d0d0du);
    if (NAME) ws |= __vcmpeq4(v, 0x20202020u) | __vcmpeq4(v, 0x09090909u);
    return v;
  }
};

template <int G>
__global__ void __launch_bounds__(256)
fq_enc_records_kernel(const FqArgs a, const unsigned long long* __restrict__ rec_off, uint8_t* __restrict__ out, uint32_t* __restrict__ err) {
  const int lane = threadIdx.x & 31, gl = lane % G;
  const uint32_t i = ((blockIdx.x * blockDim.x + threadIdx.x) >> 5) * (32 / G) + (uint32_t)(lane / G);
  if (i >= a.n_rows) return;                                 // (no group-collective operation below)
  const uint32_t row = a.row0 + i;
  uint8_t* p = out + rec_off[i];
  const int64_t rn = a.name.base + row, rs = a.seq.base + row, rq = a.qual.base + row;
  OpCheckCopy<true> cn;
  OpCheckCopy<false> cd, cs, cq;
  {
    const uint32_t n = field_len(a.name, rn);
    if (gl == 0) p[0] = '@';
    enc::grp_xform4_ref<G>(p + 1, a.name.data + a.name.off[rn], n, gl, cn);
    p += 1 + n;
  }
  if (a.has_desc) {
    const int64_t rd = a.desc.base + row;
    const uint32_t n = enc::is_valid(a.desc.valid, rd) ? field_len(a.desc, rd) : 0u;
    if (n) {
      if (gl == 0) p[0] = ' ';
      enc::grp_xform4_ref<G>(p + 1, a.desc.data + a.desc.off[rd], n, gl, cd);
      p += 1 + n;
    }
  }
  {
    const uint32_t n = field_len(a.seq, rs);
    if (gl == 0) p[0] = '\n';
    enc::grp_xform4_ref<G>(p + 1, a.seq.data + a.seq.off[rs], n, gl, cs);
    p += 1 + n;
  }
  {
    const uint32_t n = field_len(a.qual, rq);
    if (gl == 0) { p[0] = '\n'; p[1] = '+'; p[2] = '\n'; }
    enc::grp_xform4_ref<G>(p + 3, a.qual.data + a.qual.off[rq], n, gl, cq);
    if (gl == 0) p[3 + n] = '\n';
  }
  // the group's findings, OR-ed over its lanes (all G lanes of a live row are live), decide one code per row in rule order
  uint32_t bits = (cn.eol ? 1u : 0u) | (cn.ws ? 2u : 0u) | (cd.eol ? 4u : 0u) | (cs.eol ? 8u : 0u) | (cq.eol ? 16u : 0u);
  const uint32_t gmask = G == 32 ? enc::FULLMASK : (((1u << G) - 1u) << (lane - gl));
  #pragma unroll
  for (int o = G / 2; o; o >>= 1) bits |= __shfl_xor_sync(gmask, bits, o, G);
  if (bits && gl == 0) enc::report(err, FQ_ERR_EOL_NAME + (uint32_t)(__ffs((int)bits) - 1), row);
}

}  // namespace fqenc
}  // namespace bamscan
