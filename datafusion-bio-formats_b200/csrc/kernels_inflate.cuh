// kernels_inflate.cuh -- block-parallel raw-DEFLATE (RFC 1951) inflate + CRC-32 for BGZF members.
//
// Replaces: noodles-bgzf 0.49.0 io::Reader block inflate + libdeflate `deflate_decompress`/`crc32`
// (reference call sites: datafusion/bio-format-bam/src/storage.rs:161-169, physical_exec.rs:409).
//
// Two kernels share the table builder, the header parser and the CRC code; engine.cu::launch_inflate picks one per launch:
//
//   inflate_kernel     "latency" kernel: one WARP decodes one BGZF member, 48 warps / SM.  Per-warp Huffman state in shared
//                      memory (~3.9 KB): 9-bit litlen LUT + 7-bit distance LUT of self-contained 32-bit entries, canonical
//                      (sorted-symbol) arrays for the rare longer codes.  The symbol loop is warp-uniform; LZ77 copies are
//                      done by all 32 lanes; CRC-32 of the member is computed by the same warp.  Issue bound (all 32 lanes
//                      repeat the same decode), but a member is done in ~7 ms: used for launches of up to two of its waves
//                      (region queries, tail chunks).
//   inflate_lg_kernel  "throughput" kernel: FOUR LANES decode one member, eight members per warp, 152 members / SM (16-bit
//                      LUT entries, 1456 B per member).  One pass of the predicated loop body advances every group by up to
//                      three symbols, so an issued instruction serves eight DEFLATE streams: 2.3x fewer instructions per
//                      byte.  Used for whole waves (22 496 members on a B200).  Details at its definition below.
//   crc_kernel         CRC-32 of each member after inflate_lg_kernel (one warp per member).
//
// Common: members are pulled from a global atomic ticket by a persistent grid; tables are built warp-cooperatively
// (match_any ranks, brev canonical codes, strided fill); CRC-32 is slicing-by-4 on 32 lane-chunks combined with
// x^(8k) mod P multiplies; every loop is bounded by the member's input length and ISIZE (corrupt data ends in an error code,
// never in a fault).
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

#include "inflate_cta_core.h"

namespace bamscan {

struct BlockDesc {        // one BGZF member of the chunk (host-built from the BSIZE chain)
  uint32_t cdata_off;     // byte offset of the raw-deflate payload inside the chunk's compressed buffer
  uint32_t cdata_len;     // payload bytes (BSIZE+1 - header - 8)
  uint32_t isize;         // expected inflated size (trailer ISIZE)
  uint32_t crc;           // expected CRC-32 (trailer)
  uint32_t uoff;          // offset of this member's output inside the chunk's inflated buffer
};

enum InflateStatus : uint32_t {
  INF_OK = 0, INF_ERR_BTYPE = 1, INF_ERR_STORED = 2, INF_ERR_TABLE = 3, INF_ERR_SYMBOL = 4,
  INF_ERR_DIST = 5, INF_ERR_OVERRUN = 6, INF_ERR_ISIZE = 7, INF_ERR_CRC = 8, INF_ERR_INPUT = 9
};

constexpr int INF_WARPS = 8;                 // warps per CTA
constexpr int INF_CTAS_PER_SM = 6;
#ifndef BAMSCAN_D_BITS
#define BAMSCAN_D_BITS 7
#endif
constexpr int INF_LL_BITS = 9, INF_D_BITS = BAMSCAN_D_BITS;
constexpr uint32_t FULL = 0xffffffffu;

// 32-bit LUT entry, decoded without table look-ups or branches:
//   [3:0]  code length (0 = invalid code)      [7:4] number of extra bits
//   [10:8] kind bits: 0x100 length / distance, 0x200 end of block, 0x400 code longer than the LUT index (canonical walk) or invalid
//   [30:16] literal byte | base length | base distance        [31] literal flag (sign test on the hot path)
// value = base + ((bits >> code_len) & mask(extra)) ; bits consumed = code_len + extra
constexpr uint32_t E_LIT = 0x80000000u, E_SYM = 1u << 8, E_EOB = 2u << 8, E_LONG = 4u << 8;   // one bit each: single-instruction tests

struct WarpTables {
  uint32_t lut_ll[1 << INF_LL_BITS];
  uint32_t lut_d[1 << INF_D_BITS];
  uint16_t sorted_ll[288];
  uint16_t sorted_d[32];
  uint16_t first_ll[16], offs_ll[16], cnt_ll[16];
  uint16_t first_d[16], offs_d[16], cnt_d[16];
  uint16_t nxt[16];
  uint8_t cl[320];          // code lengths being assembled (litlen then dist)
};

struct InflateShared {
  uint32_t crc_tab[4][256];
  WarpTables wt[INF_WARPS];
};

__constant__ uint8_t c_clc_order[19] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};
// x^(8 * 2^j) mod P (reflected CRC-32 domain), j = 0..17 ; filled by the host at init
__constant__ uint32_t c_crc_xpow8[18];

enum TableKind { TK_LITLEN = 0, TK_DIST = 1, TK_PRECODE = 2 };

// LUT entry of symbol `sym` with code length `len` (RFC 1951 3.2.5 base/extra tables, computed arithmetically)
template <int TK>
__device__ __forceinline__ uint32_t make_entry(uint32_t sym, uint32_t len) {
  if (TK == TK_PRECODE) return E_SYM | len | (sym << 16);
  if (TK == TK_LITLEN) {
    if (sym < 256u) return E_LIT | len | (sym << 16);
    if (sym == 256u) return E_EOB | len;
    uint32_t s = sym - 257u;
    if (s > 28u) return E_LONG;                                   // 286, 287: invalid
    uint32_t extra = (s < 8u || s == 28u) ? 0u : (s - 4u) >> 2;
    uint32_t base = s == 28u ? 258u : (s < 8u ? 3u + s : 3u + ((4u + (s & 3u)) << extra));
    return E_SYM | len | (extra << 4) | (base << 16);
  }
  if (sym > 29u) return E_LONG;
  uint32_t extra = sym < 4u ? 0u : (sym - 2u) >> 1;
  uint32_t base = sym < 4u ? 1u + sym : 1u + ((2u + (sym & 1u)) << extra);
  return E_SYM | len | (extra << 4) | (base << 16);
}

// ---------------------------------------------------------------------------------------------
// warp-uniform bit reader: every lane holds the same 64-bit window (lo:hi) plus one prefetched word.  Refills are
// plain warp-uniform loads (one 32-byte sector, L1-resident after the first touch of a line), issued one word ahead
// so their latency is off the critical path.  Invariant after init()/consume(): bp < 32 => peek() returns 32 valid bits.
struct BitReader {
  const uint32_t* base;   // 4-byte aligned start
  uint32_t lo, hi, nxt;   // words wi-3, wi-2, wi-1
  uint32_t bp;            // 0..31: position of the next unread bit inside lo
  uint32_t wi;            // index of the next word to load
  uint32_t limit_words;   // words that may legitimately be touched (+ slack)

  __device__ __forceinline__ void init(const uint8_t* p, uint32_t nbytes) {
    uintptr_t a = reinterpret_cast<uintptr_t>(p);
    base = reinterpret_cast<const uint32_t*>(a & ~uintptr_t(3));
    bp = uint32_t(a & 3) * 8;
    limit_words = (uint32_t(a & 3) + nbytes + 3) / 4 + 6;
    lo = __ldg(base); hi = __ldg(base + 1); nxt = __ldg(base + 2);
    wi = 3;
  }
  __device__ __forceinline__ uint32_t peek() const { return __funnelshift_r(lo, hi, bp); }
  __device__ __forceinline__ void consume(uint32_t n) {   // n <= 32
    bp += n;
    if (bp >= 32u) { lo = hi; hi = nxt; nxt = __ldg(base + wi); wi++; bp -= 32u; }
  }
  __device__ __forceinline__ uint32_t take(uint32_t n) {   // n < 32
    uint32_t v = peek() & ((1u << n) - 1u);
    consume(n);
    return v;
  }
  __device__ __forceinline__ bool exhausted() const { return wi > limit_words; }
  // byte address of the next unread bit (must be byte aligned)
  __device__ __forceinline__ const uint8_t* byte_ptr() const {
    return reinterpret_cast<const uint8_t*>(base + (wi - 3)) + (bp >> 3);
  }
};

// ---------------------------------------------------------------------------------------------
// Canonical Huffman table build, warp-cooperative.  cl[0..n) code lengths (0 = unused).
// Returns false when the code is over-subscribed or incomplete (icta::code_complete_ok; the code-length code must be complete).
template <int PBITS, int TK>
__device__ __forceinline__ bool build_table(const uint8_t* cl, int n, uint32_t* lut, uint16_t* sorted,
                                            uint16_t* first, uint16_t* offs, uint16_t* cnt, uint16_t* nxt, int lane) {
  if (lane < 16) { cnt[lane] = 0; nxt[lane] = 0; }
  for (int i = lane; i < (1 << PBITS); i += 32) lut[i] = E_LONG;          // kind LONG with length 0 = invalid code
  __syncwarp();
  for (int s = lane; s < n; s += 32) {
    uint32_t L = cl[s];
    if (L) atomicAdd(reinterpret_cast<unsigned int*>(cnt) + (L >> 1), (L & 1) ? 0x10000u : 1u);   // 16-bit counters packed in pairs
  }
  __syncwarp();
  // every lane derives first codes / offsets redundantly; lane == len stores its row
  uint32_t code = 0, off = 0, left = 1;
  bool over = false;
  for (int len = 1; len <= 15; len++) {
    uint32_t c = cnt[len];
    code = (code + cnt[len - 1]) << 1;
    left <<= 1;
    if (c > left) over = true;
    left -= c;
    if (lane == len) { first[len] = (uint16_t)code; offs[len] = (uint16_t)off; }
    off += c;
  }
  if (over) return false;
  if (TK == TK_PRECODE ? left != 0u : !icta::code_complete_ok(left, off, cnt[1])) return false;   // incomplete
  __syncwarp();
  const uint32_t lt = (1u << lane) - 1u;
  for (int b = 0; b < n; b += 32) {
    int s = b + lane;
    uint32_t L = (s < n) ? cl[s] : 0u;
    uint32_t m = __match_any_sync(FULL, L);
    uint32_t r = nxt[L] + __popc(m & lt);
    __syncwarp();
    if (L && (m & lt) == 0) nxt[L] = (uint16_t)(nxt[L] + __popc(m));
    __syncwarp();
    if (L) {
      sorted[offs[L] + r] = (uint16_t)s;
      uint32_t cd = first[L] + r;
      uint32_t rev = __brev(cd) >> (32 - L);
      if (L <= (uint32_t)PBITS) {
        uint32_t e = make_entry<TK>((uint32_t)s, L);
        for (uint32_t idx = rev; idx < (1u << PBITS); idx += (1u << L)) lut[idx] = e;
      } else {
        lut[rev & ((1u << PBITS) - 1u)] = E_LONG | 1u;   // long-code marker (length field != 0)
      }
    }
  }
  __syncwarp();
  return true;
}

// Canonical walk for codes longer than the LUT index.  Returns E_LONG (length 0) for an invalid code.
template <int PBITS, int TK>
__device__ __noinline__ uint32_t decode_long(uint32_t bits, const uint16_t* sorted, const uint16_t* first, const uint16_t* offs, const uint16_t* cnt) {
  uint32_t rb = __brev(bits);
  for (uint32_t len = PBITS + 1; len <= 15; len++) {
    uint32_t d = (rb >> (32 - len)) - first[len];
    if (d < cnt[len]) return make_entry<TK>(sorted[offs[len] + d], len);
  }
  return E_LONG;
}

__device__ __forceinline__ uint32_t crc_mulmod(uint32_t a, uint32_t b) {   // a*b mod P, reflected domain
  uint32_t p = 0;
  #pragma unroll 4
  for (int i = 0; i < 32; i++) {
    p ^= (b & 0x80000000u) ? a : 0u;
    a = (a >> 1) ^ ((a & 1u) ? 0xEDB88320u : 0u);
    b <<= 1;
  }
  return p;
}
__device__ __forceinline__ uint32_t crc_shift(uint32_t crc, uint32_t nbytes) {   // crc * x^(8*nbytes)
  for (int j = 0; nbytes; j++, nbytes >>= 1)
    if (nbytes & 1u) crc = crc_mulmod(crc, c_crc_xpow8[j]);
  return crc;
}

// CRC-32 (IEEE, reflected, init/final 0xffffffff) of out[0..n) by one warp.
__device__ __noinline__ uint32_t warp_crc32(const uint8_t* out, uint32_t n, const uint32_t (*tab)[256], int lane) {
  uint32_t chunk = ((n + 31) / 32 + 3) & ~3u;
  uint32_t b = min(n, chunk * lane), e = min(n, b + chunk);
  uint32_t st = (lane == 0) ? 0xffffffffu : 0u;
  const uint8_t* p = out + b;
  uint32_t len = e - b;
  while (len && (reinterpret_cast<uintptr_t>(p) & 3)) { st = tab[0][(st ^ *p) & 0xff] ^ (st >> 8); p++; len--; }
  const uint32_t* pw = reinterpret_cast<const uint32_t*>(p);
#define CRC_WORD(w) { st ^= (w); st = tab[3][st & 0xff] ^ tab[2][(st >> 8) & 0xff] ^ tab[1][(st >> 16) & 0xff] ^ tab[0][st >> 24]; }
  for (; len >= 4 && (reinterpret_cast<uintptr_t>(pw) & 15); len -= 4) CRC_WORD(*pw++);
  for (; len >= 16; len -= 16) {                            // 16-byte loads: a quarter of the load instructions, next one in flight
    const uint4 v = *reinterpret_cast<const uint4*>(pw); pw += 4;
    CRC_WORD(v.x); CRC_WORD(v.y); CRC_WORD(v.z); CRC_WORD(v.w);
  }
  for (; len >= 4; len -= 4) CRC_WORD(*pw++);
#undef CRC_WORD
  p = reinterpret_cast<const uint8_t*>(pw);
  while (len) { st = tab[0][(st ^ *p) & 0xff] ^ (st >> 8); p++; len--; }
  st = crc_shift(st, n - e);
  #pragma unroll
  for (int o = 16; o; o >>= 1) st ^= __shfl_xor_sync(FULL, st, o);
  return ~st;
}

// Reads the dynamic-block header (HLIT/HDIST/HCLEN + code lengths) into T.cl.  Returns an InflateStatus.
template <class TT>
__device__ __forceinline__ uint32_t read_dynamic_header(BitReader& br, TT& T, int lane, int* n_ll_out, int* n_d_out) {
  uint32_t h = br.take(14);
  int n_ll = (int)(h & 31u) + 257, n_d = (int)((h >> 5) & 31u) + 1;
  int n_clc = (int)(h >> 10) + 4;
  if (n_ll > 286 || n_d > 30) return INF_ERR_TABLE;
  if (lane < 19) T.cl[lane] = 0;
  __syncwarp();
  for (int i = 0; i < n_clc; i++) {
    uint32_t v = br.take(3);
    if (lane == 0) T.cl[c_clc_order[i]] = (uint8_t)v;
  }
  __syncwarp();
  // pre-code (max length 7) goes into lut_d; the decoded lengths then overwrite cl[]
  if (!build_table<7, TK_PRECODE>(T.cl, 19, T.lut_d, T.sorted_d, T.first_d, T.offs_d, T.cnt_d, T.nxt, lane)) return INF_ERR_TABLE;
  int total = n_ll + n_d, i = 0;
  uint32_t prev = 0;
  while (i < total) {
    uint32_t bits = br.peek();
    uint32_t e = T.lut_d[bits & 127u];
    uint32_t L = e & 15u, s = e >> 16;
    if (L == 0) return INF_ERR_TABLE;
    uint32_t rep, val, xb;
    if (s < 16) { rep = 1; val = s; prev = s; xb = 0; }
    else if (s == 16) { if (i == 0) return INF_ERR_TABLE; xb = 2; rep = 3 + ((bits >> L) & 3u); val = prev; }
    else if (s == 17) { xb = 3; rep = 3 + ((bits >> L) & 7u); val = 0; prev = 0; }
    else { xb = 7; rep = 11 + ((bits >> L) & 127u); val = 0; prev = 0; }
    br.consume(L + xb);
    if (i + (int)rep > total) return INF_ERR_TABLE;
    for (uint32_t k = lane; k < rep; k += 32) T.cl[i + k] = (uint8_t)val;
    i += (int)rep;
  }
  __syncwarp();
  if (T.cl[256] == 0) return INF_ERR_TABLE;
  *n_ll_out = n_ll; *n_d_out = n_d;
  return INF_OK;
}

// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(INF_WARPS * 32, INF_CTAS_PER_SM)
inflate_kernel(const uint8_t* __restrict__ comp, const BlockDesc* __restrict__ blocks, uint32_t n_blocks,
               uint8_t* __restrict__ infl, uint32_t* __restrict__ status, uint32_t* __restrict__ ticket,
               uint32_t* __restrict__ err_flag, int check_crc, uint32_t only_status) {
  // only_status != 0xffffffff: redo only the members whose status[] holds that value (the CTA-per-member kernel's INF_RETRY)
  extern __shared__ __align__(16) unsigned char smem_raw[];
  InflateShared& sh = *reinterpret_cast<InflateShared*>(smem_raw);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  // CRC tables (slicing-by-4)
  for (int i = threadIdx.x; i < 256; i += blockDim.x) {
    uint32_t c = (uint32_t)i;
    for (int k = 0; k < 8; k++) c = (c >> 1) ^ ((c & 1u) ? 0xEDB88320u : 0u);
    sh.crc_tab[0][i] = c;
  }
  __syncthreads();
  for (int i = threadIdx.x; i < 256; i += blockDim.x) {
    uint32_t c = sh.crc_tab[0][i];
    for (int t = 1; t < 4; t++) { c = sh.crc_tab[0][c & 0xff] ^ (c >> 8); sh.crc_tab[t][i] = c; }
  }
  __syncthreads();
  WarpTables& T = sh.wt[warp];
  const bool lane0 = lane == 0;

  for (;;) {
    uint32_t bi = 0;
    if (lane0) bi = atomicAdd(ticket, 1u);
    bi = __shfl_sync(FULL, bi, 0);
    if (bi >= n_blocks) break;
    if (only_status != 0xffffffffu && status[bi] != only_status) continue;
    const BlockDesc bd = blocks[bi];
    uint8_t* const out = infl + bd.uoff;
    const uint32_t isize = bd.isize;
    uint32_t outpos = 0, err = INF_OK;
    BitReader br;
    br.init(comp + bd.cdata_off, bd.cdata_len);
    const uint32_t obase = bd.uoff;                 // infl[obase + k]: uniform base + 32-bit offset addressing
    bool final_block = false;

    while (!final_block && err == INF_OK) {
      if (br.exhausted()) { err = INF_ERR_INPUT; break; }   // every path below consumes input, so this bounds the loop
      uint32_t hdr = br.take(3);
      final_block = hdr & 1u;
      uint32_t btype = hdr >> 1;
      if (btype == 0) {
        // stored: skip to byte boundary, LEN / NLEN, raw copy
        br.consume((8 - (br.bp & 7)) & 7);
        uint32_t len = br.take(16), nlen = br.take(16);
        if ((len ^ nlen) != 0xffffu || outpos + len > isize) { err = INF_ERR_STORED; break; }
        const uint8_t* src = br.byte_ptr();
        uint32_t used = (uint32_t)(src + len - (comp + bd.cdata_off));
        if (used > bd.cdata_len) { err = INF_ERR_INPUT; break; }
        for (uint32_t i = lane; i < len; i += 32) out[outpos + i] = src[i];
        outpos += len;
        br.init(src + len, bd.cdata_len - used);
        continue;
      }
      if (btype == 3) { err = INF_ERR_BTYPE; break; }
      int n_ll = 288, n_d = 32;
      if (btype == 1) {
        for (int i = lane; i < 288; i += 32) T.cl[i] = i < 144 ? 8 : i < 256 ? 9 : i < 280 ? 7 : 8;
        T.cl[288 + lane] = 5;                          // all 32 distance codes: complete, and 30 / 31 decode as invalid
        __syncwarp();
      } else {
        err = read_dynamic_header(br, T, lane, &n_ll, &n_d);
        if (err) break;
      }
      if (!build_table<INF_LL_BITS, TK_LITLEN>(T.cl, n_ll, T.lut_ll, T.sorted_ll, T.first_ll, T.offs_ll, T.cnt_ll, T.nxt, lane)) { err = INF_ERR_TABLE; break; }
      if (!build_table<INF_D_BITS, TK_DIST>(T.cl + n_ll, n_d, T.lut_d, T.sorted_d, T.first_d, T.offs_d, T.cnt_d, T.nxt, lane)) { err = INF_ERR_TABLE; break; }

      // ---------------- symbol loop (warp-uniform; one look-up decodes code + extra bits) ----------------
      // The reader state lives in plain registers here; refills are real (rare) branches so the common path stays short.
      // Output overrun is checked at every match and at the end of the member (the inflated buffer carries slack for
      // literal runs); the loop is bounded by the input: the refill path stops at the member's last word (+ slack).
      {
        uint32_t lo = br.lo, hi = br.hi, nxt = br.nxt, bp = br.bp, wi = br.wi;
        const uint32_t* const wbase = br.base;
        const uint32_t wlimit = br.limit_words;
        const uint32_t* const lut_ll = T.lut_ll;
        const uint32_t* const lut_d = T.lut_d;
        uint8_t* outl = infl + obase + outpos + lane;        // this lane's byte of the next output stripe
#define INF_REFILL()                                                                         \
        if (bp >= 32u) {                                                                     \
          lo = hi; hi = nxt; nxt = __ldg(wbase + wi); wi++; bp -= 32u;                        \
          if (wi > wlimit) { err = INF_ERR_INPUT; break; }                                    \
        }
        for (;;) {
          uint32_t bits = __funnelshift_r(lo, hi, bp);
          uint32_t e = lut_ll[bits & ((1u << INF_LL_BITS) - 1u)];
          if ((int32_t)e < 0) {                                // literal
            if (lane0) *outl = (uint8_t)(e >> 16);
            outl++; outpos++;
            bp += e & 15u;
            INF_REFILL();
            continue;
          }
          if (!(e & E_SYM)) {                                  // rare: code longer than the LUT index, end of block, invalid code
            if (e & E_LONG) {
              e = decode_long<INF_LL_BITS, TK_LITLEN>(bits, T.sorted_ll, T.first_ll, T.offs_ll, T.cnt_ll);
              if ((int32_t)e < 0) {
                if (lane0) *outl = (uint8_t)(e >> 16);
                outl++; outpos++;
                bp += e & 15u;
                INF_REFILL();
                continue;
              }
            }
            if (!(e & E_SYM)) {
              bp += e & 15u;
              if ((e & 15u) == 0) err = INF_ERR_SYMBOL;
              break;
            }
          }
          {
            const uint32_t nb = e & 15u, xb = (e >> 4) & 15u;
            const uint32_t len = (e >> 16) + ((bits >> nb) & ((1u << xb) - 1u));
            bp += nb + xb;
            INF_REFILL();
            bits = __funnelshift_r(lo, hi, bp);
            uint32_t de = lut_d[bits & ((1u << INF_D_BITS) - 1u)];
            if (de & E_LONG) de = decode_long<INF_D_BITS, TK_DIST>(bits, T.sorted_d, T.first_d, T.offs_d, T.cnt_d);
            const uint32_t dnb = de & 15u, dxb = (de >> 4) & 15u;
            const uint32_t dist = (de >> 16) + ((bits >> dnb) & ((1u << dxb) - 1u));
            bp += dnb + dxb;
            if (dnb == 0 || dist > outpos || outpos + len > isize) { err = (dnb == 0 || dist > outpos) ? INF_ERR_DIST : INF_ERR_OVERRUN; break; }
            __syncwarp();                                   // earlier stores (other lanes) become visible to the loads below
            // byte i of the match is src[i mod dist]: only bytes that already exist are read, whatever dist/len are
            if (dist >= len && len <= 32u) {                // the common case: one stripe, no overlap
              const uint8_t v = *(outl - dist);
              if ((uint32_t)lane < len) *outl = v;
            } else {
              uint8_t* const d0 = outl - lane;
              const uint8_t* const s0 = d0 - dist;
              if (dist >= len) { for (uint32_t i = lane; i < len; i += 32) d0[i] = s0[i]; }
              else if (dist == 1) { const uint8_t v = s0[0]; for (uint32_t i = lane; i < len; i += 32) d0[i] = v; }
              else { for (uint32_t i = lane; i < len; i += 32) d0[i] = s0[i % dist]; }
            }
            outl += len; outpos += len;
            INF_REFILL();
          }
        }
#undef INF_REFILL
        br.lo = lo; br.hi = hi; br.nxt = nxt; br.bp = bp; br.wi = wi;
        // normalise (a block may end with bp in [32, 47))
        if (br.bp >= 32u) { br.lo = br.hi; br.hi = br.nxt; br.nxt = __ldg(br.base + br.wi); br.wi++; br.bp -= 32u; }
      }
      if (br.exhausted() && err == INF_OK) err = INF_ERR_INPUT;
    }
    __syncwarp();
    if (err == INF_OK && outpos != isize) err = outpos > isize ? INF_ERR_OVERRUN : INF_ERR_ISIZE;
    if (err == INF_OK && check_crc) {
      uint32_t crc = warp_crc32(out, isize, sh.crc_tab, lane);
      if (crc != bd.crc) err = INF_ERR_CRC;
    }
    if (lane0) {
      status[bi] = err;
      if (err) atomicCAS(err_flag, 0u, (bi << 4) | err | 0x80000000u);
    }
    __syncwarp();
  }
}

// =============================================================================================
// Lane-group inflate.  The warp-per-member kernel above spends all 32 lanes' issue slots on ONE symbol at a time and is
// issue bound.  Here a warp carries 32/G members at once: G lanes form a group that owns one member, every lane of a
// group holds the same reader state, and one pass through the (warp-uniform, predicated) loop body decodes up to
// NLIT + 1 symbols for EVERY group, so an instruction issued once advances 32/G independent DEFLATE streams.  The G
// lanes of a group share the LZ77 copy: it is cut into chunks of <= 16 bytes per pass (a longer copy continues in the next
// pass instead of decoding), the source bytes are loaded into registers and stored two match passes later (two ping-pong
// slots; a chunk that would read bytes still held in a slot retires the slots first), so the L2 / DRAM round trip of
// the history read overlaps the following Huffman decode.  The compressed stream is read through a 64-byte shared-memory
// ring per member that is topped up through a register one pass ahead.  Tables are 16-bit entries; with the canonical
// rows and the ring a member needs 1456 B, so 152 members fit in one SM's shared memory.  The rare canonical walk for
// codes longer than the LUT index takes its rows from shared memory and the symbol entry from a small global scratch (L2).
// Block headers, table builds, stored blocks and member hand-over are done by the whole warp for one group at a time
// (`service`), exactly as parallel as in the warp-per-member kernel.  CRC-32 moves to crc_kernel.
//
// 16-bit LUT entries:
//   litlen  literal : 0x8000 | byte << 4 | nb                       length : (base - 3) << 7 | xb << 4 | nb   (xb <= 5)
//           end of block : 0x0070 | nb        not in the LUT (longer code / unused prefix) : 0x0060
//   dist    m << 8 | xb << 4 | nb  with distance = 1 + (m << xb) + extra            not in the LUT : 0
//   precode sym << 4 | nb
constexpr uint32_t L16_LIT = 0x8000u, L16_EOB = 0x0070u, L16_MISS = 0x0060u;
constexpr int LG_SORTED = 320;                    // u16 entries per member slot: 288 litlen + 32 distance
constexpr int LG_SLOT_BYTES = LG_SORTED * 2;                 // global scratch per member slot: sorted16[]
constexpr int LG_RING_BYTES = 64;                // compressed-stream ring per member: four 16-byte chunks
constexpr int LG_CANON_LL = 15 - INF_LL_BITS, LG_CANON_D = 15 - INF_D_BITS;   // canonical rows kept in shared memory (lengths above the LUT index)

template <int TK>
__device__ __forceinline__ uint32_t make_entry16(uint32_t sym, uint32_t len) {
  if (TK == TK_PRECODE) return (sym << 4) | len;
  if (TK == TK_LITLEN) {
    if (sym < 256u) return L16_LIT | (sym << 4) | len;
    if (sym == 256u) return L16_EOB | len;
    uint32_t s = sym - 257u;
    if (s > 28u) return L16_MISS;
    uint32_t extra = (s < 8u || s == 28u) ? 0u : (s - 4u) >> 2;
    uint32_t base = s == 28u ? 258u : (s < 8u ? 3u + s : 3u + ((4u + (s & 3u)) << extra));
    return ((base - 3u) << 7) | (extra << 4) | len;
  }
  if (sym > 29u) return 0u;
  uint32_t extra = sym < 4u ? 0u : (sym - 2u) >> 1;
  uint32_t m = sym < 4u ? sym : 2u + (sym & 1u);
  return (m << 8) | (extra << 4) | len;
}

struct WarpScratch16 {
  uint16_t nxt[16], cnt[16], first[16], offs[16];
  uint8_t cl[320];
};

// Canonical Huffman build into a 16-bit LUT + the long-code arrays (canon[len] = first | cnt << 16 | offs << 32, sorted16[]).
template <int PBITS, int TK>
__device__ __forceinline__ bool build_table16(const uint8_t* cl, int n, uint16_t* lut, uint16_t* sorted, unsigned long long* canon,
                                              WarpScratch16& S, int lane) {
  constexpr uint32_t MISS = TK == TK_LITLEN ? L16_MISS : 0u;
  if (lane < 16) { S.cnt[lane] = 0; S.nxt[lane] = 0; }
  for (int i = lane; i < (1 << PBITS) / 2; i += 32) reinterpret_cast<uint32_t*>(lut)[i] = MISS | (MISS << 16);
  __syncwarp();
  for (int s = lane; s < n; s += 32) {
    uint32_t L = cl[s];
    if (L) atomicAdd(reinterpret_cast<unsigned int*>(S.cnt) + (L >> 1), (L & 1) ? 0x10000u : 1u);
  }
  __syncwarp();
  uint32_t code = 0, off = 0, left = 1;
  bool over = false;
  for (int len = 1; len <= 15; len++) {
    uint32_t c = S.cnt[len];
    code = (code + S.cnt[len - 1]) << 1;
    left <<= 1;
    if (c > left) over = true;
    left -= c;
    if (lane == len) {
      S.first[len] = (uint16_t)code; S.offs[len] = (uint16_t)off;
      if (len > PBITS) canon[len - PBITS - 1] = (unsigned long long)code | ((unsigned long long)c << 16) | ((unsigned long long)off << 32);
    }
    off += c;
  }
  if (over) return false;
  if (TK == TK_PRECODE ? left != 0u : !icta::code_complete_ok(left, off, S.cnt[1])) return false;   // incomplete
  __syncwarp();
  const uint32_t lt = (1u << lane) - 1u;
  for (int b = 0; b < n; b += 32) {
    int s = b + lane;
    uint32_t L = (s < n) ? cl[s] : 0u;
    uint32_t m = __match_any_sync(FULL, L);
    uint32_t r = S.nxt[L] + __popc(m & lt);
    __syncwarp();
    if (L && (m & lt) == 0) S.nxt[L] = (uint16_t)(S.nxt[L] + __popc(m));
    __syncwarp();
    if (L) {
      const uint32_t e = make_entry16<TK>((uint32_t)s, L);
      sorted[S.offs[L] + r] = (uint16_t)e;
      uint32_t cd = S.first[L] + r;
      uint32_t rev = __brev(cd) >> (32 - L);
      if (L <= (uint32_t)PBITS)
        for (uint32_t idx = rev; idx < (1u << PBITS); idx += (1u << L)) lut[idx] = (uint16_t)e;
    }
  }
  __syncwarp();
  return true;
}

__device__ __forceinline__ uint32_t lds_u16(uint32_t saddr) { uint16_t v; asm volatile("ld.shared.u16 %0, [%1];" : "=h"(v) : "r"(saddr)); return v; }
__device__ __forceinline__ unsigned long long lds_u64(uint32_t saddr) { unsigned long long v; asm volatile("ld.shared.u64 %0, [%1];" : "=l"(v) : "r"(saddr)); return v; }

// Canonical walk for codes longer than the LUT index; returns the 16-bit entry, or the "miss" value for an invalid code.
// canon_s: shared-window address of the rows first | cnt << 16 | offs << 32 for lengths PBITS+1 .. 15.
template <int PBITS, int TK>
__device__ __forceinline__ uint32_t decode_long16(uint32_t bits, uint32_t canon_s, const uint16_t* __restrict__ sorted) {
  const uint32_t c15 = __brev(bits) >> 17;
  #pragma unroll
  for (int len = PBITS + 1; len <= 15; len++) {
    const unsigned long long q = lds_u64(canon_s + 8u * (uint32_t)(len - PBITS - 1));
    const uint32_t d = (c15 >> (15 - len)) - (uint32_t)(q & 0xffffu);
    if (d < (uint32_t)((q >> 16) & 0xffffu)) return sorted[(uint32_t)(q >> 32) + d];
  }
  return TK == TK_LITLEN ? L16_MISS : 0u;
}

struct Tables16 { uint16_t* lut_ll; uint16_t* lut_d; uint16_t* sorted_ll; uint16_t* sorted_d; unsigned long long* canon_ll; unsigned long long* canon_d; };

__device__ __forceinline__ uint32_t read_dynamic_header16(BitReader& br, const Tables16& T, WarpScratch16& S, int lane, int* n_ll_out, int* n_d_out) {
  uint32_t h = br.take(14);
  int n_ll = (int)(h & 31u) + 257, n_d = (int)((h >> 5) & 31u) + 1;
  int n_clc = (int)(h >> 10) + 4;
  if (n_ll > 286 || n_d > 30) return INF_ERR_TABLE;
  if (lane < 19) S.cl[lane] = 0;
  __syncwarp();
  for (int i = 0; i < n_clc; i++) {
    uint32_t v = br.take(3);
    if (lane == 0) S.cl[c_clc_order[i]] = (uint8_t)v;
  }
  __syncwarp();
  // pre-code (max length 7) goes into the distance LUT; the decoded lengths then overwrite cl[]
  if (!build_table16<7, TK_PRECODE>(S.cl, 19, T.lut_d, T.sorted_d, T.canon_d, S, lane)) return INF_ERR_TABLE;
  int total = n_ll + n_d, i = 0;
  uint32_t prev = 0;
  while (i < total) {
    uint32_t bits = br.peek();
    uint32_t e = T.lut_d[bits & 127u];
    uint32_t L = e & 15u, s = e >> 4;
    if (L == 0) return INF_ERR_TABLE;
    uint32_t rep, val, xb;
    if (s < 16) { rep = 1; val = s; prev = s; xb = 0; }
    else if (s == 16) { if (i == 0) return INF_ERR_TABLE; xb = 2; rep = 3 + ((bits >> L) & 3u); val = prev; }
    else if (s == 17) { xb = 3; rep = 3 + ((bits >> L) & 7u); val = 0; prev = 0; }
    else { xb = 7; rep = 11 + ((bits >> L) & 127u); val = 0; prev = 0; }
    br.consume(L + xb);
    if (i + (int)rep > total) return INF_ERR_TABLE;
    for (uint32_t k = lane; k < rep; k += 32) S.cl[i + k] = (uint8_t)val;
    i += (int)rep;
  }
  __syncwarp();
  if (S.cl[256] == 0) return INF_ERR_TABLE;
  *n_ll_out = n_ll; *n_d_out = n_d;
  return INF_OK;
}

template <int G, int W> struct LgConfig {
  static constexpr int GROUPS = 32 / G;
  static constexpr int THREADS = W * 32;
  static constexpr size_t LUT_BYTES = 2 * ((1 << INF_LL_BITS) + (1 << INF_D_BITS));
  static constexpr size_t RING_OFF = LUT_BYTES + 8 * (LG_CANON_LL + LG_CANON_D);
  static constexpr size_t MEMBER_SMEM = RING_OFF + LG_RING_BYTES;
  static constexpr size_t SMEM = (size_t)W * (GROUPS * MEMBER_SMEM + sizeof(WarpScratch16));
};

enum : uint32_t { ST_SYMBOLS = 0, ST_HEADER = 1, ST_MEMBER = 2, ST_DONE = 3 };

template <int G, int W, int NLIT, int CTAS>
__global__ void __launch_bounds__(W * 32, CTAS)
inflate_lg_kernel(const uint8_t* __restrict__ comp, const BlockDesc* __restrict__ blocks, uint32_t n_blocks,
                  uint8_t* __restrict__ infl, uint32_t* __restrict__ status, uint32_t* __restrict__ ticket,
                  uint32_t* __restrict__ err_flag, uint8_t* __restrict__ slot_scratch) {
  constexpr int GROUPS = 32 / G;
  constexpr int U = (16 / G) < 1 ? 1 : (16 / G);                 // deferred bytes per lane: one pass covers 16 bytes
  constexpr uint32_t LLMASK = (1u << INF_LL_BITS) - 1u, DMASK = (1u << INF_D_BITS) - 1u;
  constexpr uint32_t MEMBER_SMEM = (uint32_t)LgConfig<G, W>::MEMBER_SMEM;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int grp = lane / G;
  int glane = lane % G;
  asm volatile("" : "+r"(glane));                               // keep it in a register (the compiler would re-read %tid in every pass)
  unsigned char* const wtab = smem_raw + (size_t)warp * GROUPS * MEMBER_SMEM;
  WarpScratch16& WS = *reinterpret_cast<WarpScratch16*>(smem_raw + (size_t)W * GROUPS * MEMBER_SMEM + (size_t)warp * sizeof(WarpScratch16));
  uint8_t* const wslots = slot_scratch + (size_t)(blockIdx.x * W + warp) * GROUPS * LG_SLOT_BYTES;
  uint32_t ll_s = (uint32_t)__cvta_generic_to_shared(wtab + grp * MEMBER_SMEM);   // shared-window address of this group's tables
  asm volatile("" : "+r"(ll_s));
#define LL16(i) lds_u16(ll_s + ((i) << 1))
#define D16(i) lds_u16(ll_s + (2u << INF_LL_BITS) + ((i) << 1))
  unsigned long long my_slot_bits = reinterpret_cast<unsigned long long>(wslots + (size_t)grp * LG_SLOT_BYTES);
  asm volatile("" : "+l"(my_slot_bits));                        // opaque: keep it in registers instead of re-deriving it every pass
  const uint16_t* const my_sorted = reinterpret_cast<const uint16_t*>(my_slot_bits);
  const uint32_t my_canon = ll_s + (uint32_t)LgConfig<G, W>::LUT_BYTES;     // shared-window address of the canonical rows

  // member state, replicated over the G lanes of the group
  const uint32_t* wbase = reinterpret_cast<const uint32_t*>(blocks);   // any valid, aligned address until a member is taken
  // reader: lo:hi hold the two current words; the following words come from the member's shared-memory ring, which is
  // kept 2-3 chunks ahead by loads that are given a whole pass to complete (see the ring top-up at the end of a pass).
  // wbase is 16-byte aligned; wi = index (from wbase) of the word after hi; fill = next 16-byte chunk to fetch.
  uint32_t lo = 0, hi = 0, bp = 0, wi = 0, wlimit = 0, fill = 0;
  uint32_t rq[4 / G + (4 % G != 0)], rq_slot = 0xffffffffu;     // ring chunk in flight (one word per lane) and its slot
  const uint32_t my_ring = ll_s + (uint32_t)LgConfig<G, W>::RING_OFF;
  uint32_t outpos = 0, isize = 0, bi = 0, err = INF_OK, state = ST_MEMBER, final_block = 0;
  uint8_t* obase = infl;
  // deferred copy: U bytes per lane loaded in the previous pass, not yet stored
  // two deferred copies per group (q0 older, q1 newer): position in the member, length, U bytes per lane
  uint32_t ppos0 = 0, plen0 = 0, ppos1 = 0, plen1 = 0; uint8_t pv0[U], pv1[U];
  uint32_t rem = 0, cdist = 0;                                  // a copy longer than one chunk continues in the next passes
  uint32_t tog = 0;                                             // warp-uniform: which deferred slot is the older one
  #pragma unroll
  for (int k = 0; k < U; k++) { pv0[k] = 0; pv1[k] = 0; }

  for (;;) {
    // ---------------- service: one group at a time, whole warp ----------------
    uint32_t need = __ballot_sync(FULL, state == ST_HEADER || state == ST_MEMBER);
    while (need) {
      const int src = __ffs(need) - 1;               // first lane of the group
      const int g = src / G;
      need &= ~(((G == 32) ? FULL : ((1u << G) - 1u)) << (g * G));
      BitReader br;
      {
        unsigned long long a = reinterpret_cast<unsigned long long>(wbase);
        a = __shfl_sync(FULL, a, src);
        br.base = reinterpret_cast<const uint32_t*>(a);
      }
      br.lo = __shfl_sync(FULL, lo, src); br.hi = __shfl_sync(FULL, hi, src);
      br.bp = __shfl_sync(FULL, bp, src); br.wi = __shfl_sync(FULL, wi, src); br.limit_words = __shfl_sync(FULL, wlimit, src) + 1u;
      br.nxt = __ldg(br.base + br.wi); br.wi += 1u;          // back to the three-word reader of the header code
      uint32_t s_outpos = __shfl_sync(FULL, outpos, src), s_isize = __shfl_sync(FULL, isize, src), s_bi = __shfl_sync(FULL, bi, src);
      uint32_t s_err = __shfl_sync(FULL, err, src), s_state = __shfl_sync(FULL, state, src), s_final = __shfl_sync(FULL, final_block, src);
      unsigned long long s_ob = __shfl_sync(FULL, reinterpret_cast<unsigned long long>(obase), src);
      uint8_t* s_obase = reinterpret_cast<uint8_t*>(s_ob);
      Tables16 T;
      T.lut_ll = reinterpret_cast<uint16_t*>(wtab + g * MEMBER_SMEM); T.lut_d = T.lut_ll + (1 << INF_LL_BITS);
      T.canon_ll = reinterpret_cast<unsigned long long*>(wtab + g * MEMBER_SMEM + LgConfig<G, W>::LUT_BYTES); T.canon_d = T.canon_ll + LG_CANON_LL;
      T.sorted_ll = reinterpret_cast<uint16_t*>(wslots + (size_t)g * LG_SLOT_BYTES); T.sorted_d = T.sorted_ll + 288;

      for (;;) {
        if (s_state == ST_MEMBER) {
          uint32_t t = 0;
          if (lane == 0) t = atomicAdd(ticket, 1u);
          t = __shfl_sync(FULL, t, 0);
          if (t >= n_blocks) { s_state = ST_DONE; break; }
          const BlockDesc bd = blocks[t];
          s_bi = t; s_obase = infl + bd.uoff; s_isize = bd.isize; s_outpos = 0; s_final = 0; s_err = INF_OK;
          br.init(comp + bd.cdata_off, bd.cdata_len);
          s_state = ST_HEADER;
        }
        if (s_err == INF_OK && s_final && s_outpos != s_isize) s_err = s_outpos > s_isize ? INF_ERR_OVERRUN : INF_ERR_ISIZE;
        if (s_err != INF_OK || s_final) {             // member finished (or failed): publish, take the next one
          if (lane == 0) {
            status[s_bi] = s_err;
            if (s_err) atomicCAS(err_flag, 0u, (s_bi << 4) | s_err | 0x80000000u);
          }
          s_state = ST_MEMBER;
          continue;
        }
        if (br.exhausted()) { s_err = INF_ERR_INPUT; continue; }
        const uint32_t hdr = br.take(3);
        s_final = hdr & 1u;
        const uint32_t btype = hdr >> 1;
        if (btype == 0) {
          br.consume((8 - (br.bp & 7)) & 7);
          const uint32_t len = br.take(16), nlen = br.take(16);
          if ((len ^ nlen) != 0xffffu || s_outpos + len > s_isize) { s_err = INF_ERR_STORED; continue; }
          const BlockDesc bd = blocks[s_bi];
          const uint8_t* sp = br.byte_ptr();
          const uint32_t used = (uint32_t)(sp + len - (comp + bd.cdata_off));
          if (used > bd.cdata_len) { s_err = INF_ERR_INPUT; continue; }
          for (uint32_t i = lane; i < len; i += 32) s_obase[s_outpos + i] = sp[i];
          s_outpos += len;
          br.init(sp + len, bd.cdata_len - used);
          continue;
        }
        if (btype == 3) { s_err = INF_ERR_BTYPE; continue; }
        int n_ll = 288, n_d = 32;
        __syncwarp();
        if (btype == 1) {
          for (int i = lane; i < 288; i += 32) WS.cl[i] = i < 144 ? 8 : i < 256 ? 9 : i < 280 ? 7 : 8;
          WS.cl[288 + lane] = 5;                         // all 32 distance codes: complete, and 30 / 31 decode as invalid
          __syncwarp();
        } else {
          s_err = read_dynamic_header16(br, T, WS, lane, &n_ll, &n_d);
          if (s_err) continue;
        }
        if (!build_table16<INF_LL_BITS, TK_LITLEN>(WS.cl, n_ll, T.lut_ll, T.sorted_ll, T.canon_ll, WS, lane)) { s_err = INF_ERR_TABLE; continue; }
        if (!build_table16<INF_D_BITS, TK_DIST>(WS.cl + n_ll, n_d, T.lut_d, T.sorted_d, T.canon_d, WS, lane)) { s_err = INF_ERR_TABLE; continue; }
        s_state = ST_SYMBOLS;
        break;
      }
      // re-base the reader on a 16-byte boundary and prime the ring with the first three chunks
      const uint32_t* s_wbase; uint32_t s_wi, s_wlimit;
      {
        const uint32_t* const plo = br.base + (br.wi - 3u);                   // the word held in lo
        const unsigned long long a16 = reinterpret_cast<unsigned long long>(plo) & ~15ull;
        const uint32_t k0 = (uint32_t)((reinterpret_cast<unsigned long long>(plo) - a16) >> 2);
        s_wbase = reinterpret_cast<const uint32_t*>(a16);
        s_wi = k0 + 2u;
        s_wlimit = br.limit_words - ((br.wi - 3u) - k0) - 1u;
        uint32_t* const rg = reinterpret_cast<uint32_t*>(wtab + g * MEMBER_SMEM + LgConfig<G, W>::RING_OFF);
        if (s_state == ST_SYMBOLS && lane < 12) rg[lane] = __ldg(s_wbase + lane);
      }
      if (grp == g) {
        wbase = s_wbase; lo = br.lo; hi = br.hi; bp = br.bp; wi = s_wi; wlimit = s_wlimit; fill = 3u; rq_slot = 0xffffffffu;
        outpos = s_outpos; isize = s_isize; bi = s_bi; err = s_err; state = s_state; final_block = s_final; obase = s_obase; rem = 0;
      }
      __syncwarp();
    }
    if (__all_sync(FULL, state == ST_DONE)) break;

    // ---------------- symbols: every group advances by up to NLIT + 1 symbols per pass ----------------
    // Branch-free refill from the ring: bp < 64 here.
#define LG_REFILL()                                                                                              \
    {                                                                                                            \
      const bool rf = bp >= 32u;                                                                                 \
      lo = rf ? hi : lo;                                                                                         \
      asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.u32 p, %1, 0;\n\t@p ld.shared.u32 %0, [%2];\n\t}"              \
                   : "+r"(hi) : "r"((uint32_t)rf), "r"(my_ring + ((wi & 15u) << 2)));                             \
      wi += bp >> 5; bp &= 31u;                                                                                  \
    }
#define LG_STORE(PPOS, PLEN, PV)                                                                                 \
    if (PLEN) {                                                                                                  \
      uint8_t* const pd = obase + PPOS + glane;                                                                  \
      _Pragma("unroll")                                                                                          \
      for (int k = 0; k < U; k++) if ((uint32_t)(glane + k * G) < PLEN) pd[k * G] = PV[k];                       \
      PLEN = 0;                                                                                                  \
    }
    // One chunk (<= U*G bytes per group) of LZ77 copy.  Slot X holds the copy deferred two match passes ago: it is stored
    // now and refilled with this pass's loads; slot Y (one pass old) is stored too only when a new chunk reads bytes that
    // are still deferred.  Byte i of a chunk is src[i mod dist], so only bytes that already exist are ever read.
#define LG_COPY(PX, LX, VX, PY, LY, VY)                                                                          \
    {                                                                                                            \
      const uint32_t pmin = LX ? PX : (LY ? PY : 0xffffffffu);                                                   \
      const bool hazard = cur != 0 && outpos - dist + cur > pmin;                                                \
      LG_STORE(PX, LX, VX);                                                                                      \
      if (__any_sync(FULL, hazard)) { LG_STORE(PY, LY, VY); }                                                    \
      __syncwarp();                                                                                              \
      const uint8_t* const s0 = obase + outpos - dist;                                                           \
      if (!__any_sync(FULL, dist < cur)) {                                                                       \
        _Pragma("unroll")                                                                                        \
        for (int k = 0; k < U; k++) if ((uint32_t)(glane + k * G) < cur) VX[k] = __ldcg(s0 + glane + k * G);     \
      } else {                                                                                                   \
        const bool ovl = dist < cur;                                                                             \
        _Pragma("unroll")                                                                                        \
        for (int k = 0; k < U; k++) {                                                                            \
          const uint32_t i = glane + k * G;                                                                      \
          if (i < cur) VX[k] = __ldcg(s0 + (ovl ? i % dist : i));                                                \
        }                                                                                                        \
      }                                                                                                          \
      PX = outpos; LX = cur;                                                                                     \
    }
    for (;;) {
      const bool act = state == ST_SYMBOLS;
      const bool dec = act && rem == 0;                     // a group in the middle of a long copy does not decode this pass
      uint32_t bits = __funnelshift_r(lo, hi, bp);
      uint32_t e = LL16(bits & LLMASK);
      #pragma unroll
      for (int k = 0; k < NLIT; k++) {
        if (dec && (e & L16_LIT)) {
          if (glane == 0) obase[outpos] = (uint8_t)(e >> 4);
          outpos++;
          bp += e & 15u;
          LG_REFILL();
          bits = __funnelshift_r(lo, hi, bp);
          e = LL16(bits & LLMASK);
        }
      }
      uint32_t len = 0;
      if (dec) {
        if ((e & (L16_LIT | 0x70u)) == L16_MISS) e = decode_long16<INF_LL_BITS, TK_LITLEN>(bits, my_canon, my_sorted);
        if (e & L16_LIT) {
          if (glane == 0) obase[outpos] = (uint8_t)(e >> 4);
          outpos++;
          bp += e & 15u;
        } else if ((e & 0x60u) != 0x60u) {
          const uint32_t nb = e & 15u, xb = (e >> 4) & 7u;
          len = (e >> 7) + 3u + ((bits >> nb) & ~(0xffffffffu << xb));
          bp += nb + xb;
        } else {                                            // end of block, or an invalid code
          bp += e & 15u;
          if ((e & 15u) == 0) err = INF_ERR_SYMBOL;
          state = ST_HEADER;
        }
        LG_REFILL();
      }
      if (__any_sync(FULL, (len | rem) != 0)) {
        if (len) {
          bits = __funnelshift_r(lo, hi, bp);
          uint32_t de = D16(bits & DMASK);
          if ((de & 15u) == 0) de = decode_long16<INF_D_BITS, TK_DIST>(bits, my_canon + 8u * LG_CANON_LL, my_sorted + 288);
          const uint32_t dnb = de & 15u, dxb = (de >> 4) & 15u;
          const uint32_t d = 1u + ((de >> 8) << dxb) + ((bits >> dnb) & ~(0xffffffffu << dxb));
          bp += dnb + dxb;
          if (dnb == 0 || d > outpos || outpos + len > isize) {
            err = (dnb == 0 || d > outpos) ? INF_ERR_DIST : INF_ERR_OVERRUN;
            state = ST_HEADER;
          } else { rem = len; cdist = d; }
        }
        const uint32_t cur = min(rem, (uint32_t)(U * G));
        const uint32_t dist = rem ? cdist : 0u;
        if (tog) { LG_COPY(ppos1, plen1, pv1, ppos0, plen0, pv0); } else { LG_COPY(ppos0, plen0, pv0, ppos1, plen1, pv1); }
        tog ^= 1u;
        outpos += cur; rem -= cur;
        LG_REFILL();
      }
      if (wi > wlimit && act) { if (state == ST_SYMBOLS) err = INF_ERR_INPUT; state = ST_HEADER; rem = 0; }
      // ring top-up, software pipelined through one register per lane: the chunk loaded one pass ago goes into its slot now
      // (its four words sit in the group's G lanes), then the next chunk is requested when its slot is free (every word of
      // the chunk it replaces has been consumed).  The load has a whole pass to complete.
      if (rq_slot != 0xffffffffu) {
        #pragma unroll
        for (int k = 0; k < 4 / G + (4 % G != 0); k++)
          if (glane + k * G < 4) asm volatile("st.shared.u32 [%0], %1;" :: "r"(my_ring + (rq_slot << 4) + ((glane + k * G) << 2)), "r"(rq[k]) : "memory");
        rq_slot = 0xffffffffu;
      }
      if (act && 4u * fill <= wi + 10u) {
        #pragma unroll
        for (int k = 0; k < 4 / G + (4 % G != 0); k++)
          if (glane + k * G < 4) rq[k] = __ldg(wbase + 4u * fill + glane + k * G);
        rq_slot = fill & 3u;
        fill++;
      }
      __syncwarp();
      if (__any_sync(FULL, state == ST_HEADER)) break;
    }

    LG_STORE(ppos0, plen0, pv0);
    LG_STORE(ppos1, plen1, pv1);
#undef LG_COPY
#undef LL16
#undef D16
#undef LG_REFILL
#undef LG_STORE
  }
}

// CRC-32 of every inflated member against its BGZF trailer: one warp per member (32 lane-chunks by slicing-by-4, combined
// with x^(8k) mod P multiplies).  Runs right behind the inflate kernel while the bytes are still in L2.  The four 256-entry
// tables are replicated per lane (entry (t, v) of lane l at word ((t * 256 + v) * 32 + l): bank == lane), so the 32
// data-dependent look-ups of a warp never conflict: 128 KB of shared memory, one CTA of 32 warps per SM.
constexpr int CRC_WARPS = 32;
constexpr size_t CRC_SMEM = 4 * 256 * 32 * sizeof(uint32_t);

__global__ void __launch_bounds__(CRC_WARPS * 32, 1)
crc_kernel(const BlockDesc* __restrict__ blocks, uint32_t n_blocks, const uint8_t* __restrict__ infl,
           uint32_t* __restrict__ status, uint32_t* __restrict__ err_flag) {
  extern __shared__ __align__(16) uint32_t ctab[];
  const int lane = threadIdx.x & 31;
  for (int v = threadIdx.x >> 5; v < 256; v += CRC_WARPS) {           // tab[0][v], one copy per lane
    uint32_t c = (uint32_t)v;
    for (int k = 0; k < 8; k++) c = (c >> 1) ^ ((c & 1u) ? 0xEDB88320u : 0u);
    ctab[(v << 5) + lane] = c;
  }
  __syncthreads();
  for (int v = threadIdx.x >> 5; v < 256; v += CRC_WARPS) {
    uint32_t c = ctab[(v << 5) + lane];
    for (int t = 1; t < 4; t++) { c = ctab[((c & 0xffu) << 5) + lane] ^ (c >> 8); ctab[(((t << 8) + v) << 5) + lane] = c; }
  }
  __syncthreads();
  const uint32_t* const T = ctab + lane;
#define CRC_T(t, b) T[(((t) << 8) + (b)) << 5]
#define CRC_BYTE(x) { st = CRC_T(0, (st ^ (x)) & 0xffu) ^ (st >> 8); }
#define CRC_WORD(w) { st ^= (w); st = CRC_T(3, st & 0xffu) ^ CRC_T(2, (st >> 8) & 0xffu) ^ CRC_T(1, (st >> 16) & 0xffu) ^ CRC_T(0, st >> 24); }
  const uint32_t wpg = gridDim.x * CRC_WARPS;
  for (uint32_t bi = blockIdx.x * CRC_WARPS + (threadIdx.x >> 5); bi < n_blocks; bi += wpg) {
    if (status[bi] != INF_OK) continue;
    const BlockDesc bd = blocks[bi];
    const uint32_t n = bd.isize;
    const uint32_t chunk = ((n + 31) / 32 + 15) & ~15u;               // lane chunks of whole 16-byte units
    const uint32_t b = min(n, chunk * lane), e = min(n, b + chunk);
    uint32_t st = (lane == 0) ? 0xffffffffu : 0u;
    const uint8_t* p = infl + bd.uoff + b;
    uint32_t len = e - b;
    while (len && (reinterpret_cast<uintptr_t>(p) & 15)) { CRC_BYTE(*p); p++; len--; }
    const uint4* pq = reinterpret_cast<const uint4*>(p);
    for (; len >= 16; len -= 16) { const uint4 v = *pq++; CRC_WORD(v.x); CRC_WORD(v.y); CRC_WORD(v.z); CRC_WORD(v.w); }
    p = reinterpret_cast<const uint8_t*>(pq);
    while (len) { CRC_BYTE(*p); p++; len--; }
    st = crc_shift(st, n - e);
    #pragma unroll
    for (int o = 16; o; o >>= 1) st ^= __shfl_xor_sync(FULL, st, o);
    if (~st != bd.crc && lane == 0) {
      status[bi] = INF_ERR_CRC;
      atomicCAS(err_flag, 0u, (bi << 4) | INF_ERR_CRC | 0x80000000u);
    }
  }
#undef CRC_T
#undef CRC_BYTE
#undef CRC_WORD
}

}  // namespace bamscan
