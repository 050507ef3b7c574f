// kernels_deflate.cuh -- BGZF member compressor on the device (SURVEY 8 f4, the write path), sm_100a.
//
// Replaces: noodles-bgzf 0.49.0 io::Writer (0xff00-byte members, libdeflate level 6) behind bam::io::Writer
// (datafusion/bio-format-bam/src/writer.rs:62-113).  The compressed bytes are not the reference's (any conformant DEFLATE
// stream of the same data is equivalent; the reference's own tests are write -> read round trips); the inflated stream is.
//
// bgzf_deflate_kernel: one CTA (384 threads, two CTAs per SM, persistent grid + atomic ticket) per member.
//   0  the member's <= 65 280 inflated bytes come into shared memory with 16-byte loads; CRC-32: every thread takes one
//      contiguous piece (table look-ups from shared memory), the pieces are shifted by x^(8 * bytes behind them) and folded;
//   A  LZ77: the member is cut into 12 regions, one per warp; a warp takes 32 consecutive positions per step: every lane
//      hashes its 4 bytes into the REGION'S OWN slice of the hash table (buckets of the two most recent positions, 16 bit; the
//      slice is pre-seeded with the last 1 KB in front of the region), extends the candidates (and the run candidate p - 1) word by word
//      up to 32 bytes, gives way to a literal when the next position starts a longer match (lazy evaluation: every lane already
//      knows its match), and the warp picks the greedy non-overlapping parse of the 32 positions by pointer jumping over the
//      lanes (5 shuffle rounds); the step's last token is extended to 258 bytes by the whole warp.  Tokens go to an L2-resident
//      scratch slot, symbol counts to per-warp histograms (packed 16-bit counters) in shared memory.  Matches do not cross a
//      region's end, so every region's token list stands alone.  (A table shared by all warps was the first version: positions
//      that other regions insert concurrently -- useless to a region in front of them -- evict the entries a region needs;
//      region-local slices took the file from 1.29 x to 1.10 x the size of zlib level 6, profiles/r2_write.md);
//   B  dynamic Huffman codes (RFC 1951 3.2.7): symbols ranked by count in parallel, the two-queue merge by one thread per
//      tree (litlen / distance side by side), depths in parallel, lengths limited to 15 by moving leaves up from the deepest
//      level (Kraft sum kept exact), canonical codes in parallel.  The code lengths are sent with a flat 4-bit code-length
//      code (no run-length symbols: 158 bytes per member, < 1 % of a typical member);
//   C  every warp turns its tokens into bits at the offset its histogram predicts (warp prefix sums of the token widths,
//      shared-memory atomicOr into the member image, which reuses the input buffer), end-of-block, CRC-32 + ISIZE trailer,
//      and the finished member (gzip header with the BC extra field included) leaves with 16-byte stores.
//   A member that would not shrink is written as a stored block.
// cta_scan_kernel (kernels_scan.cuh) / bgzf_gather_kernel: exclusive scan of the member sizes, then the members are packed back to back.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

#include "kernels_scan.cuh"

namespace bamscan {
namespace dfl {

#ifndef BAMSCAN_DFL_NT
#define BAMSCAN_DFL_NT 384
#endif
constexpr int NT = BAMSCAN_DFL_NT, WARPS = NT / 32;   // threads per CTA (one LZ77 region per warp); A/B: profiles/r2_write.md
constexpr uint32_t BLOCK = 0xff00;           // inflated bytes per member (noodles-bgzf MAX_BUF_SIZE)
constexpr uint32_t SLOT = 65536;             // bytes per member slot in the output staging area
constexpr uint32_t HASH_BITS = 13;
#ifndef BAMSCAN_DFL_LOCAL_HASH
#define BAMSCAN_DFL_LOCAL_HASH 1
#endif
#ifndef BAMSCAN_DFL_HTAB
#define BAMSCAN_DFL_HTAB 16896
#endif
constexpr uint32_t HTAB_ENTRIES = BAMSCAN_DFL_HTAB;                         // 16-bit entries of the hash table (all regions together)
#ifndef BAMSCAN_DFL_WAYS
#define BAMSCAN_DFL_WAYS 2
#endif
constexpr uint32_t WAYS = BAMSCAN_DFL_WAYS;                                // candidates per hash bucket (the most recent positions);
                                                                           // host model tools/deflate_sim.cpp: 2 / 4 / 8 ways in the same memory = -2.2 / -4.0 / -5.1 % bytes
constexpr uint32_t LOCAL_SLOTS = HTAB_ENTRIES / WARPS / WAYS;             // buckets per region
#ifndef BAMSCAN_DFL_PRESEED
#define BAMSCAN_DFL_PRESEED 1024
#endif
constexpr uint32_t PRESEED = BAMSCAN_DFL_PRESEED;                  // per-region slice of the hash table (A/B switch above)
constexpr uint32_t D0 = 288;                 // distance symbols live at [D0, D0 + 30) of the combined tables
constexpr uint32_t NSYM = 320;
constexpr uint32_t FULL = 0xffffffffu;

__constant__ uint32_t c_xpow8[18];           // x^(8 * 2^j) mod P, reflected (writer.cu fills it)

struct Smem {
  uint32_t buf[SLOT / 4 + 8];                // input bytes (zero padded), later the member image
  union {                                    // the hash table is dead when the trees are built: their scratch lives in its place
    uint16_t htab[HTAB_ENTRIES];
    struct {
      uint16_t sorted[2][288];               // used symbols by (count, symbol) ascending
      uint32_t weight[2][576];               // leaves [0, m), internal nodes [m, 2m - 1)
      uint16_t parent[2][576];
      uint8_t depth[2][576];
    } t;
  };
  uint32_t hist[WARPS][NSYM / 2];            // per-warp symbol counts, two 16-bit counters per word (a region holds < 65536 tokens)
  uint32_t freq[NSYM];                       // counts the trees are built from (>= 2 symbols per tree forced)
  uint16_t code[NSYM];                       // bit-reversed canonical codes
  uint8_t len[NSYM];
  uint32_t n_used[2];
  uint16_t first[2][16];                     // first canonical code per length (advanced while the codes are handed out)
  uint32_t crc_tab[256];
  uint32_t crc_part[WARPS];
  uint32_t warp_bits[WARPS];
  uint32_t warp_tok[WARPS];
  uint32_t ticket, total_bits;
};

__device__ __forceinline__ void hist_add(uint32_t* H, uint32_t s) { atomicAdd(H + (s >> 1), 1u << (16u * (s & 1u))); }
__device__ __forceinline__ uint32_t hist_get(const uint32_t* H, uint32_t s) { return (H[s >> 1] >> (16u * (s & 1u))) & 0xffffu; }
__device__ __forceinline__ uint32_t ld4(const uint32_t* buf, uint32_t p) { return __funnelshift_r(buf[p >> 2], buf[(p >> 2) + 1], (p & 3u) * 8u); }
__device__ __forceinline__ uint32_t crc_mul(uint32_t a, uint32_t b) {
  uint32_t p = 0;
  #pragma unroll 4
  for (int i = 0; i < 32; i++) { p ^= (b & 0x80000000u) ? a : 0u; a = (a >> 1) ^ ((a & 1u) ? 0xEDB88320u : 0u); b <<= 1; }
  return p;
}
__device__ __forceinline__ void len_symbol(uint32_t L, uint32_t& sym, uint32_t& eb, uint32_t& ev) {
  const uint32_t l = L - 3u;
  if (L == 258u) { sym = 285; eb = 0; ev = 0; }
  else if (l < 8u) { sym = 257u + l; eb = 0; ev = 0; }
  else { const uint32_t nb = 31u - __clz(l); eb = nb - 2u; sym = 257u + 4u * eb + 4u + ((l >> eb) & 3u); ev = l & ((1u << eb) - 1u); }
}
__device__ __forceinline__ void dist_symbol(uint32_t D, uint32_t& sym, uint32_t& eb, uint32_t& ev) {
  const uint32_t d = D - 1u;
  if (d < 4u) { sym = d; eb = 0; ev = 0; }
  else { const uint32_t nb = 31u - __clz(d); eb = nb - 1u; sym = 2u * nb + ((d >> eb) & 1u); ev = d & ((1u << eb) - 1u); }
}
__device__ __forceinline__ uint32_t extra_bits_of(uint32_t s) {          // s in the combined symbol space
  if (s >= D0) { const uint32_t d = s - D0; return d < 4u ? 0u : (d >> 1) - 1u; }
  return (s >= 265u && s < 285u) ? (s - 261u) >> 2 : 0u;
}
// n <= 48 bits of v at bit position pos of the member image
__device__ __forceinline__ void put_bits(uint32_t* buf, uint32_t pos, unsigned long long v, uint32_t n) {
  if (!n) return;
  const uint32_t w = pos >> 5, s = pos & 31u;
  atomicOr(buf + w, (uint32_t)(v << s));
  if (s + n > 32u) atomicOr(buf + w + 1, (uint32_t)(v >> (32u - s)));
  if (s + n > 64u) atomicOr(buf + w + 2, (uint32_t)(v >> (64u - s)));
}

// Code lengths (<= 15) and canonical codes of BOTH trees from S.freq, side by side: tree 0 = literal/length symbols [0, 286),
// tree 1 = distance symbols [D0, D0 + 30).  The serial steps of the two trees run on two threads of different warps at the
// same time; the canonical codes are assigned by one warp per tree, 32 symbols per step (`match_any` ranks).
__device__ __forceinline__ void build_trees(Smem& S, int tid) {
  const int lane = tid & 31, warp = tid >> 5;
  // (a) rank the used symbols by (count, symbol): thread s < 286 takes litlen symbol s, thread 286 + d distance symbol d
  if (tid < 2) S.n_used[tid] = 0;
  __syncthreads();
  static_assert(NT >= 316, "one thread per symbol of both alphabets");
  static_assert(sizeof(S.t) <= sizeof(S.htab), "tree scratch fits the hash table");
  if (tid < 316) {
    const int T = tid < 286 ? 0 : 1;
    const uint32_t base = T ? D0 : 0u, n = T ? 30u : 286u, s = T ? (uint32_t)tid - 286u : (uint32_t)tid;
    const uint32_t f = S.freq[base + s];
    S.len[base + s] = 0;
    if (f) {
      uint32_t r = 0;
      for (uint32_t u = 0; u < n; u++) { const uint32_t g = S.freq[base + u]; r += (g && (g < f || (g == f && u < s))) ? 1u : 0u; }
      S.t.sorted[T][r] = (uint16_t)s; S.t.weight[T][r] = f;
      atomicAdd(&S.n_used[T], 1u);
    }
  }
  __syncthreads();
  // (b) two-queue merge, one thread per tree; then the depth of every internal node from the root down
  if (tid == 0 || tid == 32) {
    const int T = tid >> 5;
    const uint32_t m = S.n_used[T];
    uint32_t i = 0, j = m;                         // next unused leaf / internal node
    for (uint32_t k = 0; k + 1 < m; k++) {
      const uint32_t node = m + k;
      uint32_t w = 0;
      #pragma unroll
      for (int c = 0; c < 2; c++) {
        uint32_t pick;
        if (i < m && (j >= node || S.t.weight[T][i] <= S.t.weight[T][j])) pick = i++; else pick = j++;
        w += S.t.weight[T][pick]; S.t.parent[T][pick] = (uint16_t)node;
      }
      S.t.weight[T][node] = w;
    }
    const uint32_t root = 2 * m - 2;
    S.t.depth[T][root] = 0;
    for (uint32_t k = root; k-- > m;) S.t.depth[T][k] = (uint8_t)min(60u, (uint32_t)S.t.depth[T][S.t.parent[T][k]] + 1u);
  }
  __syncthreads();
  if (tid < 316) {
    const int T = tid < 286 ? 0 : 1;
    const uint32_t i = T ? (uint32_t)tid - 286u : (uint32_t)tid;
    if (i < S.n_used[T]) S.t.depth[T][i] = (uint8_t)min(60u, (uint32_t)S.t.depth[T][S.t.parent[T][i]] + 1u);
  }
  __syncthreads();
  // (c) limit to 15 bits: counts per length, overflow folded into 15, Kraft sum repaired by splitting a shallower leaf;
  //     S.first[T][l] = first canonical code of length l
  if (tid == 0 || tid == 32) {
    const int T = tid >> 5;
    const uint32_t base = T ? D0 : 0u, m = S.n_used[T];
    uint32_t bl[64];
    for (int l = 0; l < 64; l++) bl[l] = 0;
    for (uint32_t i = 0; i < m; i++) bl[S.t.depth[T][i]]++;
    for (int l = 16; l < 64; l++) { bl[15] += bl[l]; bl[l] = 0; }
    unsigned long long kraft = 0;
    for (int l = 1; l <= 15; l++) kraft += (unsigned long long)bl[l] << (15 - l);
    while (kraft > (1ull << 15)) {
      bl[15]--;
      for (int l = 14; l >= 1; l--) if (bl[l]) { bl[l]--; bl[l + 1] += 2; break; }
      kraft--;
    }
    // leaves are sorted by count ascending: the rarest take the longest codes
    uint32_t i = 0;
    for (int l = 15; l >= 1; l--) for (uint32_t c = 0; c < bl[l]; c++, i++) S.len[base + S.t.sorted[T][i]] = (uint8_t)l;
    uint32_t code = 0;
    S.first[T][0] = 0;
    for (int l = 1; l <= 15; l++) { code = (code + (l > 1 ? bl[l - 1] : 0u)) << 1; S.first[T][l] = (uint16_t)code; }
  }
  __syncthreads();
  // (d) canonical codes (symbols of one length in symbol order), bit-reversed for the LSB-first bit stream: warp T, 32 symbols a step
  if (warp < 2) {
    const int T = warp;
    const uint32_t base = T ? D0 : 0u, n = T ? 30u : 286u;
    for (uint32_t s0 = 0; s0 < n; s0 += 32) {
      const uint32_t s = s0 + (uint32_t)lane;
      const uint32_t L = s < n ? S.len[base + s] : 0u;
      const uint32_t grp = __match_any_sync(FULL, L);
      const uint32_t rank = __popc(grp & ((1u << lane) - 1u));
      const uint32_t code = (uint32_t)S.first[T][L] + rank;
      __syncwarp();
      if (L && rank == 0) S.first[T][L] = (uint16_t)(S.first[T][L] + __popc(grp));     // the group's first lane moves the counter on
      __syncwarp();
      if (s < n) S.code[base + s] = L ? (uint16_t)(__brev(code) >> (32u - L)) : (uint16_t)0;
    }
  }
  __syncthreads();
}

__global__ void __launch_bounds__(NT, 2)
bgzf_deflate_kernel(const uint8_t* __restrict__ stream, unsigned long long stream_bytes, uint32_t n_members, uint8_t* __restrict__ slots,
                    uint32_t* __restrict__ sizes, uint32_t* __restrict__ tok_scratch, uint32_t* __restrict__ ticket, int stored_only) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  Smem& S = *reinterpret_cast<Smem*>(smem_raw);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  uint32_t* const tok_base = tok_scratch + (size_t)blockIdx.x * SLOT;
  for (int i = tid; i < 256; i += NT) {
    uint32_t c = (uint32_t)i;
    #pragma unroll
    for (int k = 0; k < 8; k++) c = (c >> 1) ^ ((c & 1u) ? 0xEDB88320u : 0u);
    S.crc_tab[i] = c;
  }
  // x^(8 * bytes behind this thread's CRC piece) for a full member, once per CTA (every member but the file's last is full)
  uint32_t pow_full;
  {
    const uint32_t seg = (((BLOCK + NT - 1) / NT) + 3u) & ~3u;
    const uint32_t b1 = min(BLOCK, min(BLOCK, (uint32_t)tid * seg) + seg);
    uint32_t rem = BLOCK - b1, p = 0x80000000u;                               // x^0
    for (int j = 0; rem; j++, rem >>= 1) if (rem & 1u) p = crc_mul(p, c_xpow8[j]);
    pow_full = p;
  }
  for (;;) {
    __syncthreads();
    if (tid == 0) S.ticket = atomicAdd(ticket, 1u);
    __syncthreads();
    const uint32_t m = S.ticket;
    if (m >= n_members) break;
    const unsigned long long beg = (unsigned long long)m * BLOCK;
    const uint32_t isize = (uint32_t)min((unsigned long long)BLOCK, stream_bytes - beg);
    uint8_t* const slot = slots + (size_t)m * SLOT;
    // ---- 0: load + CRC-32 ----
    {
      const uint4* src = reinterpret_cast<const uint4*>(stream + beg);
      uint4* dst = reinterpret_cast<uint4*>(S.buf);
      const uint32_t n16 = (isize + 15u) >> 4;
      for (uint32_t i = tid; i < (SLOT / 16) + 2; i += NT) dst[i] = i < n16 ? src[i] : make_uint4(0, 0, 0, 0);   // (the stream buffer is padded to 16 bytes)
      for (uint32_t i = tid; i < HTAB_ENTRIES; i += NT) S.htab[i] = 0xffff;
      for (uint32_t i = tid; i < WARPS * (NSYM / 2); i += NT) (&S.hist[0][0])[i] = 0;
    }
    __syncthreads();
    if ((isize & 15u) && tid == 0) {                                        // bytes behind isize inside the last 16-byte load: zero them
      uint8_t* b = reinterpret_cast<uint8_t*>(S.buf);
      for (uint32_t k = isize; k < ((isize + 15u) & ~15u); k++) b[k] = 0;
    }
    __syncthreads();
    uint32_t crc;
    {
      const uint32_t seg = (((isize + NT - 1) / NT) + 3u) & ~3u;
      const uint32_t b0 = min(isize, (uint32_t)tid * seg), b1 = min(isize, b0 + seg);
      uint32_t st = tid == 0 ? 0xffffffffu : 0u;
      const uint8_t* bytes = reinterpret_cast<const uint8_t*>(S.buf);
      uint32_t k = b0;
      for (; k + 4 <= b1; k += 4) {
        st ^= S.buf[k >> 2];
        #pragma unroll
        for (int q = 0; q < 4; q++) st = S.crc_tab[st & 0xffu] ^ (st >> 8);
      }
      for (; k < b1; k++) st = S.crc_tab[(st ^ bytes[k]) & 0xffu] ^ (st >> 8);
      if (isize == BLOCK) st = crc_mul(st, pow_full);
      else { uint32_t rem = isize - b1; for (int j = 0; rem; j++, rem >>= 1) if (rem & 1u) st = crc_mul(st, c_xpow8[j]); }   // bytes behind this piece
      if (b0 == b1 && tid != 0) st = 0;
      #pragma unroll
      for (int o = 16; o; o >>= 1) st ^= __shfl_xor_sync(FULL, st, o);
      if (lane == 0) S.crc_part[warp] = st;
      __syncthreads();
      crc = 0;
      #pragma unroll
      for (int w = 0; w < WARPS; w++) crc ^= S.crc_part[w];
      crc = ~crc;
    }
    bool stored = stored_only != 0 || isize < 64u;
    uint32_t total_bits = 0, hdr_bits = 0;
    if (!stored) {
      // ---- A: LZ77, one region per warp ----
      const uint32_t reg_len = (((isize + WARPS - 1) / WARPS) + 31u) & ~31u;
      const uint32_t rbeg = min(isize, (uint32_t)warp * reg_len), rend = min(isize, rbeg + reg_len);
      uint32_t* const tok = tok_base + rbeg;
      uint32_t* const H = S.hist[warp];
      uint32_t ntok = 0, skip = 0;
#if BAMSCAN_DFL_LOCAL_HASH
      // the region's table starts with the last PRESEED bytes in front of the region (the previous region's tail), so that its
      // first records find their predecessors too
      for (uint32_t q0 = rbeg > PRESEED ? rbeg - PRESEED : 0u; q0 < rbeg; q0 += 32) {
        const uint32_t q = q0 + lane;
        if (q + 4u <= rbeg) {
          uint16_t* B = S.htab + ((uint32_t)warp * LOCAL_SLOTS + __umulhi(ld4(S.buf, q) * 2654435761u, LOCAL_SLOTS)) * WAYS;
          #pragma unroll
          for (int k = WAYS - 1; k > 0; k--) B[k] = B[k - 1];
          B[0] = (uint16_t)q;
        }
        __syncwarp();
      }
#endif
      for (uint32_t pos = rbeg; pos < rend; pos += 32) {
        const uint32_t p = pos + lane;
        const bool in = p < rend;
        const bool can = in && p + 4u <= rend;
        const uint32_t w4 = ld4(S.buf, min(p, SLOT));
        uint32_t h = 0, cand = 0xffffu;
#if BAMSCAN_DFL_LOCAL_HASH && BAMSCAN_DFL_WAYS > 1
        uint32_t cands[WAYS];
        #pragma unroll
        for (int k = 0; k < (int)WAYS; k++) cands[k] = 0xffffu;
        if (can) {
          h = ((uint32_t)warp * LOCAL_SLOTS + __umulhi(w4 * 2654435761u, LOCAL_SLOTS)) * WAYS;
          #pragma unroll
          for (int k = 0; k < (int)WAYS; k++) cands[k] = S.htab[h + k];
        }
        __syncwarp();
        if (can) {                                      // the bucket ages by one: lanes of one step that share it race, any order is fine
          #pragma unroll
          for (int k = WAYS - 1; k > 0; k--) S.htab[h + k] = (uint16_t)cands[k - 1];
          S.htab[h] = (uint16_t)p;
        }
        cand = cands[0];
#elif BAMSCAN_DFL_LOCAL_HASH
        // one table slice per region: every candidate is an earlier position of the SAME region (the shared table also offers
        // other regions' positions, but concurrently inserted later ones evict the useful entries)
        if (can) { h = (uint32_t)warp * LOCAL_SLOTS + __umulhi(w4 * 2654435761u, LOCAL_SLOTS); cand = S.htab[h]; }
#else
        if (can) { h = (w4 * 2654435761u) >> (32u - HASH_BITS); cand = S.htab[h]; }
#endif
#if !(BAMSCAN_DFL_LOCAL_HASH && BAMSCAN_DFL_WAYS > 1)
        __syncwarp();
        if (can) S.htab[h] = (uint16_t)p;
#endif
        if (skip >= 32u) { skip -= 32u; continue; }                             // the whole step lies inside the previous token
        // matches are first measured up to 32 bytes only: a match that long reaches the end of the step, so it is the step's LAST
        // token whenever it is chosen, and only that one token is then extended to 258 bytes -- by the whole warp, 128 bytes per
        // round -- instead of every lane walking its own long match (runs of equal qualities cost 65 divergent rounds per lane)
        uint32_t L = 1, D = 0;
        if (can) {
          const uint32_t maxlen = min(32u, rend - p);
          uint32_t best = 0;
          if (cand < p && p - cand <= 32768u) {
            uint32_t n = 0;
            while (n < maxlen) { const uint32_t x = ld4(S.buf, cand + n) ^ ld4(S.buf, p + n); if (x) { n += (uint32_t)(__ffs((int)x) - 1) >> 3; break; } n += 4; }
            n = min(n, maxlen);
            if (n >= 4u) { best = n; D = p - cand; }
          }
#if BAMSCAN_DFL_LOCAL_HASH && BAMSCAN_DFL_WAYS > 1
          #pragma unroll
          for (int k = 1; k < (int)WAYS; k++) {                                    // the older entries of the bucket
            const uint32_t c2 = cands[k];
            if (best < maxlen && c2 < p && p - c2 <= 32768u && ld4(S.buf, c2) == w4) {
              uint32_t n = 4;
              while (n < maxlen) { const uint32_t x = ld4(S.buf, c2 + n) ^ ld4(S.buf, p + n); if (x) { n += (uint32_t)(__ffs((int)x) - 1) >> 3; break; } n += 4; }
              n = min(n, maxlen);
              if (n > best) { best = n; D = p - c2; }
            }
          }
#endif
          if (p > 0u && ld4(S.buf, p - 1u) == w4 && best < maxlen) {            // run candidate (sources inside this step are not in the table yet)
            uint32_t n = 4;
            while (n < maxlen) { const uint32_t x = ld4(S.buf, p - 1u + n) ^ ld4(S.buf, p + n); if (x) { n += (uint32_t)(__ffs((int)x) - 1) >> 3; break; } n += 4; }
            n = min(n, maxlen);
            if (n > best) { best = n; D = 1; }
          }
          if (best >= 4u) L = best;
        }
        // lazy evaluation for free (every lane already knows its own match): a match gives way to a literal when the next
        // position starts a longer one (zlib's deflate_slow rule)
        {
          const uint32_t Ln = __shfl_down_sync(FULL, L, 1);
          if (lane < 31 && L >= 4u && Ln > L) L = 1;
        }
        // greedy parse of the 32 positions: lane i jumps to lane i + L_i; the lanes on the path from `skip` are the tokens
        uint32_t endl = (uint32_t)lane + L;
        uint32_t nxt = min(endl, 32u), reach = 1u << lane;
        #pragma unroll
        for (int r = 0; r < 5; r++) {
          const uint32_t rn = __shfl_sync(FULL, reach, nxt & 31u), nn = __shfl_sync(FULL, nxt, nxt & 31u);
          if (nxt < 32u) { reach |= rn; nxt = nn; }
        }
        const uint32_t inmask = __ballot_sync(FULL, in);
        const uint32_t sel = __shfl_sync(FULL, reach, skip) & inmask;
        if (!sel) { skip = 0; continue; }
        {
          // the last token: if it stopped at the 32-byte cap, the warp extends it (lane j compares bytes 32 + 4 j + 128 r ...)
          const int last = 31 - __clz(sel);
          const uint32_t lL = __shfl_sync(FULL, L, last), lD = __shfl_sync(FULL, D, last), lp = pos + (uint32_t)last;
          if (lL == 32u) {
            const uint32_t lmax = min(258u, rend - lp);
            uint32_t ext = 32;
            for (uint32_t b = 32; b < lmax; b += 128) {
              const uint32_t o = b + 4u * (uint32_t)lane;
              uint32_t x = 0xffffffffu;
              if (o < lmax) x = ld4(S.buf, lp - lD + o) ^ ld4(S.buf, lp + o);
              const uint32_t bal = __ballot_sync(FULL, x != 0u);                   // (lanes past lmax count as mismatches)
              if (bal) {
                const int fl = __ffs((int)bal) - 1;
                const uint32_t fx = __shfl_sync(FULL, x, fl), fo = b + 4u * (uint32_t)fl;
                ext = fo < lmax ? min(lmax, fo + ((uint32_t)(__ffs((int)fx) - 1) >> 3)) : lmax;
                break;
              }
              ext = min(lmax, b + 128u);
            }
            if (lane == last) { L = ext; endl = (uint32_t)lane + L; }
          }
        }
        if ((sel >> lane) & 1u) {
          const uint32_t idx = ntok + __popc(sel & ((1u << lane) - 1u));
          if (L >= 4u) {
            tok[idx] = 0x80000000u | ((L - 3u) << 16) | (D - 1u);
            uint32_t sy, eb, ev;
            len_symbol(L, sy, eb, ev); hist_add(H, sy);
            dist_symbol(D, sy, eb, ev); hist_add(H, D0 + sy);
          } else {
            const uint32_t b = w4 & 0xffu;
            tok[idx] = b; hist_add(H, b);
          }
        }
        ntok += __popc(sel);
        const uint32_t last_end = __shfl_sync(FULL, endl, 31 - __clz(sel));
        skip = last_end > 32u ? last_end - 32u : 0u;
      }
      if (lane == 0) S.warp_tok[warp] = ntok;
      __syncthreads();
      // ---- B: Huffman codes ----
      for (uint32_t s = tid; s < NSYM; s += NT) {
        uint32_t c = 0;
        #pragma unroll
        for (int w = 0; w < WARPS; w++) c += hist_get(S.hist[w], s);
        if (s == 256u) c = 1;
        uint32_t f = c;
        if ((s == 0u || s == D0 || s == D0 + 1u) && f == 0u) f = 1;        // >= 2 used symbols per tree: complete codes
        if (s >= 286u && s < D0) f = 0;
        if (s >= D0 + 30u) f = 0;
        S.freq[s] = f;
      }
      __syncthreads();
      build_trees(S, tid);
      // widths: per warp (emit offsets) and in total
      {
        uint32_t bits = 0;
        for (uint32_t s = lane; s < NSYM; s += 32) bits += hist_get(S.hist[warp], s) * ((uint32_t)S.len[s] + extra_bits_of(s));
        #pragma unroll
        for (int o = 16; o; o >>= 1) bits += __shfl_xor_sync(FULL, bits, o);
        if (lane == 0) S.warp_bits[warp] = bits;
      }
      __syncthreads();
      hdr_bits = 3u + 5u + 5u + 4u + 19u * 3u + (286u + 30u) * 4u;
      total_bits = hdr_bits + (uint32_t)S.len[256];
      #pragma unroll
      for (int w = 0; w < WARPS; w++) total_bits += S.warp_bits[w];
      if (((total_bits + 7u) >> 3) >= isize) stored = true;
    }
    const uint32_t clen = stored ? isize + 5u : (total_bits + 7u) >> 3;
    const uint32_t msize = 18u + clen + 8u;
    if (stored) {
      __syncthreads();
      const uint8_t* bytes = reinterpret_cast<const uint8_t*>(S.buf);
      if (tid < 23) {
        const uint8_t hdr[23] = {0x1f, 0x8b, 8, 4, 0, 0, 0, 0, 0, 0xff, 6, 0, 'B', 'C', 2, 0, (uint8_t)(msize - 1u), (uint8_t)((msize - 1u) >> 8),
                                 1, (uint8_t)isize, (uint8_t)(isize >> 8), (uint8_t)~isize, (uint8_t)(~isize >> 8)};
        slot[tid] = hdr[tid];
      }
      for (uint32_t k = tid; k < isize; k += NT) slot[23u + k] = bytes[k];
      if (tid < 8) slot[23u + isize + tid] = (uint8_t)((tid < 4 ? crc : isize) >> (8 * (tid & 3)));
      if (tid == 0) sizes[m] = msize;
      continue;
    }
    // ---- C: the member image ----
    __syncthreads();
    for (uint32_t i = tid; i < SLOT / 4 + 8; i += NT) S.buf[i] = 0;
    __syncthreads();
    {
      const uint32_t B0 = 144u;                                              // bits of the 18-byte gzip header
      if (tid == 0) {
        S.buf[0] = 0x04088b1fu; S.buf[1] = 0; S.buf[2] = 0x0006ff00u; S.buf[3] = 0x00024342u;
        atomicOr(S.buf + 4, (msize - 1u) & 0xffffu);                       // (the deflate bits of other threads share this word)
        // BFINAL = 1, BTYPE = 10, HLIT = 29, HDIST = 29, HCLEN = 15; code-length code: 16, 17, 18 unused, 0..15 four bits each
        unsigned long long h = 1ull | (2ull << 1) | (29ull << 3) | (29ull << 8) | (15ull << 13);
        put_bits(S.buf, B0, h, 17);
        unsigned long long cl = 0;
        for (int k = 3; k < 19; k++) cl |= 4ull << (3 * (k - 3));
        put_bits(S.buf, B0 + 17u + 9u, cl, 48);
      }
      for (uint32_t s = tid; s < 316u; s += NT) {
        const uint32_t L = S.len[s < 286u ? s : D0 + (s - 286u)];
        put_bits(S.buf, B0 + 17u + 57u + 4u * s, __brev(L) >> 28, 4);
      }
      uint32_t base = B0 + hdr_bits;
      for (int w = 0; w < warp; w++) base += S.warp_bits[w];
      const uint32_t reg_len = (((isize + WARPS - 1) / WARPS) + 31u) & ~31u;
      const uint32_t* const tok = tok_base + min(isize, (uint32_t)warp * reg_len);
      const uint32_t ntok = S.warp_tok[warp];
      for (uint32_t t0 = 0; t0 < ntok; t0 += 32) {
        const uint32_t t = t0 + lane;
        unsigned long long v = 0; uint32_t n = 0;
        if (t < ntok) {
          const uint32_t k = tok[t];
          if (k & 0x80000000u) {
            uint32_t sy, eb, ev;
            len_symbol(((k >> 16) & 0xffu) + 3u, sy, eb, ev);
            v = S.code[sy]; n = S.len[sy];
            v |= (unsigned long long)ev << n; n += eb;
            dist_symbol((k & 0x7fffu) + 1u, sy, eb, ev);
            v |= (unsigned long long)S.code[D0 + sy] << n; n += S.len[D0 + sy];
            v |= (unsigned long long)ev << n; n += eb;
          } else { v = S.code[k]; n = S.len[k]; }
        }
        uint32_t incl = n;
        #pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const uint32_t y = __shfl_up_sync(FULL, incl, o); if (lane >= o) incl += y; }
        put_bits(S.buf, base + incl - n, v, n);
        base += __shfl_sync(FULL, incl, 31);
      }
      if (tid == 0) put_bits(S.buf, B0 + total_bits - (uint32_t)S.len[256], S.code[256], S.len[256]);
    }
    __syncthreads();
    if (tid < 8) reinterpret_cast<uint8_t*>(S.buf)[18u + clen + tid] = (uint8_t)((tid < 4 ? crc : isize) >> (8 * (tid & 3)));
    __syncthreads();
    {
      const uint4* src = reinterpret_cast<const uint4*>(S.buf);
      uint4* dst = reinterpret_cast<uint4*>(slot);
      for (uint32_t i = tid; i < (msize + 15u) >> 4; i += NT) dst[i] = src[i];
    }
    if (tid == 0) sizes[m] = msize;
  }
}

__global__ void __launch_bounds__(256)
bgzf_gather_kernel(const uint8_t* __restrict__ slots, const uint32_t* __restrict__ sizes, const unsigned long long* __restrict__ offsets, uint8_t* __restrict__ out) {
  const uint32_t m = blockIdx.x, n = sizes[m];
  const uint8_t* src = slots + (size_t)m * SLOT;
  uint8_t* dst = out + offsets[m];
  // destination-aligned words: head bytes, then 4-byte words assembled from two aligned source words, then the tail
  const uint32_t head = min(n, (uint32_t)((4u - (reinterpret_cast<uintptr_t>(dst) & 3u)) & 3u));
  if (threadIdx.x < head) dst[threadIdx.x] = src[threadIdx.x];
  const uint32_t nw = (n - head) >> 2;
  const uint32_t* sw = reinterpret_cast<const uint32_t*>(src);
  uint32_t* dw = reinterpret_cast<uint32_t*>(dst + head);
  const uint32_t sh = head * 8u;
  for (uint32_t i = threadIdx.x; i < nw; i += blockDim.x) dw[i] = sh ? __funnelshift_r(sw[i], sw[i + 1], sh) : sw[i];
  const uint32_t done = head + 4u * nw;
  if (threadIdx.x < n - done) dst[done + threadIdx.x] = src[done + threadIdx.x];
}

// exclusive scan of the record lengths of one slice -> 64-bit offsets (offsets[n] = total); one CTA per 4096 rows + a tile pass
__global__ void __launch_bounds__(256)
len_tile_sums_kernel(const uint32_t* __restrict__ len, uint32_t n, unsigned long long* __restrict__ tile_sums) {
  __shared__ unsigned long long ws[8];
  const uint32_t base = blockIdx.x * 4096u + threadIdx.x * 16u;
  unsigned long long s = 0;
  #pragma unroll
  for (int k = 0; k < 16; k++) if (base + k < n) s += len[base + k];
  const unsigned long long t = block_sum<256>(s, ws);
  if (threadIdx.x == 0) tile_sums[blockIdx.x] = t;
}
__global__ void __launch_bounds__(256)
len_offsets_kernel(const uint32_t* __restrict__ len, uint32_t n, const unsigned long long* __restrict__ tile_offsets, unsigned long long first,
                   unsigned long long* __restrict__ offsets) {
  __shared__ unsigned long long ws[8];
  const uint32_t base = blockIdx.x * 4096u + threadIdx.x * 16u;
  uint32_t v[16]; unsigned long long s = 0;
  #pragma unroll
  for (int k = 0; k < 16; k++) { v[k] = base + k < n ? len[base + k] : 0u; s += v[k]; }
  unsigned long long run = first + tile_offsets[blockIdx.x] + block_exclusive_scan<256>(s, ws);
  #pragma unroll
  for (int k = 0; k < 16; k++) { if (base + k <= n) offsets[base + k] = run; run += v[k]; }
}

}  // namespace dfl
}  // namespace bamscan
