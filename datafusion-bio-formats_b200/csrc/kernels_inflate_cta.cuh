// kernels_inflate_cta.cuh -- CTA-per-member raw-DEFLATE inflate for BGZF, parallel INSIDE the member, sm_100a.
//
// Replaces: noodles-bgzf 0.49.0 io::Reader block inflate + libdeflate `deflate_decompress` / `crc32`
// (reference call sites: datafusion/bio-format-bam/src/storage.rs:161-169, physical_exec.rs:409).
//
// One CTA of two teams (two CTAs per SM) holds two BGZF members at a time (persistent grid, atomic ticket).
// PRODUCER team (warps 0-7, NT_P threads), member k+1:
//   1. the deflate payload is brought into shared memory by ONE cp.async.bulk (TMA) + mbarrier;
//   2. per deflate block: warp 0 reads the block header, warps 0/1 build two-level Huffman LUTs in shared memory;
//   3. the block's symbol stream is cut into NT_P sub-streams which all lanes decode speculatively and then re-anchor on
//      their predecessor's end until nothing changes (inflate_cta_core.h explains why that converges in ~2 rounds);
//   4. a team scan of the per-lane byte counts gives output offsets; the lanes decode again and EMIT literals and parked
//      matches into the member's 64 KB OUTPUT WINDOW, which lives in shared memory.
// CONSUMER team (warps 8-11, NT_C threads), member k:
//   5. RESOLVE the parked matches in output order, in batches of at most LIST_CAP matches, each warp over its own part of
//      the window, ordered by per-piece map bits (every LZ77 source read is a shared-memory read);
//   6. CRC-32 is computed from the window (no second pass over HBM), ISIZE is checked, and the window leaves the SM once:
//      cp.async.bulk shared -> global for the 16-byte aligned body, byte stores for the ragged ends.
// Steps 1-3 never touch the window or its head bitmap and steps 5-6 never touch the payload or the LUTs, so the producer's
// header / tables / count of member k+1 run while the consumer resolves member k.  The window (with the head bitmap) is
// handed over by two named barriers: FULL (producer -> consumer, with a hand-off record) and EMPTY (consumer -> producer).
// HBM traffic is the algorithmic minimum: payload read once, inflated bytes written once.
//
// Members this kernel cannot take (ISIZE > 65536, a Huffman code whose second-level tables exceed the shared-memory budget:
// in practice only a distance code, see SUB_D) are flagged INF_RETRY in status[], counted in *retry_count and redone by the
// warp-per-member kernel of kernels_inflate.cuh.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

#include "inflate_cta_core.h"
#include "kernels_inflate.cuh"

namespace bamscan {
namespace icta {

constexpr uint32_t INF_RETRY = 15;          // status: redo this member with the warp-per-member kernel
constexpr uint32_t FRONT_DONE = 0xffffffffu;
#ifndef BAMSCAN_ICTA_MIN_SUB_BITS
#define BAMSCAN_ICTA_MIN_SUB_BITS 64
#endif
constexpr uint32_t MIN_SUB_BITS = BAMSCAN_ICTA_MIN_SUB_BITS;      // shortest sub-stream a lane is given
#ifndef BAMSCAN_ICTA_WARMUP_BITS
#define BAMSCAN_ICTA_WARMUP_BITS 640
#endif
constexpr uint32_t WARMUP_BITS = BAMSCAN_ICTA_WARMUP_BITS;
#ifndef BAMSCAN_ICTA_WARMUP_MIN_BITS
#define BAMSCAN_ICTA_WARMUP_MIN_BITS 192
#endif
constexpr uint32_t WARMUP_MIN_BITS = BAMSCAN_ICTA_WARMUP_MIN_BITS;
#ifndef BAMSCAN_ICTA_PAY_KB
#define BAMSCAN_ICTA_PAY_KB 24
#endif

// the two teams of a CTA
constexpr int NT_P = 256, NT_C = 128, NT = NT_P + NT_C;
constexpr int RWARPS = NT_C / 32;                                 // resolver warps = the consumer team
// named barriers (0 is __syncthreads, used only before the teams split)
constexpr uint32_t BAR_P = 1, BAR_C = 2, BAR_FULL = 3, BAR_EMPTY = 4;

// global constant tables of the CRC stage, filled once per device by crc_tables_init_kernel:
//   [0, 1024)     four 256-entry tables of the operator "multiply by x^(32*NT)" (strided slicing-by-4)
//   [1024, 1024+NT] x^(32*j) mod P for j = 0..NT
template <int NT> struct CrcTabs { static constexpr uint32_t WORDS = 1024 + NT + 1; };

struct Cfg {
  static constexpr uint32_t WIN_BYTES = 65536 + 32;
  static constexpr uint32_t HB_WORDS = 2052;                  // head bitmap: one bit per window byte
  static constexpr uint32_t CCTL_BYTES = 256;
  static constexpr uint32_t CTL_BYTES = 1024;
  static constexpr uint32_t PAY_BYTES = BAMSCAN_ICTA_PAY_KB * 1024;   // payload buffer (larger payloads are streamed through it)
  static constexpr uint32_t PAY_SLACK = 64;
  static constexpr uint32_t LUT_LL_WORDS = ROOT_LL + SUB_LL, LUT_D_WORDS = ROOT_D + SUB_D;
  static constexpr uint32_t SMEM_MAX = 113 * 1024;            // two CTAs per SM
  // consumer-owned while it holds the window: window, head / unresolved bitmap, consumer control block, match list
  static constexpr uint32_t OFF_WIN = 16;                     // (the resolver gathers up to 3 bytes in front of the window's first word)
  static constexpr uint32_t OFF_HB = OFF_WIN + WIN_BYTES;
  static constexpr uint32_t OFF_CCTL = OFF_HB + HB_WORDS * 4;
  static constexpr uint32_t OFF_LIST = OFF_CCTL + CCTL_BYTES;
  // producer-owned: payload, LUTs, lane arrays, producer control block; the match list takes what is left
  static constexpr uint32_t PROD_BYTES = PAY_BYTES + PAY_SLACK + (LUT_LL_WORDS + LUT_D_WORDS) * 4 + 2 * NT_P * 4 + CTL_BYTES;
  static constexpr uint32_t LIST_CAP = ((SMEM_MAX - OFF_LIST - PROD_BYTES) / 2) & ~7u;   // u16 entries, 16-byte multiple
  static constexpr uint32_t OFF_PAY = OFF_LIST + LIST_CAP * 2;
  static constexpr uint32_t OFF_LUT_LL = OFF_PAY + PAY_BYTES + PAY_SLACK;
  static constexpr uint32_t OFF_LUT_D = OFF_LUT_LL + LUT_LL_WORDS * 4;
  static constexpr uint32_t OFF_LANE_E = OFF_LUT_D + LUT_D_WORDS * 4;
  static constexpr uint32_t OFF_LANE_N = OFF_LANE_E + NT_P * 4;
  static constexpr uint32_t OFF_CTL = OFF_LANE_N + NT_P * 4;
  static constexpr uint32_t SMEM = OFF_CTL + CTL_BYTES;
  static_assert(OFF_PAY % 16 == 0, "cp.async.bulk destination");
  static_assert(LIST_CAP >= 2048, "match list");
  static_assert(SMEM <= SMEM_MAX, "two CTAs per SM");
};

// producer control block
struct Ctl {
  unsigned long long mbar;
  uint32_t ticket, err, btype, final_block, hdr_end, stored_len, n_ll, n_d;
  uint32_t first_term[2];            // lowest lane whose chain does not hand over (double buffered per round)
  uint32_t last_lane, last_info;
  uint32_t warp_tot[NT_P / 32];
  uint16_t cnt[2][16], first[2][16], nxt[2][16], offs[2][16];
  uint8_t cl[320];
};
static_assert(sizeof(Ctl) <= Cfg::CTL_BYTES, "Ctl fits its slot");

// window hand-off record, producer -> consumer (bi == HANDOFF_END: no more members)
constexpr uint32_t HANDOFF_END = 0xffffffffu;
struct Handoff { uint32_t bi, obase, isize, crc, uoff; };

// consumer control block
struct CCtl {
  unsigned long long psel[8];        // psel[d]: sixteen nibbles k mod d (byte selectors of a period-d piece, resolve stage)
  uint32_t err;
  uint32_t warp_tot[RWARPS];
  uint32_t crc_part[RWARPS];
  Handoff h;
};
static_assert(sizeof(CCtl) <= Cfg::CCTL_BYTES, "CCtl fits its slot");

// ---- PTX helpers: mbarrier + 1-D bulk copies (TMA) ----
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned long long* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(unsigned long long* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
// bounded: a transfer that never completes becomes an error code instead of a hung kernel
__device__ __forceinline__ bool mbar_wait(unsigned long long* bar, uint32_t parity) {
  for (uint32_t tries = 0; tries < (1u << 22); tries++) {
    uint32_t ok;
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                 : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    if (ok) return true;
  }
  return false;
}
__device__ __forceinline__ void bulk_load(void* dst_smem, const void* src_gmem, uint32_t bytes, unsigned long long* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(smem_u32(dst_smem)), "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void bulk_store(void* dst_gmem, const void* src_smem, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst_gmem), "r"(smem_u32(src_smem)), "r"(bytes) : "memory");
  asm volatile("cp.async.bulk.commit_group;" ::: "memory");
}
__device__ __forceinline__ void bulk_store_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// named barriers: a team's own barrier, and the arrive / wait halves of the window hand-off
template <uint32_t ID, uint32_t N> __device__ __forceinline__ void bar_sync() { asm volatile("bar.sync %0, %1;" ::"n"(ID), "n"(N) : "memory"); }
template <uint32_t ID, uint32_t N> __device__ __forceinline__ void bar_arrive() { asm volatile("bar.arrive %0, %1;" ::"n"(ID), "n"(N) : "memory"); }
template <uint32_t ID, uint32_t N> __device__ __forceinline__ bool bar_or(bool v) {
  uint32_t r;
  asm volatile("{\n\t.reg .pred p, q;\n\tsetp.ne.u32 p, %1, 0;\n\tbar.red.or.pred q, %2, %3, p;\n\tselp.u32 %0, 1, 0, q;\n\t}"
               : "=r"(r) : "r"((uint32_t)v), "n"(ID), "n"(N) : "memory");
  return r != 0u;
}
__device__ __forceinline__ void psync() { bar_sync<BAR_P, NT_P>(); }
__device__ __forceinline__ void csync() { bar_sync<BAR_C, NT_C>(); }

__device__ __forceinline__ void sts_u32(uint32_t a, uint32_t v) { asm volatile("st.shared.u32 [%0], %1;" ::"r"(a), "r"(v) : "memory"); }
__device__ __forceinline__ uint32_t lds_u16(uint32_t a) { uint32_t v; asm volatile("ld.shared.u16 %0, [%1];" : "=r"(v) : "r"(a) : "memory"); return v; }
// (predicated inside the asm: an `if` around a volatile asm compiles to a branch + reconvergence barrier per statement)
__device__ __forceinline__ void and_shared_if(uint32_t a, uint32_t v, bool on) { asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.u32 p, %2, 0;\n\t@p red.shared.and.b32 [%0], %1;\n\t}" ::"r"(a), "r"(v), "r"((uint32_t)on) : "memory"); }
__device__ __forceinline__ void red_and_shared(uint32_t a, uint32_t v) { asm volatile("red.shared.and.b32 [%0], %1;" ::"r"(a), "r"(v) : "memory"); }

__device__ __forceinline__ uint32_t brev_n(uint32_t v, uint32_t bits) { return __brev(v) >> (32u - bits); }

// Canonical Huffman build into a two-level LUT (format: inflate_cta_core.h), in three steps:
//   lut_prepare_warp  one warp per table: counts, first codes, every symbol's code and the symbols sorted by (length, symbol);
//   lut_fill_root     ALL threads: root entry idx is decoded canonically (<= RBITS steps) -- perfectly balanced, where a
//                     symbol-centric fill leaves one lane writing 2^(RBITS - len) entries for the shortest code;
//   lut_sub_warp      one warp per table: second-level tables for the codes longer than RBITS bits.
// `S` selects the scratch rows of Ctl.  Error codes: INF_ERR_TABLE for an over-subscribed or incomplete code
// (code_complete_ok), INF_RETRY when the second-level tables do not fit.
template <int RBITS>
__device__ __forceinline__ uint32_t lut_prepare_warp(const uint8_t* cl, int n, Ctl* C, int S, uint16_t* sorted, uint16_t* codes, int lane) {
  uint16_t* cnt = C->cnt[S]; uint16_t* first = C->first[S]; uint16_t* nxt = C->nxt[S]; uint16_t* offs = C->offs[S];
  if (lane < 16) { cnt[lane] = 0; nxt[lane] = 0; }
  __syncwarp();
  for (int s = lane; s < n; s += 32) {
    const uint32_t L = cl[s];
    if (L) atomicAdd(reinterpret_cast<unsigned int*>(cnt) + (L >> 1), (L & 1) ? 0x10000u : 1u);   // 16-bit counters packed in pairs
  }
  __syncwarp();
  uint32_t code = 0, left = 1, off = 0;
  bool over = false;
  for (int len = 1; len <= 15; len++) {
    const uint32_t c = cnt[len];
    code = (code + cnt[len - 1]) << 1;
    left <<= 1;
    if (c > left) over = true;
    left -= c;
    if (lane == len) { first[len] = (uint16_t)code; offs[len] = (uint16_t)off; }
    off += c;
  }
  if (over || !code_complete_ok(left, off, cnt[1])) return INF_ERR_TABLE;
  __syncwarp();
  const uint32_t lt = (1u << lane) - 1u;
  #pragma unroll
  for (int b = 0; b < 9; b++) {
    if (b * 32 >= n) break;                                    // (uniform: the distance alphabet needs one pass)
    const int s = b * 32 + lane;
    const uint32_t L = (s < n) ? cl[s] : 0u;
    const uint32_t m = __match_any_sync(FULL, L);
    const uint32_t r = nxt[L] + __popc(m & lt);
    __syncwarp();
    if (L && (m & lt) == 0) nxt[L] = (uint16_t)(nxt[L] + __popc(m));
    __syncwarp();
    if (L) { sorted[offs[L] + r] = (uint16_t)s; codes[s] = (uint16_t)(first[L] + r); }
  }
  return INF_OK;
}

template <int RBITS, bool DIST, int NT>
__device__ __forceinline__ void lut_fill_root(uint32_t* lut, uint32_t sub_cap, const Ctl* C, int S, const uint16_t* sorted, int tid) {
  constexpr uint32_t ROOT = 1u << RBITS;
  const uint16_t* cnt = C->cnt[S]; const uint16_t* first = C->first[S]; const uint16_t* offs = C->offs[S];
  for (uint32_t idx = tid; idx < ROOT; idx += NT) {
    const uint32_t rev = __brev(idx) >> (32 - RBITS);          // the code bits, first bit on top
    uint32_t hl = 0, hd = 0;
    #pragma unroll
    for (int L = 1; L <= RBITS; L++) {
      const uint32_t d = (rev >> (RBITS - L)) - first[L];
      if (d < cnt[L]) { hl = L; hd = d + offs[L]; }            // (prefix code: at most one length matches)
    }
    uint32_t e = E_BAD;
    if (hl) { const uint32_t sy = sorted[hd]; e = DIST ? entry_dist(sy, hl) : entry_litlen(sy, hl); }
    lut[idx] = e;
  }
  for (uint32_t i = ROOT + tid; i < ROOT + sub_cap; i += NT) lut[i] = E_BAD;
}

template <int RBITS, bool DIST>
__device__ __forceinline__ uint32_t lut_sub_warp(const uint8_t* cl, int n, uint32_t* lut, uint32_t sub_cap, Ctl* C, int S, const uint16_t* codes, int lane) {
  constexpr uint32_t ROOT = 1u << RBITS;
  const uint16_t* cnt = C->cnt[S]; const uint16_t* first = C->first[S];
  uint32_t any_long = 0;
  for (int len = RBITS + 1; len <= 15; len++) any_long += cnt[len];
  if (!any_long) return INF_OK;
  // per root prefix of a long code, the widest remainder (atomicMax on the root slot, E_SUB | bits > E_BAD)
  for (int s = lane; s < n; s += 32) {
    const uint32_t L = cl[s];
    if (L > (uint32_t)RBITS) atomicMax(lut + brev_n((uint32_t)codes[s] >> (L - RBITS), RBITS), E_SUB | (L - RBITS));
  }
  __syncwarp();
  // one second-level table per root prefix that carries long codes; prefixes of long codes are the top of the code space
  const uint32_t q_min = (uint32_t)first[RBITS + 1] >> 1;
  uint32_t base = ROOT;
  for (uint32_t q0 = q_min; q0 < ROOT; q0 += 32) {
    const uint32_t q = q0 + lane;
    uint32_t slot = 0, sz = 0, sb = 0;
    if (q < ROOT) {
      slot = brev_n(q, RBITS);
      const uint32_t e = lut[slot];
      if (e & E_SUB) { sb = e & 31u; sz = 1u << sb; }
    }
    uint32_t incl = sz;
    #pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const uint32_t v = __shfl_up_sync(FULL, incl, o); if (lane >= o) incl += v; }
    if (sz && base + incl <= ROOT + sub_cap) lut[slot] = entry_sub((uint32_t)RBITS, sb, base + incl - sz);
    base += __shfl_sync(FULL, incl, 31);
  }
  if (base > ROOT + sub_cap) return INF_RETRY;
  __syncwarp();
  for (int s = lane; s < n; s += 32) {
    const uint32_t L = cl[s];
    if (L > (uint32_t)RBITS) {
      const uint32_t cd = codes[s], l2 = L - RBITS;
      const uint32_t pe = lut[brev_n(cd >> l2, RBITS)];
      const uint32_t sbits = pe & 31u, sbase = pe >> 16;
      const uint32_t e = DIST ? entry_dist((uint32_t)s, L) : entry_litlen((uint32_t)s, L);
      for (uint32_t idx = brev_n(cd & ((1u << l2) - 1u), l2); idx < (1u << sbits); idx += (1u << l2)) lut[sbase + idx] = e;
    }
  }
  __syncwarp();
  return INF_OK;
}

// warp-uniform bit reader over the payload words in shared memory (block headers only)
struct SBits {
  const uint32_t* w; uint32_t pos;
  __device__ __forceinline__ uint32_t peek() const { return __funnelshift_r(w[pos >> 5], w[(pos >> 5) + 1], pos & 31u); }
  __device__ __forceinline__ uint32_t take(uint32_t n) { const uint32_t v = peek() & ((1u << n) - 1u); pos += n; return v; }
};

// Dynamic block header (RFC 1951 3.2.7), part 1, one warp: HLIT / HDIST / HCLEN, the code-length code and its 7-bit LUT
// (128 entries at `plut`: length | symbol << 16, 0 = unused).  Leaves br.pos at the first code-length symbol.
__device__ __noinline__ uint32_t read_precode_warp(SBits& br, uint32_t* plut, Ctl* C, int lane) {
  const uint32_t h = br.take(14);
  const int n_ll = (int)(h & 31u) + 257, n_d = (int)((h >> 5) & 31u) + 1, n_clc = (int)(h >> 10) + 4;
  if (n_ll > 286 || n_d > 30) return INF_ERR_TABLE;
  if (lane < 19) C->cl[lane] = 0;
  __syncwarp();
  {
    const uint32_t v = (lane < n_clc) ? ((__funnelshift_r(br.w[(br.pos + 3u * lane) >> 5], br.w[((br.pos + 3u * lane) >> 5) + 1], (br.pos + 3u * lane) & 31u)) & 7u) : 0u;
    if (lane < n_clc) C->cl[c_clc_order[lane]] = (uint8_t)v;
    br.pos += 3u * (uint32_t)n_clc;
  }
  __syncwarp();
  uint16_t* cnt = C->cnt[1]; uint16_t* first = C->first[1];
  if (lane < 16) cnt[lane] = 0;
  for (int i = lane; i < 128; i += 32) plut[i] = 0;
  __syncwarp();
  const uint32_t L = lane < 19 ? C->cl[lane] : 0u;
  if (L) atomicAdd(reinterpret_cast<unsigned int*>(cnt) + (L >> 1), (L & 1) ? 0x10000u : 1u);
  __syncwarp();
  uint32_t code = 0, left = 1; bool over = false;
  for (int len = 1; len <= 7; len++) {
    const uint32_t c = cnt[len];
    code = (code + cnt[len - 1]) << 1; left <<= 1;
    if (c > left) over = true;
    left -= c;
    if (lane == len) first[len] = (uint16_t)code;
  }
  if (over || left != 0) return INF_ERR_TABLE;                  // the code-length code must be complete (no exceptions)
  __syncwarp();
  const uint32_t m = __match_any_sync(FULL, L);
  const uint32_t r = __popc(m & ((1u << lane) - 1u));
  if (L) {
    const uint32_t cd = first[L] + r;
    for (uint32_t idx = brev_n(cd, L); idx < 128u; idx += (1u << L)) plut[idx] = L | ((uint32_t)lane << 16);
  }
  __syncwarp();
  C->n_ll = (uint32_t)n_ll; C->n_d = (uint32_t)n_d;
  return INF_OK;
}

// Part 2, whole producer team (NT threads): the run-length coded code lengths.  One code-length symbol takes a warp ~300 cycles when it is decoded
// serially (one LUT look-up per symbol on a dependent chain, sharing the issue slots with 15 other warps), and a member has
// ~500 of them.  Here every thread decodes the symbol that WOULD start at its bit offsets (a table of 16-bit records:
// bits consumed - 1 [3:0], kind [5:4] = 0 length / 1 repeat previous / 2 zeros / 3 invalid, value or run length [13:6]),
// one thread then follows the chain of real symbols through that table (a handful of instructions per symbol), and all
// threads expand the runs into C->cl.  Returns the error code; *end_pos = bit position behind the code lengths.
template <int NT>
__device__ __forceinline__ uint32_t read_code_lengths_cta(const uint32_t* pay, uint32_t start_pos, uint32_t limit_pos, const uint32_t* plut,
                                                          uint16_t* tab, uint32_t tab_cap, uint32_t* chain, Ctl* C, int tid, uint32_t* end_pos) {
  const uint32_t total = C->n_ll + C->n_d;
  const uint32_t n_tab = min(tab_cap, limit_pos > start_pos ? limit_pos - start_pos : 0u);
  for (uint32_t q = tid; q < n_tab; q += NT) {
    const uint32_t p = start_pos + q;
    const uint32_t bits = __funnelshift_r(pay[p >> 5], pay[(p >> 5) + 1], p & 31u);
    const uint32_t e = plut[bits & 127u];
    const uint32_t L = e & 15u, sy = e >> 16;
    uint32_t rec;
    if (L == 0) rec = (3u << 4) | (255u << 6);
    else if (sy < 16u) rec = (L - 1u) | (sy << 6);
    else if (sy == 16u) rec = (L + 2u - 1u) | (1u << 4) | ((3u + ((bits >> L) & 3u)) << 6);
    else if (sy == 17u) rec = (L + 3u - 1u) | (2u << 4) | ((3u + ((bits >> L) & 7u)) << 6);
    else rec = (L + 7u - 1u) | (2u << 4) | ((11u + ((bits >> L) & 127u)) << 6);
    tab[q] = (uint16_t)rec;
  }
  bar_sync<BAR_P, NT>();
  if (tid < 32) {
    // Follow the chain of real symbols through the table: warp 0, 32 segments of 64 bit positions at a time.  Every lane walks
    // its segment from the segment's first position (lane 0: from the true entry) and keeps the visited positions as a 64-bit
    // mask; the code-length code self-synchronises within a few symbols, so when a lane is then given its true entry (its
    // predecessor's exit) it only re-walks until it meets a position it has already visited.  Repeat until every lane's entry
    // equals its predecessor's exit (lane 0 is exact, hence all are): two rounds in practice, ~45 cycles per step and ~20
    // steps per lane instead of ~400 steps in a row.  Validity, "repeat previous" values and the expansion come below.
    const int lane = tid;
    constexpr uint32_t SEG = 64;
    uint32_t win_q = 0, entry0 = 0, i_base = 0, k_base = 0, q_end = 0;
    bool done = false;
    while (!done) {
      const uint32_t lo = win_q + (uint32_t)lane * SEG, hi = lo + SEG;
      auto walk = [&](uint32_t from, unsigned long long old, unsigned long long& m, uint32_t& ex) {
        // from `from` until the segment is left, the table ends, or a position of `old` is met (then the old tail is kept)
        uint32_t q = from; unsigned long long nm = 0;
        while (q < hi && q < n_tab && !((old >> (q - lo)) & 1ull)) { nm |= 1ull << (q - lo); q += (tab[q] & 15u) + 1u; }
        if (q < hi && q < n_tab) m = nm | (old & (~0ull << (q - lo)));      // met the old chain at q: its exit stands
        else { m = nm; ex = q; }
      };
      unsigned long long mask = 0; uint32_t exit_q = 0;
      uint32_t entry = lane == 0 ? entry0 : lo;
      walk(min(entry, hi), 0ull, mask, exit_q);
      if (entry >= hi) { mask = 0; exit_q = entry; }                        // (lane 0 only: the entry lies beyond its segment)
      for (int round = 0; round < 34; round++) {
        const uint32_t x = __shfl_up_sync(FULL, exit_q, 1);
        bool changed = false;
        if (lane > 0 && x != entry) {
          entry = x; changed = true;
          if (x >= hi) { mask = 0; exit_q = x; }                            // the chain steps over this whole segment
          else walk(x, mask, mask, exit_q);
        }
        if (!__any_sync(FULL, changed)) break;
      }
      // symbols and code lengths per lane, then their prefix sums
      uint32_t nsym = (uint32_t)__popcll(mask), nlen = 0;
      for (unsigned long long m = mask; m; m &= m - 1ull) {
        const uint32_t t = tab[lo + (uint32_t)__ffsll((long long)m) - 1u];
        nlen += ((t >> 4) & 3u) ? (t >> 6) : 1u;
      }
      uint32_t ks = nsym, is = nlen;
      #pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const uint32_t a = __shfl_up_sync(FULL, ks, o), c = __shfl_up_sync(FULL, is, o);
        if (lane >= o) { ks += a; is += c; }
      }
      uint32_t k = k_base + ks - nsym, i = i_base + is - nlen;
      // records: symbols that start while i < total
      uint32_t last_q = 0xffffffffu;
      for (unsigned long long m = mask; m && i < total; m &= m - 1ull) {
        const uint32_t q = lo + (uint32_t)__ffsll((long long)m) - 1u, t = tab[q];
        chain[k++] = t | (i << 16);
        i += ((t >> 4) & 3u) ? (t >> 6) : 1u;
        if (i >= total) last_q = q + (t & 15u) + 1u;                        // this symbol completes the code lengths
      }
      const uint32_t fin = __ballot_sync(FULL, last_q != 0xffffffffu);
      const uint32_t tot_i = __shfl_sync(FULL, i_base + is, 31), tot_k = __shfl_sync(FULL, k_base + ks, 31), ex31 = __shfl_sync(FULL, exit_q, 31);
      if (fin) {
        const int fl = __ffs((int)fin) - 1;
        q_end = __shfl_sync(FULL, last_q, fl); k_base = __shfl_sync(FULL, k, fl);
        done = true;
      } else {
        i_base = tot_i; k_base = tot_k; entry0 = ex31; win_q += 32u * SEG; q_end = ex31;
        if (entry0 >= n_tab || win_q >= n_tab) done = true;                 // out of table / input with i < total
        if (done && lane == 0) C->err = n_tab == tab_cap ? INF_RETRY : INF_ERR_INPUT;    // (a format error found below wins)
      }
    }
    if (lane == 0) { C->last_lane = k_base; C->last_info = q_end; }
  }
  bar_sync<BAR_P, NT>();
  const uint32_t k = C->last_lane;
  for (uint32_t j = tid; j < k; j += NT) {
    const uint32_t c = chain[j];
    const uint32_t i0 = c >> 16, kind = (c >> 4) & 3u, pl = (c >> 6) & 255u, rep = kind ? pl : 1u;
    if (kind == 3u || (kind == 1u && i0 == 0u) || i0 + rep > total) { C->err = INF_ERR_TABLE; continue; }
    uint32_t val = kind == 0u ? pl : 0u;
    if (kind == 1u) {                  // repeat previous: the value of the nearest earlier symbol that is not a repeat
      uint32_t jj = j - 1u, cc = chain[jj];
      while (((cc >> 4) & 3u) == 1u && jj > 0u) cc = chain[--jj];
      val = ((cc >> 4) & 3u) == 0u ? (cc >> 6) & 255u : 0u;
    }
    for (uint32_t r = 0; r < rep; r++) C->cl[i0 + r] = (uint8_t)val;
  }
  bar_sync<BAR_P, NT>();
  if (C->err) return C->err;
  *end_pos = start_pos + C->last_info;
  if (C->cl[256] == 0) return INF_ERR_TABLE;
  return INF_OK;
}


// RESOLVE stage C: dataflow over the in-order match list.  RWARPS warps x 32 lanes x SLOTS matches are in flight,
// dealt statically (thread t, slot m takes the matches t + T m, + T SLOTS, ... with T = 32 RWARPS: the lowest
// unresolved match of the member is therefore always in flight and its sources are final, so the stage always makes
// progress).  The LZ77 dependency chains of sorted BAM data are 90-190 pieces deep per member (a record copies from the
// record in front of it): this stage is a latency chain, not a bandwidth problem, and what counts is the length of one
// hop = the dependent instructions of one loop iteration.  Hence: descriptors are prefetched one match ahead, the source is
// gathered in the DESTINATION's word frame (one funnel shift per word, no second alignment pass), periods < 8 are expanded
// in registers with byte permutes, all stores are predicated inside the asm (no branches), and a slot tests the map bits of
// exactly the source bytes it needs (partial pieces go as soon as their bytes are final).
// Ordering: a writer stores the piece and then clears its map bits; a reader loads the map and then the bytes.  Both are
// shared-memory accesses of one SM, performed in program order per warp; every member's CRC-32 is checked behind this stage.
__device__ __forceinline__ void sts_u32_if(uint32_t a, uint32_t v, bool on) { asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.u32 p, %2, 0;\n\t@p st.shared.u32 [%0], %1;\n\t}" ::"r"(a), "r"(v), "r"((uint32_t)on) : "memory"); }
__device__ __forceinline__ void sts_u8_if(uint32_t a, uint32_t v, bool on) { asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.u32 p, %2, 0;\n\t@p st.shared.u8 [%0], %1;\n\t}" ::"r"(a), "r"(v), "r"((uint32_t)on) : "memory"); }
template <int SLOTS, int RWARPS>
__device__ __forceinline__ void resolve_dataflow(uint32_t win_s, uint32_t hb_s, uint32_t list_s, uint32_t psel_s, uint32_t obase, uint32_t total, int tid, uint32_t* err) {
  constexpr uint32_t T = 32u * RWARPS;
  uint32_t o[SLOTS], dist[SLOTS], len[SLOTS], done[SLOTS], no[SLOTS], nv[SLOTS], nr[SLOTS];
  bool pend[SLOTS];
  auto load_desc = [&](uint32_t r, uint32_t& oo, uint32_t& vv) {
    oo = obase + lds_u16(list_s + r * 2u);
    const uint32_t a = win_s + (oo & ~3u);
    vv = __funnelshift_r(lds_u32(a), lds_u32(a + 4u), (oo & 3u) * 8u) & 0xffffffu;
  };
  #pragma unroll
  for (int m = 0; m < SLOTS; m++) {
    const uint32_t r = (uint32_t)tid + T * m;
    uint32_t v = 0;
    pend[m] = r < total; o[m] = obase + 4u; no[m] = obase + 4u; nv[m] = 0;
    if (pend[m]) load_desc(r, o[m], v);
    dist[m] = pend[m] ? (v & 0x7fffu) + 1u : 1u; len[m] = pend[m] ? (v >> 15) + 3u : 0u; done[m] = 0;
    nr[m] = r + T * SLOTS;
    if (nr[m] < total) load_desc(nr[m], no[m], nv[m]);
  }
  uint32_t spins = 0;
  for (;;) {
    bool anyp = false;
    #pragma unroll
    for (int m = 0; m < SLOTS; m++) anyp |= pend[m];
    if (!__any_sync(FULL, anyp)) break;
    uint32_t cur[SLOTS], sa[SLOTS], x[SLOTS], n[SLOTS], D[SLOTS][5];
    // phase 1: map bits of the source
    #pragma unroll
    for (int m = 0; m < SLOTS; m++) {
      cur[m] = o[m] + done[m];
      sa[m] = cur[m] - dist[m];
      const uint32_t wa = hb_s + ((sa[m] >> 5) << 2);
      x[m] = __funnelshift_r(lds_u32(wa), lds_u32(wa + 4u), sa[m] & 31u);
    }
    // phase 2: gather in the destination's word frame: D[j] = the source bytes that land in the word at (cur & ~3) + 4 j
    #pragma unroll
    for (int m = 0; m < SLOTS; m++) {
      const uint32_t f = sa[m] - (cur[m] & 3u);                      // (>= obase - 3: the window starts 16 bytes into shared memory)
      const uint32_t a = win_s + (f & ~3u), s8 = (f & 3u) * 8u;
      const uint32_t w0 = lds_u32(a), w1 = lds_u32(a + 4u), w2 = lds_u32(a + 8u), w3 = lds_u32(a + 12u), w4 = lds_u32(a + 16u), w5 = lds_u32(a + 20u);
      D[m][0] = __funnelshift_r(w0, w1, s8); D[m][1] = __funnelshift_r(w1, w2, s8); D[m][2] = __funnelshift_r(w2, w3, s8);
      D[m][3] = __funnelshift_r(w3, w4, s8); D[m][4] = __funnelshift_r(w4, w5, s8);
    }
    // phase 3: how many bytes of the piece can go now
    bool anyn = false, anywrap = false;
    #pragma unroll
    for (int m = 0; m < SLOTS; m++) {
      uint32_t want = min(len[m] - done[m], RESOLVE_PIECE);
      if (dist[m] < want && dist[m] >= 8u) want = dist[m];                         // (only periods < 8 are expanded in registers)
      const uint32_t outn = min(want, dist[m]);                                    // the piece's bytes that come from outside itself
      const uint32_t avail = x[m] ? (uint32_t)__ffs((int)x[m]) - 1u : 32u;         // final source bytes from sa on
      n[m] = avail >= outn ? want : (dist[m] >= want ? avail : 0u);
      if (!pend[m]) n[m] = 0;
      anyn |= n[m] != 0u; anywrap |= n[m] > dist[m];
    }
    if (!__any_sync(FULL, anyn)) {                                                 // nothing ready in this warp: another warp's piece comes first
      if (RWARPS == 1 || ++spins > (1u << 22)) { *err = INF_ERR_INPUT; break; }  // (one warp: cannot happen; else a safety valve, never taken)
      continue;
    }
    if (__any_sync(FULL, anywrap)) {                                               // a piece longer than its period: byte k is src[k mod dist]
      #pragma unroll
      for (int m = 0; m < SLOTS; m++) if (n[m] > dist[m]) {
        const uint32_t h8 = (cur[m] & 3u) * 8u;
        const uint32_t s0 = __funnelshift_r(D[m][0], D[m][1], h8), s1 = __funnelshift_r(D[m][1], D[m][2], h8);   // the 8 bytes at sa
        const uint32_t m0 = lds_u32(psel_s + dist[m] * 8u), m1 = lds_u32(psel_s + dist[m] * 8u + 4u);
        const uint32_t V0 = __byte_perm(s0, s1, m0 & 0xffffu), V1 = __byte_perm(s0, s1, m0 >> 16), V2 = __byte_perm(s0, s1, m1 & 0xffffu), V3 = __byte_perm(s0, s1, m1 >> 16);
        D[m][0] = V0 << h8; D[m][1] = __funnelshift_l(V0, V1, h8); D[m][2] = __funnelshift_l(V1, V2, h8); D[m][3] = __funnelshift_l(V2, V3, h8); D[m][4] = __funnelshift_l(V3, 0u, h8);
      }
    }
    // phase 4: store.  Word j holds the piece's bytes [4j - sh, 4j - sh + 4); whole words, then the ragged head and tail as bytes
    #pragma unroll
    for (int m = 0; m < SLOTS; m++) {
      const uint32_t sh = cur[m] & 3u, A = win_s + (cur[m] & ~3u), e = sh + n[m], ca = win_s + cur[m];
      sts_u32_if(A, D[m][0], sh == 0u && n[m] >= 4u);
      sts_u32_if(A + 4u, D[m][1], e >= 8u);
      sts_u32_if(A + 8u, D[m][2], e >= 12u);
      sts_u32_if(A + 12u, D[m][3], e >= 16u);
      sts_u32_if(A + 16u, D[m][4], e >= 20u);
      const uint32_t h = sh ? min(n[m], 4u - sh) : 0u, hv = D[m][0] >> (sh * 8u);
      sts_u8_if(ca, hv, h > 0u); sts_u8_if(ca + 1u, hv >> 8, h > 1u); sts_u8_if(ca + 2u, hv >> 16, h > 2u);
      const uint32_t jt = e >> 2, t = (e >= 4u || sh == 0u) ? (e & 3u) : 0u;
      const uint32_t Dt = jt == 0u ? D[m][0] : jt == 1u ? D[m][1] : jt == 2u ? D[m][2] : jt == 3u ? D[m][3] : D[m][4];
      const uint32_t ta = A + 4u * jt;
      sts_u8_if(ta, Dt, t > 0u); sts_u8_if(ta + 1u, Dt >> 8, t > 1u); sts_u8_if(ta + 2u, Dt >> 16, t > 2u);
    }
    // phase 5: the piece's bytes are final
    #pragma unroll
    for (int m = 0; m < SLOTS; m++) {
      const uint32_t wa = hb_s + ((cur[m] >> 5) << 2), b = cur[m] & 31u, mk = (1u << n[m]) - 1u;      // n <= 16
      and_shared_if(wa, ~(mk << b), n[m] != 0u);
      and_shared_if(wa + 4u, ~__funnelshift_r(mk, 0u, 32u - b), b + n[m] > 32u);
    }
    // phase 6: a finished slot adopts its prefetched next match and prefetches the one after
    #pragma unroll
    for (int m = 0; m < SLOTS; m++) {
      done[m] += n[m];
      if (pend[m] && done[m] == len[m]) {
        pend[m] = nr[m] < total;
        o[m] = no[m]; done[m] = 0;
        dist[m] = pend[m] ? (nv[m] & 0x7fffu) + 1u : 1u; len[m] = pend[m] ? (nv[m] >> 15) + 3u : 0u;
        nr[m] += T * SLOTS;
        if (nr[m] < total) load_desc(nr[m], no[m], nv[m]);
      }
    }
  }
}

// RESOLVE, whole member, consumer team (NTC threads).  `hb` holds one bit per parked match head on entry and is all zero
// on return.  The matches are taken in output-ordered batches of at most `list_cap`; this is exact, because a match's
// source bytes lie in front of its own bytes and hence in front of every later match.  Per batch:
//   A  every thread ranks the heads of its share of the bitmap words; a team scan turns the first list_cap of them into an
//      in-order list of head positions (u16, relative to obase) and clears their bits (later heads stay for the next batch);
//   B  the bitmap becomes the UNRESOLVED map of the batch: every byte of every listed match is flagged;
//   C  dataflow (resolve_dataflow above): a lane copies a piece (<= 16 bytes) of its match as soon as the map shows that the
//      piece's source bytes are final, then clears the piece's bits.  The lowest unresolved piece of the batch always has
//      final sources (earlier batches are done), so every iteration makes progress.
// Returns the number of batches.
template <int NTC>
__device__ __forceinline__ uint32_t resolve_member(uint8_t* win, uint32_t* hb, uint16_t* list, uint32_t list_cap, CCtl* CC,
                                                   uint32_t obase, uint32_t olimit, int tid) {
  constexpr int WARPS = NTC / 32;
  const int lane = tid & 31, warp = tid >> 5;
  const uint32_t wend = (olimit + 31u) >> 5;
  uint32_t wbeg = obase >> 5;
  for (uint32_t batch = 1;; batch++) {
    const uint32_t WPT = (wend - wbeg + NTC - 1) / NTC;             // bitmap words per thread (<= 17)
    // ---- A: rank + list
    const uint32_t w0 = wbeg + (uint32_t)tid * WPT, w1 = min(wend, w0 + WPT);
    uint32_t cnt = 0;
    for (uint32_t w = w0; w < w1; w++) cnt += __popc(hb[w]);
    uint32_t incl = cnt;
    #pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const uint32_t v = __shfl_up_sync(FULL, incl, o); if (lane >= o) incl += v; }
    if (lane == 31) CC->warp_tot[warp] = incl;
    bar_sync<BAR_C, NTC>();
    uint32_t base = 0, total = 0;
    #pragma unroll
    for (int w = 0; w < WARPS; w++) { const uint32_t t = CC->warp_tot[w]; if (w < warp) base += t; total += t; }
    const uint32_t n = min(total, list_cap);
    {
      uint32_t k = base + incl - cnt;
      for (uint32_t w = w0; w < w1 && k < n; w++) {
        uint32_t bits = hb[w];
        while (bits && k < n) { list[k++] = (uint16_t)(w * 32u + (uint32_t)__ffs((int)bits) - 1u - obase); bits &= bits - 1u; }
        hb[w] = bits;
      }
    }
    bar_sync<BAR_C, NTC>();
    // ---- B: unresolved map
    for (uint32_t r = tid; r < n; r += NTC) {
      const uint32_t o = obase + list[r];
      const uint32_t len = ((((uint32_t)win[o + 1] << 8) | ((uint32_t)win[o + 2] << 16)) >> 15) + 3u;
      uint32_t w = o >> 5, b = o & 31u, rem = len;
      while (rem) {
        const uint32_t m = min(rem, 32u - b);
        atomicOr(hb + w, (m == 32u ? 0xffffffffu : ((1u << m) - 1u)) << b);
        rem -= m; w++; b = 0;
      }
    }
    bar_sync<BAR_C, NTC>();
    // ---- C: dataflow
    resolve_dataflow<1, WARPS>(smem_u32(win), smem_u32(hb), smem_u32(list), smem_u32(CC->psel), obase, n, tid, &CC->err);
    if (total <= list_cap) return batch;                             // (uniform)
    bar_sync<BAR_C, NTC>();                                          // the list and the map are free again
    if (CC->err) return batch;
    wbeg = (obase + list[n - 1u]) >> 5;                              // the next batch's first head lies in this word or behind it
  }
}

// CRC tables of the strided CRC (see Cfg / the CRC stage below); one launch per device at init.
template <int NT>
__global__ void crc_tables_init_kernel(uint32_t* __restrict__ tabs) {
  const int t = threadIdx.x;      // 256 threads
  // standard byte table
  uint32_t c = (uint32_t)t;
  for (int k = 0; k < 8; k++) c = (c >> 1) ^ ((c & 1u) ? 0xEDB88320u : 0u);
  __shared__ uint32_t t0[256];
  t0[t] = c;
  __syncthreads();
  // x^(32*j) mod P: x^32 is the state after feeding 0x00000001... use repeated multiplication by x^32
  const uint32_t x32 = crc_mulmod(0x00800000u, crc_mulmod(0x00800000u, crc_mulmod(0x00800000u, 0x00800000u)));   // (x^8)^4
  if (t == 0) {
    uint32_t p = 0x80000000u;     // x^0 in the reflected domain
    for (int j = 0; j <= NT; j++) { tabs[1024 + j] = p; p = crc_mulmod(p, x32); }
  }
  __syncthreads();
  __threadfence();
  // slicing-by-4 tables T_k[b] = (b * x^(8k+8)) * x^(32*(NT-1)): standard tables times the stride operator
  uint32_t e = t0[t];
  const uint32_t stride = tabs[1024 + NT - 1];
  for (int k = 0; k < 4; k++) {
    tabs[k * 256 + t] = crc_mulmod(e, stride);
    e = t0[e & 0xffu] ^ (e >> 8);
  }
}

__device__ __forceinline__ uint32_t crc_byte_bitwise(uint32_t st, uint32_t b) {
  st ^= b;
  #pragma unroll
  for (int k = 0; k < 8; k++) st = (st >> 1) ^ ((st & 1u) ? 0xEDB88320u : 0u);
  return st;
}

// =============================================================================================
__global__ void __launch_bounds__(NT, 2)
inflate_cta_kernel(const uint8_t* __restrict__ comp, const BlockDesc* __restrict__ blocks, uint32_t n_blocks,
                   uint8_t* __restrict__ infl, uint32_t* __restrict__ status, uint32_t* __restrict__ ticket,
                   uint32_t* __restrict__ err_flag, uint32_t* __restrict__ retry_count, const uint32_t* __restrict__ crc_tabs, int check_crc,
                   unsigned long long* __restrict__ prof) {
  // prof (optional, profiling builds of the bench only): per-phase clock64() sums of producer thread 0 and consumer thread
  // NT_P, 16 slots per CTA: 0-5 producer phases, 6-8 consumer phases, 9 producer waits for the window, 10 consumer waits for
  // a member, 11 resolve batches, 12 count rounds, 13 members
  using K = Cfg;
  extern __shared__ __align__(128) unsigned char smem[];
  uint8_t* const win = smem + K::OFF_WIN;
  uint32_t* const hb = reinterpret_cast<uint32_t*>(smem + K::OFF_HB);
  CCtl* const CC = reinterpret_cast<CCtl*>(smem + K::OFF_CCTL);
  uint32_t* const pay = reinterpret_cast<uint32_t*>(smem + K::OFF_PAY);
  uint32_t* const lut_ll = reinterpret_cast<uint32_t*>(smem + K::OFF_LUT_LL);
  uint32_t* const lut_d = reinterpret_cast<uint32_t*>(smem + K::OFF_LUT_D);
  uint32_t* const laneE = reinterpret_cast<uint32_t*>(smem + K::OFF_LANE_E);
  Ctl* const C = reinterpret_cast<Ctl*>(smem + K::OFF_CTL);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const uint32_t win_s = smem_u32(win), pay_s = smem_u32(pay), hb_s = smem_u32(hb), ll_s = smem_u32(lut_ll), d_s = smem_u32(lut_d);

  for (uint32_t i = tid; i < K::HB_WORDS; i += NT) hb[i] = 0;
  if (tid == 0) mbar_init(&C->mbar, 1);
  if (tid < 8) {
    unsigned long long m = 0;
    for (uint32_t k = 0; k < 16; k++) m |= (unsigned long long)(tid ? k % (uint32_t)tid : 0u) << (4u * k);
    CC->psel[tid] = m;
  }
  if (tid == 0) CC->err = INF_OK;
  __syncthreads();                                                   // (the last CTA-wide barrier: from here on each team has its own)
  long long t_prev = prof ? clock64() : 0;
#define ICTA_PROF(slot) do { if (prof && (tid == 0 || tid == NT_P)) { const long long t_now = clock64(); prof[blockIdx.x * 16 + (slot)] += (unsigned long long)(t_now - t_prev); t_prev = t_now; } } while (0)

  if (warp < NT_P / 32) {
    // ================= PRODUCER: ticket, payload, headers, tables, count, emit =================
    uint32_t bar_parity = 0;
    bool have_win = false;                                           // (uniform over the team)
    auto acquire_window = [&]() {                                    // before the first window write of a member
      if (have_win) return;
      bar_sync<BAR_EMPTY, NT>();
      have_win = true;
      ICTA_PROF(9);
    };
    for (;;) {
      if (tid == 0) { C->ticket = atomicAdd(ticket, 1u); C->err = INF_OK; }
      psync();
      const uint32_t bi = C->ticket;
      if (bi >= n_blocks) break;
      const BlockDesc bd = blocks[bi];
      const uint8_t* const gpay = comp + bd.cdata_off;
      const uint32_t isize = bd.isize, clen = bd.cdata_len;
      const uint32_t obase = bd.uoff & 15u, olimit = obase + isize;
      uint32_t err = INF_OK;
      if (isize > 65536u) err = INF_RETRY;

      // ---- payload window: buffer byte 0 <-> payload byte buf_lo (negative: bytes in front of the payload, for 16-byte alignment)
      int32_t buf_lo = 0; uint32_t loaded = 0;
      auto load_payload = [&](uint32_t from_byte) {
        const uintptr_t a = reinterpret_cast<uintptr_t>(gpay + from_byte);
        const uint32_t ph = (uint32_t)(a & 15u);
        buf_lo = (int32_t)from_byte - (int32_t)ph;
        const uint32_t want = (clen - from_byte) + ph + 32u;                  // + slack: the reader looks up to 18 bytes ahead
        loaded = min((want + 15u) & ~15u, K::PAY_BYTES);
        psync();                                                             // everyone is done with the old contents
        if (tid == 0) {
          fence_proxy_async();
          mbar_expect_tx(&C->mbar, loaded);
          bulk_load(pay, reinterpret_cast<const void*>(a - ph), loaded, &C->mbar);
        }
        if (!mbar_wait(&C->mbar, bar_parity)) C->err = INF_ERR_INPUT;
        bar_parity ^= 1u;
        psync();
        if (C->err) err = C->err;
      };
      uint32_t abs_bit = 0;                                                  // position in the payload, in bits
      const uint32_t end_bit = clen * 8u;
      ICTA_PROF(0);
      if (!err) load_payload(0);
      ICTA_PROF(1);
      auto buf_bit = [&](uint32_t abit) { return abit - (uint32_t)(buf_lo * 8); };   // payload bit -> buffer bit (two's complement handles buf_lo < 0)
      auto has_tail = [&]() { return (int64_t)buf_lo + (int64_t)loaded >= (int64_t)clen + 32; };   // the buffer reaches the end of the payload
      auto covers = [&](uint32_t abit_end) {                                  // is [.., abit_end) inside the buffer (with look-ahead margin)?
        return has_tail() ? abit_end <= end_bit : (int64_t)abit_end <= ((int64_t)buf_lo + (int64_t)loaded - 32) * 8;
      };

      uint32_t outpos = obase;
      bool final_block = false;
      while (!final_block && !err) {
        // ---- block header (warp 0) ----
        if (abs_bit + 3u > end_bit) { err = INF_ERR_INPUT; break; }
        if (!covers(min(end_bit, abs_bit + 8u * 1024u))) { load_payload(abs_bit >> 3); if (err) break; }
        if (warp == 0) {
          SBits br; br.w = pay; br.pos = buf_bit(abs_bit);
          const uint32_t hdr = br.take(3);
          uint32_t e = INF_OK, btype = hdr >> 1, slen = 0;
          if (btype == 3) e = INF_ERR_BTYPE;
          else if (btype == 0) {
            br.pos = (br.pos + 7u) & ~7u;
            const uint32_t len = br.take(16), nlen = br.take(16);
            slen = len;
            if ((len ^ nlen) != 0xffffu) e = INF_ERR_STORED;
          } else if (btype == 1) {
            for (int i = lane; i < 288; i += 32) C->cl[i] = i < 144 ? 8 : i < 256 ? 9 : i < 280 ? 7 : 8;
            C->cl[288 + lane] = 5;                                 // all 32 distance codes: complete, and 30 / 31 decode as invalid
            if (lane == 0) { C->n_ll = 288; C->n_d = 32; }
          } else {
            e = read_precode_warp(br, lut_d + ROOT_D, C, lane);
          }
          if (lane == 0) { C->btype = btype; C->final_block = hdr & 1u; C->hdr_end = br.pos + (uint32_t)(buf_lo * 8); C->stored_len = slen; if (e) C->err = e; }
        }
        psync();
        if (C->btype == 2u && !C->err) {
          // code lengths, whole team; the symbol table aliases the (not yet built) LUTs, the chain records the lane arrays
          uint32_t endp = 0;
          const uint32_t e = read_code_lengths_cta<NT_P>(pay, buf_bit(C->hdr_end), buf_bit(end_bit), lut_d + ROOT_D, reinterpret_cast<uint16_t*>(lut_ll),
                                                         (K::LUT_LL_WORDS + ROOT_D) * 2u, laneE, C, tid, &endp);
          if (tid == 0) { if (e) C->err = e; else C->hdr_end = endp + (uint32_t)(buf_lo * 8); }
        }
        psync();
        ICTA_PROF(2);
        err = C->err;
        if (err) break;
        final_block = C->final_block != 0;
        abs_bit = C->hdr_end;
        const uint32_t btype = C->btype;
        if (btype == 0) {
          const uint32_t len = C->stored_len, from = abs_bit >> 3;
          if (from + len > clen || outpos + len > olimit) { err = INF_ERR_STORED; break; }
          acquire_window();
          for (uint32_t i = tid; i < len; i += NT_P) win[outpos + i] = __ldg(gpay + from + i);     // straight from global: any length
          outpos += len; abs_bit += 8u * len;
          psync();
          continue;
        }
        // ---- tables: prepared by warps 0 (litlen) and 1 (distance), root LUTs filled by everyone, second levels by warps 0 / 1 ----
        {
          const int n_ll = (int)C->n_ll, n_d = (int)C->n_d;
          // scratch in the lane arrays (free until the count pass): symbols sorted by (length, symbol) and every symbol's code
          uint16_t* const sorted_ll = reinterpret_cast<uint16_t*>(laneE), *const codes_ll = sorted_ll + 288, *const sorted_d = codes_ll + 288, *const codes_d = sorted_d + 32;
          uint32_t e = INF_OK;
          if (warp == 0) e = lut_prepare_warp<R_LL>(C->cl, n_ll, C, 0, sorted_ll, codes_ll, lane);
          else if (warp == 1) e = lut_prepare_warp<R_D>(C->cl + n_ll, n_d, C, 1, sorted_d, codes_d, lane);
          if (e && lane == 0) atomicMax(&C->err, e);
          psync();
          if (!C->err) {
            lut_fill_root<R_LL, false, NT_P>(lut_ll, SUB_LL, C, 0, sorted_ll, tid);
            lut_fill_root<R_D, true, NT_P>(lut_d, SUB_D, C, 1, sorted_d, tid);
          }
          psync();
          if (!C->err) {
            e = INF_OK;
            if (warp == 0) e = lut_sub_warp<R_LL, false>(C->cl, n_ll, lut_ll, SUB_LL, C, 0, codes_ll, lane);
            else if (warp == 1) e = lut_sub_warp<R_D, true>(C->cl + n_ll, n_d, lut_d, SUB_D, C, 1, codes_d, lane);
            if (e && lane == 0) atomicMax(&C->err, e);        // INF_RETRY (15) wins over a format error of the other table
          }
          psync();
          ICTA_PROF(3);
          err = C->err;
          if (err) break;
        }
        // ---- spans of the symbol stream ----
        bool block_done = false;
        while (!block_done && !err) {
          if (abs_bit >= end_bit) { err = INF_ERR_INPUT; break; }
          if (!has_tail() && !covers(abs_bit + (K::PAY_BYTES / 2u) * 8u)) { load_payload(abs_bit >> 3); if (err) break; }
          const uint32_t span_beg = buf_bit(abs_bit);
          const bool to_end = has_tail();
          const uint32_t span_end = to_end ? buf_bit(end_bit) : (uint32_t)(((int64_t)loaded - 32) * 8);
          uint32_t S = (span_end - span_beg + NT_P - 1) / NT_P;
          if (S < MIN_SUB_BITS) S = MIN_SUB_BITS;
          const uint32_t my_p = span_beg + (uint32_t)tid * S;
          const bool active = my_p < span_end;
          const uint32_t my_stop = min(my_p + S, span_end);
          // round 0 starts every lane but the first `ov` bits EARLY and only warms the chain up until the lane's own cut is
          // reached: by then it is almost always the true chain (self-synchronisation), so most spans need no second round
          const uint32_t ov = min(WARMUP_BITS, max(S, WARMUP_MIN_BITS));
          uint32_t my_s = (tid == 0 || my_p - span_beg <= ov) ? span_beg : my_p - ov;
          bool need = active;
          uint32_t my_e = 0, my_t = T_CROSS, my_n = 0, F = 0;
          for (int round = 0;; round++) {
            if (__any_sync(FULL, need)) {                       // (all lanes of a warp enter together: see decode_sub)
              const uint32_t from = round == 0 ? (tid == 0 ? span_beg : my_p) : my_s;
              const SubResult r = decode_sub<false>(need, pay_s, ll_s, d_s, my_s, from, my_stop, 0, 0, 0, 0, 0, nullptr);
              if (need) {
                my_e = r.end_bit; my_t = r.term; my_n = r.n_out;
                if (round == 0) {
                  my_s = r.first_bit;                           // 0xffffffff (chain ended inside the warm-up) never equals a predecessor's end
                  if (r.first_bit == 0xffffffffu) { my_e = my_p; my_t = T_CROSS; my_n = 0; }
                }
                laneE[tid] = my_e;
              }
            }
            if (tid == 0) C->first_term[round & 1] = NT_P - 1;
            psync();
            {
              const uint32_t m = __ballot_sync(FULL, !active || my_t != T_CROSS);
              if (m && lane == 0) {
                const int l = __ffs((int)m) - 1;
                atomicMin(&C->first_term[round & 1], (uint32_t)(warp * 32 + l));
              }
            }
            psync();
            // the lane found above is either inactive (chain ends one before it) or terminates the chain itself
            F = C->first_term[round & 1];
            need = false;
            if (active && tid > 0 && (uint32_t)tid <= F) {
              const uint32_t pe = laneE[tid - 1];
              if (pe != my_s) { my_s = pe; need = true; }
            }
            if (prof && tid == 0) prof[blockIdx.x * 16 + 12] += 1;
            if (!bar_or<BAR_P, NT_P>(need)) break;
            if (round > NT_P + 2) { err = INF_ERR_INPUT; break; }
          }
          ICTA_PROF(4);
          if (err) break;
          // F may name the first INACTIVE lane: the chain then ends at F - 1
          if ((uint32_t)tid == F) C->last_lane = active ? F : F - 1;
          psync();
          const uint32_t last = C->last_lane;
          if ((uint32_t)tid == last) C->last_info = my_t | (my_e << 2);
          // ---- exclusive scan of the byte counts of lanes 0..last ----
          const uint32_t cnt_n = ((uint32_t)tid <= last) ? my_n : 0u;
          uint32_t incl = cnt_n;
          #pragma unroll
          for (int o = 1; o < 32; o <<= 1) { const uint32_t v = __shfl_up_sync(FULL, incl, o); if (lane >= o) incl += v; }
          if (lane == 31) C->warp_tot[warp] = incl;
          psync();
          uint32_t wbase = 0, total = 0;
          #pragma unroll
          for (int w = 0; w < NT_P / 32; w++) { const uint32_t t = C->warp_tot[w]; if (w < warp) wbase += t; total += t; }
          const uint32_t last_t = C->last_info & 3u, last_e = C->last_info >> 2;
          if (last_t == T_BAD) { err = INF_ERR_SYMBOL; break; }
          if (outpos + total > olimit || total > 65536u) { err = INF_ERR_OVERRUN; break; }
          // ---- emit ----
          acquire_window();
          if ((uint32_t)(warp * 32) <= last) {
            uint32_t e2 = 0;
            decode_sub<true>((uint32_t)tid <= last, pay_s, ll_s, d_s, my_s, my_s, my_stop, win_s, hb_s, outpos + wbase + incl - cnt_n, obase, olimit, &e2);
            if (e2) atomicMax(&C->err, e2);
          }
          psync();
          ICTA_PROF(5);
          err = C->err;
          if (err) break;
          outpos += total;
          abs_bit = last_e + (uint32_t)(buf_lo * 8);
          if (last_t == T_EOB) block_done = true;
          else if (to_end) { err = INF_ERR_INPUT; break; }
        }
      }
      if (!err && outpos != olimit) err = outpos > olimit ? INF_ERR_OVERRUN : INF_ERR_ISIZE;

      if (!err) {
        // ---- hand the window over: the consumer resolves, checks and stores this member while the next one is decoded ----
        acquire_window();                                                    // (an empty member writes nothing, but is handed over all the same)
        fence_proxy_async();                                                 // window bytes -> the consumer's cp.async.bulk store
        if (tid == 0) { CC->h.bi = bi; CC->h.obase = obase; CC->h.isize = isize; CC->h.crc = bd.crc; CC->h.uoff = bd.uoff; }
        bar_arrive<BAR_FULL, NT>();
        have_win = false;
      } else {
        // rejected: leave clean state behind (no head bits); the producer keeps the window
        psync();
        if (have_win) for (uint32_t i = tid; i < K::HB_WORDS; i += NT_P) hb[i] = 0;
        if (tid == 0) {
          status[bi] = err;
          if (err == INF_RETRY) atomicAdd(retry_count, 1u);
          else atomicCAS(err_flag, 0u, (bi << 4) | err | 0x80000000u);
        }
      }
      if (prof && tid == 0) prof[blockIdx.x * 16 + 13] += 1;
      psync();
    }
    // end of the ticket stream
    acquire_window();
    if (tid == 0) CC->h.bi = HANDOFF_END;
    bar_arrive<BAR_FULL, NT>();
  } else {
    // ================= CONSUMER: resolve, CRC-32, ISIZE, store, status =================
    const int ct = tid - NT_P, cwarp = ct >> 5;
    uint16_t* const list = reinterpret_cast<uint16_t*>(smem + K::OFF_LIST);
    bar_arrive<BAR_EMPTY, NT>();                                             // the window starts empty
    for (;;) {
      bar_sync<BAR_FULL, NT>();
      ICTA_PROF(10);
      const Handoff h = CC->h;
      if (h.bi == HANDOFF_END) break;
      const uint32_t obase = h.obase, isize = h.isize;
      // ---- resolve ----
      const uint32_t nbatch = resolve_member<NT_C>(win, hb, list, K::LIST_CAP, CC, obase, obase + isize, ct);
      csync();
      uint32_t err = CC->err;
      if (prof && ct == 0) prof[blockIdx.x * 16 + 11] += nbatch;
      ICTA_PROF(6);

      // ---- CRC-32 from the window (strided slicing-by-4: thread t owns words t, t+NT_C, ...; tables read through L1) ----
      if (check_crc && !err) {
        const uint32_t* const ctab = crc_tabs;
        const uint32_t head = min(isize, (4u - (obase & 3u)) & 3u);           // bytes in front of the first aligned word
        const uint32_t nw = (isize - head) >> 2, tail = (isize - head) & 3u;
        const uint32_t* const words = reinterpret_cast<const uint32_t*>(win + obase + head);
        uint32_t st = 0;
        if (ct == 0) { st = 0xffffffffu; for (uint32_t k = 0; k < head; k++) st = crc_byte_bitwise(st, win[obase + k]); }
        uint32_t acc = 0, part = 0;
        if ((uint32_t)ct < nw) {
          acc = words[ct] ^ st;                                                // the running state folds into the first word
          uint32_t k = ct + NT_C;
          for (; k < nw; k += NT_C) {
            acc = __ldg(ctab + 3 * 256 + (acc & 0xffu)) ^ __ldg(ctab + 2 * 256 + ((acc >> 8) & 0xffu)) ^ __ldg(ctab + 256 + ((acc >> 16) & 0xffu)) ^ __ldg(ctab + (acc >> 24));
            acc ^= words[k];
          }
          // acc sits at word k_last = k - NT_C; it still has to cross (nw - k_last) words
          part = crc_mulmod(acc, __ldg(ctab + 1024 + (nw - (k - NT_C))));
        } else if (ct == 0) {
          part = st;                                                           // fewer than one word: only the head bytes
        }
        #pragma unroll
        for (int o = 16; o; o >>= 1) part ^= __shfl_xor_sync(FULL, part, o);
        if (lane == 0) CC->crc_part[cwarp] = part;
        csync();
        if (ct == 0) {
          uint32_t crc = 0;
          for (int w = 0; w < RWARPS; w++) crc ^= CC->crc_part[w];
          for (uint32_t k = 0; k < tail; k++) crc = crc_byte_bitwise(crc, win[obase + head + 4u * nw + k]);
          if (~crc != h.crc) CC->err = INF_ERR_CRC;
        }
        csync();
        err = CC->err;
        ICTA_PROF(7);
      }
      if (!err) {
        // ---- the window leaves the SM once: 16-byte aligned body by cp.async.bulk, ragged ends by byte stores ----
        uint8_t* const gout = infl + h.uoff;                                   // (gout + k) and (win + obase + k) are congruent mod 16
        const uint32_t head = min(isize, (16u - obase) & 15u);
        const uint32_t body = (isize - head) & ~15u, tailb = isize - head - body;
        if ((uint32_t)ct < head) gout[ct] = win[obase + ct];
        if ((uint32_t)ct < tailb) gout[head + body + ct] = win[obase + head + body + ct];
        if (body) {
          fence_proxy_async();
          csync();
          if (ct == 0) { bulk_store(gout + head, win + obase + head, body); bulk_store_wait_read(); }
        }
      } else {
        // leave clean state behind: no head or map bits
        for (uint32_t i = ct; i < K::HB_WORDS; i += NT_C) hb[i] = 0;
      }
      if (ct == 0) {
        status[h.bi] = err;
        if (err) { atomicCAS(err_flag, 0u, (h.bi << 4) | err | 0x80000000u); CC->err = INF_OK; }
      }
      csync();                                                               // (the store has read the window)
      ICTA_PROF(8);
      bar_arrive<BAR_EMPTY, NT>();
    }
    // a bulk store must have finished reading shared memory before the CTA exits; writes complete with the grid
    if (ct == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
  }
#undef ICTA_PROF
}

}  // namespace icta
}  // namespace bamscan
