// inflate_cta_core.h -- per-lane building blocks of the CTA-per-member inflate kernel (kernels_inflate_cta.cuh).
//
// Replaces (together with the kernel): noodles-bgzf 0.49.0 io::Reader block inflate + libdeflate `deflate_decompress`
// (reference call sites: datafusion/bio-format-bam/src/storage.rs:161-169, physical_exec.rs:409).
//
// Everything here is plain integer code over arrays (`pay` = the member's deflate payload as little-endian 32-bit words,
// `win` = the member's output window, `hb` = one "a parked match starts here" bit per window byte), written so that the SAME source is
// compiled into the kernel (arrays in shared memory, one call per thread) and into tools/inflate_sim.cpp, a host program
// that runs the lanes of a CTA in a loop -- the algorithm can be checked against zlib without a GPU.
//
// The algorithm (one CTA of NT lanes per BGZF member, all state in shared memory):
//   * a deflate block's symbol stream is cut into NT sub-streams at fixed bit positions; every lane decodes its own
//     sub-stream speculatively from the cut.  Huffman streams self-synchronise (measured on BAM data: half of the false
//     starts are on the true symbol chain after 6 symbols, 99 % after 46), so a lane's END position -- the first symbol
//     boundary at or after the next cut -- is almost always the true one even when its start was not;
//   * lanes then restart from their predecessor's end until nothing changes (lane 0 is exact, so lane i is exact after
//     at most i rounds; in practice two rounds).  This yields every lane's true start, its output byte count and the
//     lane holding the end-of-block symbol;
//   * an exclusive scan of the byte counts gives every lane its output offset; the lanes decode once more and EMIT:
//     literals go straight into the window, a match (len, dist) is parked in the first three bytes of its own
//     destination and its first byte is flagged in the head bitmap `hb`;
//   * RESOLVE (one warp, whole member, in output order): the head bitmap is read 32 words at a time, the matches of
//     the stripe are dealt to the lanes 32 at a time in position order, and a lane copies a piece (<= 16 bytes) of
//     its match as soon as the piece's source lies below the FRONTIER (the position of the first unfinished byte of
//     the batch: everything below it is final).  Measured on sorted BAM data the LZ77 dependency chains are ~120-190
//     matches deep per member (every record copies from the one before), i.e. ~33 independent matches per level:
//     one warp is the parallelism this stage has, and the frontier rule needs no flags, fences or polling.
#pragma once
#include <cstdint>

#if defined(__CUDACC__)
#define ICTA_HD __host__ __device__ __forceinline__
#else
#define ICTA_HD inline
#endif

namespace bamscan {
namespace icta {

constexpr int R_LL = 10, R_D = 8;                       // root LUT index bits (litlen / distance)
constexpr uint32_t ROOT_LL = 1u << R_LL, ROOT_D = 1u << R_D;
constexpr uint32_t SUB_LL = 512, SUB_D = 128;           // second-level entries available (a table that needs more is refused;
                                                        // a canonical lit/len code over <= 286 symbols never needs 512)

// 32-bit LUT entry (laid out for the fewest instructions in the decode step):
//   [4:0]   bits this half-token consumes: code length + extra bits (0 = unused code); E_SUB: index bits of the second level
//   [8:5]   code length (whole code, also in second-level entries)
//   [9] E_LIT literal   [10] E_SYM length / distance symbol   [11] E_EOB end of block   [12] E_SUB pointer to a second-level table
//   [31:16] literal byte | base length | base distance | E_SUB: index of the second-level table inside the LUT array
//   value = [31:16] + ((bits & mask([4:0])) >> [8:5])
constexpr uint32_t E_LIT = 1u << 9, E_SYM = 1u << 10, E_EOB = 1u << 11, E_SUB = 1u << 12, E_BAD = 0u;

enum Term : uint32_t { T_CROSS = 0, T_EOB = 1, T_BAD = 2 };    // how a lane's sub-stream decode ended
enum CoreErr : uint32_t { CE_OK = 0, CE_DIST = 5, CE_OVERRUN = 6 };   // values of InflateStatus (kernels_inflate.cuh)

ICTA_HD uint32_t entry_litlen(uint32_t sym, uint32_t len) {     // RFC 1951 3.2.5, computed arithmetically
  if (sym < 256u) return E_LIT | (len << 5) | len | (sym << 16);
  if (sym == 256u) return E_EOB | (len << 5) | len;
  const uint32_t s = sym - 257u;
  if (s > 28u) return E_BAD;
  const uint32_t extra = (s < 8u || s == 28u) ? 0u : (s - 4u) >> 2;
  const uint32_t base = s == 28u ? 258u : (s < 8u ? 3u + s : 3u + ((4u + (s & 3u)) << extra));
  return E_SYM | (len << 5) | (len + extra) | (base << 16);
}
ICTA_HD uint32_t entry_dist(uint32_t sym, uint32_t len) {
  if (sym > 29u) return E_BAD;
  const uint32_t extra = sym < 4u ? 0u : (sym - 2u) >> 1;
  const uint32_t base = sym < 4u ? 1u + sym : 1u + ((2u + (sym & 1u)) << extra);
  return E_SYM | (len << 5) | (len + extra) | (base << 16);
}
// Completeness rule of a lit/len or distance code, as zlib (inftrees.c) and libdeflate apply it.  `left` is the code space
// the lengths leave unused (0: complete), `n_codes` the number of used symbols, `n_len1` those of length 1.  An incomplete
// code is rejected unless it is empty (a distance code of a block without matches) or a single code of length 1 (its
// codeword is the bit 0; the bit 1 is an invalid code).  Over-subscription is checked separately.
ICTA_HD bool code_complete_ok(uint32_t left, uint32_t n_codes, uint32_t n_len1) {
  return left == 0u || n_codes == 0u || (n_codes == 1u && n_len1 == 1u);
}
ICTA_HD uint32_t entry_sub(uint32_t root_bits, uint32_t sub_bits, uint32_t index) { return E_SUB | (root_bits << 5) | sub_bits | (index << 16); }

#if defined(__CUDA_ARCH__)
ICTA_HD void bm_or(uint32_t* p, uint32_t m) { atomicOr(p, m); }
ICTA_HD void bm_and(uint32_t* p, uint32_t m) { atomicAnd(p, m); }
ICTA_HD void fence_cta() { __threadfence_block(); }
ICTA_HD uint32_t ld_volatile(const uint32_t* p) { return *reinterpret_cast<const volatile uint32_t*>(p); }
ICTA_HD uint32_t ffs32(uint32_t v) { return (uint32_t)__ffs((int)v); }
#else
ICTA_HD void bm_or(uint32_t* p, uint32_t m) { *p |= m; }
ICTA_HD void bm_and(uint32_t* p, uint32_t m) { *p &= m; }
ICTA_HD void fence_cta() {}
ICTA_HD uint32_t ld_volatile(const uint32_t* p) { return *p; }
ICTA_HD uint32_t ffs32(uint32_t v) { return (uint32_t)__builtin_ffs((int)v); }
#endif

struct SubResult { uint32_t end_bit, term, n_out, first_bit; };   // first_bit: first token boundary at or after count_from (0xffffffff: the chain ended before it)

// Decodes tokens from bit `start_bit` of `pay` until the first token boundary at or after `stop_bit`, an end-of-block
// symbol or an unused code.  EMIT = false: count only.  EMIT = true: literals and parked matches go into win[opos...]
// (obase = window offset of the member's first byte, olimit = window offset one past the member's last byte).
// A token is at most 48 bits; the caller guarantees that `pay` is readable 18 bytes past stop_bit.
//
// On the device ALL 32 lanes of a warp call this together (`enabled` = false for a lane with nothing to do): the loop
// condition is a warp vote, so the lanes re-converge after every token.  (A per-lane `while` with `continue` / `break`
// compiles to code whose lanes never re-converge inside the loop: measured, one active thread per issued instruction.)
#if !defined(__CUDACC__)
template <bool EMIT>
inline SubResult decode_sub(bool enabled, const uint32_t* pay, const uint32_t* lut_ll, const uint32_t* lut_d,
                            uint32_t start_bit, uint32_t count_from, uint32_t stop_bit,
                            uint8_t* win, uint32_t* hb, uint32_t opos, uint32_t obase, uint32_t olimit, uint32_t* err) {
  uint32_t wi = enabled ? (start_bit >> 5) : 0u;
  const uint32_t sh = start_bit & 31u;
  uint64_t buf = (((uint64_t)pay[wi + 1] << 32) | pay[wi]) >> sh;
  uint32_t cnt = 64u - sh;                                   // valid bits in buf
  wi += 2;
  uint32_t pos = start_bit, n_out = 0, term = T_CROSS, first_bit = 0xffffffffu;
  bool live = enabled && pos < stop_bit;
  while (live) {
    const bool counting = pos >= count_from;                 // tokens in front of count_from only warm the chain up
    if (counting && first_bit == 0xffffffffu) first_bit = pos;
    if (cnt <= 32u) { buf |= (uint64_t)pay[wi] << cnt; cnt += 32u; wi++; }
    uint32_t bits = (uint32_t)buf;
    uint32_t e = lut_ll[bits & (ROOT_LL - 1u)];
    if (e & E_SUB) e = lut_ll[(e >> 16) + ((bits >> R_LL) & ~(~0u << (e & 31u)))];
    uint32_t tot = e & 31u;
    const uint32_t len = (e >> 16) + ((bits & ~(~0u << tot)) >> ((e >> 5) & 15u));   // literal: its byte
    buf >>= tot; cnt -= tot; pos += tot;
    if (e & E_LIT) {
      if (EMIT) {
        if (opos >= olimit) { *err = CE_OVERRUN; term = T_BAD; }
        else { win[opos] = (uint8_t)len; opos++; }
      }
      if (counting) n_out++;
    } else if (e & E_SYM) {
      if (cnt <= 32u) { buf |= (uint64_t)pay[wi] << cnt; cnt += 32u; wi++; }
      bits = (uint32_t)buf;
      uint32_t de = lut_d[bits & (ROOT_D - 1u)];
      if (de & E_SUB) de = lut_d[(de >> 16) + ((bits >> R_D) & ~(~0u << (de & 31u)))];
      if (!(de & E_SYM)) term = T_BAD;
      else {
        tot = de & 31u;
        const uint32_t dist = (de >> 16) + ((bits & ~(~0u << tot)) >> ((de >> 5) & 15u));
        buf >>= tot; cnt -= tot; pos += tot;
        if (EMIT) {
          if (dist > opos - obase) { *err = CE_DIST; term = T_BAD; }
          else if (opos + len > olimit) { *err = CE_OVERRUN; term = T_BAD; }
          else {
            const uint32_t v = (dist - 1u) | ((len - 3u) << 15);   // parked in the match's own first three bytes
            win[opos] = (uint8_t)v; win[opos + 1] = (uint8_t)(v >> 8); win[opos + 2] = (uint8_t)(v >> 16);
            hb[opos >> 5] |= 1u << (opos & 31u);                    // head bit
            opos += len;
          }
        }
        if (counting) n_out += len;
      }
    } else {
      term = (e & E_EOB) ? T_EOB : T_BAD;
    }
    live = term == T_CROSS && pos < stop_bit;
  }
  if (first_bit == 0xffffffffu && term == T_CROSS && pos >= count_from) first_bit = pos;
  SubResult r; r.end_bit = pos; r.term = term; r.n_out = n_out; r.first_bit = first_bit;
  return r;
}
#else
// Device version: same contract, shared-memory state addresses (32-bit shared-window addresses), and ALL 32 lanes of a warp
// call it together (`enabled` = false for a lane with nothing to do).  The loop condition is a warp vote, so the lanes
// re-converge after every token; the body is straight-line predicated code: literal/length half, then the distance half,
// which every lane executes (a literal lane discards it).  A per-lane `while` with `continue` / `break` compiles to code
// whose lanes never re-converge inside the loop (measured: one active thread per issued instruction).
__device__ __forceinline__ uint32_t lds_u32(uint32_t a) { uint32_t v; asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(a)); return v; }
__device__ __forceinline__ void sts_u8(uint32_t a, uint32_t v) { asm volatile("st.shared.u8 [%0], %1;" ::"r"(a), "r"(v) : "memory"); }
template <bool EMIT>
__device__ __forceinline__ SubResult decode_sub_c(bool enabled, uint32_t pay_s, uint32_t ll_s, uint32_t d_s,
                                                uint32_t start_bit, uint32_t count_from, uint32_t stop_bit,
                                                uint32_t win_s, uint32_t hb_s, uint32_t opos, uint32_t obase, uint32_t olimit, uint32_t* err) {
  // One SYMBOL per iteration (literal/length or distance, selected by the lane's state), not one token: 63 % of the tokens
  // of BAM data are literals, and a token-per-iteration body makes every literal lane sit through the distance half.
  // The body is written for instruction count (it is ~45 % of the kernel's issued instructions): the table base, root mask
  // and root width of the lane's state live in registers, how the chain ended is worked out after the loop from the
  // entry that ended it, and a finished lane keeps executing with tot = 0.
  uint32_t wa = pay_s + ((enabled ? start_bit : 0u) >> 5) * 4u;
  const uint32_t sh = start_bit & 31u;
  uint64_t buf = (((uint64_t)lds_u32(wa + 4u) << 32) | lds_u32(wa)) >> sh;
  uint32_t cnt = 64u - sh;
  wa += 8u;
  uint32_t pos = start_bit, n_out = 0, first_bit = 0xffffffffu, len = 0, end_e = 0, emit_err = 0;
  uint32_t tb = ll_s, rmask = (ROOT_LL - 1u) << 2, rb = (uint32_t)R_LL;      // state 0: a token starts (literal/length table)
  bool st1 = false, ended = false;                                          // st1: the distance symbol of a match comes next
  bool live = enabled && pos < stop_bit;
  if (!EMIT) {
    // warm-up: symbols in front of count_from only bring the lane onto the true chain; nothing but their bit lengths matters
    bool warm = live && pos < count_from;
    while (__any_sync(0xffffffffu, warm)) {
      if (cnt <= 32u) { buf |= (uint64_t)lds_u32(wa) << cnt; cnt += 32u; wa += 4u; }
      const uint32_t bits = (uint32_t)buf;
      uint32_t e = lds_u32(tb + ((bits << 2) & rmask));
      if (e & E_SUB) e = lds_u32(tb + (((e >> 16) + ((bits >> rb) & ~(~0u << (e & 31u)))) << 2));
      const uint32_t tot = warm ? (e & 31u) : 0u;
      buf >>= tot; cnt -= tot; pos += tot;
      const bool sym = (e & E_SYM) != 0u;
      if (warm && !sym && (st1 || !(e & E_LIT))) { warm = false; live = false; ended = true; end_e = st1 ? 0u : e; }
      st1 = warm && sym && !st1;
      tb = st1 ? d_s : ll_s; rmask = st1 ? ((ROOT_D - 1u) << 2) : ((ROOT_LL - 1u) << 2); rb = st1 ? (uint32_t)R_D : (uint32_t)R_LL;
      warm = warm && (st1 || pos < count_from);
    }
    if (live) first_bit = pos;                                   // first token boundary at or after count_from
    live = live && pos < stop_bit;
  } else {
    if (live) first_bit = pos;
  }
  while (__any_sync(0xffffffffu, live)) {
    if (cnt <= 32u) { buf |= (uint64_t)lds_u32(wa) << cnt; cnt += 32u; wa += 4u; }            // (a symbol is at most 28 bits)
    const uint32_t bits = (uint32_t)buf;
    uint32_t e = lds_u32(tb + ((bits << 2) & rmask));
    if (e & E_SUB) e = lds_u32(tb + (((e >> 16) + ((bits >> rb) & ~(~0u << (e & 31u)))) << 2));
    const uint32_t tot = live ? (e & 31u) : 0u;
    const uint32_t val = (e >> 16) + ((bits & ~(~0u << tot)) >> ((e >> 5) & 15u));
    buf >>= tot; cnt -= tot; pos += tot;
    const bool sym = (e & E_SYM) != 0u;
    const bool lit = !st1 && (e & E_LIT) != 0u;
    if (live && !sym && !lit) { live = false; ended = true; end_e = st1 ? 0u : e; }            // end of block, or an unused code
    if (EMIT) {
      if (live && lit) {
        if (opos >= olimit) { emit_err = CE_OVERRUN; live = false; }
        else { sts_u8(win_s + opos, val); opos++; }
      }
      if (live && st1) {                                       // the distance symbol completes a match
        if (val > opos - obase) { emit_err = CE_DIST; live = false; }
        else if (opos + len > olimit) { emit_err = CE_OVERRUN; live = false; }
        else {
          const uint32_t v = (val - 1u) | ((len - 3u) << 15);     // parked in the match's own first three bytes
          sts_u8(win_s + opos, v); sts_u8(win_s + opos + 1u, v >> 8); sts_u8(win_s + opos + 2u, v >> 16);
          asm volatile("red.shared.or.b32 [%0], %1;" ::"r"(hb_s + ((opos >> 5) << 2)), "r"(1u << (opos & 31u)) : "memory");   // head bit
          opos += len;
        }
      }
    }
    if (live) n_out += st1 ? len : (lit ? 1u : 0u);
    if (!st1) len = val;
    st1 = live && sym && !st1;
    tb = st1 ? d_s : ll_s; rmask = st1 ? ((ROOT_D - 1u) << 2) : ((ROOT_LL - 1u) << 2); rb = st1 ? (uint32_t)R_D : (uint32_t)R_LL;
    live = live && (st1 || pos < stop_bit);
  }
  uint32_t term = T_CROSS;
  if (ended) term = (end_e & E_EOB) ? T_EOB : T_BAD;
  if (EMIT && emit_err) { *err = emit_err; term = T_BAD; }
  SubResult r; r.end_bit = pos; r.term = term; r.n_out = n_out; r.first_bit = first_bit;
  return r;
}

// The same three loops written in PTX.  The C++ version above (decode_sub_c, compiled with -DBAMSCAN_ICTA_DECODE_C) is
// the specification; nvcc turns its lane state into byte-sized booleans in general registers and spends 63-64 instructions
// per symbol in the warm-up and count loops and 102 in the emit loop.  Hand-scheduled predicates bring that down to
// 41 / 49 / 78.  Flag bits of a table entry: 512 literal, 1024 length/distance symbol, 2048 end of block, 4096 second level.
// A lane's state is the table it reads next: tb == ll_s <=> a token starts here.
#define ICTA_PTX_REGS \
  ".reg .pred pa, pany, pr, psub, psym, plit, pnl, pst, pend, pns, pc, pal, pm, pli, povr, pbd, pbl, pe;\n\t" \
  ".reg .b32 w, bits, idx, e, t, x, tot, v, a2, pk;\n\t" \
  ".reg .b64 w64;\n\t"
// refill + root look-up + second level; `pa` = lane active.  Leaves e, bits, tot.
#define ICTA_PTX_CORE \
  "setp.le.u32 pr, %1, 32;\n\t" \
  "@pr ld.shared.u32 w, [%2];\n\t" \
  "@pr cvt.u64.u32 w64, w;\n\t" \
  "@pr shl.b64 w64, w64, %1;\n\t" \
  "@pr or.b64 %0, %0, w64;\n\t" \
  "@pr add.u32 %1, %1, 32;\n\t" \
  "@pr add.u32 %2, %2, 4;\n\t" \
  "cvt.u32.u64 bits, %0;\n\t" \
  "shl.b32 idx, bits, 2;\n\t" \
  "and.b32 idx, idx, %5;\n\t" \
  "add.u32 idx, idx, %4;\n\t" \
  "ld.shared.u32 e, [idx];\n\t" \
  "and.b32 t, e, 4096;\n\t" \
  "setp.ne.u32 psub, t, 0;\n\t" \
  "@psub shr.u32 x, bits, %6;\n\t" \
  "@psub and.b32 t, e, 31;\n\t" \
  "@psub shl.b32 t, -1, t;\n\t" \
  "@psub not.b32 t, t;\n\t" \
  "@psub and.b32 x, x, t;\n\t" \
  "@psub shr.u32 t, e, 16;\n\t" \
  "@psub add.u32 x, x, t;\n\t" \
  "@psub shl.b32 x, x, 2;\n\t" \
  "@psub add.u32 x, x, %4;\n\t" \
  "@psub ld.shared.u32 e, [x];\n\t" \
  "and.b32 tot, e, 31;\n\t" \
  "selp.u32 tot, tot, 0, pa;\n\t"
// value of the symbol: base + extra bits
#define ICTA_PTX_VAL \
  "shl.b32 v, -1, tot;\n\t" \
  "not.b32 v, v;\n\t" \
  "and.b32 v, v, bits;\n\t" \
  "shr.u32 t, e, 5;\n\t" \
  "and.b32 t, t, 15;\n\t" \
  "shr.u32 v, v, t;\n\t" \
  "shr.u32 t, e, 16;\n\t" \
  "add.u32 v, v, t;\n\t"
#define ICTA_PTX_CONSUME \
  "shr.b64 %0, %0, tot;\n\t" \
  "sub.u32 %1, %1, tot;\n\t" \
  "add.u32 %3, %3, tot;\n\t"
// classification: psym, plit, pst (old state), pend (chain ends here), pal (still alive)
#define ICTA_PTX_CLASS(LIVE) \
  "and.b32 t, e, 1024;\n\t" \
  "setp.ne.u32 psym, t, 0;\n\t" \
  "and.b32 t, e, 512;\n\t" \
  "setp.ne.u32 plit, t, 0;\n\t" \
  "and.b32 t, e, 1536;\n\t" \
  "setp.eq.u32 pnl, t, 0;\n\t" \
  "and.pred pend, pa, pnl;\n\t" \
  "@pend mov.u32 " LIVE ", 0;\n\t" \
  "@pend mov.u32 %8, 1;\n\t" \
  "@pend mov.u32 %9, e;\n\t" \
  "setp.ne.u32 pst, %4, %15;\n\t" \
  "and.pred pal, pa, !pnl;\n\t"
// next state from pns
#define ICTA_PTX_NEXT \
  "selp.u32 %4, %16, %15, pns;\n\t" \
  "selp.u32 %5, 1020, 4092, pns;\n\t" \
  "selp.u32 %6, 8, 10, pns;\n\t"

template <bool EMIT>
__device__ __forceinline__ SubResult decode_sub(bool enabled, uint32_t pay_s, uint32_t ll_s, uint32_t d_s,
                                                uint32_t start_bit, uint32_t count_from, uint32_t stop_bit,
                                                uint32_t win_s, uint32_t hb_s, uint32_t opos, uint32_t obase, uint32_t olimit, uint32_t* err) {
#if defined(BAMSCAN_ICTA_DECODE_C)
  return decode_sub_c<EMIT>(enabled, pay_s, ll_s, d_s, start_bit, count_from, stop_bit, win_s, hb_s, opos, obase, olimit, err);
#else
  static_assert(R_LL == 10 && R_D == 8 && E_LIT == 512u && E_SYM == 1024u && E_EOB == 2048u && E_SUB == 4096u, "the PTX loops hard-code the table format");
  uint32_t wa = pay_s + ((enabled ? start_bit : 0u) >> 5) * 4u;
  const uint32_t sh = start_bit & 31u;
  unsigned long long buf = (((unsigned long long)lds_u32(wa + 4u) << 32) | lds_u32(wa)) >> sh;
  uint32_t cnt = 64u - sh;
  wa += 8u;
  uint32_t pos = start_bit, n_out = 0, first_bit = 0xffffffffu, len = 0, end_e = 0, emit_err = 0, ended = 0;
  uint32_t tb = ll_s, rmask = (ROOT_LL - 1u) << 2, rb = (uint32_t)R_LL;
  uint32_t live = (enabled && pos < stop_bit) ? 1u : 0u;
  // (read-only operands are passed "+r" too: a plain input whose value equals a read-write operand's -- tb starts as ll_s -- may be given the same register)
  uint32_t warm = 0;     // (operand numbers are shared by the three loops: %0 buf %1 cnt %2 wa %3 pos %4 tb %5 rmask %6 rb %7 live %8 ended %9 end_e
                         //  %10 warm %11 n_out %12 len %13 opos %14 emit_err | %15 ll_s %16 d_s %17 limit %18 win_s %19 hb_s %20 obase %21 olimit)
  if (!EMIT) {
    warm = (live && pos < count_from) ? 1u : 0u;
    asm volatile("{\n\t" ICTA_PTX_REGS
      "WLOOP:\n\t"
      "setp.ne.u32 pa, %10, 0;\n\t"
      "vote.sync.any.pred pany, pa, 0xffffffff;\n\t"
      "@!pany bra WDONE;\n\t"
      ICTA_PTX_CORE ICTA_PTX_CONSUME ICTA_PTX_CLASS("%10")
      "@pend mov.u32 %7, 0;\n\t"
      "and.pred pns, pal, psym;\n\t"
      "and.pred pns, pns, !pst;\n\t"
      ICTA_PTX_NEXT
      "setp.lt.u32 pc, %3, %17;\n\t"
      "or.pred pc, pc, pns;\n\t"
      "@!pc mov.u32 %10, 0;\n\t"
      "bra WLOOP;\n\t"
      "WDONE:\n\t}"
      : "+l"(buf), "+r"(cnt), "+r"(wa), "+r"(pos), "+r"(tb), "+r"(rmask), "+r"(rb), "+r"(live), "+r"(ended), "+r"(end_e), "+r"(warm), "+r"(n_out), "+r"(len), "+r"(opos), "+r"(emit_err),
        "+r"(ll_s), "+r"(d_s), "+r"(count_from), "+r"(win_s), "+r"(hb_s), "+r"(obase), "+r"(olimit) :: "memory");
    if (live) first_bit = pos;                                   // first token boundary at or after count_from
    live = (live && pos < stop_bit) ? 1u : 0u;
    // (the count loop stays C++: nvcc's version of it is 63 instructions, the PTX one 70)
    {
      bool st1 = false, lv = live != 0u;
      while (__any_sync(0xffffffffu, lv)) {
        if (cnt <= 32u) { buf |= (unsigned long long)lds_u32(wa) << cnt; cnt += 32u; wa += 4u; }
        const uint32_t bits = (uint32_t)buf;
        uint32_t e = lds_u32(tb + ((bits << 2) & rmask));
        if (e & E_SUB) e = lds_u32(tb + (((e >> 16) + ((bits >> rb) & ~(~0u << (e & 31u)))) << 2));
        const uint32_t tot = lv ? (e & 31u) : 0u;
        const uint32_t val = (e >> 16) + ((bits & ~(~0u << tot)) >> ((e >> 5) & 15u));
        buf >>= tot; cnt -= tot; pos += tot;
        const bool sym = (e & E_SYM) != 0u;
        const bool lit = (e & E_LIT) != 0u;
        if (lv && !sym && !lit) { lv = false; ended = 1u; end_e = e; }            // end of block, or an unused code
        if (lv) n_out += st1 ? len : (lit ? 1u : 0u);
        if (!st1) len = val;
        st1 = lv && sym && !st1;
        tb = st1 ? d_s : ll_s; rmask = st1 ? ((ROOT_D - 1u) << 2) : ((ROOT_LL - 1u) << 2); rb = st1 ? (uint32_t)R_D : (uint32_t)R_LL;
        lv = lv && (st1 || pos < stop_bit);
      }
    }
  } else {
    asm volatile("{\n\t" ICTA_PTX_REGS
      "ELOOP:\n\t"
      "setp.ne.u32 pa, %7, 0;\n\t"
      "vote.sync.any.pred pany, pa, 0xffffffff;\n\t"
      "@!pany bra EDONE;\n\t"
      ICTA_PTX_CORE ICTA_PTX_VAL ICTA_PTX_CONSUME ICTA_PTX_CLASS("%7")
      // literal: one byte into the window
      "and.pred pli, pal, plit;\n\t"
      "setp.ge.u32 povr, %13, %21;\n\t"
      "and.pred pe, pli, povr;\n\t"
      "@pe mov.u32 %14, 6;\n\t"
      "and.pred pli, pli, !povr;\n\t"
      "add.u32 a2, %18, %13;\n\t"
      "@pli st.shared.u8 [a2], v;\n\t"
      "@pli add.u32 %13, %13, 1;\n\t"
      // match (the distance symbol completes it): parked in its own first three bytes + head bit
      "and.pred pm, pal, pst;\n\t"
      "sub.u32 t, %13, %20;\n\t"
      "setp.gt.u32 pbd, v, t;\n\t"
      "add.u32 t, %13, %12;\n\t"
      "setp.gt.u32 pbl, t, %21;\n\t"
      "and.pred pbd, pbd, pm;\n\t"
      "@pbd mov.u32 %14, 5;\n\t"
      "and.pred pbl, pbl, pm;\n\t"
      "and.pred pbl, pbl, !pbd;\n\t"
      "@pbl mov.u32 %14, 6;\n\t"
      "or.pred pe, pe, pbd;\n\t"
      "or.pred pe, pe, pbl;\n\t"
      "@pe mov.u32 %7, 0;\n\t"
      "and.pred pm, pm, !pe;\n\t"
      "sub.u32 pk, %12, 3;\n\t"
      "shl.b32 pk, pk, 15;\n\t"
      "add.u32 pk, pk, v;\n\t"
      "sub.u32 pk, pk, 1;\n\t"
      "@pm st.shared.u8 [a2], pk;\n\t"
      "shr.u32 t, pk, 8;\n\t"
      "@pm st.shared.u8 [a2+1], t;\n\t"
      "shr.u32 t, pk, 16;\n\t"
      "@pm st.shared.u8 [a2+2], t;\n\t"
      "shr.u32 t, %13, 5;\n\t"
      "shl.b32 t, t, 2;\n\t"
      "add.u32 t, t, %19;\n\t"
      "and.b32 x, %13, 31;\n\t"
      "shl.b32 x, 1, x;\n\t"
      "@pm red.shared.or.b32 [t], x;\n\t"
      "@pm add.u32 %13, %13, %12;\n\t"
      "@!pst mov.u32 %12, v;\n\t"
      "and.pred pns, pal, psym;\n\t"
      "and.pred pns, pns, !pst;\n\t"
      "and.pred pns, pns, !pe;\n\t"
      ICTA_PTX_NEXT
      "setp.lt.u32 pc, %3, %17;\n\t"
      "or.pred pc, pc, pns;\n\t"
      "@!pc mov.u32 %7, 0;\n\t"
      "bra ELOOP;\n\t"
      "EDONE:\n\t}"
      : "+l"(buf), "+r"(cnt), "+r"(wa), "+r"(pos), "+r"(tb), "+r"(rmask), "+r"(rb), "+r"(live), "+r"(ended), "+r"(end_e), "+r"(warm), "+r"(n_out), "+r"(len), "+r"(opos), "+r"(emit_err),
        "+r"(ll_s), "+r"(d_s), "+r"(stop_bit), "+r"(win_s), "+r"(hb_s), "+r"(obase), "+r"(olimit) :: "memory");
  }
  uint32_t term = T_CROSS;
  if (ended) term = (end_e & E_EOB) ? T_EOB : T_BAD;
  if (EMIT && emit_err) { *err = emit_err; term = T_BAD; }
  SubResult r; r.end_bit = pos; r.term = term; r.n_out = n_out; r.first_bit = first_bit;
  return r;
#endif
}
#endif

constexpr uint32_t RESOLVE_PIECE = 16;   // bytes a lane copies per round of the resolver (longer matches continue in the next round)

}  // namespace icta
}  // namespace bamscan
