// inflate_sim.cpp -- host model of the CTA-per-member inflate kernel (kernels_inflate_cta.cuh).
//
// Runs the kernel's algorithm (speculative sub-stream decode -> restart rounds -> scan -> emit -> resolve) with the
// lanes of a CTA executed in a loop, using the very same per-lane code (csrc/inflate_cta_core.h), and compares every
// BGZF member of a file with zlib.  Test/verification tool only: nothing in the product links it.
//
//   inflate_sim file.bam [--lanes 256] [--max-members N] [--span-bytes B] [--overlap BITS] [--stats]
//                        [--resolve MODE] [--piece BYTES] [--rlanes N] [--gate G] [--group-sync] [--list-cap N]
// --resolve: 0 the round-2 v3 resolver (eight polling warps, groups of 32), 1 / 2 one warp in order with the frontier rule
// (groups / rolling), 3 rolling + exact readiness, 4 static lane-strided + exact readiness, 6 the COMMITTED resolver (all warps,
// static, exact readiness; --gate models the measured-and-dropped gate; --list-cap N resolves in output-ordered batches of at most
// N matches, as the kernel does), 7 list-free dealing by bitmap word (292 rounds: dropped).
#include <zlib.h>

#include <algorithm>
#include <array>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "../datafusion-bio-formats_b200/csrc/inflate_cta_core.h"

using namespace bamscan::icta;

static const uint8_t kClcOrder[19] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};

struct Bits {
  const uint32_t* w; uint32_t pos;
  uint32_t peek(int n) const { uint64_t v = (((uint64_t)w[(pos >> 5) + 1] << 32) | w[pos >> 5]) >> (pos & 31); return (uint32_t)(v & ((1ull << n) - 1)); }
  uint32_t take(int n) { uint32_t v = peek(n); pos += n; return v; }
};

// serial canonical build in the kernel's table format: root LUT of RBITS index bits + second-level tables behind it.
// Returns 0 ok, 1 over-subscribed or incomplete (code_complete_ok), 2 second-level space exhausted.
template <int RBITS, bool DIST>
static int build_lut(const uint8_t* cl, int n, uint32_t* lut, uint32_t sub_cap) {
  const uint32_t ROOT = 1u << RBITS;
  int cnt[16] = {0};
  for (int i = 0; i < n; i++) cnt[cl[i]]++;
  cnt[0] = 0;
  uint32_t first[17], code = 0; int left = 1;
  for (int L = 1; L <= 15; L++) { code = (code + (L > 1 ? cnt[L - 1] : 0)) << 1; first[L] = code; left <<= 1; left -= cnt[L]; if (left < 0) return 1; }
  uint32_t n_codes = 0; for (int L = 1; L <= 15; L++) n_codes += cnt[L];
  if (!code_complete_ok((uint32_t)left, n_codes, (uint32_t)cnt[1])) return 1;
  for (uint32_t i = 0; i < ROOT + sub_cap; i++) lut[i] = E_BAD;
  uint32_t next[16]; for (int L = 1; L <= 15; L++) next[L] = first[L];
  // per root prefix: index bits of its second-level table
  std::vector<uint8_t> sub_bits(ROOT, 0);
  std::vector<uint32_t> codes(n, 0);
  for (int s = 0; s < n; s++) {
    int L = cl[s]; if (!L) continue;
    uint32_t c = next[L]++; codes[s] = c;
    if (L > RBITS) { uint32_t q = c >> (L - RBITS); sub_bits[q] = std::max<uint8_t>(sub_bits[q], (uint8_t)(L - RBITS)); }
  }
  std::vector<uint32_t> sub_base(ROOT, 0);
  uint32_t used = 0;
  for (uint32_t q = 0; q < ROOT; q++) if (sub_bits[q]) { sub_base[q] = ROOT + used; used += 1u << sub_bits[q]; }
  if (used > sub_cap) return 2;
  auto rev = [](uint32_t v, int bits) { uint32_t r = 0; for (int i = 0; i < bits; i++) r |= ((v >> i) & 1u) << (bits - 1 - i); return r; };
  for (uint32_t q = 0; q < ROOT; q++) if (sub_bits[q]) lut[rev(q, RBITS)] = entry_sub(RBITS, sub_bits[q], sub_base[q]);
  for (int s = 0; s < n; s++) {
    int L = cl[s]; if (!L) continue;
    uint32_t e = DIST ? entry_dist((uint32_t)s, (uint32_t)L) : entry_litlen((uint32_t)s, (uint32_t)L);
    uint32_t c = codes[s];
    if (L <= RBITS) { for (uint32_t idx = rev(c, L); idx < ROOT; idx += 1u << L) lut[idx] = e; }
    else {
      uint32_t q = c >> (L - RBITS); int sb = sub_bits[q], l2 = L - RBITS;
      uint32_t low = rev(c & ((1u << l2) - 1), l2);
      for (uint32_t idx = low; idx < (1u << sb); idx += 1u << l2) lut[sub_base[q] + idx] = e;
    }
  }
  return 0;
}

struct Stats { long members = 0, blocks = 0, spans = 0, rounds = 0, lane_decodes = 0, lane_slots = 0, resolve_iters = 0, resolve_steps_max = 0, sub_overflow = 0, resolve_batches = 0, matches_max = 0, list_batches = 0; };


// Host model of the kernel's resolver (resolve_member in kernels_inflate_cta.cuh): in-order list of match heads, the
// head bitmap turned into an "unresolved" map, then W warps taking groups of 32 consecutive matches round-robin.  The
// warps are stepped one iteration at a time in turn, so a lane really does wait for another warp's progress here.
static int resolve_member_model(uint8_t* win, uint32_t* hb, uint32_t obase, uint32_t olimit, int W, Stats& S) {
  const uint32_t wbeg = obase >> 5, wend = (olimit + 31) >> 5;
  std::vector<uint16_t> list;
  for (uint32_t w = wbeg; w < wend; w++) { uint32_t bits = hb[w]; hb[w] = 0; while (bits) { list.push_back((uint16_t)(w * 32 + __builtin_ctz(bits) - obase)); bits &= bits - 1; } }
  const uint32_t total = (uint32_t)list.size();
  for (uint32_t r = 0; r < total; r++) {
    uint32_t o = obase + list[r], len = (((win[o + 1] << 8) | (win[o + 2] << 16)) >> 15) + 3;
    for (uint32_t k = 0; k < len; k++) hb[(o + k) >> 5] |= 1u << ((o + k) & 31);
  }
  struct Lane { uint32_t o, dist, len, done; bool pend; };
  struct Warp { uint32_t g; bool loaded, finished; Lane l[32]; };
  std::vector<Warp> ws(W);
  for (int w = 0; w < W; w++) { ws[w].g = w; ws[w].loaded = false; ws[w].finished = (uint32_t)w * 32 >= total; }
  int left = 0; for (auto& w : ws) if (!w.finished) left++;
  long idle_turns = 0;
  while (left) {
    bool progressed = false;
    for (int wi = 0; wi < W; wi++) {
      Warp& w = ws[wi];
      if (w.finished) continue;
      if (!w.loaded) {
        for (int l = 0; l < 32; l++) {
          uint32_t r = w.g * 32 + l; Lane& L = w.l[l]; L.pend = r < total; L.done = 0; L.o = 0; L.dist = 1; L.len = 0;
          if (L.pend) { L.o = obase + list[r]; uint32_t v = win[L.o] | (win[L.o + 1] << 8) | (win[L.o + 2] << 16); L.dist = (v & 0x7fff) + 1; L.len = (v >> 15) + 3; }
        }
        w.loaded = true; S.resolve_batches++;
      }
      // one iteration of the warp's loop
      bool ok[32]; uint32_t n[32]; bool any_ok = false, any_pend = false;
      for (int l = 0; l < 32; l++) {
        Lane& L = w.l[l]; ok[l] = false; n[l] = 0;
        if (!L.pend) continue;
        any_pend = true;
        uint32_t cur = L.o + L.done; n[l] = std::min(L.len - L.done, RESOLVE_PIECE);
        uint32_t sa = cur - L.dist, sb = std::min(cur, sa + n[l]);
        bool clear = true; for (uint32_t x = sa; x < sb; x++) if (hb[x >> 5] >> (x & 31) & 1) clear = false;
        ok[l] = clear; any_ok |= clear;
      }
      if (!any_pend) { w.g += W; w.loaded = false; if (w.g * 32 >= total) { w.finished = true; left--; } progressed = true; continue; }
      S.resolve_iters++;
      if (!any_ok) continue;
      progressed = true;
      for (int l = 0; l < 32; l++) if (ok[l]) {            // loads first (all sources are final), then stores
        Lane& L = w.l[l]; uint32_t cur = L.o + L.done, sa = cur - L.dist; uint8_t v[16]; uint32_t j = 0;
        for (uint32_t k = 0; k < n[l]; k++) { v[k] = win[sa + j]; if (++j == L.dist) j = 0; }
        for (uint32_t k = 0; k < n[l]; k++) win[cur + k] = v[k];
      }
      for (int l = 0; l < 32; l++) if (ok[l]) {
        Lane& L = w.l[l]; uint32_t cur = L.o + L.done;
        for (uint32_t k = 0; k < n[l]; k++) hb[(cur + k) >> 5] &= ~(1u << ((cur + k) & 31));
        L.done += n[l]; L.pend = L.done < L.len;
      }
    }
    if (!progressed && ++idle_turns > 4) return 52;       // stalled: cannot happen (the lowest unresolved piece is always ready)
    if (progressed) idle_turns = 0;
  }
  return 0;
}


// Host model of the IN-ORDER resolver (one warp, frontier rule).  mode 1: a group of 32 consecutive matches at a time;
// mode 2: rolling (a lane that finishes takes the next match of the list at once).  Returns warp iterations via S.
static uint32_t g_piece = 16; static int g_lanes = 32;
static int resolve_inorder_model(uint8_t* win, uint32_t* hb, uint32_t obase, uint32_t olimit, int mode, Stats& S) {
  const uint32_t wbeg = obase >> 5, wend = (olimit + 31) >> 5;
  std::vector<uint16_t> list;
  for (uint32_t w = wbeg; w < wend; w++) { uint32_t bits = hb[w]; hb[w] = 0; while (bits) { list.push_back((uint16_t)(w * 32 + __builtin_ctz(bits) - obase)); bits &= bits - 1; } }
  const uint32_t total = (uint32_t)list.size();
  struct Lane { uint32_t o, dist, len, done; bool pend; };
  std::vector<Lane> L(g_lanes); for (auto& l : L) l.pend = false;
  std::vector<uint8_t> fin(olimit + 64, 1);
  if (mode >= 3) for (uint32_t r = 0; r < total; r++) { uint32_t o = obase + list[r], len = (((win[o + 1] << 8) | (win[o + 2] << 16)) >> 15) + 3; for (uint32_t k = 0; k < len; k++) fin[o + k] = 0; }
  uint32_t next = 0;
  std::vector<uint32_t> lane_next(g_lanes); for (int i = 0; i < g_lanes; i++) lane_next[i] = i;
  auto fetch_static = [&](Lane& l, int i) { if (lane_next[i] >= total) return; l.o = obase + list[lane_next[i]]; lane_next[i] += g_lanes; uint32_t v = win[l.o] | (win[l.o + 1] << 8) | (win[l.o + 2] << 16); l.dist = (v & 0x7fff) + 1; l.len = (v >> 15) + 3; l.done = 0; l.pend = true; };
  auto fetch = [&](Lane& l) { if (next >= total) return; l.o = obase + list[next++]; uint32_t v = win[l.o] | (win[l.o + 1] << 8) | (win[l.o + 2] << 16); l.dist = (v & 0x7fff) + 1; l.len = (v >> 15) + 3; l.done = 0; l.pend = true; };
  for (;;) {
    bool any = false; for (auto& l : L) any |= l.pend;
    if (mode == 1) { if (!any) { if (next >= total) break; for (auto& l : L) fetch(l); S.resolve_batches++; } }
    else if (mode == 4) { for (int i = 0; i < g_lanes; i++) if (!L[i].pend) fetch_static(L[i], i); any = false; for (auto& l : L) any |= l.pend; if (!any) break; }
    else { for (auto& l : L) if (!l.pend) fetch(l); any = false; for (auto& l : L) any |= l.pend; if (!any) break; }
    S.resolve_iters++;
    uint32_t F = 0xffffffffu; for (auto& l : L) if (l.pend) F = std::min(F, l.o + l.done);
    std::vector<uint32_t> n(g_lanes); int nok = 0;
    for (int i = 0; i < g_lanes; i++) {
      Lane& l = L[i]; n[i] = 0; if (!l.pend) continue;
      uint32_t cur = l.o + l.done, sa = cur - l.dist, want = std::min(l.len - l.done, g_piece);
      if (mode >= 3) { uint32_t k = 0; while (k < want && (sa + k >= cur || fin[sa + k])) k++; n[i] = k; }
      else if (sa >= l.o || F >= cur) n[i] = want; else if (F > sa) n[i] = std::min(want, F - sa);
      if (n[i]) nok++;
    }
    if (!nok) return 52;
        std::vector<std::array<uint8_t,64>> v(g_lanes);
    for (int i = 0; i < g_lanes; i++) if (n[i]) { Lane& l = L[i]; uint32_t cur = l.o + l.done, sa = cur - l.dist, j = 0; for (uint32_t k = 0; k < n[i]; k++) { v[i][k] = win[sa + j]; if (++j == l.dist) j = 0; } }
    for (int i = 0; i < g_lanes; i++) if (n[i]) { Lane& l = L[i]; uint32_t cur = l.o + l.done; for (uint32_t k = 0; k < n[i]; k++) { win[cur + k] = v[i][k]; fin[cur + k] = 1; } l.done += n[i]; l.pend = l.done < l.len; }
  }
  return 0;
}

// Host model of the multi-warp STATIC dataflow resolver (resolve_dataflow in kernels_inflate_cta.cuh): W warps x 32 lanes,
// thread t takes matches t, t + 32 W, ...  `group_sync`: a warp adopts its next 32 matches only when all 32 current ones
// are done, and (gate >= 0) starts polling a group only when the group `gate` groups in front of it is complete.
// All warps execute one iteration per round (lockstep): rounds ~ latency, polls ~ issued iterations.
// `list_cap` > 0: the kernel's batched form -- the matches in output order, at most list_cap at a time, each batch's map built
// only when the batch before it is done (exact: a match's sources lie in front of it, hence in front of every later match).
static int g_gate = -1; static bool g_group_sync = false; static uint32_t g_list_cap = 0;
static int resolve_static_batch(uint8_t* win, const uint16_t* list, uint32_t total, uint32_t obase, uint32_t olimit, int W, Stats& S);
static int resolve_static_model(uint8_t* win, uint32_t* hb, uint32_t obase, uint32_t olimit, int W, Stats& S) {
  const uint32_t wbeg = obase >> 5, wend = (olimit + 31) >> 5;
  std::vector<uint16_t> list;
  for (uint32_t w = wbeg; w < wend; w++) { uint32_t bits = hb[w]; hb[w] = 0; while (bits) { list.push_back((uint16_t)(w * 32 + __builtin_ctz(bits) - obase)); bits &= bits - 1; } }
  const uint32_t all = (uint32_t)list.size(), cap = g_list_cap ? g_list_cap : std::max(1u, all);
  S.matches_max = std::max<long>(S.matches_max, all);
  for (uint32_t b = 0; b < all; b += cap) {
    S.list_batches++;
    if (int rc = resolve_static_batch(win, list.data() + b, std::min(cap, all - b), obase, olimit, W, S)) return rc;
  }
  return 0;
}
static int resolve_static_batch(uint8_t* win, const uint16_t* list, uint32_t total, uint32_t obase, uint32_t olimit, int W, Stats& S) {
  std::vector<uint8_t> fin(olimit + 64, 1);
  for (uint32_t r = 0; r < total; r++) { uint32_t o = obase + list[r], len = (((win[o + 1] << 8) | (win[o + 2] << 16)) >> 15) + 3; for (uint32_t k = 0; k < len; k++) fin[o + k] = 0; }
  const int T = 32 * W;
  struct Lane { uint32_t o, dist, len, done, r; bool pend; };
  std::vector<Lane> L(T);
  const uint32_t ngroups = (total + 31) / 32;
  std::vector<uint32_t> grp_left(ngroups + 1, 0);
  for (uint32_t r = 0; r < total; r++) grp_left[r / 32]++;
  auto load = [&](Lane& l, uint32_t r) { l.r = r; l.pend = r < total; l.done = 0; if (!l.pend) return; l.o = obase + list[r]; uint32_t v = win[l.o] | (win[l.o + 1] << 8) | (win[l.o + 2] << 16); l.dist = (v & 0x7fff) + 1; l.len = (v >> 15) + 3; };
  for (int t = 0; t < T; t++) load(L[t], t);
  long rounds = 0, polls = 0, cheap = 0;
  for (;;) {
    bool any = false; for (auto& l : L) any |= l.pend;
    if (!any) break;
    rounds++;
    std::vector<std::pair<int, uint32_t>> todo;   // decisions from the state at the start of the round
    std::vector<char> warp_real(W, 0);
    for (int w = 0; w < W; w++) {
      bool wp = false; uint32_t ming = 0xffffffffu;
      for (int l = 0; l < 32; l++) if (L[w * 32 + l].pend) { wp = true; ming = std::min(ming, L[w * 32 + l].r / 32); }
      if (!wp) continue;
      if (g_gate >= 0 && ming >= (uint32_t)g_gate && grp_left[ming - g_gate] != 0) { cheap++; continue; }   // gated: one-word poll
      polls++; warp_real[w] = 1;
      for (int l = 0; l < 32; l++) {
        Lane& a = L[w * 32 + l]; if (!a.pend) continue;
        uint32_t cur = a.o + a.done, sa = cur - a.dist, want = std::min(a.len - a.done, g_piece);
        if (a.dist < want && a.dist >= 8) want = a.dist;
        uint32_t outn = std::min(want, a.dist), k = 0; while (k < outn && fin[sa + k]) k++;
        uint32_t n = k >= outn ? want : (a.dist >= want ? k : 0);
        if (n) { todo.push_back({w * 32 + l, n}); warp_real[w] = 2; }
      }
    }
    if (todo.empty() && cheap > 100000000) return 52;
    for (auto& td : todo) { Lane& a = L[td.first]; uint32_t cur = a.o + a.done, sa = cur - a.dist, j = 0; uint8_t v[64]; for (uint32_t k = 0; k < td.second; k++) { v[k] = win[sa + j]; if (++j == a.dist) j = 0; } for (uint32_t k = 0; k < td.second; k++) { win[cur + k] = v[k]; fin[cur + k] = 1; } a.done += td.second; if (a.done == a.len) { a.pend = false; grp_left[a.r / 32]--; } }
    for (int w = 0; w < W; w++) {
      if (g_group_sync) { bool wp = false; for (int l = 0; l < 32; l++) wp |= L[w * 32 + l].pend; if (!wp) for (int l = 0; l < 32; l++) { Lane& a = L[w * 32 + l]; if (a.r < total) load(a, a.r + T); } }
      else for (int l = 0; l < 32; l++) { Lane& a = L[w * 32 + l]; if (!a.pend && a.r < total) load(a, a.r + T); }
    }
    if (rounds > 10000000) return 52;
  }
  S.resolve_iters += polls; S.resolve_batches += rounds; S.lane_slots += cheap;
  return 0;
}

// Host model of a LIST-FREE resolver: the matches are dealt by head-bitmap WORD (32 output bytes): thread t owns the words
// t, t + T, ... and resolves the matches whose heads lie in its current word one after the other, then moves to its next
// word.  Lock-step rounds as in resolve_static_model.
static int resolve_word_model(uint8_t* win, uint32_t* hb, uint32_t obase, uint32_t olimit, int W, Stats& S) {
  const uint32_t wbeg = obase >> 5, wend = (olimit + 31) >> 5;
  std::vector<uint32_t> heads(hb + wbeg, hb + wend);
  std::vector<uint8_t> fin(olimit + 64, 1);
  for (uint32_t w = wbeg; w < wend; w++) { uint32_t bits = hb[w]; hb[w] = 0; while (bits) { uint32_t o = w * 32 + __builtin_ctz(bits); bits &= bits - 1; uint32_t len = (((win[o + 1] << 8) | (win[o + 2] << 16)) >> 15) + 3; for (uint32_t k = 0; k < len; k++) fin[o + k] = 0; } }
  const int T = 32 * W;
  struct Lane { uint32_t w, bits, o, dist, len, done; bool pend; };
  std::vector<Lane> L(T);
  const uint32_t nw = wend - wbeg;
  auto next_match = [&](Lane& l) {   // take the next head of the current word, or move on to the next owned word
    for (;;) {
      if (l.bits) { l.o = (wbeg + l.w) * 32 + __builtin_ctz(l.bits); l.bits &= l.bits - 1; uint32_t v = win[l.o] | (win[l.o + 1] << 8) | (win[l.o + 2] << 16); l.dist = (v & 0x7fff) + 1; l.len = (v >> 15) + 3; l.done = 0; l.pend = true; return; }
      l.w += T; if (l.w >= nw) { l.pend = false; l.w = nw; return; } l.bits = heads[l.w];
    }
  };
  for (int t = 0; t < T; t++) { L[t].w = t; L[t].pend = false; if ((uint32_t)t < nw) { L[t].bits = heads[t]; next_match(L[t]); } else L[t].w = nw; }
  long rounds = 0, polls = 0;
  for (;;) {
    bool any = false; for (auto& l : L) any |= l.pend;
    if (!any) break;
    rounds++;
    std::vector<std::pair<int, uint32_t>> todo;
    for (int w = 0; w < W; w++) {
      bool wp = false;
      for (int l = 0; l < 32; l++) {
        Lane& a = L[w * 32 + l]; if (!a.pend) continue; wp = true;
        uint32_t cur = a.o + a.done, sa = cur - a.dist, want = std::min(a.len - a.done, g_piece);
        if (a.dist < want && a.dist >= 8) want = a.dist;
        uint32_t outn = std::min(want, a.dist), k = 0; while (k < outn && fin[sa + k]) k++;
        uint32_t n = k >= outn ? want : (a.dist >= want ? k : 0);
        if (n) todo.push_back({w * 32 + l, n});
      }
      if (wp) polls++;
    }
    if (todo.empty()) return 52;
    for (auto& td : todo) { Lane& a = L[td.first]; uint32_t cur = a.o + a.done, sa = cur - a.dist, j = 0; uint8_t v[64]; for (uint32_t k = 0; k < td.second; k++) { v[k] = win[sa + j]; if (++j == a.dist) j = 0; } for (uint32_t k = 0; k < td.second; k++) { win[cur + k] = v[k]; fin[cur + k] = 1; } a.done += td.second; if (a.done == a.len) { a.pend = false; } }
    for (auto& l : L) if (!l.pend && l.w < nw) next_match(l);
    if (rounds > 10000000) return 52;
  }
  S.resolve_iters += polls; S.resolve_batches += rounds;
  return 0;
}

// One member through the modelled CTA.  Returns 0 ok, else an error code (string in *why).
static uint32_t overlap = 448;
static int g_rmode = 0;
static int inflate_member_sim(const uint8_t* payload, uint32_t clen, uint32_t isize, int NT, uint32_t span_bytes, std::vector<uint8_t>& out, Stats& S, std::string* why) {
  // payload as words, with slack
  std::vector<uint32_t> pay((clen + 3) / 4 + 16, 0);
  memcpy(pay.data(), payload, clen);
  const uint32_t obase = 5;                                     // any window offset (the kernel uses uoff & 15)
  std::vector<uint8_t> win(obase + 65536 + 64, 0);
  std::vector<uint32_t> bm((obase + 65536) / 32 + 4, 0);
  std::vector<uint32_t> lut_ll(ROOT_LL + SUB_LL), lut_d(ROOT_D + SUB_D);
  const uint32_t olimit = obase + isize;
  const uint32_t end_bit = clen * 8;
  uint32_t outpos = obase;
  Bits br{pay.data(), 0};
  bool final_block = false;
  S.members++;
  while (!final_block) {
    if (br.pos + 3 > end_bit) { *why = "input exhausted at block header"; return 9; }
    uint32_t hdr = br.take(3); final_block = hdr & 1; uint32_t btype = hdr >> 1;
    S.blocks++;
    if (btype == 3) { *why = "btype 3"; return 1; }
    if (btype == 0) {
      br.pos = (br.pos + 7) & ~7u;
      if (br.pos + 32 > end_bit) { *why = "stored header past end"; return 9; }
      uint32_t len = br.take(16), nlen = br.take(16);
      if ((len ^ nlen) != 0xffff || outpos + len > olimit || br.pos / 8 + len > clen) { *why = "stored"; return 2; }
      memcpy(win.data() + outpos, payload + br.pos / 8, len);
      outpos += len; br.pos += 8 * len;
      continue;
    }
    uint8_t cl[320] = {0}; int n_ll = 288, n_d = 32;   // fixed code: all 32 distance codes (complete; 30 / 31 decode as invalid)
    if (btype == 1) { for (int i = 0; i < 288; i++) cl[i] = i < 144 ? 8 : i < 256 ? 9 : i < 280 ? 7 : 8; for (int i = 0; i < 32; i++) cl[288 + i] = 5; }
    else {
      uint32_t h = br.take(14); n_ll = (h & 31) + 257; n_d = ((h >> 5) & 31) + 1; int n_clc = (h >> 10) + 4;
      if (n_ll > 286 || n_d > 30) { *why = "hlit/hdist"; return 3; }
      uint8_t pcl[19] = {0}; for (int i = 0; i < n_clc; i++) pcl[kClcOrder[i]] = (uint8_t)br.take(3);
      std::vector<uint32_t> plut(128 + 8);
      // precode: 7-bit root, no second level needed (max length 7)
      {
        int cnt[8] = {0}; for (int i = 0; i < 19; i++) cnt[pcl[i]]++; cnt[0] = 0;
        uint32_t code = 0, first[8]; int left = 1;
        for (int L = 1; L <= 7; L++) { code = (code + (L > 1 ? cnt[L - 1] : 0)) << 1; first[L] = code; left <<= 1; left -= cnt[L]; if (left < 0) { *why = "precode oversubscribed"; return 3; } }
        if (left != 0) { *why = "precode incomplete"; return 3; }
        for (auto& v : plut) v = 0;
        for (int s = 0; s < 19; s++) { int L = pcl[s]; if (!L) continue; uint32_t c = first[L]++; uint32_t r = 0; for (int i = 0; i < L; i++) r |= ((c >> i) & 1u) << (L - 1 - i); for (uint32_t idx = r; idx < 128; idx += 1u << L) plut[idx] = (uint32_t)L | ((uint32_t)s << 16); }
      }
      int i = 0, total = n_ll + n_d; uint32_t prev = 0;
      while (i < total) {
        if (br.pos > end_bit) { *why = "input exhausted in code lengths"; return 9; }
        uint32_t e = plut[br.peek(7)]; uint32_t L = e & 15, s = e >> 16;
        if (!L) { *why = "bad precode"; return 3; }
        br.pos += L;
        uint32_t rep, val;
        if (s < 16) { rep = 1; val = s; prev = s; }
        else if (s == 16) { if (i == 0) { *why = "rep at 0"; return 3; } rep = 3 + br.take(2); val = prev; }
        else if (s == 17) { rep = 3 + br.take(3); val = 0; prev = 0; }
        else { rep = 11 + br.take(7); val = 0; prev = 0; }
        if (i + (int)rep > total) { *why = "code lengths overrun"; return 3; }
        while (rep--) cl[i++] = (uint8_t)val;
      }
      if (cl[256] == 0) { *why = "no EOB code"; return 3; }
    }
    int rc = build_lut<R_LL, false>(cl, n_ll, lut_ll.data(), SUB_LL);
    if (!rc) rc = build_lut<R_D, true>(cl + n_ll, n_d, lut_d.data(), SUB_D);
    if (rc == 2) { S.sub_overflow++; *why = "second-level table space exhausted"; return 100; }
    if (rc) { *why = "over-subscribed or incomplete code"; return 3; }

    // ---- spans: the symbol stream of this block, NT lanes at a time ----
    uint32_t cur = br.pos;
    bool block_done = false;
    while (!block_done) {
      S.spans++;
      const uint32_t span_end = std::min<uint64_t>(end_bit, (uint64_t)cur + (uint64_t)span_bytes * 8);
      if (cur >= end_bit) { *why = "input exhausted before end of block"; return 9; }
      uint32_t Sbits = (span_end - cur + NT - 1) / NT; if (Sbits < 256) Sbits = 256;
      std::vector<uint32_t> ls(NT), le(NT), lt(NT), ln(NT); std::vector<char> active(NT), need(NT);
      std::vector<uint32_t> lp(NT);
      for (int i = 0; i < NT; i++) { uint64_t p = (uint64_t)cur + (uint64_t)i * Sbits; active[i] = p < span_end; lp[i] = ls[i] = (uint32_t)p; need[i] = active[i]; }
      int F = 0;
      for (int round = 0;; round++) {
        S.rounds++;
        for (int i = 0; i < NT; i++) {
          S.lane_slots++;
          if (!need[i]) continue;
          S.lane_decodes++;
          uint32_t stop = std::min<uint64_t>(span_end, (uint64_t)cur + (uint64_t)(i + 1) * Sbits);
          SubResult r;
          if (round == 0 && i > 0) {
            // warm-up: start `overlap` bits early so that the chain is (almost always) the true one when it reaches the lane's cut
            const uint32_t from = lp[i] - cur > overlap ? lp[i] - overlap : cur;
            r = decode_sub<false>(true, pay.data(), lut_ll.data(), lut_d.data(), from, lp[i], stop, nullptr, nullptr, 0, 0, 0, nullptr);
            ls[i] = r.first_bit;                      // 0xffffffff: ended during the warm-up -> never equals a predecessor's end
            if (r.first_bit == 0xffffffffu) { r.term = T_CROSS; r.end_bit = lp[i]; r.n_out = 0; }
          } else {
            r = decode_sub<false>(true, pay.data(), lut_ll.data(), lut_d.data(), ls[i], ls[i], stop, nullptr, nullptr, 0, 0, 0, nullptr);
          }
          le[i] = r.end_bit; lt[i] = r.term; ln[i] = r.n_out;
        }
        // first lane of the chain that does not hand over to a successor
        F = NT - 1;
        for (int i = 0; i < NT; i++) if (!active[i]) { F = i - 1; break; } else if (lt[i] != T_CROSS) { F = i; break; }
        bool any = false;
        for (int i = 0; i < NT; i++) {
          need[i] = 0;
          if (i == 0 || i > F) continue;
          if (le[i - 1] != ls[i]) {
            // the predecessor's chain may step over this lane's whole sub-stream (a long token): then this lane owns nothing
            ls[i] = le[i - 1]; need[i] = 1; any = true;
          }
        }
        if (!any) break;
        if (round > NT + 2) { *why = "restart rounds did not converge"; return 50; }
      }
      // lanes 0..F are the true chain
      if (lt[F] == T_BAD) { *why = "unused code on the true chain"; return 4; }
      uint64_t total = 0; std::vector<uint32_t> lo(NT, 0);
      for (int i = 0; i <= F; i++) { lo[i] = outpos + (uint32_t)total; total += ln[i]; }
      if (outpos + total > olimit) { *why = "output overrun"; return 6; }
      uint32_t err = 0;
      for (int i = 0; i <= F; i++) {
        uint32_t stop = std::min<uint64_t>(span_end, (uint64_t)cur + (uint64_t)(i + 1) * Sbits);
        SubResult r = decode_sub<true>(true, pay.data(), lut_ll.data(), lut_d.data(), ls[i], ls[i], stop, win.data(), bm.data(), lo[i], obase, olimit, &err);
        if (err) { *why = err == CE_DIST ? "distance too far back" : "overrun in emit"; return (int)err; }
        if (r.end_bit != le[i] || r.n_out != ln[i]) { *why = "emit pass disagrees with count pass"; return 51; }
      }
      outpos += (uint32_t)total;
      if (lt[F] == T_EOB) { block_done = true; br.pos = le[F]; }
      else {
        cur = le[F];
        if (span_end >= end_bit) { *why = "input exhausted before end of block"; return 9; }
      }
    }
  }
  if (outpos != olimit) { *why = "isize mismatch"; return 7; }
  if (int rr = g_rmode == 7 ? resolve_word_model(win.data(), bm.data(), obase, olimit, NT / 32, S) : g_rmode == 6 ? resolve_static_model(win.data(), bm.data(), obase, olimit, NT / 32, S) : g_rmode ? resolve_inorder_model(win.data(), bm.data(), obase, olimit, g_rmode, S) : resolve_member_model(win.data(), bm.data(), obase, olimit, NT / 32, S)) { *why = "resolver"; return rr; }
  for (auto v : bm) if (v) { *why = "head bits left"; return 53; }
  out.assign(win.begin() + obase, win.begin() + obase + isize);
  return 0;
}

int main(int argc, char** argv) {
  if (argc < 2) { fprintf(stderr, "usage: inflate_sim file.bam [--lanes N] [--max-members N] [--span-bytes B] [--stats]\n"); return 2; }
  int NT = 256; long maxm = 1L << 40; uint32_t span_bytes = 28 * 1024; bool stats = false;
  for (int i = 2; i < argc; i++) {
    std::string a = argv[i];
    if (a == "--lanes") NT = atoi(argv[++i]); else if (a == "--max-members") maxm = atol(argv[++i]);
    else if (a == "--span-bytes") span_bytes = (uint32_t)atol(argv[++i]); else if (a == "--overlap") overlap = (uint32_t)atol(argv[++i]); else if (a == "--stats") stats = true; else if (a == "--resolve") g_rmode = atoi(argv[++i]); else if (a == "--gate") g_gate = atoi(argv[++i]); else if (a == "--group-sync") g_group_sync = true; else if (a == "--rlanes") g_lanes = atoi(argv[++i]); else if (a == "--piece") g_piece = (uint32_t)atol(argv[++i]); else if (a == "--list-cap") g_list_cap = (uint32_t)atol(argv[++i]);
  }
  FILE* f = fopen(argv[1], "rb"); if (!f) { perror("open"); return 2; }
  fseek(f, 0, SEEK_END); long sz = ftell(f); fseek(f, 0, SEEK_SET);
  std::vector<uint8_t> d(sz + 64, 0); if (fread(d.data(), 1, sz, f) != (size_t)sz) return 2; fclose(f);
  Stats S; long off = 0, nm = 0, bad = 0; std::vector<uint8_t> out, ref(65536 + 16);
  while (off + 28 <= sz && nm < maxm) {
    if (d[off] != 0x1f || d[off + 1] != 0x8b) { fprintf(stderr, "not a gzip member at %ld\n", off); return 2; }
    uint32_t xlen = d[off + 10] | (d[off + 11] << 8);
    uint32_t bsize = 0; for (uint32_t x = 0; x + 4 <= xlen;) { const uint8_t* p = &d[off + 12 + x]; uint32_t slen = p[2] | (p[3] << 8); if (p[0] == 'B' && p[1] == 'C') bsize = p[4] | (p[5] << 8); x += 4 + slen; }
    uint32_t hdr = 12 + xlen, clen = bsize + 1 - hdr - 8;
    const uint8_t* payload = &d[off + hdr];
    uint32_t isize; memcpy(&isize, &d[off + bsize + 1 - 4], 4);
    if (isize) {
      z_stream zs; memset(&zs, 0, sizeof zs); inflateInit2(&zs, -15);
      zs.next_in = (Bytef*)payload; zs.avail_in = clen; zs.next_out = ref.data(); zs.avail_out = 65536 + 16;
      int zr = inflate(&zs, Z_FINISH); inflateEnd(&zs);
      std::string why;
      int rc = inflate_member_sim(payload, clen, isize, NT, span_bytes, out, S, &why);
      bool zok = zr == Z_STREAM_END && zs.total_out == isize;
      if (rc == 100) { /* refused: second-level space */ }
      else if (zok && (rc != 0 || memcmp(out.data(), ref.data(), isize))) { bad++; if (bad < 10) fprintf(stderr, "member %ld at %ld: MISMATCH rc=%d (%s)\n", nm, off, rc, why.c_str()); }
      else if (!zok && rc == 0) { bad++; if (bad < 10) fprintf(stderr, "member %ld: zlib failed (%d) but the model succeeded\n", nm, zr); }
    }
    off += bsize + 1; nm++;
  }
  printf("%s: members=%ld bad=%ld refused(sub-table)=%ld | deflate blocks=%ld spans=%ld rounds/span=%.2f lane-decodes/span=%.1f (of %d) resolver warp-iterations/member=%.0f groups/member=%.0f", argv[1], S.members, bad, S.sub_overflow,
         S.blocks, S.spans, (double)S.rounds / std::max(1L, S.spans), (double)S.lane_decodes / std::max(1L, S.spans), NT, (double)S.resolve_iters / std::max(1L, S.members), (double)S.resolve_batches / std::max(1L, S.members));
  if (g_rmode == 6) printf(" matches/member(max)=%ld list-batches=%ld", S.matches_max, S.list_batches);
  printf("\n");
  (void)stats;
  return bad ? 1 : 0;
}
