// f32_parse.h -- decimal text -> the nearest f32, as Rust's `f32::from_str` (the SAM `f` aux type and `B:f` elements).
//
// Grammar (core::num::dec2flt): [+-]? then "inf" | "infinity" | "nan" (any case), or digits [. digits] | . digits, followed by an
// optional [eE][+-]?digits.  The result is the f32 nearest to the EXACT decimal value, ties to even; a value at or above the
// halfway point between f32::MAX and 2^128 is infinity, one at or below half the smallest subnormal is zero.
//
// Fast path: at most 7 significant digits and a decimal exponent in [-10, 10].  The digits and 10^|e| are then exact f32s and one
// IEEE f32 multiplication or division rounds once, correctly.  Everything else takes the exact path: a candidate from a double
// approximation, then exact big-integer comparisons of the value with the halfway points around the candidate, moving it one ulp
// at a time.  Rounding through a double alone is not used: that rounds twice and is wrong next to f32 halfway points.
// Compiles for host and device (no library calls; the device's f32 division is IEEE round-to-nearest).
#pragma once
#include <cstdint>
#include <cstring>

#if defined(__CUDACC__)
#define F32P_HD __host__ __device__
#define F32P_NOINLINE __noinline__
#else
#define F32P_HD
#define F32P_NOINLINE
#endif

namespace bamscan {

constexpr int F32P_MAX_DIGITS = 120;   // f32 halfway points have at most 112 significant digits; later digits only break ties

struct F32PBig {                       // little-endian base 2^32; 40 words hold 10^120 * 2^151 and 2^25 * 10^166 with room
  static constexpr int W = 40;
  uint32_t w[W];
  F32P_HD void set(uint32_t v) { for (int i = 0; i < W; i++) w[i] = 0; w[0] = v; }
  F32P_HD void mul_add(uint32_t k, uint32_t a) { uint64_t c = a; for (int i = 0; i < W; i++) { c += (uint64_t)w[i] * k; w[i] = (uint32_t)c; c >>= 32; } }
  F32P_HD void mul_pow10(int e) { while (e >= 9) { mul_add(1000000000u, 0); e -= 9; } uint32_t p = 1; while (e-- > 0) p *= 10; mul_add(p, 0); }
  F32P_HD void shl(int bits) {
    const int words = bits >> 5, b = bits & 31;
    for (int i = W - 1; i >= 0; i--) {
      const uint32_t hi = i - words >= 0 ? w[i - words] : 0u, lo = i - words - 1 >= 0 ? w[i - words - 1] : 0u;
      w[i] = b ? (hi << b) | (lo >> (32 - b)) : hi;
    }
  }
  F32P_HD int cmp(const F32PBig& o) const { for (int i = W - 1; i >= 0; i--) if (w[i] != o.w[i]) return w[i] < o.w[i] ? -1 : 1; return 0; }
};

struct F32PDec {
  const char* s;          // text
  uint32_t d0, d1;        // the significant digits are the digit characters of s[d0 .. d1) (the '.' skipped)
  int nd;                 // how many of them are used (<= F32P_MAX_DIGITS)
  bool sticky;            // a non-zero digit was dropped behind those
  int e;                  // value = (used digits as an integer) * 10^e
};

// sign(V - H) where V = the decimal, H = the halfway point between f32 `bits` and the next one up: (2m + 1) * 2^(ex - 1)
F32P_HD F32P_NOINLINE inline int f32p_cmp_half(const F32PDec& D, uint32_t bits) {
  const uint32_t fe = bits >> 23, fm = bits & 0x7fffffu;
  const uint32_t m = fe ? fm | 0x800000u : fm;
  const int ex = fe ? (int)fe - 150 : -149;
  F32PBig A, B;
  A.set(0);
  int used = 0;
  for (uint32_t k = D.d0; k < D.d1 && used < D.nd; k++) { if (D.s[k] == '.') continue; A.mul_add(10, (uint32_t)(D.s[k] - '0')); used++; }
  B.set(2 * m + 1);
  if (D.e >= 0) A.mul_pow10(D.e); else B.mul_pow10(-D.e);
  if (ex - 1 >= 0) B.shl(ex - 1); else A.shl(1 - ex);
  const int c = A.cmp(B);
  return (c == 0 && D.sticky) ? 1 : c;
}

// Parses s[0 .. n).  Returns false when the text is not a float; *bits receives the f32's bit pattern.
F32P_HD F32P_NOINLINE inline bool f32_parse(const char* s, uint32_t n, uint32_t* bits) {
  uint32_t k = 0, sign = 0;
  if (k < n && (s[k] == '+' || s[k] == '-')) { sign = s[k] == '-' ? 0x80000000u : 0u; k++; }
  {   // inf / infinity / nan
    auto word = [&](const char* w) { uint32_t i = 0; for (; w[i]; i++) { if (k + i >= n || (s[k + i] | 0x20) != w[i]) return false; } return k + i == n; };
    if (word("inf") || word("infinity")) { *bits = sign | 0x7f800000u; return true; }
    if (word("nan")) { *bits = sign | 0x7fc00000u; return true; }
  }
  F32PDec D; D.s = s; D.nd = 0; D.sticky = false;
  int digits = 0, frac = 0, lead = -1;     // digit characters, of them behind the '.', index (in digits) of the first non-zero
  bool dot = false;
  uint32_t first = 0;
  uint64_t m19 = 0; int n19 = 0;
  for (; k < n; k++) {
    const char c = s[k];
    if (c == '.') { if (dot) return false; dot = true; continue; }
    if (c < '0' || c > '9') break;
    if (lead < 0 && c != '0') { lead = digits; first = k; }
    if (lead >= 0) {
      if (D.nd < F32P_MAX_DIGITS) { D.nd++; D.d1 = k + 1; } else if (c != '0') D.sticky = true;
      if (n19 < 19) { m19 = m19 * 10 + (uint64_t)(c - '0'); n19++; }
    }
    digits++; if (dot) frac++;
  }
  if (digits == 0) return false;
  long long ex = 0;
  if (k < n) {
    if (s[k] != 'e' && s[k] != 'E') return false;
    k++;
    bool neg = false;
    if (k < n && (s[k] == '+' || s[k] == '-')) { neg = s[k] == '-'; k++; }
    if (k >= n) return false;
    for (; k < n; k++) { if (s[k] < '0' || s[k] > '9') return false; if (ex < 100000) ex = ex * 10 + (s[k] - '0'); }
    if (neg) ex = -ex;
  }
  if (lead < 0) { *bits = sign; return true; }                       // zero
  D.d0 = first;
  // value = (first nd significant digits) * 10^e: the digits in front of the first used one are zeros
  const int int_digits_after = digits - frac;                        // digit characters in front of the '.'
  const long long e = ex + (long long)int_digits_after - (long long)lead - (long long)D.nd;
  const long long mag = e + D.nd;                                    // value in [10^(mag-1), 10^mag)
  if (mag > 39) { *bits = sign | 0x7f800000u; return true; }         // >= 10^39 > f32::MAX
  if (mag < -45) { *bits = sign; return true; }                      // < 10^-46 < half the smallest subnormal (7.0e-46)
  D.e = (int)e;
  if (!D.sticky && D.nd <= 7 && D.e >= -10 && D.e <= 10) {
    const float p10[11] = {1e0f, 1e1f, 1e2f, 1e3f, 1e4f, 1e5f, 1e6f, 1e7f, 1e8f, 1e9f, 1e10f};
    const float v = D.e >= 0 ? (float)m19 * p10[D.e] : (float)m19 / p10[-D.e];
    uint32_t b; memcpy(&b, &v, 4);
    *bits = sign | b;
    return true;
  }
  // candidate: the double nearest-ish to the value, rounded to f32 by bits (within an ulp or two of the answer)
  double approx = (double)m19;
  int e19 = D.e + (D.nd - n19);
  while (e19 > 0) { approx *= 10.0; e19--; }
  while (e19 < 0) { approx /= 10.0; e19++; }
  uint32_t b;
  if (approx >= 3.4028234663852886e38) b = 0x7f7fffffu;
  else { const float f = (float)approx; memcpy(&b, &f, 4); }
  for (;;) {
    if (b < 0x7f800000u) {
      const int up = f32p_cmp_half(D, b);                            // V against the halfway point above b
      if (up > 0 || (up == 0 && (b & 1u))) { b++; continue; }
    }
    if (b > 0) {
      const int dn = f32p_cmp_half(D, b - 1);                        // V against the halfway point below b
      if (dn < 0 || (dn == 0 && (b & 1u))) { b--; continue; }
    }
    break;
  }
  *bits = sign | b;
  return true;
}

}  // namespace bamscan
