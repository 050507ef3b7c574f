// f32_text.h -- a float tag rendered into a Utf8 column: Rust's `f32::to_string()` (sam_tag_io.rs:670-676).
//
// Rust prints the SHORTEST decimal that parses back to the same f32, without an exponent ("0.0000001", "100000000000000000000"):
// the fewest significant digits of any decimal inside the float's rounding interval, and of two such decimals the closer
// (the even last digit on a tie).  Computed here as: the smallest number N <= 9 of significant digits for which the value,
// correctly rounded to N digits (round-half-even on the EXACT binary value), reads back as the same float -- or, when that
// rounded down at a power of two (m = 2^23, where the float below is half as far away as the one above), the N-digit value
// one unit above, which can lie inside the wider upper half when the rounded one misses the narrow lower half (2^87:
// 1.5474250e26 does not read back, 1.5474251e26 does).  Then those digits in plain positional notation.  The exact
// reference is oracle/f32_exact.py::display (tests/test_f32_exact.py).
//
// No floating point and no library: the exact decimal expansion of m * 2^e is built with a small big-integer (m * 5^-e for
// e < 0, at most 370 bits), rounded on its digit string, and the round-trip test |R - v| < half an ulp (ties: even mantissa)
// is a comparison of digit strings.  One thread per value; this is a rare path (a float tag read into a Utf8 column happens
// only for tags outside the registry with inference off), so clarity wins over speed.  Compiles for host and device.
#pragma once
#include <cstdint>

#if defined(__CUDACC__)
#define F32T_HD __host__ __device__
#define F32T_NOINLINE __noinline__      // a rare path: its registers and stack must not be charged to the decode kernels' main loops
#else
#define F32T_HD
#define F32T_NOINLINE
#endif

namespace bamscan {

struct F32Big {                       // little-endian base 2^32, enough for 24 + 346 bits and a factor 100
  static constexpr int W = 14;
  uint32_t w[W];
  F32T_HD void set(uint32_t v) { for (int i = 0; i < W; i++) w[i] = 0; w[0] = v; }
  F32T_HD void mul_small(uint32_t k) { uint64_t c = 0; for (int i = 0; i < W; i++) { c += (uint64_t)w[i] * k; w[i] = (uint32_t)c; c >>= 32; } }
  F32T_HD void shl(uint32_t bits) { for (uint32_t b = 0; b < bits; b++) { uint32_t c = 0; for (int i = 0; i < W; i++) { const uint32_t n = w[i] >> 31; w[i] = (w[i] << 1) | c; c = n; } } }
  F32T_HD uint32_t divmod_small(uint32_t k) { uint64_t r = 0; for (int i = W - 1; i >= 0; i--) { r = (r << 32) | w[i]; w[i] = (uint32_t)(r / k); r %= k; } return (uint32_t)r; }
  F32T_HD bool is_zero() const { for (int i = 0; i < W; i++) if (w[i]) return false; return true; }
  // decimal digits, most significant first; returns the count (>= 1)
  F32T_HD int digits(uint8_t* out) {
    uint8_t tmp[140]; int n = 0;
    while (!is_zero()) { uint32_t r = divmod_small(1000000000u); for (int k = 0; k < 9; k++) { tmp[n++] = (uint8_t)(r % 10u); r /= 10u; } }
    while (n > 1 && tmp[n - 1] == 0) n--;
    if (n == 0) { tmp[0] = 0; n = 1; }
    for (int i = 0; i < n; i++) out[i] = tmp[n - 1 - i];
    return n;
  }
};

// compares two digit strings (no leading zeros except a lone 0): -1, 0, 1
F32T_HD inline int f32t_cmp(const uint8_t* a, int na, const uint8_t* b, int nb) {
  while (na > 1 && a[0] == 0) { a++; na--; }
  while (nb > 1 && b[0] == 0) { b++; nb--; }
  if (na != nb) return na < nb ? -1 : 1;
  for (int i = 0; i < na; i++) if (a[i] != b[i]) return a[i] < b[i] ? -1 : 1;
  return 0;
}

// Writes the text of the f32 with bit pattern `bits` to out (when out != nullptr) and returns its length (<= 64).
F32T_HD F32T_NOINLINE inline uint32_t f32_to_text(uint32_t bits, uint8_t* out) {
  const uint32_t sign = bits >> 31, ex = (bits >> 23) & 0xffu, mant = bits & 0x7fffffu;
  uint32_t o = 0;
#define F32T_PUT(c) do { if (out) out[o] = (uint8_t)(c); o++; } while (0)
  if (ex == 255u) {
    if (mant) { F32T_PUT('N'); F32T_PUT('a'); F32T_PUT('N'); return o; }
    if (sign) F32T_PUT('-');
    F32T_PUT('i'); F32T_PUT('n'); F32T_PUT('f');
    return o;
  }
  if (sign) F32T_PUT('-');
  if (ex == 0u && mant == 0u) { F32T_PUT('0'); return o; }
  const uint32_t m = ex ? (mant | 0x800000u) : mant;
  const int e = ex ? (int)ex - 150 : -149;
  const bool boundary = mant == 0u && ex > 1u;      // the float below is half as far away as the one above
  // exact value D / 10^F, unit in the last place U / 10^F
  F32Big D, Ub;
  int F = 0;
  D.set(m); Ub.set(1);
  if (e >= 0) { D.shl((uint32_t)e); Ub.shl((uint32_t)e); }
  else { F = -e; for (int k = 0; k < F; k++) { D.mul_small(5u); Ub.mul_small(5u); } }
  uint8_t dv[132], hu[136], hd[136];
  const int n = D.digits(dv);
  const int exp10 = n - 1 - F;                      // value = d.ddd * 10^exp10
  F32Big H = Ub; H.mul_small(50u);                  // half an ulp, in units of 10^-(F+2)
  const int nhu = H.digits(hu);
  H = Ub; H.mul_small(boundary ? 25u : 50u);
  const int nhd = H.digits(hd);
  // shortest N whose correctly rounded value reads back as this float
  uint8_t rv[134];                                   // candidate, n + 1 digits (rv[0] = carry out of the first digit)
  int N = 1;
  for (; N <= 9; N++) {
    rv[0] = 0;
    for (int i = 0; i < n; i++) rv[i + 1] = i < N ? dv[i] : 0;
    bool up = false;
    if (N < n) {
      if (dv[N] > 5) up = true;
      else if (dv[N] == 5) { bool rest = false; for (int i = N + 1; i < n; i++) if (dv[i]) rest = true; up = rest || (dv[N - 1] & 1); }
    }
    if (N >= n) break;                               // all digits: exact
    bool inside = false;
    for (;;) {
      if (up) { int i = N; while (i >= 0) { if (rv[i] == 9) { rv[i] = 0; i--; } else { rv[i]++; break; } } }
      // diff = |rv - dv| as n + 1 digits, then two more zeros (units of 10^-(F+2))
      uint8_t df[136];
      int borrow = 0;
      for (int i = n; i >= 0; i--) {
        const int a = up ? rv[i] : (i ? dv[i - 1] : 0), b = up ? (i ? dv[i - 1] : 0) : rv[i];
        int d = a - b - borrow;
        if (d < 0) { d += 10; borrow = 1; } else borrow = 0;
        df[i] = (uint8_t)d;
      }
      df[n + 1] = 0; df[n + 2] = 0;
      const int c = up ? f32t_cmp(df, n + 3, hu, nhu) : f32t_cmp(df, n + 3, hd, nhd);
      inside = c < 0 || (c == 0 && (m & 1u) == 0u);
      // rounded down at a power of two and outside the narrow lower half: the N-digit value one unit above v may still be
      // inside the upper half, which is twice as wide
      if (inside || up || !boundary) break;
      up = true;
    }
    if (inside) break;
  }
  if (N > 9) N = 9;
  // significant digits of the candidate and its decimal exponent
  int first = rv[0] ? 0 : 1;
  int e10 = rv[0] ? exp10 + 1 : exp10;
  int nd = (N < n ? N : n) + (rv[0] ? 1 : 0);
  if (nd > n + 1 - first) nd = n + 1 - first;
  while (nd > 1 && rv[first + nd - 1] == 0) nd--;
  if (e10 < 0) {
    F32T_PUT('0'); F32T_PUT('.');
    for (int i = 0; i < -e10 - 1; i++) F32T_PUT('0');
    for (int i = 0; i < nd; i++) F32T_PUT('0' + rv[first + i]);
  } else {
    for (int i = 0; i <= e10; i++) F32T_PUT(i < nd ? '0' + rv[first + i] : '0');
    if (nd > e10 + 1) { F32T_PUT('.'); for (int i = e10 + 1; i < nd; i++) F32T_PUT('0' + rv[first + i]); }
  }
#undef F32T_PUT
  return o;
}

}  // namespace bamscan
