// Checks csrc/f32_text.h (integer-only shortest round-trip text of an f32, what the GPU runs) against the oracle's rule
// (oracle/bam_oracle.c::rust_f32_to_string: smallest precision whose correctly rounded "%.*e" reads back with strtof, or
// when that rounded down, the value one unit above it -- the power-of-two case).
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <cstdint>
#include <random>
#include "../../datafusion-bio-formats_b200/csrc/f32_text.h"

static void next_up(const char* s, char* out, size_t cap) {
  char d[16]; int nd = 0; const char* p = s;
  for (; *p != 'e'; p++) if (*p != '.') d[nd++] = *p;
  int x = atoi(p + 1), i = nd - 1;
  while (i >= 0 && d[i] == '9') d[i--] = '0';
  if (i >= 0) d[i]++; else { d[0] = '1'; x++; }
  snprintf(out, cap, "%c.%.*se%d", d[0], nd - 1, d + 1, x);
}

static size_t oracle_rule(float v, char* out) {
  if (v != v) return (size_t)sprintf(out, "NaN");
  if (v == 1.0f / 0.0f) return (size_t)sprintf(out, "inf");
  if (v == -1.0f / 0.0f) return (size_t)sprintf(out, "-inf");
  char tmp[64], alt[64]; int prec;
  const bool minus = v < 0 || (v == 0 && 1.0f / v < 0);
  const float a = minus ? -v : v;
  for (prec = 1; prec <= 9; prec++) {
    snprintf(tmp, sizeof tmp, "%.*e", prec - 1, (double)a);
    if (strtof(tmp, NULL) == a) break;
    if (strtod(tmp, NULL) < (double)a) {
      next_up(tmp, alt, sizeof alt);
      if (strtof(alt, NULL) == a) { memcpy(tmp, alt, sizeof tmp); break; }
    }
  }
  if (minus) { memmove(tmp + 1, tmp, strlen(tmp) + 1); tmp[0] = '-'; }
  char digits[16]; int nd = 0, neg = 0; const char* s = tmp;
  if (*s == '-') { neg = 1; s++; }
  for (; *s && *s != 'e'; s++) if (*s != '.') digits[nd++] = *s;
  int exp10 = atoi(s + 1);
  while (nd > 1 && digits[nd - 1] == '0') nd--;
  size_t o = 0;
  if (neg) out[o++] = '-';
  if (nd == 1 && digits[0] == '0') { out[o++] = '0'; out[o] = 0; return o; }
  if (exp10 < 0) { out[o++] = '0'; out[o++] = '.'; for (int i = 0; i < -exp10 - 1; i++) out[o++] = '0'; for (int i = 0; i < nd; i++) out[o++] = digits[i]; }
  else { for (int i = 0; i <= exp10; i++) out[o++] = i < nd ? digits[i] : '0'; if (nd > exp10 + 1) { out[o++] = '.'; for (int i = exp10 + 1; i < nd; i++) out[o++] = digits[i]; } }
  out[o] = 0;
  return o;
}

int main(int argc, char** argv) {
  long n = argc > 1 ? atol(argv[1]) : 300000, bad = 0;
  std::mt19937 rng(12345);
  auto check = [&](uint32_t bits) {
    float v; memcpy(&v, &bits, 4);
    char want[128]; uint8_t got[128];
    size_t nw = oracle_rule(v, want);
    uint32_t ng = bamscan::f32_to_text(bits, got), ng2 = bamscan::f32_to_text(bits, nullptr);
    if (ng != nw || ng2 != ng || memcmp(got, want, nw)) { if (bad++ < 10) { got[ng] = 0; fprintf(stderr, "bits %08x: got '%s' want '%s'\n", bits, got, want); } }
  };
  const uint32_t edge[] = {0x00000000u, 0x80000000u, 0x00000001u, 0x007fffffu, 0x00800000u, 0x00800001u, 0x7f7fffffu, 0x7f800000u, 0xff800000u, 0x7fc00000u,
                           0x3f800000u, 0x3fc00000u, 0x3dcccccdu, 0x33d6bf95u, 0x60ad78ecu, 0x4b800000u, 0x4b7fffffu, 0x3f7fffffu, 0x34000000u, 0x01000000u, 0x7e800000u};
  for (uint32_t b : edge) check(b);
  for (uint32_t ex = 0; ex < 255; ex++) { check(ex << 23); check((ex << 23) | 1u); check((ex << 23) | 0x7fffffu); check((ex << 23) | 0x400000u); }
  for (long i = 0; i < n; i++) check(rng());
  for (long i = 0; i < n / 4; i++) check((uint32_t)(rng() % 0x00800000u));          // subnormals
  for (long i = 0; i < n / 4; i++) { float f = (float)((int)(rng() % 2000001) - 1000000) / 1000.0f; uint32_t b; memcpy(&b, &f, 4); check(b); }   // "human" values
  printf("checked, bad=%ld\n", bad);
  return bad ? 1 : 0;
}
