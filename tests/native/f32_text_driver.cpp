// f32_text_driver.cpp -- test-only: one hex f32 bit pattern per stdin line -> its text per stdout line, through the product's
// f32_text.h (what the scan and the SAM writer run on the device) compiled for the host.  The length-only call (out = nullptr,
// what the size passes use) must give the same length, or the line is "length <n> != <m>".
#include <cstdio>

#include "../../datafusion-bio-formats_b200/csrc/f32_text.h"

int main() {
  unsigned bits;
  uint8_t out[80];
  while (scanf("%x", &bits) == 1) {
    const uint32_t n = bamscan::f32_to_text(bits, out), n0 = bamscan::f32_to_text(bits, nullptr);
    if (n != n0) { printf("length %u != %u\n", n0, n); continue; }
    out[n] = 0;
    printf("%s\n", (const char*)out);
  }
  return 0;
}
