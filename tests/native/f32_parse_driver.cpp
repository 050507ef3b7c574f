// f32_parse_driver.cpp -- test-only: one decimal string per stdin line -> "<hex bits>" or "err" per stdout line, through the
// product's f32_parse.h (the parser the SAM transcoder runs on the device) compiled for the host.
#include <cstdio>
#include <cstring>
#include <iostream>
#include <string>

#include "../../datafusion-bio-formats_b200/csrc/f32_parse.h"

int main() {
  std::string line;
  while (std::getline(std::cin, line)) {
    uint32_t bits = 0;
    if (bamscan::f32_parse(line.data(), (uint32_t)line.size(), &bits)) printf("%08x\n", bits);
    else printf("err\n");
  }
  return 0;
}
