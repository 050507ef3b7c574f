// vcf_format_cpp_check.cpp -- compile-and-run check of bamscan.hpp's VcfTableProvider with format_fields (planning calls only: no
// GPU needed).
//   vcf_format_cpp_check <file.vcf.gz>   (tests/vcf_format_inputs.py::EDGE_FMT: 12 INFO fields, FORMAT GT, DP, AD, ...)
#include <cstdio>
#include <cstdlib>
#include <string>

#include "bamscan.hpp"

using namespace bamscan_cpp;

#define REQUIRE(c) do { if (!(c)) { fprintf(stderr, "FAILED line %d: %s\n", __LINE__, #c); return 1; } } while (0)

int main(int argc, char** argv) {
  if (argc < 2) return 2;
  ArrowSchema sc;
  VcfTableProvider none(argv[1]);
  none.schema(&sc);
  REQUIRE(sc.n_children == 20 && sc.metadata == nullptr);
  sc.release(&sc);
  VcfTableProvider t(argv[1], std::nullopt, std::nullopt, true, 0, 0, std::vector<std::string>{"PL", "GT", "DP"});
  t.schema(&sc);
  // flag 2: ARROW_FLAG_NULLABLE; the list is not nullable, its elements (and nested leaves) are
  REQUIRE(sc.n_children == 23 && std::string(sc.children[20]->name) == "format_PL" && std::string(sc.children[21]->name) == "format_GT");
  REQUIRE(std::string(sc.children[20]->format) == "+l" && !(sc.children[20]->flags & 2) && std::string(sc.children[20]->children[0]->format) == "+l" &&
          (sc.children[20]->children[0]->flags & 2) && std::string(sc.children[20]->children[0]->children[0]->format) == "i" &&
          (sc.children[20]->children[0]->children[0]->flags & 2));
  REQUIRE(std::string(sc.children[21]->children[0]->format) == "u" && std::string(sc.children[22]->children[0]->format) == "i");
  REQUIRE(sc.metadata != nullptr);
  sc.release(&sc);
  BamExec one = t.scan(std::vector<int32_t>{21}, std::nullopt);
  one.schema(&sc);
  REQUIRE(sc.n_children == 1 && std::string(sc.children[0]->name) == "format_GT");
  sc.release(&sc);
  bool threw = false;
  try { VcfTableProvider bad(argv[1], std::nullopt, std::nullopt, true, 0, 0, std::vector<std::string>{"NOPE"}); } catch (const Error& e) { threw = e.code == BAMSCAN_ERR_SCHEMA; }
  REQUIRE(threw);
  printf("vcf format cpp check ok\n");
  return 0;
}
