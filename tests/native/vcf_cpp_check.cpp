// vcf_cpp_check.cpp -- compile-and-run check of bamscan.hpp's VcfTableProvider (planning calls only: no GPU needed).
//   vcf_cpp_check <file.vcf.gz>   (a file of tests/vcf_inputs.py::sites_text: INFO DP, AF, DB, CSQ, ...)
#include <cstdio>
#include <cstdlib>
#include <string>

#include "bamscan.hpp"

using namespace bamscan_cpp;

#define REQUIRE(c) do { if (!(c)) { fprintf(stderr, "FAILED line %d: %s\n", __LINE__, #c); return 1; } } while (0)

int main(int argc, char** argv) {
  if (argc < 2) return 2;
  VcfTableProvider t(argv[1]);
  ArrowSchema sc;
  t.schema(&sc);
  REQUIRE(sc.n_children > 8 && std::string(sc.children[0]->name) == "chrom" && std::string(sc.children[7]->name) == "filter" &&
          std::string(sc.children[8]->name) == "DP");
  // flag 2: ARROW_FLAG_NULLABLE
  REQUIRE(std::string(sc.children[1]->format) == "I" && std::string(sc.children[6]->format) == "f" && (sc.children[3]->flags & 2) && !(sc.children[0]->flags & 2));
  sc.release(&sc);
  VcfTableProvider sel(argv[1], std::vector<std::string>{"CSQ", "DB"});
  sel.schema(&sc);
  REQUIRE(sc.n_children == 10 && std::string(sc.children[8]->format) == "+l" && std::string(sc.children[8]->children[0]->format) == "u" &&
          std::string(sc.children[9]->format) == "b" && !(sc.children[9]->flags & 2));
  sc.release(&sc);
  REQUIRE(std::string(t.table_type()) == "Base");
  BamExec one = t.scan(std::vector<int32_t>{2}, std::nullopt);
  REQUIRE(one.output_partition_count() == 1);
  one.schema(&sc);
  REQUIRE(sc.n_children == 1 && std::string(sc.children[0]->name) == "end");
  sc.release(&sc);
  BamExec four = t.scan(std::nullopt, 10, 4);
  REQUIRE(four.output_partition_count() == 4);
  bool threw = false;
  try { VcfTableProvider bad(argv[1], std::vector<std::string>{"NOPE"}); } catch (const Error& e) { threw = e.code == BAMSCAN_ERR_SCHEMA; }
  REQUIRE(threw);
  threw = false;
  try { VcfTableProvider missing("/nonexistent/file.vcf.gz"); } catch (const Error& e) { threw = e.code == BAMSCAN_ERR_IO; }
  REQUIRE(threw);
  printf("vcf cpp check ok\n");
  return 0;
}
