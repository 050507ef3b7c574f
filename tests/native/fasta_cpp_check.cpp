// fasta_cpp_check.cpp -- compile-and-run check of bamscan.hpp's FastaTableProvider (planning calls only: no GPU needed).
//   fasta_cpp_check <file.fa.bgz>
#include <cstdio>
#include <cstdlib>
#include <string>

#include "bamscan.hpp"

using namespace bamscan_cpp;

#define REQUIRE(c) do { if (!(c)) { fprintf(stderr, "FAILED line %d: %s\n", __LINE__, #c); return 1; } } while (0)

int main(int argc, char** argv) {
  if (argc < 2) return 2;
  FastaTableProvider t(argv[1]);
  ArrowSchema sc;
  t.schema(&sc);
  REQUIRE(sc.n_children == 3 && std::string(sc.children[0]->name) == "name" && std::string(sc.children[1]->name) == "description" &&
          std::string(sc.children[2]->name) == "sequence");
  // flag 2: ARROW_FLAG_NULLABLE
  REQUIRE(std::string(sc.children[2]->format) == "u" && (sc.children[1]->flags & 2) && !(sc.children[0]->flags & 2));
  sc.release(&sc);
  REQUIRE(std::string(t.table_type()) == "Base");
  BamExec one = t.scan(std::vector<int32_t>{2}, std::nullopt);
  REQUIRE(one.output_partition_count() == 1);
  one.schema(&sc);
  REQUIRE(sc.n_children == 1 && std::string(sc.children[0]->name) == "sequence");
  sc.release(&sc);
  BamExec four = t.scan(std::nullopt, 10, 4);
  REQUIRE(four.output_partition_count() == 4);
  bool threw = false;
  try { FastaTableProvider bad("/nonexistent/file.fa.bgz"); } catch (const Error& e) { threw = e.code == BAMSCAN_ERR_IO; }
  REQUIRE(threw);
  threw = false;
  try { FastaTableProvider remote(argv[1], std::string("{}")); } catch (const Error& e) { threw = e.code == BAMSCAN_ERR_UNSUPPORTED; }
  REQUIRE(threw);
  printf("fasta cpp check ok\n");
  return 0;
}
