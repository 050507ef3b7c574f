// sam_host_driver.cpp -- test-only driver of the product's HOST code for plain SAM (host_file.cpp::load_sam, the @SQ parser,
// the aux-text tag inference, block-range planning on line starts), linked WITHOUT the CUDA engine so that it can be built with
// -fsanitize=address,undefined.  The helpers engine.cu provides to those files are stubbed with malloc.
//   sam_host_driver file.sam
// Prints what the host made of the file; exit code 0 whether the input is accepted or refused (a sanitizer report or a crash is
// the failure the test looks for).
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>

#include "../../datafusion-bio-formats_b200/csrc/bamscan_internal.h"

namespace bamscan {
void* pinned_alloc(size_t bytes) { return calloc(1, bytes); }
void pinned_free(void* p) { free(p); }
void* map_file_pinned(const char*, uint64_t, bool*) { return nullptr; }   // never taken: load_file falls back to a private copy
void unmap_file_pinned(void*, uint64_t, bool) {}
}  // namespace bamscan

using namespace bamscan;

int main(int argc, char** argv) {
  if (argc < 2) return 2;
  BamFile f;
  f.path = argv[1];
  f.format = is_sam_path(f.path) ? 2 : 0;
  f.has_tag_fields = true; f.tag_fields = {"NM", "MD", "XA", "XB", "XF", "ZZ", "CB"};
  const int rc = load_file(&f);
  if (f.size >= (1u << 20)) { fprintf(stderr, "driver: files of 1 MiB and more are mapped by the engine; use a smaller input\n"); return 2; }
  size_t n_tags = 0;
  int partitions = 0;
  if (rc == BAMSCAN_OK) {
    BamScanOptions opt; memset(&opt, 0, sizeof opt);
    opt.struct_size = sizeof opt; opt.coordinate_system_zero_based = 1; opt.infer_tag_types = 1; opt.infer_tag_sample_size = 100; opt.has_tag_fields = 1;
    if (build_schema(&f, &opt) == BAMSCAN_OK) {
      std::map<std::string, std::pair<char, int32_t>> all;
      infer_tag_types(f, {}, 1000, &all, true);
      n_tags = all.size();
      struct ArrowSchema sc; memset(&sc, 0, sizeof sc);
      if (export_schema(f.fields, f.schema_metadata, &sc) == BAMSCAN_OK && sc.release) sc.release(&sc);
      for (int tp : {1, 3, 16}) for (int mode : {BAMSCAN_PARTITION_REFERENCE, BAMSCAN_PARTITION_BLOCK_RANGE}) {
        Plan* p = nullptr;
        if (make_plan(&f, nullptr, -1, nullptr, 0, tp, mode, &p) == BAMSCAN_OK && p) {
          for (const Partition& part : p->partitions)
            for (const ScanRange& r : part.ranges) {
              // a range starts on a line: the body start, or behind a '\n'
              if (r.first_uoff != f.first_record_uoff && (r.first_uoff == 0 || r.first_uoff > f.size || f.data[r.first_uoff - 1] != '\n')) { printf("driver: range off a line start\n"); return 1; }
              partitions++;
            }
          delete p;
        }
      }
    }
  }
  printf("driver: format=%d rc=%d header_ok=%d n_ref=%zu blocks=%zu tags=%zu ranges=%d\n", f.format, rc, f.header_ok ? 1 : 0, f.ref_names.size(), f.blocks.size(), n_tags, partitions);
  release_file(&f);
  return 0;
}
