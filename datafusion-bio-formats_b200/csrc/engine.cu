// engine.cu -- the device pipeline behind BamExec::execute, and the extern "C" entry points.
//
// Per partition (== one reference `execute(partition)` stream, physical_exec.rs:108-172) the engine walks the
// partition's BGZF block ranges in CHUNKS (default 512 MiB inflated) and, per chunk, runs on one compute stream:
//
//   H2D (side stream, pinned source, double buffered)            BASELINE north_star (1)
//   inflate_kernel              (kernels_inflate.cuh)            north_star (2)
//   carry-in copy of the previous chunk's incomplete tail record
//   seg_candidates / seg_walk / seg_check / seg_repair / seg_scan / seg_emit   north_star (3)
//   decode_fixed_kernel -> multi_scan_* -> decode_var_kernel     north_star (4)
//   D2H of the chunk's Arrow arena (side stream) while the next chunk computes
//
// Two host syncs per chunk (row count; var-len totals) size the arena exactly.  A batch is handed out one
// chunk late so its D2H overlaps the next chunk's kernels.
#include <cuda_runtime.h>
#include <nvtx3/nvToolsExt.h>
#include <fcntl.h>
#include <sys/mman.h>
#include <unistd.h>
#include <zlib.h>

#include <algorithm>
#include <atomic>
#include <functional>
#include <numeric>
#include <cstdio>
#include <cstring>
#include <ctime>
#include <mutex>
#include <thread>
#include <vector>

#include "bamscan_internal.h"
#include "kernels_decode.cuh"
#include "kernels_filter.cuh"
#include "kernels_inflate.cuh"
#include "kernels_inflate_cta.cuh"
#include "kernels_fastq.cuh"
#include "kernels_fasta.cuh"
#include "kernels_sam.cuh"
#include "kernels_vcf.cuh"
#include "kernels_vcf_format.cuh"

namespace bamscan {

const char* last_error_cstr();
bool filter_is_record_pushable(const BamFile& f, const BamScanFilter& flt);

#define CU_TRY(expr)                                                                                         \
  do {                                                                                                       \
    cudaError_t _e = (expr);                                                                                 \
    if (_e != cudaSuccess) {                                                                                 \
      set_error("CUDA error %s at %s:%d (%s)", cudaGetErrorString(_e), __FILE__, __LINE__, #expr);           \
      return BAMSCAN_ERR_CUDA;                                                                               \
    }                                                                                                        \
  } while (0)

constexpr uint32_t HEADROOM = 16u << 20;      // room in front of a chunk for the carried-over tail record
constexpr uint32_t INFL_PAD = 1u << 20;   // slack behind a chunk: literal runs of a corrupt member may overshoot before the check
constexpr uint32_t MAX_BLOCK_SIZE = 256u << 20;
constexpr int FA_HFLAGS = 620;            // FASTA flag words [16, 64) of a chunk on the mapped flags page (nothing else uses [620, 668))

static bool g_have_device = false;
// Page-locked host memory.  Without a device (planning-only use: open / schema / classify / plan) plain memory is
// handed out instead; bamscan_execute refuses to run in that case -- there is no CPU scan path.
void* pinned_alloc(size_t bytes) {
  void* p = nullptr;
  if (!g_have_device) { if (posix_memalign(&p, 4096, bytes ? bytes : 1) != 0) { set_error("out of host memory (%zu bytes)", bytes); return nullptr; } return p; }
  cudaError_t e = cudaHostAlloc(&p, bytes, cudaHostAllocPortable);
  if (e != cudaSuccess) { set_error("cudaHostAlloc(%zu) failed: %s", bytes, cudaGetErrorString(e)); return nullptr; }
  return p;
}
void pinned_free(void* p) { if (!p) return; if (g_have_device) cudaFreeHost(p); else free(p); }

// Maps the file READ-ONLY (O_RDONLY, PROT_READ): the scan never needs write permission on the user's BAM, and nothing a
// stray host or driver write could do reaches the file.  The mapping is not page-locked: compressed bytes reach the GPU
// through a small ring of pinned staging buffers (issue_h2d), so pinned memory does not grow with the file, and the
// per-GPU processes of one node share the page cache.
void* map_file_pinned(const char* path, uint64_t size, bool* registered) {
  *registered = false;
  int fd = open(path, O_RDONLY);
  if (fd < 0) return nullptr;
  void* p = mmap(nullptr, size, PROT_READ, MAP_SHARED, fd, 0);
  close(fd);
  if (p == MAP_FAILED) return nullptr;
  madvise(p, size, MADV_SEQUENTIAL);
  return p;
}
void unmap_file_pinned(void* p, uint64_t size, bool registered) {
  (void)registered;
  if (!p) return;
  munmap(p, size);
}

// memcpy with a few threads: page cache -> pinned staging runs at ~10 GB/s per core, a chunk is ~0.5 GB
static void parallel_copy(uint8_t* dst, const uint8_t* src, size_t n) {
  const size_t piece = 32u << 20;
  unsigned t = (unsigned)std::min<size_t>(4, (n + piece - 1) / piece);
  if (t <= 1) { memcpy(dst, src, n); return; }
  std::vector<std::thread> th;
  const size_t per = ((n + t - 1) / t + 4095) & ~size_t(4095);
  for (unsigned i = 0; i < t; i++) {
    const size_t a = std::min(n, (size_t)i * per), b = std::min(n, a + per);
    if (a < b) th.emplace_back([=] { memcpy(dst + a, src + a, b - a); });
  }
  for (auto& x : th) x.join();
}

// Tiny results (row counts, totals, error words) reach the host through mapped pinned memory written by a kernel:
// a cudaMemcpyAsync D2H would queue on the copy engine behind the previous chunk's multi-hundred-MB Arrow transfer.
__global__ void publish_kernel(const uint32_t* __restrict__ src, volatile uint32_t* __restrict__ dst, int n) {
  for (int i = threadIdx.x; i < n; i += blockDim.x) dst[i] = src[i];
  __threadfence_system();
}

// NVTX ranges around the pipeline steps of a chunk (host-side issue of H2D / inflate / boundaries / decode, the D2H wait):
// an nsys timeline of the end-to-end path shows where a step's wall time goes (SURVEY 5).
struct NvtxRange { explicit NvtxRange(const char* name) { nvtxRangePushA(name); } ~NvtxRange() { nvtxRangePop(); } };

struct DeviceBuf {
  void* p = nullptr; size_t cap = 0;
  int ensure(size_t n) {
    if (n <= cap) return BAMSCAN_OK;
    if (p) cudaFree(p);
    p = nullptr; cap = 0;
    size_t want = n + n / 8 + 256;
    cudaError_t e = cudaMalloc(&p, want);
    if (e != cudaSuccess) { set_error("cudaMalloc(%zu) failed: %s", want, cudaGetErrorString(e)); return BAMSCAN_ERR_CUDA; }
    cap = want;
    return BAMSCAN_OK;
  }
  void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
  template <typename T> T* as() const { return static_cast<T*>(p); }
};

// ---- pinned host arenas: pooled, reference counted by the exported Arrow arrays ----
struct HostArena { uint8_t* p = nullptr; size_t cap = 0; };
static std::mutex g_pool_mu;
static std::vector<HostArena> g_pool;
static HostArena arena_acquire(size_t bytes) {
  {
    std::lock_guard<std::mutex> lk(g_pool_mu);
    int best = -1;
    for (size_t i = 0; i < g_pool.size(); i++) if (g_pool[i].cap >= bytes && (best < 0 || g_pool[i].cap < g_pool[best].cap)) best = (int)i;
    if (best >= 0) { HostArena a = g_pool[best]; g_pool.erase(g_pool.begin() + best); return a; }
  }
  HostArena a;
  // coarse sizes, so that the slices of a scan (whose byte counts differ a little) reuse each other's arenas and the pool
  // stops allocating after the first few batches: page-locking a GB costs ~0.1 s, several times that with 8 ranks at it
  size_t cap = bytes + bytes / 8;
  cap = cap > (64u << 20) ? (cap + (64u << 20) - 1) / (64u << 20) * (64u << 20) : std::max<size_t>(cap, 1 << 16);
  a.p = (uint8_t*)pinned_alloc(cap);
  a.cap = a.p ? cap : 0;
  return a;
}
static void arena_release(HostArena a) {
  if (!a.p) return;
  std::lock_guard<std::mutex> lk(g_pool_mu);
  if (g_pool.size() < 4) { g_pool.push_back(a); return; }
  // keep the largest ones
  size_t smallest = 0;
  for (size_t i = 1; i < g_pool.size(); i++) if (g_pool[i].cap < g_pool[smallest].cap) smallest = i;
  if (g_pool[smallest].cap < a.cap) std::swap(g_pool[smallest], a);
  cudaFreeHost(a.p);
}

struct BatchOwner {
  HostArena arena;                 // host hand-off: pinned arena the batch was copied into
  void* dev = nullptr;             // device hand-off (bamscan_next_device): the batch's own device allocation ...
  cudaEvent_t dev_ready = nullptr; // ... and the event behind the kernels / copy that produced it (ArrowDeviceArray::sync_event)
  int device = 0;
  std::atomic<int> refs{0};
};
static void owner_unref(BatchOwner* o) {
  if (o->refs.fetch_sub(1) == 1) {
    arena_release(o->arena);
    if (o->dev || o->dev_ready) {
      int cur = 0; cudaGetDevice(&cur);
      if (cur != o->device) cudaSetDevice(o->device);
      if (o->dev_ready) { cudaEventSynchronize(o->dev_ready); cudaEventDestroy(o->dev_ready); }
      if (o->dev) cudaFree(o->dev);
      if (cur != o->device) cudaSetDevice(cur);
    }
    delete o;
  }
}

// one output column of a chunk (offsets into the arena; same layout on device and host)
struct ColLayout {
  int32_t schema_idx = 0, kind = 0;
  bool has_validity = false;
  size_t validity_off = 0, offsets_off = 0, values_off = 0, data_off = 0;
  uint64_t data_bytes = 0;      // var-len data bytes / list child bytes
  uint64_t child_len = 0;       // list child element count
  bool child_validity = false;  // VCF lists: the child has a validity bitmap (child_validity_off)
  size_t child_validity_off = 0, child_offsets_off = 0;   // List<Utf8>: child_offsets_off holds the child's offsets
  // VCF FORMAT List<List<...>>: the child is the middle list (child_validity_off, child_offsets_off), the leaves have their own
  // validity and their values at data_off
  uint64_t leaf_len = 0;
  size_t leaf_validity_off = 0;
  uint64_t elem_bytes = 0;      // VCF FORMAT: the bytes of the element and leaf buffers that data_bytes does not count
};

struct ChunkPlan { uint32_t b0 = 0, b1 = 0; uint64_t c0 = 0, c1 = 0, u0 = 0, ubytes = 0; bool extension = false; };

struct PendingBatch {
  BatchOwner* owner = nullptr;
  std::vector<ColLayout> cols;
  uint64_t rows = 0;
  size_t arena_bytes = 0;
  size_t err_off = 0;
  uint64_t row0 = 0;               // rows of the partition in front of this batch (FASTA error messages)
  cudaEvent_t done = nullptr;
  bool valid = false;
};

struct ReadyBatch { BatchOwner* owner; std::vector<ColLayout> cols; uint64_t rows_total, row0, nrows; };

}  // namespace bamscan

using namespace bamscan;

struct BamScanStream;
struct BamScanHandle { BamFile file; std::mutex mu; std::vector<BamScanStream*> idle_streams; };   // idle_streams: device buffers, CUDA streams and events kept for the next execute()
struct BamScanPlan { Plan* plan = nullptr; BamScanHandle* handle = nullptr; };

struct BamScanStream {
  Plan* plan = nullptr; BamFile* f = nullptr; const Partition* part = nullptr; BamScanHandle* handle = nullptr;
  bool resources_ready = false;
  uint32_t mean_record_bytes = 0;        // of the last chunk whose records were counted (segment size of the next ones)
  bool device_resident = false;
  bool device_export = false;            // batches stay in HBM and are handed out through the Arrow C Device Data Interface
  // Chunk k runs entirely on s_chunk[k & 1] (inflate, record boundaries, rows, decode): the next chunk's inflate is queued on
  // the other stream as soon as this chunk's boundaries are known, so it overlaps this chunk's decode kernels -- the inflate
  // kernel fills the SMs' shared memory but leaves registers, issue slots and nearly all of the HBM bandwidth unused.  Every
  // per-chunk device buffer is double buffered by the same slot; stream order makes the reuse two chunks later safe.
  cudaStream_t s_chunk[2] = {nullptr, nullptr}, s_compute = nullptr /* = s_chunk[0] */, s_h2d = nullptr, s_d2h = nullptr;
  cudaEvent_t ev_h2d[2] = {nullptr, nullptr}, ev_compute = nullptr, ev_flags[2] = {nullptr, nullptr}, ev_dflags = nullptr, ev_carry = nullptr, ev_t[2][6] = {}, ev_dt[2] = {};
  // iteration
  size_t range_idx = 0;
  std::vector<ChunkPlan> chunks; size_t chunk_idx = 0; bool range_open = false; bool finished = false;
  uint32_t carry_len = 0; bool have_h2d_ahead = false; uint32_t ext_blocks = 8; bool need_spec = false;
  // room in front of a chunk for the carried tail record: HEADROOM for BAM, SAM and FASTQ; a FASTA record may be far longer, so
  // for FASTA it grows to the carried record.  desc_base: the room a slot's member descriptors were built for (issue_h2d)
  uint32_t headroom = HEADROOM, desc_base[2] = {HEADROOM, HEADROOM};
  bool fa_lead_nl = true;     // FASTA: the byte in front of the next chunk is a '\n' (its first byte starts a line)
  bool fa_leading = false;    // FASTA: the range owns the file's first byte and no '>' was found yet
  int n_format = 0;           // VCF: projected FORMAT columns
  // unique decoded columns
  std::vector<int32_t> dec_cols;          // schema indices, unique
  std::vector<int32_t> out_to_dec;        // projection position -> index into dec_cols
  // device memory
  DeviceBuf d_comp[2], d_blk[2], d_infl[2], d_carry, d_status[2], d_flags[2], d_seg[2], d_recoff[2], d_recoff2[2], d_keep[2], d_tiles, d_totals, d_scratch, d_arena[2], d_refs, d_sorted;
  // SAM: per slot the parsed lines, record sizes -> offsets, "QUAL is *" flags, scan tiles and the transcoded BAM records;
  // the reference names sorted bytewise for RNAME / RNEXT lookups
  DeviceBuf d_samline[2], d_samsize[2], d_qabs[2], d_samtiles[2], d_bam[2], d_samrefs;
  // FASTA: per slot the line index of every record start and every line's destination in the sequence text
  DeviceBuf d_fastarts[2], d_faseq[2];
  cudaEvent_t ev_text_free[2] = {nullptr, nullptr}, ev_ing[2][2] = {};   // the write pass has read a slot's text; ingest copy timing
  bool tail_seen = false, range_stop = false;   // per-reference unmapped tail state (physical_exec.rs:1203-1215)
  const uint8_t* d_comp_all = nullptr; DeviceBuf d_comp_all_buf; uint64_t comp_all_c0 = 0;
  uint32_t* d_hflags = nullptr;           // device alias of h_flags (mapped)
  uint32_t* h_flags = nullptr;            // pinned mirror: [0..15] boundary flags / inflate err, [16..] totals (u64)
  BlockDesc* h_descs[2] = {nullptr, nullptr}; size_t h_descs_cap[2] = {0, 0}; uint32_t n_descs[2] = {0, 0}; uint32_t chunk_data_hi[2] = {0, 0};
  uint8_t* h_stage[2] = {nullptr, nullptr}; size_t h_stage_cap[2] = {0, 0};   // pinned staging ring for the compressed bytes (the file mapping is read-only, not page-locked)
  int arena_flip = 0;
  // rows of the current chunk that are not decoded yet: a chunk is one inflate wave, a batch is one slice of its rows
  bool slice_pending = false;    // a decode slice whose time / error word has not been collected (flush_slice)
  int64_t launched_chunk = -1;   // index in `chunks` of a chunk whose inflate + boundary kernels are already queued (run_chunk phase 1)
  struct { const uint8_t* U = nullptr; const uint32_t* recoff = nullptr; const uint8_t* qabs = nullptr; uint32_t n = 0, pos = 0, rows_per_slice = 0; bool long_records = false; uint64_t ubytes = 0; cudaStream_t cs = nullptr;
           // FASTA: the chunk's lines, their destinations, the newline scan's tile bases and the decode slices (first record, first byte)
           const uint32_t* fa_lines = nullptr; const uint32_t* fa_seqpos = nullptr; const uint32_t* fa_tile_base = nullptr; uint32_t fa_lo = 0, fa_hi = 0;
           uint32_t fa_slice_rec[FA_MAX_SLICES + 1] = {}, fa_slice_byte[FA_MAX_SLICES + 1] = {}, fa_slice = 0; } cur;
  PendingBatch pending;
  std::vector<ReadyBatch> ready; size_t ready_pos = 0;
  BamScanStats st{};
  int error = 0;
};

namespace bamscan {

static inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }
static double wall_ms() { timespec ts; clock_gettime(CLOCK_MONOTONIC, &ts); return ts.tv_sec * 1e3 + ts.tv_nsec * 1e-6; }

static bool g_crc_init[64] = {};
static uint32_t* g_crc_tabs[64] = {};
static unsigned long long* g_icta_prof = nullptr;   // bamscan_bench_inflate with BAMSCAN_ICTA_PROF=1: per-phase cycle counters             // per device: tables of the in-window CRC stage (kernels_inflate_cta.cuh)
static int init_device_constants(int dev) {
  if (dev >= 64) { set_error("device id %d out of range", dev); return BAMSCAN_ERR_CUDA; }
  if (g_crc_init[dev]) return BAMSCAN_OK;
  CU_TRY(cudaMalloc((void**)&g_crc_tabs[dev], icta::CrcTabs<icta::NT_C>::WORDS * 4));
  icta::crc_tables_init_kernel<icta::NT_C><<<1, 256>>>(g_crc_tabs[dev]);
  CU_TRY(cudaDeviceSynchronize());
  // x^(8 * 2^j) mod P in the reflected domain
  auto mulmod = [](uint32_t a, uint32_t b) { uint32_t p = 0; for (int i = 0; i < 32; i++) { if (b & 0x80000000u) p ^= a; a = (a >> 1) ^ ((a & 1u) ? 0xEDB88320u : 0u); b <<= 1; } return p; };
  uint32_t tab[18];
  tab[0] = 0x00800000u;   // x^8
  for (int j = 1; j < 18; j++) tab[j] = mulmod(tab[j - 1], tab[j - 1]);
  CU_TRY(cudaMemcpyToSymbol(c_crc_xpow8, tab, sizeof tab));
  g_crc_init[dev] = true;
  return BAMSCAN_OK;
}

// ---- inflate: three kernels, one picked per launch ----
//   inflate_cta_kernel   parallel INSIDE the member, two members per CTA (kernels_inflate_cta.cuh): 592 members in flight, a member
//                        is done in ~0.3 ms.  Members it refuses (INF_RETRY) are redone by inflate_kernel.  Picked for every
//                        launch of up to ICTA_MAX_MEMBERS members: region queries, tail chunks, small and long-read files.
//   inflate_lg_kernel    4 lanes per member, 152 members per SM (22 496 in flight), a member takes ~17 ms: more members per
//                        second on a FULL wave (15.9 ms against 20.1 ms measured), so whole-wave chunks of a big scan use it.
//   inflate_kernel       a warp per member: the retry path of the first.
//   debug_flags: bit 2 forces inflate_kernel, bit 3 inflate_lg_kernel, bit 4 inflate_cta_kernel (tests and A/B runs).
constexpr uint32_t ICTA_MAX_MEMBERS = 0xffffffffu;   // (every launch: since round 2 the CTA kernel is also the faster one on full waves, 15.3 ms against 15.9 ms)
#ifndef BAMSCAN_LG_W
#define BAMSCAN_LG_W 19
#endif
#ifndef BAMSCAN_LG_NLIT
#define BAMSCAN_LG_NLIT 2
#endif
constexpr int LG_G = 4, LG_W = BAMSCAN_LG_W, LG_NLIT = BAMSCAN_LG_NLIT;
using LgCfg = LgConfig<LG_G, LG_W>;
static int device_sms(int device) { int sms = 148; cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device); return sms; }

// Inflates the nb members described by d_blk (and verifies their CRC-32 unless skip_crc) on stream cs.
// d_retry_ticket, d_retries: zeroed words (ticket of the retry launch; members the CTA kernel refused, counted by it).
static int launch_inflate(const BamFile* f, cudaStream_t cs, const uint8_t* d_comp, const BlockDesc* d_blk, uint32_t nb, uint8_t* U,
                          uint32_t* d_status, uint32_t* d_ticket, uint32_t* d_err, uint32_t* d_retry_ticket, uint32_t* d_retries,
                          DeviceBuf* slots, int* launches) {
  const uint32_t sms = (uint32_t)device_sms(f->device);
  const int check_crc = f->skip_crc ? 0 : 1;
  if (f->debug_flags & 4) {          // tests: the warp-per-member kernel on everything
    uint32_t grid = std::min<uint32_t>((nb + INF_WARPS - 1) / INF_WARPS, sms * INF_CTAS_PER_SM);
    inflate_kernel<<<grid, INF_WARPS * 32, sizeof(InflateShared), cs>>>(d_comp, d_blk, nb, U, d_status, d_ticket, d_err, check_crc, 0xffffffffu);
    *launches += 1;
    return BAMSCAN_OK;
  }
  if ((f->debug_flags & 8) || (!(f->debug_flags & 16) && nb > ICTA_MAX_MEMBERS)) {   // lane-group kernel + separate CRC kernel
    const uint32_t per_cta = (uint32_t)(LgCfg::GROUPS * LG_W);
    const uint32_t grid = std::min<uint32_t>((nb + per_cta - 1) / per_cta, sms);
    int rc = slots->ensure((size_t)sms * per_cta * LG_SLOT_BYTES);
    if (rc) return rc;
    inflate_lg_kernel<LG_G, LG_W, LG_NLIT, 1><<<grid, LG_W * 32, LgCfg::SMEM, cs>>>(d_comp, d_blk, nb, U, d_status, d_ticket, d_err, slots->as<uint8_t>());
    *launches += 1;
    if (check_crc) {
      crc_kernel<<<std::min<uint32_t>((nb + CRC_WARPS - 1) / CRC_WARPS, sms), CRC_WARPS * 32, CRC_SMEM, cs>>>(d_blk, nb, U, d_status, d_err);
      *launches += 1;
    }
    return BAMSCAN_OK;
  }
  {
    const uint32_t grid = std::min<uint32_t>(nb, sms * 2u);
    icta::inflate_cta_kernel<<<grid, icta::NT, icta::Cfg::SMEM, cs>>>(d_comp, d_blk, nb, U, d_status, d_ticket, d_err, d_retries, g_crc_tabs[f->device], check_crc, g_icta_prof);
    *launches += 1;
    // members flagged INF_RETRY (none on ordinary files); the launch finds nothing to do otherwise
    uint32_t rgrid = std::min<uint32_t>((nb + INF_WARPS - 1) / INF_WARPS, sms);
    inflate_kernel<<<rgrid, INF_WARPS * 32, sizeof(InflateShared), cs>>>(d_comp, d_blk, nb, U, d_status, d_retry_ticket, d_err, check_crc, icta::INF_RETRY);
    *launches += 1;
  }
  return BAMSCAN_OK;
}

static int stream_init(BamScanStream* s) {
  BamFile* f = s->f;
  CU_TRY(cudaSetDevice(f->device));
  int rc = BAMSCAN_OK;
  // per-scan state
  s->range_idx = 0; s->chunks.clear(); s->chunk_idx = 0; s->range_open = false; s->finished = false;
  s->carry_len = 0; s->have_h2d_ahead = false; s->ext_blocks = 8; s->need_spec = false; s->tail_seen = false; s->range_stop = false;
  s->headroom = HEADROOM; s->desc_base[0] = s->desc_base[1] = HEADROOM;
  s->dec_cols.clear(); s->out_to_dec.clear(); s->arena_flip = 0; s->cur.n = s->cur.pos = 0; s->launched_chunk = -1; s->slice_pending = false; s->pending = PendingBatch(); s->ready.clear(); s->ready_pos = 0;
  s->st = BamScanStats{}; s->st.first_record_uoff = ~0ull; s->error = 0; s->d_comp_all = nullptr; s->comp_all_c0 = 0;
  if (!s->resources_ready) {
  rc = init_device_constants(f->device);
  if (rc) return rc;
  for (auto& st : s->s_chunk) CU_TRY(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
  s->s_compute = s->s_chunk[0];
  CU_TRY(cudaStreamCreateWithFlags(&s->s_h2d, cudaStreamNonBlocking));
  CU_TRY(cudaStreamCreateWithFlags(&s->s_d2h, cudaStreamNonBlocking));
  for (int i = 0; i < 2; i++) CU_TRY(cudaEventCreateWithFlags(&s->ev_h2d[i], cudaEventDisableTiming));
  CU_TRY(cudaEventCreateWithFlags(&s->ev_compute, cudaEventDisableTiming));
  for (auto& e : s->ev_flags) CU_TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
  CU_TRY(cudaEventCreateWithFlags(&s->ev_dflags, cudaEventDisableTiming));
  CU_TRY(cudaEventCreateWithFlags(&s->ev_carry, cudaEventDisableTiming));
  for (auto& row : s->ev_t) for (auto& e : row) CU_TRY(cudaEventCreate(&e));
  for (auto& e : s->ev_dt) CU_TRY(cudaEventCreate(&e));
  for (auto& e : s->ev_text_free) CU_TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
  for (auto& row : s->ev_ing) for (auto& e : row) CU_TRY(cudaEventCreate(&e));
  CU_TRY(cudaHostAlloc((void**)&s->h_flags, 4096, cudaHostAllocPortable | cudaHostAllocMapped));
  CU_TRY(cudaHostGetDevicePointer((void**)&s->d_hflags, s->h_flags, 0));
  CU_TRY(cudaFuncSetAttribute(inflate_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(InflateShared)));
  CU_TRY(cudaFuncSetAttribute(inflate_lg_kernel<LG_G, LG_W, LG_NLIT, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)LgCfg::SMEM));
  CU_TRY(cudaFuncSetAttribute(crc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)CRC_SMEM));
  CU_TRY(cudaFuncSetAttribute(icta::inflate_cta_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)icta::Cfg::SMEM));
  CU_TRY(cudaFuncSetAttribute(icta::inflate_cta_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, 100));
  // reference dictionary: lengths + names blob
  size_t n_ref = f->ref_names.size();
  std::vector<uint32_t> offs(n_ref + 1, 0);
  std::string blob;
  for (size_t i = 0; i < n_ref; i++) { offs[i] = (uint32_t)blob.size(); blob += f->ref_names[i]; }
  offs[n_ref] = (uint32_t)blob.size();
  size_t o_len = 0, o_off = align_up(4 * n_ref + 4, 16), o_blob = o_off + align_up(4 * (n_ref + 1), 16);
  rc = s->d_refs.ensure(o_blob + blob.size() + 16);
  if (rc) return rc;
  if (n_ref) CU_TRY(cudaMemcpy(s->d_refs.as<uint8_t>() + o_len, f->ref_lens.data(), 4 * n_ref, cudaMemcpyHostToDevice));
  CU_TRY(cudaMemcpy(s->d_refs.as<uint8_t>() + o_off, offs.data(), 4 * (n_ref + 1), cudaMemcpyHostToDevice));
  if (!blob.empty()) CU_TRY(cudaMemcpy(s->d_refs.as<uint8_t>() + o_blob, blob.data(), blob.size(), cudaMemcpyHostToDevice));
  if (f->format == FMT_SAM) {
    // SAM: names sorted bytewise + their ids (enc::lookup_ref), laid out as [offsets n_ref + 1][ids n_ref][names]
    std::vector<int32_t> ids(n_ref);
    std::iota(ids.begin(), ids.end(), 0);
    std::sort(ids.begin(), ids.end(), [&](int32_t a, int32_t b) { return f->ref_names[a] < f->ref_names[b]; });
    std::vector<int32_t> soff(n_ref + 1, 0);
    std::string sblob;
    for (size_t i = 0; i < n_ref; i++) { soff[i] = (int32_t)sblob.size(); sblob += f->ref_names[ids[i]]; }
    soff[n_ref] = (int32_t)sblob.size();
    const size_t o_ids = align_up(4 * (n_ref + 1), 16), o_names = o_ids + align_up(4 * n_ref + 4, 16);
    rc = s->d_samrefs.ensure(o_names + sblob.size() + 16);
    if (rc) return rc;
    CU_TRY(cudaMemcpy(s->d_samrefs.p, soff.data(), 4 * (n_ref + 1), cudaMemcpyHostToDevice));
    if (n_ref) CU_TRY(cudaMemcpy(s->d_samrefs.as<uint8_t>() + o_ids, ids.data(), 4 * n_ref, cudaMemcpyHostToDevice));
    if (!sblob.empty()) CU_TRY(cudaMemcpy(s->d_samrefs.as<uint8_t>() + o_names, sblob.data(), sblob.size(), cudaMemcpyHostToDevice));
  }
  s->resources_ready = true;
  }
  // unique decode columns
  const Plan* P = s->plan;
  std::vector<int32_t> proj;
  if (P->has_projection) proj = P->projection; else for (size_t i = 0; i < f->fields.size(); i++) proj.push_back((int32_t)i);
  for (int32_t c : proj) {
    auto it = std::find(s->dec_cols.begin(), s->dec_cols.end(), c);
    if (it == s->dec_cols.end()) { s->out_to_dec.push_back((int32_t)s->dec_cols.size()); s->dec_cols.push_back(c); }
    else s->out_to_dec.push_back((int32_t)(it - s->dec_cols.begin()));
  }
  if (f->format == FMT_VCF) {
    int n_info = 0;
    s->n_format = 0;
    for (int32_t c : s->dec_cols) {                               // INFO columns follow the eight fixed ones, FORMAT columns them
      if (c >= f->vcf_info_end) s->n_format++;
      else if (c >= 8) n_info++;
    }
    if (n_info > vcf::MAX_INFO) { set_error("more than %d projected INFO columns are not supported by this build", vcf::MAX_INFO); return BAMSCAN_ERR_UNSUPPORTED; }
    return BAMSCAN_OK;
  }
  int n_tag_cols = 0;
  for (int32_t c : s->dec_cols) if (c >= 12) n_tag_cols++;
  if (f->decode_all_tags && n_tag_cols) {
    // reference quirk (sam_tag_io.rs:42-52): any projected tag makes the reader decode EVERY tag_fields entry; the extra columns
    // are decoded (and their coercions checked) but never exported: no projection position maps to them
    for (int32_t c = 12; c < (int32_t)f->fields.size(); c++)
      if (std::find(s->dec_cols.begin(), s->dec_cols.end(), c) == s->dec_cols.end()) { s->dec_cols.push_back(c); n_tag_cols++; }
  }
  if (n_tag_cols > MAX_TAGS) { set_error("more than %d projected tag columns are not supported by this build", MAX_TAGS); return BAMSCAN_ERR_UNSUPPORTED; }
  return BAMSCAN_OK;
}

static void stream_destroy(BamScanStream* s, bool recycle = true) {
  if (!s) return;
  cudaSetDevice(s->f->device);
  for (auto st : s->s_chunk) if (st) cudaStreamSynchronize(st);
  if (s->s_h2d) cudaStreamSynchronize(s->s_h2d);
  if (s->s_d2h) cudaStreamSynchronize(s->s_d2h);
  if (s->pending.valid) { owner_unref(s->pending.owner); if (s->pending.done) cudaEventDestroy(s->pending.done); }
  for (size_t i = s->ready_pos; i < s->ready.size(); i++) owner_unref(s->ready[i].owner);
  s->pending = PendingBatch(); s->ready.clear(); s->ready_pos = 0;
  s->d_comp_all_buf.release();     // the staged copy of a whole partition is never kept
  if (recycle && s->resources_ready && s->handle && cudaGetLastError() == cudaSuccess) {
    std::lock_guard<std::mutex> lk(s->handle->mu);
    if (s->handle->idle_streams.size() < 2) { s->handle->idle_streams.push_back(s); return; }
  }
  for (auto* b : {&s->d_comp[0], &s->d_comp[1], &s->d_blk[0], &s->d_blk[1], &s->d_infl[0], &s->d_infl[1], &s->d_carry, &s->d_status[0], &s->d_status[1], &s->d_flags[0], &s->d_flags[1], &s->d_seg[0], &s->d_seg[1],
                  &s->d_recoff[0], &s->d_recoff[1], &s->d_recoff2[0], &s->d_recoff2[1], &s->d_keep[0], &s->d_keep[1], &s->d_tiles, &s->d_totals, &s->d_scratch, &s->d_arena[0], &s->d_arena[1], &s->d_refs, &s->d_comp_all_buf, &s->d_sorted,
                  &s->d_samline[0], &s->d_samline[1], &s->d_samsize[0], &s->d_samsize[1], &s->d_qabs[0], &s->d_qabs[1], &s->d_samtiles[0], &s->d_samtiles[1], &s->d_bam[0], &s->d_bam[1], &s->d_samrefs,
                  &s->d_fastarts[0], &s->d_fastarts[1], &s->d_faseq[0], &s->d_faseq[1]}) b->release();
  if (s->h_flags) cudaFreeHost(s->h_flags);
  for (auto& hd : s->h_descs) if (hd) cudaFreeHost(hd);
  for (auto& hs : s->h_stage) if (hs) cudaFreeHost(hs);
  for (auto& e : s->ev_h2d) if (e) cudaEventDestroy(e);
  if (s->ev_compute) cudaEventDestroy(s->ev_compute);
  for (auto& e : s->ev_flags) if (e) cudaEventDestroy(e);
  if (s->ev_dflags) cudaEventDestroy(s->ev_dflags);
  if (s->ev_carry) cudaEventDestroy(s->ev_carry);
  for (auto& row : s->ev_t) for (auto& e : row) if (e) cudaEventDestroy(e);
  for (auto& e : s->ev_dt) if (e) cudaEventDestroy(e);
  for (auto& e : s->ev_text_free) if (e) cudaEventDestroy(e);
  for (auto& row : s->ev_ing) for (auto& e : row) if (e) cudaEventDestroy(e);
  for (auto st : s->s_chunk) if (st) cudaStreamDestroy(st);
  if (s->s_h2d) cudaStreamDestroy(s->s_h2d);
  if (s->s_d2h) cudaStreamDestroy(s->s_d2h);
  delete s;
}

// Members the throughput inflate kernel keeps in flight (one per lane group).  A member takes milliseconds, so a chunk whose
// member count is not a whole number of such waves leaves most of the GPU idle in its last wave.
static uint32_t inflate_wave_members(int device) { return (uint32_t)device_sms(device) * LgCfg::GROUPS * LG_W; }

// A chunk is the unit of H2D, inflate and record-boundary resolution; its rows are decoded in slices of <= SLICE_BYTES
// inflated (Arrow offsets are i32).  Default: one whole inflate wave per chunk (a member takes milliseconds, so a chunk
// that is not a whole number of waves leaves most of the GPU idle in its last wave); chunk_inflated_bytes overrides it.
static const uint64_t SLICE_BYTES = 768ull << 20;
static const uint64_t FMT_SLICE_ELEMS = 1ull << 24;
static uint64_t chunk_cap_bytes(const BamFile& f) {
  if (f.chunk_bytes) return f.chunk_bytes;
  if (f.format == FMT_SAM) return 512ull << 20;    // SAM: text bytes per chunk (no inflate wave to fill)
  // FASTA: the carried record (up to 1 GiB) sits in front of the chunk, and chunk offsets are u32
  return std::min<uint64_t>((uint64_t)inflate_wave_members(f.device) * 65280ull + 65536ull, f.format == FMT_FASTA ? 2ull << 30 : 3ull << 30);
}
static void plan_chunks(const BamFile& f, uint32_t b0, uint32_t b1, bool extension, std::vector<ChunkPlan>* out) {
  const uint32_t wave = inflate_wave_members(f.device);
  const uint64_t cap = chunk_cap_bytes(f);
  const uint64_t waves = cap / ((uint64_t)wave * 65280ull);
  const uint32_t member_cap = waves >= 1 ? (uint32_t)waves * wave : 0xffffffffu;   // small (test) chunk sizes: bytes only
  uint32_t b = b0;
  while (b < b1) {
    ChunkPlan c; c.b0 = b; c.u0 = f.blocks[b].uoff; c.c0 = f.blocks[b].coff; c.extension = extension;
    uint64_t ub = 0; uint32_t members = 0;
    while (b < b1 && (ub == 0 || (ub + f.blocks[b].isize <= cap && members < member_cap))) { ub += f.blocks[b].isize; members += f.blocks[b].isize ? 1u : 0u; b++; }
    c.b1 = b; c.ubytes = ub; c.c1 = f.blocks[b - 1].coff + f.blocks[b - 1].csize;
    out->push_back(c);
  }
}

// An empty member (ISIZE 0) gives the inflate kernels nothing to do, so it has no descriptor; it is still a member of the
// file, and zlib and the reference's reader reject it unless its CRC-32 is 0 and its payload inflates to nothing.  It is
// checked on the host (it is a few bytes; host zlib) when the chunk that holds it is staged: a scan fails on the empty
// members of the blocks it reads, and a region query never looks at members outside its blocks.
static int check_empty_member(const BamFile* f, uint32_t b) {
  const BgzfBlock& B = f->blocks[b];
  const char* why = nullptr;
  if (B.crc != 0) why = "CRC32 mismatch";
  else {
    z_stream zs; memset(&zs, 0, sizeof zs);
    uint8_t out = 0;
    if (inflateInit2(&zs, -15) != Z_OK) { set_error("zlib initialisation failed"); return BAMSCAN_ERR_IO; }
    zs.next_in = const_cast<Bytef*>(f->data + B.coff + B.cdata_off); zs.avail_in = B.csize - B.cdata_off - 8;
    zs.next_out = &out; zs.avail_out = 1;
    const int zr = inflate(&zs, Z_FINISH);
    if (zs.total_out) why = "ISIZE mismatch";
    else if (zr != Z_STREAM_END) why = "invalid deflate stream";
    inflateEnd(&zs);
  }
  if (!why) return BAMSCAN_OK;
  set_error("BAM read error: BGZF member %u (file offset %llu): inflate failed: %s", b, (unsigned long long)B.coff, why);
  return BAMSCAN_ERR_CRC;
}

// page cache -> the slot's pinned staging buffer (its previous transfer has long finished)
static int stage_bytes(BamScanStream* s, uint64_t c0, size_t bytes, int slot) {
  CU_TRY(cudaEventSynchronize(s->ev_h2d[slot]));
  if (s->h_stage_cap[slot] < bytes) {
    if (s->h_stage[slot]) cudaFreeHost(s->h_stage[slot]);
    const size_t cap = bytes + bytes / 8 + 4096;
    s->h_stage[slot] = (uint8_t*)pinned_alloc(cap);
    if (!s->h_stage[slot]) { s->h_stage_cap[slot] = 0; return BAMSCAN_ERR_CUDA; }
    s->h_stage_cap[slot] = cap;
  }
  parallel_copy(s->h_stage[slot], s->f->data + c0, bytes);
  return BAMSCAN_OK;
}

// SAM: the chunk's text goes straight into its buffer behind the carry headroom with one copy (H2D from the staging ring, or
// device to device from the staged partition of a device-resident run).  No descriptors, no inflate.
static int issue_h2d_text(BamScanStream* s, const ChunkPlan& c, int slot) {
  const size_t bytes = (size_t)(c.c1 - c.c0);
  int rc;
  s->n_descs[slot] = 0; s->chunk_data_hi[slot] = HEADROOM + (uint32_t)bytes;
  if ((rc = s->d_infl[slot].ensure((size_t)HEADROOM + bytes + INFL_PAD))) return rc;
  uint8_t* dst = s->d_infl[slot].as<uint8_t>() + HEADROOM;
  CU_TRY(cudaStreamWaitEvent(s->s_h2d, s->ev_text_free[slot], 0));     // the write pass of the chunk two back has read this buffer
  if (!s->device_resident && (rc = stage_bytes(s, c.c0, bytes, slot))) return rc;
  CU_TRY(cudaEventRecord(s->ev_ing[slot][0], s->s_h2d));
  if (s->device_resident) CU_TRY(cudaMemcpyAsync(dst, s->d_comp_all + (c.c0 - s->comp_all_c0), bytes, cudaMemcpyDeviceToDevice, s->s_h2d));
  else { CU_TRY(cudaMemcpyAsync(dst, s->h_stage[slot], bytes, cudaMemcpyHostToDevice, s->s_h2d)); s->st.h2d_bytes += bytes; }
  CU_TRY(cudaEventRecord(s->ev_ing[slot][1], s->s_h2d));
  CU_TRY(cudaEventRecord(s->ev_h2d[slot], s->s_h2d));
  return BAMSCAN_OK;
}

// Builds the chunk's member descriptors in pinned memory and queues them, with the compressed bytes, on the H2D stream.
// Everything the compute stream needs from the host for this chunk travels here, so the copy engine never makes the
// kernels of the previous chunk wait (a pageable copy issued on the compute stream would queue behind the big transfer).
static int issue_h2d(BamScanStream* s, const ChunkPlan& c, int slot) {
  NvtxRange nv("bamscan: stage + H2D of a chunk's compressed members");
  const BamFile* f = s->f;
  if (f->format == FMT_SAM) return issue_h2d_text(s, c, slot);
  const uint32_t nb_all = c.b1 - c.b0;
  if (s->h_descs_cap[slot] < nb_all) {
    if (s->h_descs[slot]) cudaFreeHost(s->h_descs[slot]);
    size_t cap = std::max<size_t>(nb_all + nb_all / 4, 1024);
    s->h_descs[slot] = (BlockDesc*)pinned_alloc(cap * sizeof(BlockDesc));
    if (!s->h_descs[slot]) { s->h_descs_cap[slot] = 0; return BAMSCAN_ERR_CUDA; }
    s->h_descs_cap[slot] = cap;
  }
  BlockDesc* descs = s->h_descs[slot];
  uint32_t uoff = s->headroom, nb = 0;
  s->desc_base[slot] = s->headroom;
  for (uint32_t b = c.b0; b < c.b1; b++) {
    const BgzfBlock& B = f->blocks[b];
    if (B.isize) { BlockDesc d; d.cdata_off = (uint32_t)(B.coff - c.c0) + B.cdata_off; d.cdata_len = B.csize - B.cdata_off - 8; d.isize = B.isize; d.crc = B.crc; d.uoff = uoff; descs[nb++] = d; }
    else if (int rc = check_empty_member(f, b)) return rc;
    uoff += B.isize;
  }
  s->n_descs[slot] = nb; s->chunk_data_hi[slot] = uoff;
  int rc = s->d_blk[slot].ensure(sizeof(BlockDesc) * std::max<uint32_t>(nb, 1));
  if (rc) return rc;
  if (nb) CU_TRY(cudaMemcpyAsync(s->d_blk[slot].p, descs, sizeof(BlockDesc) * nb, cudaMemcpyHostToDevice, s->s_h2d));
  if (!s->device_resident) {
    size_t bytes = (size_t)(c.c1 - c.c0);
    if ((rc = s->d_comp[slot].ensure(bytes + 1024))) return rc;
    // page cache -> pinned staging buffer of this slot -> one async copy
    if ((rc = stage_bytes(s, c.c0, bytes, slot))) return rc;
    CU_TRY(cudaMemcpyAsync(s->d_comp[slot].p, s->h_stage[slot], bytes, cudaMemcpyHostToDevice, s->s_h2d));
    CU_TRY(cudaMemsetAsync(s->d_comp[slot].as<uint8_t>() + bytes, 0, 1024, s->s_h2d));   // the bit reader may look a few words past the last member
    s->st.h2d_bytes += bytes;
  }
  CU_TRY(cudaEventRecord(s->ev_h2d[slot], s->s_h2d));
  return BAMSCAN_OK;
}

struct ArenaBuilder {
  size_t pos = 0;
  size_t take(size_t bytes) { size_t o = pos; pos = align_up(pos + bytes, 256); return o; }
};

// Collects the time and, for device-resident runs, the error word of the decode slice queued last (decode_slice).
static int flush_slice(BamScanStream* s) {
  if (!s->slice_pending) return BAMSCAN_OK;
  s->slice_pending = false;
  CU_TRY(cudaEventSynchronize(s->ev_dt[1]));
  { float d = 0; cudaEventElapsedTime(&d, s->ev_dt[0], s->ev_dt[1]); s->st.ms_decode += d; }
  if (s->device_resident && s->h_flags[512]) { set_error("decode error %u at row %u", s->h_flags[512], s->h_flags[513]); return BAMSCAN_ERR_FORMAT; }
  return BAMSCAN_OK;
}

// Arrow offsets from per-row lengths (kernels_decode.cuh phase 2): every column of SC is exclusive-scanned in place, column k's
// total -> totals[k].  tiles holds the tile sums and is sized here.
static int launch_offsets_scan(BamScanStream* s, cudaStream_t cs, const ScanCols& SC, DeviceBuf& tiles, uint64_t* totals) {
  const uint32_t n_tiles = (SC.n + SCAN_TILE - 1) / SCAN_TILE;
  if (int rc = tiles.ensure(8ull * n_tiles * SC.n_cols)) return rc;
  uint64_t* d_tiles = tiles.as<uint64_t>();
  multi_scan_reduce_kernel<<<dim3(n_tiles, SC.n_cols), SCAN_TPB, 0, cs>>>(SC, d_tiles, n_tiles);
  cta_scan_kernel<<<SC.n_cols, CTA_SCAN_THREADS, 0, cs>>>(d_tiles, d_tiles, n_tiles, totals);
  multi_scan_apply_kernel<<<dim3(n_tiles, SC.n_cols), SCAN_TPB, 0, cs>>>(SC, d_tiles, n_tiles);
  s->st.kernel_launches += 3;
  return BAMSCAN_OK;
}

// Hands a decoded slice's arena A (rows n, arena_bytes, error word at err_off) to the consumer: kept in HBM (device-resident runs),
// copied into the batch's own device allocation (device export), or copied to a pinned host arena; queued as s->pending.
static int hand_off_batch(BamScanStream* s, cudaStream_t cs, uint8_t* A, const std::vector<ColLayout>& cols, uint32_t n, size_t arena_bytes,
                          size_t err_off, uint64_t row0, bool* produced) {
  const BamFile* f = s->f;
  if (s->device_resident) {
    // keep everything in HBM: only the decode error word travels
    publish_kernel<<<1, 32, 0, cs>>>(reinterpret_cast<const uint32_t*>(A + err_off), s->d_hflags + 512, 2);     // (checked by flush_slice)
  } else if (s->device_export) {
    // device hand-off: the batch gets its own exactly-sized device allocation (a device-to-device copy on the side
    // stream, ~3 TB/s); only the decode error word travels to the host
    CU_TRY(cudaEventRecord(s->ev_compute, cs));
    PendingBatch& P = s->pending;
    P.owner = new BatchOwner();
    P.owner->device = f->device; P.owner->refs = 1;
    if (cudaMalloc(&P.owner->dev, arena_bytes) != cudaSuccess) { delete P.owner; P.owner = nullptr; set_error("cudaMalloc(%zu) for a device batch failed", arena_bytes); return BAMSCAN_ERR_CUDA; }
    P.cols = cols; P.rows = n; P.arena_bytes = arena_bytes; P.err_off = err_off; P.row0 = row0; P.valid = true;
    if (!P.done) CU_TRY(cudaEventCreateWithFlags(&P.done, cudaEventDisableTiming));
    CU_TRY(cudaEventCreateWithFlags(&P.owner->dev_ready, cudaEventDisableTiming));
    CU_TRY(cudaStreamWaitEvent(s->s_d2h, s->ev_compute, 0));
    CU_TRY(cudaMemcpyAsync(P.owner->dev, A, arena_bytes, cudaMemcpyDeviceToDevice, s->s_d2h));
    CU_TRY(cudaMemcpyAsync(s->h_flags + 514, A + err_off, 8, cudaMemcpyDeviceToHost, s->s_d2h));
    CU_TRY(cudaEventRecord(P.owner->dev_ready, s->s_d2h));
    CU_TRY(cudaEventRecord(P.done, s->s_d2h));
    s->arena_flip ^= 1;
    *produced = true;
  } else {
    CU_TRY(cudaEventRecord(s->ev_compute, cs));
    PendingBatch& P = s->pending;
    P.owner = new BatchOwner();
    P.owner->arena = arena_acquire(arena_bytes);
    if (!P.owner->arena.p) { delete P.owner; P.owner = nullptr; return BAMSCAN_ERR_CUDA; }
    P.owner->refs = 1;
    P.cols = cols; P.rows = n; P.arena_bytes = arena_bytes; P.err_off = err_off; P.row0 = row0; P.valid = true;
    if (!P.done) CU_TRY(cudaEventCreateWithFlags(&P.done, cudaEventDisableTiming));
    CU_TRY(cudaStreamWaitEvent(s->s_d2h, s->ev_compute, 0));
    CU_TRY(cudaMemcpyAsync(P.owner->arena.p, A, arena_bytes, cudaMemcpyDeviceToHost, s->s_d2h));
    CU_TRY(cudaEventRecord(P.done, s->s_d2h));
    s->st.d2h_bytes += arena_bytes;
    s->arena_flip ^= 1;
    // the next chunk must not overwrite this arena before the copy has read it: arenas are double buffered and the
    // batch before this one has already been waited for (see bamscan_next)
    *produced = true;
  }
  return BAMSCAN_OK;
}

// ---- decode slices: one function per format picks the slice's rows, binds its kernels to the arena and launches them; the arena
// steps are shared.  Region A (the error word, then per column its validity words and its offsets or fixed values) is laid out
// before the count kernels run, region B (variable-length data, list children) once the scanned totals are known.

static bool is_var(int32_t kind) { return kind == HK_Utf8 || kind == HK_Binary || kind >= HK_ListInt8; }     // Arrow offsets + data
static size_t fixed_bytes(int32_t kind, uint32_t n) { return kind == HK_Boolean ? 4ull * ((n + 31) / 32) : 4ull * n; }   // Boolean: bitmap words
// A column's buffers in the arena at A: valid is null without a validity bitmap, data until region B is laid out (region A starts
// with the error word, so no data lies at offset 0)
struct ColPtrs { uint32_t* valid; int32_t* offs; uint32_t* vals; uint8_t* data; };
static ColPtrs col_ptrs(uint8_t* A, const ColLayout& L) {
  return {L.has_validity ? reinterpret_cast<uint32_t*>(A + L.validity_off) : nullptr, reinterpret_cast<int32_t*>(A + L.offsets_off),
          reinterpret_cast<uint32_t*>(A + L.values_off), L.data_off ? A + L.data_off : nullptr};
}

struct Slice {
  uint32_t n = 0;                  // rows
  std::vector<ColLayout> cols;     // one per s->dec_cols
  ArenaBuilder AB;
  size_t err_off = 0, region_a = 0;
  uint8_t* A = nullptr;            // s->d_arena[s->arena_flip]
};
struct CountCol { int32_t* counts; size_t col; uint32_t len = 0; };   // a count column, scanned in place, its index in Slice::cols, and
                                                                      // its entries (0: the slice's rows + 1)

// Region A of an n-row slice, in an arena that holds it (a first sizing guess, grown by layout_region_b), with the error word
// cleared.  has_validity: the format's rule for which columns carry a validity bitmap; more (optional): buffers of a column whose
// sizes the row count decides besides its validity and offsets or values.
static int layout_region_a(BamScanStream* s, Slice& S, uint32_t n, bool (*has_validity)(const BamFile&, int32_t),
                           const std::function<void(ColLayout&)>& more = nullptr) {
  S.n = n;
  S.err_off = S.AB.take(64);
  S.cols.resize(s->dec_cols.size());
  for (size_t i = 0; i < S.cols.size(); i++) {
    ColLayout& L = S.cols[i]; L.schema_idx = s->dec_cols[i]; L.kind = s->f->fields[L.schema_idx].kind;
    L.has_validity = has_validity(*s->f, L.schema_idx);
    if (L.has_validity) L.validity_off = S.AB.take(4ull * ((n + 31) / 32));
    if (is_var(L.kind)) L.offsets_off = S.AB.take(4ull * (n + 1)); else L.values_off = S.AB.take(fixed_bytes(L.kind, n));
    if (more) more(L);
  }
  S.region_a = S.AB.pos;
  DeviceBuf& arena = s->d_arena[s->arena_flip];
  if (arena.cap < S.region_a) { if (int rc = arena.ensure(S.region_a + (size_t)s->cur.ubytes * 2)) return rc; }
  S.A = arena.as<uint8_t>();
  CU_TRY(cudaMemsetAsync(S.A + S.err_off, 0, 64, s->cur.cs));
  return BAMSCAN_OK;
}

// The count columns of BAM, SAM, FASTQ and FASTA: the offsets of every variable-length column
static std::vector<CountCol> offset_counts(const Slice& S) {
  std::vector<CountCol> counts;
  for (size_t i = 0; i < S.cols.size(); i++) if (is_var(S.cols[i].kind)) counts.push_back({reinterpret_cast<int32_t*>(S.A + S.cols[i].offsets_off), i});
  return counts;
}

// Count columns -> Arrow offsets, in launches of up to MAX_SCAN_COLS columns of equal length.  The totals reach the host through the
// mapped flags page at [16, 16 + 2 * counts) (VCF's 229 INFO and 16 FORMAT columns at most stay below the decode error words at
// [512, 516)) with one host sync, and each is held to Arrow's 2^31-1 limit.  *T: the totals, in the order of counts.
static int scan_counts(BamScanStream* s, const Slice& S, const std::vector<CountCol>& counts, const uint64_t** T) {
  cudaStream_t cs = s->cur.cs;
  const size_t n_scan = counts.size();
  int rc;
  if ((rc = s->d_totals.ensure(8 * n_scan))) return rc;
  for (size_t k0 = 0; k0 < n_scan;) {
    ScanCols SC; memset(&SC, 0, sizeof SC); SC.n = counts[k0].len ? counts[k0].len : S.n + 1;
    size_t k = k0;
    for (; k < n_scan && k < k0 + MAX_SCAN_COLS && (counts[k].len ? counts[k].len : S.n + 1) == SC.n; k++) SC.col[SC.n_cols++] = counts[k].counts;
    if ((rc = launch_offsets_scan(s, cs, SC, s->d_tiles, s->d_totals.as<uint64_t>() + k0))) return rc;
    k0 = k;
  }
  publish_kernel<<<1, 256, 0, cs>>>(s->d_totals.as<uint32_t>(), s->d_hflags + 16, (int)(2 * n_scan));
  CU_TRY(cudaEventRecord(s->ev_dflags, cs));
  CU_TRY(cudaEventSynchronize(s->ev_dflags));
  CU_TRY(cudaGetLastError());
  *T = reinterpret_cast<const uint64_t*>(s->h_flags + 16);
  for (size_t k = 0; k < n_scan; k++)
    if ((*T)[k] > 0x7fffffffull) { set_error("column '%s' exceeds 2^31-1 bytes in one batch; lower chunk_inflated_bytes", s->f->fields[S.cols[counts[k].col].schema_idx].name.c_str()); return BAMSCAN_ERR_UNSUPPORTED; }
  return BAMSCAN_OK;
}

// Region B per count column: the total's bytes (Utf8, Binary) or, for a list, the child validity words when list_child_validity
// (VCF; BAM tag lists have none), then the child values, or for List<Utf8> the child offsets and the bytes the next count column
// totals.
static void layout_counts(Slice& S, const std::vector<CountCol>& counts, const uint64_t* T, bool list_child_validity) {
  for (size_t k = 0; k < counts.size(); k++) {
    ColLayout& L = S.cols[counts[k].col];
    uint64_t bytes = T[k];
    if (L.kind >= HK_ListInt8) {
      L.child_len = T[k];
      if (list_child_validity) { L.child_validity = true; L.child_validity_off = S.AB.take(4 * ((T[k] + 31) / 32)); }
      if (L.kind == HK_ListUtf8) { L.child_offsets_off = S.AB.take(4 * (T[k] + 1)); bytes = T[++k]; }
      else bytes *= (L.kind == HK_ListInt8 || L.kind == HK_ListUInt8) ? 1 : (L.kind == HK_ListInt16 || L.kind == HK_ListUInt16) ? 2 : 4;
    }
    L.data_bytes = bytes;
    L.data_off = S.AB.take((size_t)bytes + 16);
  }
}

// The arena grows when region B does not fit, keeping region A; the format binds its kernels again afterwards.
static int fit_region_b(BamScanStream* s, Slice& S) {
  DeviceBuf& arena = s->d_arena[s->arena_flip];
  if (S.AB.pos > arena.cap) {
    DeviceBuf bigger;
    if (int rc = bigger.ensure(S.AB.pos)) return rc;
    CU_TRY(cudaMemcpyAsync(bigger.p, arena.p, S.region_a, cudaMemcpyDeviceToDevice, s->cur.cs));
    CU_TRY(cudaStreamSynchronize(s->cur.cs));
    arena.release(); arena = bigger;
    S.A = arena.as<uint8_t>();
  }
  return BAMSCAN_OK;
}

// Count columns -> Arrow offsets, then region B laid out behind region A
static int layout_region_b(BamScanStream* s, Slice& S, const std::vector<CountCol>& counts, bool list_child_validity) {
  const uint64_t* T = nullptr;
  if (int rc = scan_counts(s, S, counts, &T)) return rc;
  layout_counts(S, counts, T, list_child_validity);
  return fit_region_b(s, S);
}

// FASTQ: fq_lengths -> scan -> fq_copy.  name, description, sequence and quality_scores (schema 0-3) are Utf8; description is the
// nullable one.
static int decode_fastq(BamScanStream* s, Slice& S) {
  cudaStream_t cs = s->cur.cs;
  const uint32_t n = std::min<uint32_t>(s->cur.rows_per_slice, s->cur.n - s->cur.pos);
  int rc;
  if ((rc = layout_region_a(s, S, n, [](const BamFile&, int32_t c) { return c == 1; }))) return rc;
  FastqCols FC{s->cur.U, s->cur.recoff + 4ull * s->cur.pos, n};        // (the column pointers: bind)
  s->cur.pos += n;
  auto bind = [&](uint8_t* A) {
    FC.err = reinterpret_cast<uint32_t*>(A + S.err_off);
    for (const ColLayout& L : S.cols) {
      const ColPtrs c = col_ptrs(A, L);
      switch (L.schema_idx) {
        case 0: FC.l_name = c.offs; FC.d_name = c.data; break;
        case 1: FC.l_desc = c.offs; FC.v_desc = c.valid; FC.d_desc = c.data; break;
        case 2: FC.l_seq = c.offs; FC.d_seq = c.data; break;
        case 3: FC.l_qual = c.offs; FC.d_qual = c.data; break;
      }
    }
  };
  bind(S.A);
  fq_lengths_kernel<<<(n + 255) / 256, 256, 0, cs>>>(FC);
  s->st.kernel_launches++;
  const std::vector<CountCol> counts = offset_counts(S);
  if (counts.empty() || (rc = layout_region_b(s, S, counts, false))) return rc;
  bind(S.A);
  fq_copy_kernel<8><<<(uint32_t)(((uint64_t)n * 8 + 255) / 256), 256, 0, cs>>>(FC);
  s->st.kernel_launches++;
  return BAMSCAN_OK;
}

// FASTA: fa_lengths -> scan -> fa_copy (name, description) and fa_seq (the sequence lines joined).  The slices are the ones
// frame_fasta cut: whole records, about SLICE_BYTES of text each.
static int decode_fasta(BamScanStream* s, Slice& S) {
  cudaStream_t cs = s->cur.cs;
  const uint32_t k = s->cur.fa_slice++;
  const uint32_t n = s->cur.fa_slice_rec[k + 1] - s->cur.pos, b0 = s->cur.fa_slice_byte[k], b1 = s->cur.fa_slice_byte[k + 1];
  int rc;
  if ((rc = layout_region_a(s, S, n, [](const BamFile&, int32_t c) { return c == 1; }))) return rc;
  const uint32_t* rec = s->cur.recoff + s->cur.pos;
  s->cur.pos += n;
  FastaCols AC{s->cur.U, s->cur.fa_lines, rec, s->cur.fa_seqpos, n};
  FastaSeq SQ{s->cur.U, s->cur.fa_lines, s->cur.fa_seqpos, s->cur.fa_tile_base, rec, n, s->cur.fa_lo, s->cur.fa_hi, (b0 - s->cur.fa_lo) / FQ_TILE, nullptr, nullptr};
  auto bind = [&](uint8_t* A) {
    AC.err = SQ.err = reinterpret_cast<uint32_t*>(A + S.err_off);
    for (const ColLayout& L : S.cols) {
      const ColPtrs c = col_ptrs(A, L);
      switch (L.schema_idx) {
        case 0: AC.l_name = c.offs; AC.d_name = c.data; break;
        case 1: AC.l_desc = c.offs; AC.v_desc = c.valid; AC.d_desc = c.data; break;
        case 2: AC.l_seq = c.offs; SQ.dst = c.data; break;
      }
    }
  };
  bind(S.A);
  fa_lengths_kernel<<<(n + 255) / 256, 256, 0, cs>>>(AC);
  s->st.kernel_launches++;
  const std::vector<CountCol> counts = offset_counts(S);
  if (counts.empty() || (rc = layout_region_b(s, S, counts, false))) return rc;
  bind(S.A);
  if (AC.d_name || AC.d_desc) { fa_copy_kernel<8><<<(uint32_t)(((uint64_t)n * 8 + 255) / 256), 256, 0, cs>>>(AC); s->st.kernel_launches++; }
  if (SQ.dst && b1 > b0) { fa_seq_kernel<<<(b1 - s->cur.fa_lo + FQ_TILE - 1) / FQ_TILE - SQ.t0, 256, 0, cs>>>(SQ); s->st.kernel_launches++; }
  return BAMSCAN_OK;
}

// BAM and SAM (lines that transcode_sam turned into BAM records): decode_fixed -> scan -> decode_var.  Short records take 8 lanes
// each, long records (and debug_flags bit 1) a warp.
static int decode_bam(BamScanStream* s, Slice& S) {
  const BamFile* f = s->f;
  cudaStream_t cs = s->cur.cs;
  const uint32_t n = std::min<uint32_t>(s->cur.rows_per_slice, s->cur.n - s->cur.pos);
  int rc;
  if ((rc = layout_region_a(s, S, n, [](const BamFile&, int32_t c) { return c >= 12 || c == 1 || c == 2 || c == 3 || c == 7 || c == 8; }))) return rc;
  // scratch: per variable-length tag column, each row's aux field offset in U
  std::vector<size_t> src_off(S.cols.size(), 0);
  size_t scratch = 0;
  for (size_t i = 0; i < S.cols.size(); i++) if (S.cols[i].schema_idx >= 12 && is_var(S.cols[i].kind)) { src_off[i] = scratch; scratch += align_up(4ull * n, 256); }
  if ((rc = s->d_scratch.ensure(scratch + 256))) return rc;
  DecodeParams DP{};
  DP.U = s->cur.U; DP.rec_off = s->cur.recoff + s->cur.pos; DP.n = n; DP.zero_based = f->zero_based; DP.binary_cigar = f->binary_cigar;
  const size_t n_ref = f->ref_names.size(); DP.n_ref = (int32_t)n_ref;
  DP.end_zero_span = f->format == FMT_SAM; DP.qual_absent = s->cur.qabs ? s->cur.qabs + s->cur.pos : nullptr;
  DP.ref_name_off = reinterpret_cast<const uint32_t*>(s->d_refs.as<uint8_t>() + align_up(4 * n_ref + 4, 16));
  DP.ref_names = s->d_refs.as<uint8_t>() + align_up(4 * n_ref + 4, 16) + align_up(4 * (n_ref + 1), 16);
  s->cur.pos += n;
  auto bind = [&](uint8_t* A) {
    DP.err = reinterpret_cast<uint32_t*>(A + S.err_off);
    DP.n_tags = 0;
    for (size_t i = 0; i < S.cols.size(); i++) {
      const ColLayout& L = S.cols[i];
      const ColPtrs c = col_ptrs(A, L);
      switch (L.schema_idx) {
        case 0: DP.l_name = c.offs; DP.d_name = c.data; break;
        case 1: DP.l_chrom = c.offs; DP.v_chrom = c.valid; DP.d_chrom = c.data; break;
        case 2: DP.start = c.vals; DP.v_start = c.valid; break;
        case 3: DP.end = c.vals; DP.v_end = c.valid; break;
        case 4: DP.flags = c.vals; break;
        case 5: DP.l_cigar = c.offs; DP.d_cigar = c.data; break;
        case 6: DP.mapq = c.vals; break;
        case 7: DP.l_mchrom = c.offs; DP.v_mchrom = c.valid; DP.d_mchrom = c.data; break;
        case 8: DP.mate_start = c.vals; DP.v_mstart = c.valid; break;
        case 9: DP.l_seq = c.offs; DP.d_seq = c.data; break;
        case 10: DP.l_qual = c.offs; DP.d_qual = c.data; break;
        case 11: DP.tlen = reinterpret_cast<int32_t*>(c.vals); break;
        default: {
          TagPlan& T = DP.tags[DP.n_tags++];
          const std::string& tg = f->fields[L.schema_idx].name;
          T.tag = tg.size() == 2 ? (uint16_t)((uint8_t)tg[0] | ((uint16_t)(uint8_t)tg[1] << 8)) : 0xffffu;   // names that are not 2 bytes never match (sam_tag_io.rs:58-68)
          T.kind = L.kind; T.valid = c.valid;
          if (is_var(L.kind)) { T.lens = c.offs; T.src = reinterpret_cast<uint32_t*>(s->d_scratch.as<uint8_t>() + src_off[i]); T.data = c.data; }
          else T.values = c.vals;
        }
      }
    }
  };
  bind(S.A);
  if (s->cur.long_records) {
    CU_TRY(cudaMemsetAsync(S.A, 0, S.region_a, cs));                                     // validity words are OR-ed in
    decode_fixed_warp_kernel<<<(uint32_t)(((uint64_t)n * 32 + 255) / 256), 256, 0, cs>>>(DP);     // a warp per row, lanes co-operate inside the record
  }
  else
    decode_fixed_kernel<<<(n + 255) / 256, 256, 0, cs>>>(DP);
  s->st.kernel_launches++;
  const std::vector<CountCol> counts = offset_counts(S);
  if (counts.empty() || (rc = layout_region_b(s, S, counts, false))) return rc;
  bind(S.A);
  if (s->cur.long_records)
    decode_var_kernel<32><<<std::min<uint32_t>((n + VAR_WARPS - 1) / VAR_WARPS, 148u * 8u * 4u), VAR_WARPS * 32, 0, cs>>>(DP);
  else
    decode_var_kernel<8><<<std::min<uint32_t>((n + VAR_WARPS * 4 - 1) / (VAR_WARPS * 4), 148u * 8u * 4u), VAR_WARPS * 32, 0, cs>>>(DP);
  s->st.kernel_launches++;
  return BAMSCAN_OK;
}

// VCF: vcf_fields -> vcf_rows -> scan -> vcf_write (kernels_vcf.cuh).  The count columns are the Utf8 bytes and list elements, and
// for List<Utf8> also the elements' bytes.  Projected FORMAT columns add vcf_samples and vcf_values in front of the scan and
// vcf_fmt_write behind it (kernels_vcf_format.cuh); their count columns are element-level (n * S + 1 entries) and share the
// scan's host sync.
static int decode_vcf(BamScanStream* s, Slice& S) {
  const BamFile* f = s->f;
  cudaStream_t cs = s->cur.cs;
  const uint32_t n = std::min<uint32_t>(s->cur.rows_per_slice, s->cur.n - s->cur.pos);
  const uint32_t* lines = s->cur.recoff + s->cur.pos;
  s->cur.pos += n;
  int rc;
  const int32_t info_end = f->vcf_info_end;
  const uint32_t n_smp = (uint32_t)f->vcf_samples.size();
  const uint64_t nel = (uint64_t)n * n_smp;          // FORMAT elements (< 2^31: run_chunk cuts the slices so)
  // FORMAT columns: besides their outer offsets, region A holds the element validity and the Int32 / Float32 values or the
  // element counts (-> offsets) of Utf8 and nested columns, all sized by n * S
  auto fmt_elems = [&](ColLayout& L) {
    if (L.schema_idx < info_end) return;
    L.child_validity = true; L.child_len = nel;
    L.child_validity_off = S.AB.take(4 * ((nel + 31) / 32));
    L.elem_bytes = (nel + 7) / 8;
    if (L.kind == HK_ListInt32 || L.kind == HK_ListFloat32) { L.data_bytes = 4 * nel; L.data_off = S.AB.take(4 * nel + 16); }
    else { L.child_offsets_off = S.AB.take(4 * (nel + 1)); L.elem_bytes += 4 * (nel + 1); }
  };
  if ((rc = layout_region_a(s, S, n, [](const BamFile& file, int32_t c) { return file.fields[c].nullable; }, fmt_elems))) return rc;
  const size_t n_dec = S.cols.size();
  // keys: the projected INFO IDs (key k is INFO column k), then END unless it is one of them
  std::vector<int> info_col(n_dec, -1);           // column -> INFO column (key) index
  std::vector<std::string> keys;
  for (size_t i = 0; i < n_dec; i++) if (S.cols[i].schema_idx >= 8 && S.cols[i].schema_idx < info_end) { info_col[i] = (int)keys.size(); keys.push_back(f->fields[S.cols[i].schema_idx].name); }
  const int n_info = (int)keys.size();
  int end_key = (int)(std::find(keys.begin(), keys.end(), std::string("END")) - keys.begin());
  if (end_key == (int)keys.size()) keys.push_back("END");
  // Keys::off and Params::cols hold MAX_INFO + 1 keys (stream_init refuses more projected INFO columns)
  if (keys.size() > (size_t)vcf::MAX_INFO + 1) { set_error("more than %d projected INFO columns are not supported by this build", vcf::MAX_INFO); return BAMSCAN_ERR_UNSUPPORTED; }
  std::unique_ptr<vcf::Params> P(new vcf::Params());
  memset(P.get(), 0, sizeof(vcf::Params));
  vcf::Keys& K = P->keys;
  uint32_t blob = 0;
  for (size_t k = 0; k < keys.size(); k++) {
    if (blob + keys[k].size() > (size_t)vcf::KEY_BLOB) { set_error("the projected INFO IDs exceed %d bytes, which is not supported by this build", vcf::KEY_BLOB); return BAMSCAN_ERR_UNSUPPORTED; }
    K.off[k] = (uint16_t)blob;
    memcpy(K.blob + blob, keys[k].data(), keys[k].size()); blob += (uint32_t)keys[k].size();
    uint32_t h = vcf::key_hash(reinterpret_cast<const uint8_t*>(keys[k].data()), (uint32_t)keys[k].size());
    while (K.slot[h & (vcf::KEY_SLOTS - 1)]) h++;
    K.slot[h & (vcf::KEY_SLOTS - 1)] = (uint16_t)(k + 1);
  }
  K.off[keys.size()] = (uint16_t)blob; K.n_keys = (int32_t)keys.size(); K.end_key = end_key;
  // scratch: per row the field starts, per key the value tokens, per List<Utf8> column its byte counts
  const size_t o_tok = align_up(sizeof(vcf::Row) * n, 256), o_blen = o_tok + align_up(8ull * n * keys.size(), 256);
  size_t scratch = o_blen;
  std::vector<size_t> blen_off(n_dec, 0);
  for (size_t i = 0; i < n_dec; i++) if (S.cols[i].kind == HK_ListUtf8) { blen_off[i] = scratch; scratch += align_up(4ull * (n + 1), 256); }
  // FORMAT scratch: the sample starts and the per-line key map
  const size_t o_samp = align_up(scratch, 256), o_frow = o_samp + align_up(4 * nel, 256);
  std::vector<size_t> fmt_cols;                   // FORMAT column c -> index into S.cols
  for (size_t i = 0; i < n_dec; i++) if (S.cols[i].schema_idx >= info_end) fmt_cols.push_back(i);
  if (!fmt_cols.empty()) scratch = o_frow + sizeof(vcf::FmtRow) * n;
  if ((rc = s->d_scratch.ensure(scratch + 256))) return rc;
  uint8_t* SCR = s->d_scratch.as<uint8_t>();
  std::unique_ptr<vcf::FormatParams> FP;
  if (!fmt_cols.empty()) {
    FP.reset(new vcf::FormatParams());
    memset(FP.get(), 0, sizeof(vcf::FormatParams));
    uint32_t blob = 0;
    for (size_t c = 0; c < fmt_cols.size(); c++) {
      const std::string id = f->fields[S.cols[fmt_cols[c]].schema_idx].name.substr(7);     // behind "format_"
      if (blob + id.size() > (size_t)vcf::FMT_BLOB) { set_error("the projected FORMAT IDs exceed %d bytes, which is not supported by this build", vcf::FMT_BLOB); return BAMSCAN_ERR_UNSUPPORTED; }
      FP->off[c] = (uint16_t)blob;
      memcpy(FP->blob + blob, id.data(), id.size()); blob += (uint32_t)id.size();
    }
    FP->off[fmt_cols.size()] = (uint16_t)blob;
  }
  auto bind = [&](uint8_t* A) {
    if (FP) {
      vcf::FormatParams& F = *FP;
      F.U = s->cur.U; F.lines = lines; F.rows = reinterpret_cast<const vcf::Row*>(SCR); F.n = n; F.S = n_smp; F.nf = (int32_t)fmt_cols.size();
      F.samp = reinterpret_cast<uint32_t*>(SCR + o_samp); F.frow = reinterpret_cast<vcf::FmtRow*>(SCR + o_frow);
      F.err = reinterpret_cast<uint32_t*>(A + S.err_off);
      for (size_t c = 0; c < fmt_cols.size(); c++) {
        const ColLayout& L = S.cols[fmt_cols[c]];
        vcf::FmtCol& C = F.cols[c];
        C.kind = L.kind; C.offs = reinterpret_cast<int32_t*>(A + L.offsets_off); C.valid = reinterpret_cast<uint32_t*>(A + L.child_validity_off);
        if (L.kind == HK_ListInt32 || L.kind == HK_ListFloat32) C.values = reinterpret_cast<uint32_t*>(A + L.data_off);
        else { C.counts = reinterpret_cast<int32_t*>(A + L.child_offsets_off); C.data = L.data_off ? A + L.data_off : nullptr; }
        if (L.leaf_validity_off) C.lvalid = reinterpret_cast<uint32_t*>(A + L.leaf_validity_off);
      }
    }
    P->U = s->cur.U; P->lines = lines; P->n = n; P->zero_based = f->zero_based; P->n_info = n_info;
    P->rows = reinterpret_cast<vcf::Row*>(SCR); P->err = reinterpret_cast<uint32_t*>(A + S.err_off);
    for (size_t k = 0; k < keys.size(); k++) P->cols[k].tok = reinterpret_cast<uint2*>(SCR + o_tok) + (size_t)k * n;
    for (size_t i = 0; i < n_dec; i++) {
      const ColLayout& L = S.cols[i];
      const ColPtrs c = col_ptrs(A, L);
      uint8_t* d = L.data_bytes ? c.data : nullptr;     // a fixed column without bytes in the slice (an all-'.' ID) is skipped by vcf_write_kernel
      switch (L.schema_idx) {
        case 0: P->l_chrom = c.offs; P->d_chrom = d; break;
        case 1: P->start = c.vals; break;
        case 2: P->end = c.vals; break;
        case 3: P->l_id = c.offs; P->v_id = c.valid; P->d_id = d; break;
        case 4: P->l_ref = c.offs; P->d_ref = d; break;
        case 5: P->l_alt = c.offs; P->v_alt = c.valid; P->d_alt = d; break;
        case 6: P->qual = c.vals; P->v_qual = c.valid; break;
        case 7: P->l_filter = c.offs; P->v_filter = c.valid; P->d_filter = d; break;
        default: {
          if (L.schema_idx >= info_end) break;      // (FORMAT: FP)
          vcf::InfoCol& C = P->cols[info_col[i]];
          C.kind = L.kind; C.valid = c.valid; C.data = c.data;
          if (is_var(L.kind)) C.lens = c.offs; else C.values = c.vals;
          if (L.kind == HK_ListUtf8) { C.blens = reinterpret_cast<int32_t*>(SCR + blen_off[i]); C.coffs = reinterpret_cast<int32_t*>(A + L.child_offsets_off); }
          if (L.child_validity) C.cvalid = reinterpret_cast<uint32_t*>(A + L.child_validity_off);
        }
      }
    }
  };
  bind(S.A);
  CU_TRY(cudaMemsetAsync(SCR + o_tok, 0, 8ull * n * keys.size(), cs));
  // 8 lanes per line; 32 for long lines (sam_records_kernel's rule)
  if (s->cur.long_records) vcf::vcf_fields_kernel<32><<<(uint32_t)(((uint64_t)n * 32 + 255) / 256), 256, 0, cs>>>(*P);
  else vcf::vcf_fields_kernel<8><<<(uint32_t)(((uint64_t)n * 8 + 255) / 256), 256, 0, cs>>>(*P);
  vcf::vcf_rows_kernel<<<(n + 255) / 256, 256, 0, cs>>>(*P);
  s->st.kernel_launches += 2;
  if (FP) {
    if (s->cur.long_records) vcf::vcf_samples_kernel<32><<<(uint32_t)(((uint64_t)n * 32 + 255) / 256), 256, 0, cs>>>(*FP);
    else vcf::vcf_samples_kernel<8><<<(uint32_t)(((uint64_t)n * 8 + 255) / 256), 256, 0, cs>>>(*FP);
    vcf::vcf_values_kernel<<<(uint32_t)((nel + 255) / 256), 256, 0, cs>>>(*FP);
    s->st.kernel_launches += 2;
  }
  std::vector<CountCol> counts;
  for (size_t i = 0; i < n_dec; i++) {
    if (!is_var(S.cols[i].kind) || S.cols[i].schema_idx >= info_end) continue;
    counts.push_back({reinterpret_cast<int32_t*>(S.A + S.cols[i].offsets_off), i});
    if (S.cols[i].kind == HK_ListUtf8) counts.push_back({reinterpret_cast<int32_t*>(SCR + blen_off[i]), i});
  }
  const size_t n_info_counts = counts.size();
  for (size_t i : fmt_cols)
    if (S.cols[i].kind != HK_ListInt32 && S.cols[i].kind != HK_ListFloat32) counts.push_back({reinterpret_cast<int32_t*>(S.A + S.cols[i].child_offsets_off), i, (uint32_t)nel + 1u});
  if (!counts.empty()) {
    s->st.kernel_launches++;     // the totals publish: VCF has always counted it, the other formats never have, so both stay comparable
    const uint64_t* T = nullptr;
    if ((rc = scan_counts(s, S, counts, &T))) return rc;
    layout_counts(S, std::vector<CountCol>(counts.begin(), counts.begin() + n_info_counts), T, true);
    for (size_t k = n_info_counts; k < counts.size(); k++) {
      // FORMAT: Utf8 bytes, or the leaves of a nested column (validity, values)
      ColLayout& L = S.cols[counts[k].col];
      if (L.kind == HK_ListUtf8) L.data_bytes = T[k];
      else { L.leaf_len = T[k]; L.leaf_validity_off = S.AB.take(4 * ((T[k] + 31) / 32)); L.elem_bytes += (T[k] + 7) / 8; L.data_bytes = 4 * T[k]; }
      L.data_off = S.AB.take((size_t)L.data_bytes + 16);
    }
    if ((rc = fit_region_b(s, S))) return rc;
  }
  bind(S.A);
  for (const ColLayout& L : S.cols) {
    if (L.child_validity && L.schema_idx < info_end) CU_TRY(cudaMemsetAsync(S.A + L.child_validity_off, 0, 4 * ((L.child_len + 31) / 32), cs));
    if (L.leaf_validity_off) CU_TRY(cudaMemsetAsync(S.A + L.leaf_validity_off, 0, 4 * ((L.leaf_len + 31) / 32), cs));
  }
  if (s->cur.long_records) vcf::vcf_write_kernel<32><<<(uint32_t)(((uint64_t)n * 32 + 255) / 256), 256, 0, cs>>>(*P);
  else vcf::vcf_write_kernel<8><<<(uint32_t)(((uint64_t)n * 8 + 255) / 256), 256, 0, cs>>>(*P);
  s->st.kernel_launches++;
  if (FP) { vcf::vcf_fmt_write_kernel<<<(uint32_t)((nel + 255) / 256), 256, 0, cs>>>(*FP); s->st.kernel_launches++; }
  return BAMSCAN_OK;
}

// Decodes the next slice of the current chunk's rows into the arena and queues its hand-off (one batch).  A decode slice is queued
// without waiting for it; its time (and, for device-resident runs, its error word) is collected when the next slice starts or the
// partition ends (flush_slice).
static int decode_slice(BamScanStream* s, bool* produced) {
  NvtxRange nv("bamscan: decode slice (count, scan, write) + D2H issue");
  cudaStream_t cs = s->cur.cs;
  int rc;
  if ((rc = flush_slice(s))) return rc;
  CU_TRY(cudaEventRecord(s->ev_dt[0], cs));
  Slice S;
  switch (s->f->format) {
    case FMT_BAM: case FMT_SAM: rc = decode_bam(s, S); break;
    case FMT_FASTQ: rc = decode_fastq(s, S); break;
    case FMT_FASTA: rc = decode_fasta(s, S); break;
    case FMT_VCF: rc = decode_vcf(s, S); break;
  }
  if (rc) return rc;
  const uint32_t n = S.n;
  const uint64_t row0 = s->st.rows;
  s->st.rows += n; s->st.batches++;
  for (const ColLayout& L : S.cols) s->st.arrow_bytes += (L.has_validity ? (n + 7) / 8 : 0) + (is_var(L.kind) ? 4ull * (n + 1) + L.data_bytes : fixed_bytes(L.kind, n)) + L.elem_bytes;
  if ((rc = hand_off_batch(s, cs, S.A, S.cols, n, S.AB.pos, S.err_off, row0, produced))) return rc;
  CU_TRY(cudaEventRecord(s->ev_dt[1], cs));
  s->slice_pending = true;
  return BAMSCAN_OK;
}

static int sam_error_to_rc(uint32_t code, unsigned long long rec) {
  static const char* what[] = {"?", "fewer than 11 fields", "invalid QNAME (1-254 of [!-?A-~])", "invalid FLAG (not an integer in 0..65535)",
                               "RNAME is not a reference sequence of the header", "invalid POS (not an integer in 0..2^31)",
                               "invalid MAPQ (not an integer in 0..255)", "invalid CIGAR", "CIGAR with more than 65535 operations is not supported",
                               "RNEXT is not a reference sequence of the header", "invalid PNEXT (not an integer in 0..2^31)",
                               "invalid TLEN (not an i32)", "invalid SEQ (not * or [A-Za-z=.]+)", "invalid QUAL (not * or [!-~]+)",
                               "QUAL length differs from SEQ length", "malformed aux field", "duplicate aux tag", "aux value out of range for its type"};
  set_error("SAM read error: record %llu of the partition (0-based): %s", rec, code < sizeof what / sizeof *what ? what[code] : "?");
  return code == sam::SAM_ERR_CIGAR_OPS ? BAMSCAN_ERR_UNSUPPORTED : BAMSCAN_ERR_FORMAT;
}

// SAM: the chunk's n complete owned lines -> BAM records in the slot's own buffer (kernels_sam.cuh).  One host sync: the first
// error and the total record bytes (the buffer's size).  *bam / *recoff: the records and their offsets, for the decode stage.
static int transcode_sam(BamScanStream* s, int slot, cudaStream_t cs, const uint8_t* U, const uint32_t* lines, uint32_t n,
                         const uint8_t** bam, const uint32_t** recoff) {
  NvtxRange nv("bamscan: SAM lines -> BAM records");
  const BamFile* f = s->f;
  int rc;
  if ((rc = s->d_samline[slot].ensure(sizeof(sam::SamLine) * (size_t)n)) || (rc = s->d_samsize[slot].ensure(4ull * (n + 1) + 64)) ||
      (rc = s->d_qabs[slot].ensure((size_t)n + 64))) return rc;
  uint32_t* d_flags = s->d_flags[slot].as<uint32_t>();
  uint32_t* d_err = d_flags + 24;                  // [24] first error, [25] its line, [26..27] total record bytes (u64): device only
  CU_TRY(cudaMemsetAsync(d_err, 0, 16, cs));
  const size_t n_ref = f->ref_names.size();
  const uint8_t* R = s->d_samrefs.as<uint8_t>();
  const size_t o_ids = align_up(4 * (n_ref + 1), 16), o_names = o_ids + align_up(4 * n_ref + 4, 16);
  sam::SamSizeArgs A;
  A.U = U; A.lines = lines; A.n = n;
  A.R = sam::SamRefs{R + o_names, reinterpret_cast<const int32_t*>(R), reinterpret_cast<const int32_t*>(R + o_ids), (int32_t)n_ref};
  A.out = s->d_samline[slot].as<sam::SamLine>(); A.sizes = s->d_samsize[slot].as<uint32_t>(); A.qual_absent = s->d_qabs[slot].as<uint8_t>(); A.err = d_err;
  sam::sam_size_kernel<<<(n + 255) / 256, 256, 0, cs>>>(A);
  ScanCols SC; memset(&SC, 0, sizeof SC);
  SC.col[0] = reinterpret_cast<int32_t*>(A.sizes); SC.n_cols = 1; SC.n = n + 1;
  if ((rc = launch_offsets_scan(s, cs, SC, s->d_samtiles[slot], reinterpret_cast<uint64_t*>(d_flags + 26)))) return rc;
  publish_kernel<<<1, 32, 0, cs>>>(d_err, s->d_hflags + 600, 4);     // [600, 604) of the mapped page: nothing else uses it
  s->st.kernel_launches += 2;
  CU_TRY(cudaEventRecord(s->ev_flags[slot], cs));
  CU_TRY(cudaEventSynchronize(s->ev_flags[slot]));
  CU_TRY(cudaGetLastError());
  const uint32_t* hf = s->h_flags + 600;
  if (hf[0]) return sam_error_to_rc(hf[0], (unsigned long long)s->st.rows + hf[1]);
  const uint64_t total = (uint64_t)hf[2] | ((uint64_t)hf[3] << 32);
  if (total > 0xffffffffull) { set_error("SAM chunk transcodes to more than 4 GiB of BAM records; lower chunk_inflated_bytes"); return BAMSCAN_ERR_UNSUPPORTED; }
  if ((rc = s->d_bam[slot].ensure((size_t)total + 64))) return rc;
  sam::SamWriteArgs W{U, A.out, A.sizes, n, s->d_bam[slot].as<uint8_t>()};
  // a group of 8 lanes per line (4 lines per warp); 32 when the previous chunk's lines averaged above 2 KiB, as in decode and encode
  if ((f->debug_flags & 2) || s->mean_record_bytes > 2048) sam::sam_records_kernel<32><<<(uint32_t)(((uint64_t)n * 32 + 255) / 256), 256, 0, cs>>>(W);
  else sam::sam_records_kernel<8><<<(uint32_t)(((uint64_t)n * 8 + 255) / 256), 256, 0, cs>>>(W);
  s->st.kernel_launches++;
  CU_TRY(cudaEventRecord(s->ev_text_free[slot], cs));
  *bam = s->d_bam[slot].as<uint8_t>(); *recoff = A.sizes;
  return BAMSCAN_OK;
}

// ---- chunk framing: one function per format queues the kernels that find the chunk's records behind its inflate, publishes the
// flag words (kernels_boundary.cuh's convention in [0, 16)) to the mapped page and records ev_flags[slot].

struct LineScan { uint32_t n_tiles, line_cap; uint32_t* tile_base; };

// The newline scan of FASTQ, SAM and FASTA (kernels_fastq.cuh): the line starts of U[lo, hi) -> d_recoff[slot], which holds
// (hi - lo) / line_divisor + 4096 of them (beyond that the framing kernel fails loudly); the line count -> d_flags[16].  d_seg[slot]
// holds tile_words words per tile: the newline counts, their scan (L->tile_base), then whatever the caller keeps there.
static int launch_line_scan(BamScanStream* s, int slot, cudaStream_t cs, const uint8_t* U, uint32_t lo, uint32_t hi, uint32_t tile_words,
                            uint32_t line_divisor, LineScan* L) {
  const uint32_t span = hi - lo;
  L->n_tiles = std::max<uint32_t>(1, (span + FQ_TILE - 1) / FQ_TILE);
  L->line_cap = span / line_divisor + 4096;
  int rc;
  if ((rc = s->d_seg[slot].ensure(4ull * tile_words * L->n_tiles + 64)) || (rc = s->d_recoff[slot].ensure(4ull * L->line_cap))) return rc;
  uint32_t* d_tile_count = s->d_seg[slot].as<uint32_t>();
  L->tile_base = d_tile_count + L->n_tiles;
  fq_count_kernel<<<L->n_tiles, 256, 0, cs>>>(U, lo, hi, d_tile_count);
  cta_scan_kernel<<<1, CTA_SCAN_THREADS, 0, cs>>>(d_tile_count, L->tile_base, L->n_tiles, s->d_flags[slot].as<uint32_t>() + 16);
  fq_lines_kernel<<<L->n_tiles, 256, 0, cs>>>(U, lo, hi, L->tile_base, s->d_recoff[slot].as<uint32_t>(), L->line_cap);
  s->st.kernel_launches += 3;
  return BAMSCAN_OK;
}

// BAM: record chains walked from candidate starts per segment, the seams between segments checked and repaired (kernels_boundary.cuh)
static int frame_bam(BamScanStream* s, int slot, const BoundaryParams& BP, const WalkOut& W, uint32_t* d_seg_base) {
  const BamFile* f = s->f;
  cudaStream_t cs = s->s_chunk[slot];
  const uint32_t n_seg = BP.n_seg;
  seg_candidates_kernel<<<(n_seg * 32 + 255) / 256, 256, 0, cs>>>(BP, W.seg_start, (f->debug_flags & 1) ? 1 : 0);
  seg_walk_kernel<<<(n_seg + 127) / 128, 128, 0, cs>>>(BP, W);
  seg_check_kernel<<<(n_seg + 127) / 128, 128, 0, cs>>>(BP, W);
  if (!(f->debug_flags & 64)) {
    // parallel repair rounds (no-ops when every seam agreed); debug_flags bit 6 leaves everything to the sequential repair
    for (int round = 0; round < 3; round++) {
      seg_fix_kernel<<<(n_seg + 127) / 128, 128, 0, cs>>>(BP, W, round);
      seg_reset_kernel<<<1, 1, 0, cs>>>(W);
      seg_check_kernel<<<(n_seg + 127) / 128, 128, 0, cs>>>(BP, W);
    }
    s->st.kernel_launches += 9;
  }
  seg_repair_kernel<<<1, 1, 0, cs>>>(BP, W);
  seg_scan_kernel<<<1, 1024, 0, cs>>>(W.seg_count, W.seg_start, W.seg_exit, W.seg_tail, d_seg_base, n_seg, W.flags);
  s->st.kernel_launches += 5;
  publish_kernel<<<1, 32, 0, cs>>>(W.flags, s->d_hflags, 16);
  CU_TRY(cudaEventRecord(s->ev_flags[slot], cs));
  return BAMSCAN_OK;
}

// FASTQ: line starts of the chunk -> d_recoff (kernels_fastq.cuh); the flags come out as the seg_* kernels report them
static int frame_fastq(BamScanStream* s, const ChunkPlan& c, int slot, const BoundaryParams& BP) {
  cudaStream_t cs = s->s_chunk[slot];
  uint32_t* d_flags = s->d_flags[slot].as<uint32_t>();
  LineScan L;
  // lines[] capacity: FASTQ lines average far more than 8 bytes
  if (int rc = launch_line_scan(s, slot, cs, BP.U, BP.data_lo, BP.data_hi, 2, 8, &L)) return rc;
  FastqFrame FF{BP.U, BP.data_lo, BP.data_hi, BP.own_hi, (uint32_t)(s->need_spec ? 1 : 0), (uint32_t)(c.b1 == s->f->blocks.size() ? 1 : 0), L.line_cap};
  fq_frame_kernel<<<1, 32, 0, cs>>>(FF, d_flags + 16, s->d_recoff[slot].as<uint32_t>(), d_flags);
  s->st.kernel_launches++;
  publish_kernel<<<1, 32, 0, cs>>>(d_flags, s->d_hflags, 16);
  CU_TRY(cudaEventRecord(s->ev_flags[slot], cs));
  return BAMSCAN_OK;
}

// SAM: line starts of the chunk (the newline scan), one record per line (kernels_sam.cuh)
static int frame_sam(BamScanStream* s, const ChunkPlan& c, int slot, const BoundaryParams& BP) {
  cudaStream_t cs = s->s_chunk[slot];
  uint32_t* d_flags = s->d_flags[slot].as<uint32_t>();
  LineScan L;
  // a SAM record has 11 fields: lines average far more than 8 bytes
  if (int rc = launch_line_scan(s, slot, cs, BP.U, BP.data_lo, BP.data_hi, 2, 8, &L)) return rc;
  FastqFrame FF{BP.U, BP.data_lo, BP.data_hi, BP.own_hi, 0u, (uint32_t)(c.b1 == s->f->blocks.size() ? 1 : 0), L.line_cap};
  sam::sam_frame_kernel<<<1, 32, 0, cs>>>(FF, BP.first_start, d_flags + 16, s->d_recoff[slot].as<uint32_t>(), d_flags);
  s->st.kernel_launches++;
  publish_kernel<<<1, 32, 0, cs>>>(d_flags, s->d_hflags, 16);
  CU_TRY(cudaEventRecord(s->ev_flags[slot], cs));
  return BAMSCAN_OK;
}

// VCF: a record is a line, framed as a SAM line is.  A range owns the lines that start at or after its first owned byte
// (BP.first_start): the member in front of a block range is inflated too, so that a line start there is seen behind its '\n'.  '#'
// lines and empty lines are refused by vcf_rows_kernel, which knows the record number.
static int frame_vcf(BamScanStream* s, const ChunkPlan& c, int slot, const BoundaryParams& BP) {
  return frame_sam(s, c, slot, BP);
}

// FASTA: line starts (the newline scan) and the lines that start with '>' (kernels_fasta.cuh).  Its own flag words [16, 64) go to
// [FA_HFLAGS, FA_HFLAGS + 48) of the mapped page.
static int frame_fasta(BamScanStream* s, const ChunkPlan& c, const ScanRange& range, int slot, const BoundaryParams& BP, bool first_of_range) {
  cudaStream_t cs = s->s_chunk[slot];
  uint32_t* d_flags = s->d_flags[slot].as<uint32_t>();
  const uint32_t lo = BP.data_lo, data_hi = BP.data_hi, H = BP.seg0, carry = s->carry_len;
  int rc;
  CU_TRY(cudaMemsetAsync(d_flags + 16, 0, 4 * 48, cs));
  LineScan L;
  // lines[] capacity; d_seg also holds the '>' line counts and their scan
  if ((rc = launch_line_scan(s, slot, cs, BP.U, lo, data_hi, 4, 4, &L)) || (rc = s->d_fastarts[slot].ensure(4ull * L.line_cap))) return rc;
  uint32_t* d_st_count = L.tile_base + L.n_tiles; uint32_t* d_st_base = d_st_count + L.n_tiles;
  // ownership starts at the range's first byte (the member in front of it is inflated too, and owned by the range before) or at
  // the carried record; the chunk's first byte starts a line at the file start, for a carried record, or behind a '\n'
  const uint32_t own_lo = first_of_range && !carry ? H + (uint32_t)std::min<uint64_t>(range.first_uoff - c.u0, data_hi - H) : lo;
  const uint32_t lead_ok = carry || (first_of_range ? c.u0 == 0 : s->fa_lead_nl);
  FastaFrame FF{BP.U, lo, data_hi, own_lo, BP.own_hi, lead_ok, (uint32_t)(c.b1 == s->f->blocks.size() ? 1 : 0), L.line_cap, (uint32_t)SLICE_BYTES};
  fa_count_kernel<<<L.n_tiles, 256, 0, cs>>>(FF, d_st_count);
  cta_scan_kernel<<<1, CTA_SCAN_THREADS, 0, cs>>>(d_st_count, d_st_base, L.n_tiles, d_flags + FA_F_STARTS);
  fa_starts_kernel<<<L.n_tiles, 256, 0, cs>>>(FF, L.tile_base, d_st_base, s->d_fastarts[slot].as<uint32_t>());
  fa_frame_kernel<<<1, 32, 0, cs>>>(FF, s->d_recoff[slot].as<uint32_t>(), s->d_fastarts[slot].as<uint32_t>(), d_flags);
  s->st.kernel_launches += 4;
  if (s->fa_leading) { fa_leading_kernel<<<L.n_tiles, 256, 0, cs>>>(FF, s->d_recoff[slot].as<uint32_t>(), s->d_fastarts[slot].as<uint32_t>(), d_flags); s->st.kernel_launches++; }
  publish_kernel<<<1, 32, 0, cs>>>(d_flags, s->d_hflags, 16);
  publish_kernel<<<1, 64, 0, cs>>>(d_flags + 16, s->d_hflags + FA_HFLAGS, 48);
  s->st.kernel_launches += 2;
  CU_TRY(cudaEventRecord(s->ev_flags[slot], cs));
  return BAMSCAN_OK;
}

// The host's reading of a framed chunk's flags, per format: the framing error in hf[1], FASTA's own flag words, whether the next
// chunk still has to speculate where a record starts (need_spec), and the longest record the next chunk can take in (new_carry).
static int read_frame_flags(BamScanStream* s, const ChunkPlan& c, uint32_t H, uint32_t data_lo, uint32_t data_hi, uint32_t n_rec, uint32_t new_carry) {
  const uint32_t* hf = s->h_flags;
  const bool start_known = n_rec > 0 || hf[2] != 0xffffffffu;
  auto over_headroom = [](const char* what) { set_error("%s larger than %u bytes is not supported", what, HEADROOM); return BAMSCAN_ERR_UNSUPPORTED; };
  switch (s->f->format) {
    case FMT_BAM:
      if (hf[1]) { set_error("BAM read error: invalid record block_size at inflated offset %llu", (unsigned long long)(c.u0 + ((hf[1] & ~1u) - H))); return BAMSCAN_ERR_FORMAT; }
      if (start_known) s->need_spec = false;
      if (new_carry > HEADROOM) return over_headroom("BAM record");
      break;
    case FMT_FASTQ:
      if (hf[1]) { set_error("FASTQ read error: more lines in one chunk than supported (lines shorter than 8 bytes on average)"); return BAMSCAN_ERR_UNSUPPORTED; }
      if (n_rec > 0) s->need_spec = false;
      if (new_carry > HEADROOM) return over_headroom("BAM record");
      break;
    case FMT_SAM:
      if (hf[1]) { set_error("SAM read error: lines shorter than 8 bytes on average (a SAM record has 11 fields)"); return BAMSCAN_ERR_FORMAT; }
      if (start_known) s->need_spec = false;
      if (new_carry > HEADROOM) return over_headroom("SAM line");
      break;
    case FMT_VCF:
      if (hf[1]) { set_error("VCF read error: lines shorter than 8 bytes on average (a VCF record has 8 fields)"); return BAMSCAN_ERR_FORMAT; }
      if (start_known) s->need_spec = false;
      if (new_carry > HEADROOM) return over_headroom("VCF line");
      break;
    case FMT_FASTA: {
      if (hf[1]) { set_error("FASTA read error: more lines in one chunk than supported (lines shorter than 4 bytes on average)"); return BAMSCAN_ERR_UNSUPPORTED; }
      const uint32_t* fa_hf = s->h_flags + FA_HFLAGS - 16;     // FASTA words, indexed as in d_flags
      if (fa_hf[FA_F_LEADING]) { set_error("FASTA read error: record %llu of the partition (0-based): bytes other than whitespace in front of the first '>'", (unsigned long long)s->st.rows); return BAMSCAN_ERR_FORMAT; }
      if (fa_hf[FA_F_STARTS]) s->fa_leading = false;
      if (data_hi > data_lo) s->fa_lead_nl = fa_hf[FA_F_LAST_NL] != 0;
      if (start_known) s->need_spec = false;
      if (new_carry > FA_MAX_RECORD) { set_error("FASTA read error: record %llu of the partition (0-based) is larger than %llu bytes, which is not supported", (unsigned long long)(s->st.rows + n_rec), (unsigned long long)FA_MAX_RECORD); return BAMSCAN_ERR_UNSUPPORTED; }
      if (new_carry > s->headroom) s->headroom = (uint32_t)align_up(new_carry, 1u << 20);     // the next chunk's room (this chunk's U is unchanged)
      return s->d_carry.ensure(new_carry);
    }
  }
  return BAMSCAN_OK;
}

// Runs one chunk.  On success *produced tells whether a batch went into s->pending (previous pending must have been consumed).
// phase 1 queues H2D wait + inflate + record boundaries and returns without waiting (the host can then wait for an older
// batch's D2H while the GPU works); phase 2 picks the chunk up from there; phase 0 does both.
static int run_chunk(BamScanStream* s, const ChunkPlan& c, const ScanRange& range, int slot, bool first_of_range, bool* produced, uint32_t* new_carry, bool* owned_done, int phase) {
  BamFile* f = s->f;
  *produced = false;
  NvtxRange nv(phase == 1 ? "bamscan: queue inflate + record boundaries (ahead)" : phase == 2 ? "bamscan: chunk boundaries -> rows" : "bamscan: inflate + record boundaries");
  static const bool trace2 = getenv("BAMSCAN_TRACE") && atoi(getenv("BAMSCAN_TRACE")) >= 2;
  const double tw0 = wall_ms();
  // H: room in front of the chunk (HEADROOM except for FASTA, where it grows to the carried record); the slot's member descriptors
  // were built for desc_base, so the inflate output moves up by the difference
  const uint32_t H = s->headroom, shift = H - s->desc_base[slot];
  const uint32_t data_hi = s->chunk_data_hi[slot] + shift, seg0 = H;
  const uint32_t nb = s->n_descs[slot];
  int rc;
  if ((rc = s->d_infl[slot].ensure((size_t)H + c.ubytes + INFL_PAD))) return rc;
  if ((rc = s->d_status[slot].ensure(4 * std::max<uint32_t>(nb, 1)))) return rc;
  if ((rc = s->d_flags[slot].ensure(f->format == FMT_FASTA ? 1024 : 256))) return rc;
  if ((rc = s->d_carry.ensure(H))) return rc;
  // Long records (the previous chunk's mean above 2 KiB): 64 KiB segments.  seg_candidates tests every byte offset of a segment up
  // to its first record start, i.e. about half a record per segment (and all of it when a 10 kb record covers the segment): with
  // 16 KiB segments that scan was 9.5 % of the long-read scan.
  const uint32_t seg_bytes = (!f->seg_bytes_set && s->mean_record_bytes > 2048) ? 65536u : f->seg_bytes;
  const uint32_t n_seg = std::max<uint32_t>(1, (uint32_t)((c.ubytes + seg_bytes - 1) / seg_bytes));
  // seg arrays: start, exit, count, base (u32 each) + tail (u8)
  if ((rc = s->d_seg[slot].ensure((size_t)n_seg * 17 + 64))) return rc;
  uint32_t* d_seg_start = s->d_seg[slot].as<uint32_t>();
  uint32_t* d_seg_exit = d_seg_start + n_seg;
  uint32_t* d_seg_count = d_seg_exit + n_seg;
  uint32_t* d_seg_base = d_seg_count + n_seg;
  uint8_t* d_seg_tail = reinterpret_cast<uint8_t*>(d_seg_base + n_seg);
  // [0..7] boundary / filter flags, [8] inflate ticket, [9] inflate error, [10] seams rejected, [11] first disagreeing seam,
  // [12] retry ticket, [13] first owned record, [14] FASTQ first record line, [15] members the CTA inflate kernel refused:
  // these 16 words are published to the host.  [16] line count of the newline scan (device only; FASTA publishes [16, 64)).
  uint32_t* d_flags = s->d_flags[slot].as<uint32_t>();
  const WalkOut W{d_seg_start, d_seg_exit, d_seg_count, d_seg_tail, d_flags};

  cudaStream_t cs = s->s_chunk[slot];
  const uint8_t* d_comp;
  if (s->device_resident) d_comp = s->d_comp_all + (c.c0 - s->comp_all_c0);
  else d_comp = s->d_comp[slot].as<uint8_t>();
  uint8_t* U = s->d_infl[slot].as<uint8_t>();
  const uint32_t carry = s->carry_len;
  // ---- boundaries
  BoundaryParams BP;
  BP.U = U; BP.data_lo = H - carry; BP.data_hi = data_hi; BP.seg0 = seg0; BP.seg_bytes = seg_bytes; BP.n_seg = n_seg;
  BP.n_ref = (int32_t)f->ref_names.size(); BP.ref_len = s->d_refs.as<int32_t>(); BP.max_block_size = MAX_BLOCK_SIZE;
  if (carry) BP.first_start = H - carry;
  else if (s->need_spec) BP.first_start = SEG_NONE;                 // shard without a known start: speculate
  else if (!first_of_range) BP.first_start = H;
  else BP.first_start = H + (uint32_t)(range.first_uoff - c.u0);
  // ownership bound inside this chunk
  uint64_t own = data_hi;
  if (c.extension) own = seg0;
  if (range.stop_uoff != ~0ull && range.stop_uoff < c.u0 + c.ubytes) own = std::min<uint64_t>(own, range.stop_uoff >= c.u0 ? H + (range.stop_uoff - c.u0) : seg0);
  BP.own_hi = (uint32_t)own;
  if (phase != 2) {
    CU_TRY(cudaStreamWaitEvent(cs, s->ev_h2d[slot], 0));   // descriptors (+ compressed bytes) of this chunk have landed
    CU_TRY(cudaMemsetAsync(d_flags, 0, 64, cs));
    CU_TRY(cudaMemsetAsync(d_flags + 2, 0xff, 4, cs));     // [2] tail offset
    CU_TRY(cudaMemsetAsync(d_flags + 5, 0xff, 8, cs));     // [5] first row of the target reference, [6] stop row
    CU_TRY(cudaMemsetAsync(d_flags + 11, 0xff, 4, cs));    // [11] first disagreeing seam
    CU_TRY(cudaMemsetAsync(d_flags + 13, 0xff, 4, cs));    // [13] first owned record of the chunk
    CU_TRY(cudaEventRecord(s->ev_t[slot][0], cs));
    if (nb) {
      int nl = 0;
      if ((rc = launch_inflate(f, cs, d_comp, s->d_blk[slot].as<BlockDesc>(), nb, U + shift, s->d_status[slot].as<uint32_t>(), d_flags + 8, d_flags + 9, d_flags + 12, d_flags + 15, &s->d_sorted, &nl))) return rc;
      s->st.kernel_launches += nl;
    }
    CU_TRY(cudaEventRecord(s->ev_t[slot][1], cs));
    // ---- carry-in
    if (carry) {
      CU_TRY(cudaStreamWaitEvent(cs, s->ev_carry, 0));                  // the previous chunk's tail was copied out on the other stream
      CU_TRY(cudaMemcpyAsync(U + H - carry, s->d_carry.p, carry, cudaMemcpyDeviceToDevice, cs));
    }
    switch (f->format) {
      case FMT_BAM: rc = frame_bam(s, slot, BP, W, d_seg_base); break;
      case FMT_FASTQ: rc = frame_fastq(s, c, slot, BP); break;
      case FMT_SAM: rc = frame_sam(s, c, slot, BP); break;
      case FMT_VCF: rc = frame_vcf(s, c, slot, BP); break;
      case FMT_FASTA: rc = frame_fasta(s, c, range, slot, BP, first_of_range); break;
    }
    if (rc) return rc;
    if (phase == 1) return BAMSCAN_OK;
  }
  CU_TRY(cudaEventSynchronize(s->ev_flags[slot]));
  CU_TRY(cudaGetLastError());
  // ---- host: decisions
  const uint32_t* hf = s->h_flags;
  if (hf[9]) {
    uint32_t bi = (hf[9] & 0x7fffffffu) >> 4, code = hf[9] & 15u;
    static const char* names[] = {"ok", "reserved block type", "stored block LEN/NLEN", "Huffman table", "invalid literal/length code", "invalid distance", "output overrun", "ISIZE mismatch", "CRC32 mismatch", "input overrun"};
    // bi indexes the chunk's descriptors, which skip empty members: map it back to the block table
    uint32_t blk = c.b0;
    for (uint32_t k = 0; blk < c.b1; blk++) if (f->blocks[blk].isize && k++ == bi) break;
    blk = std::min(blk, c.b1 - 1);
    set_error("BAM read error: BGZF member %u (file offset %llu): inflate failed: %s", blk, (unsigned long long)f->blocks[blk].coff, code < 10 ? names[code] : "?");
    return BAMSCAN_ERR_CRC;
  }
  const uint32_t n_rec = hf[3];
  uint32_t tail_off = hf[2] == 0xffffffffu ? data_hi : hf[2];
  if (tail_off > data_hi) tail_off = data_hi;
  *owned_done = tail_off >= BP.own_hi;
  *new_carry = *owned_done ? 0 : data_hi - tail_off;
  if ((rc = read_frame_flags(s, c, H, BP.data_lo, data_hi, n_rec, *new_carry))) return rc;
  s->st.boundary_repairs += hf[4]; s->st.boundary_seam_mismatches += hf[10]; s->st.inflate_retries += hf[15];
  if (*new_carry) { CU_TRY(cudaMemcpyAsync(s->d_carry.p, U + tail_off, *new_carry, cudaMemcpyDeviceToDevice, cs)); CU_TRY(cudaEventRecord(s->ev_carry, cs)); }
  const uint8_t* U_rows = U;               // the bytes the decode stage reads: the inflated chunk, or the SAM chunk's BAM records
  const uint32_t* sam_recoff = nullptr;
  if (f->format == FMT_SAM && n_rec > 0) {
    if ((rc = transcode_sam(s, slot, cs, U, s->d_recoff[slot].as<uint32_t>() + hf[14], n_rec, &U_rows, &sam_recoff))) return rc;
    s->cur.qabs = s->d_qabs[slot].as<uint8_t>();
  } else s->cur.qabs = nullptr;
  s->st.chunks++; s->st.blocks += nb; s->st.inflated_bytes += c.ubytes; s->st.compressed_bytes += c.c1 - c.c0;
  // seam evidence of block-range partitions (BamScanStats): where the first owned record starts, where the chain lands
  // (FASTA: the first record may have been carried in, in front of H)
  if (n_rec > 0 && s->st.first_record_uoff == ~0ull && hf[13] != 0xffffffffu && (hf[13] >= H || f->format == FMT_FASTA)) s->st.first_record_uoff = c.u0 + (uint64_t)hf[13] - H;
  // (FASTA: the chain ends at the next record start; a chunk without one says nothing about where that is)
  if (*owned_done && (f->format != FMT_FASTA || hf[2] != 0xffffffffu)) s->st.end_chain_uoff = c.u0 + (uint64_t)tail_off - H;
  CU_TRY(cudaEventRecord(s->ev_t[slot][2], cs));
  if (n_rec == 0) { CU_TRY(cudaEventRecord(s->ev_t[slot][3], cs)); goto timing; }
  {
    // ---- record offsets
    uint32_t* d_recoff = nullptr;
    switch (f->format) {
      case FMT_BAM:
        if ((rc = s->d_recoff[slot].ensure(4ull * (n_rec + 1)))) return rc;
        d_recoff = s->d_recoff[slot].as<uint32_t>();
        seg_emit_kernel<<<(n_seg + 127) / 128, 128, 0, cs>>>(BP, d_seg_start, d_seg_count, d_seg_base, d_recoff, n_rec, tail_off);
        s->st.kernel_launches++;
        break;
      case FMT_FASTQ: d_recoff = s->d_recoff[slot].as<uint32_t>() + hf[14]; break;       // lines[] from the first record's line on: 4 per row
      case FMT_SAM: d_recoff = const_cast<uint32_t*>(sam_recoff); break;
      case FMT_VCF: d_recoff = s->d_recoff[slot].as<uint32_t>() + hf[14]; break;      // line starts: row r = [lines[r], lines[r + 1])
      case FMT_FASTA: {
        // every line's destination in the chunk's sequence text: content bytes per line, scanned (the decode slices read it)
        const uint32_t* fa_hf = s->h_flags + FA_HFLAGS - 16;     // FASTA words, indexed as in d_flags
        const uint32_t n_lines = fa_hf[FA_F_LINES];
        if ((rc = s->d_faseq[slot].ensure(4ull * (n_lines + 1) + 64))) return rc;
        uint32_t* d_seqpos = s->d_faseq[slot].as<uint32_t>();
        fa_lines_kernel<<<(n_lines + 255) / 256, 256, 0, cs>>>(U, s->d_recoff[slot].as<uint32_t>(), n_lines, d_seqpos);
        s->st.kernel_launches++;
        ScanCols LC; memset(&LC, 0, sizeof LC);
        LC.col[0] = reinterpret_cast<int32_t*>(d_seqpos); LC.n_cols = 1; LC.n = n_lines + 1;
        if ((rc = s->d_totals.ensure(8ull * MAX_SCAN_COLS)) || (rc = launch_offsets_scan(s, cs, LC, s->d_tiles, s->d_totals.as<uint64_t>()))) return rc;
        d_recoff = s->d_fastarts[slot].as<uint32_t>();
        s->cur.fa_lines = s->d_recoff[slot].as<uint32_t>(); s->cur.fa_seqpos = d_seqpos;
        s->cur.fa_tile_base = s->d_seg[slot].as<uint32_t>() + std::max<uint32_t>(1, (data_hi - BP.data_lo + FQ_TILE - 1) / FQ_TILE);
        s->cur.fa_lo = BP.data_lo; s->cur.fa_hi = data_hi; s->cur.fa_slice = 0;
        const uint32_t n_sl = fa_hf[FA_F_SLICES];
        for (uint32_t k = 0; k <= n_sl; k++) { s->cur.fa_slice_rec[k] = fa_hf[FA_F_SLICE_REC + k]; s->cur.fa_slice_byte[k] = fa_hf[FA_F_SLICE_BYTE + k]; }
        break;
      }
    }
    uint32_t n = n_rec;
    if (range.region_mode > 0) {
      // ---- row rule of the indexed scan + residual filters -> compacted record list
      RowRule RR;
      memset(&RR, 0, sizeof RR);
      RR.mode = range.region_mode; RR.ref = range.region_ref; RR.start1 = (uint32_t)range.region_start; RR.end1 = (uint32_t)range.region_end;
      RR.zero_based = f->zero_based; RR.seen_before = s->tail_seen;
      for (const RecordFilter& rf : s->plan->residual) {
        if (RR.n_filters >= MAX_DEV_FILTERS || rf.nums.size() > (size_t)MAX_FILTER_VALUES || rf.strs.size() > (size_t)MAX_FILTER_VALUES) continue;   // not pushed: DataFusion re-applies it (Inexact)
        DevFilter& D = RR.f[RR.n_filters++];
        D.column = rf.column; D.op = rf.op; D.is_str = !rf.strs.empty(); D.n = (int32_t)(D.is_str ? rf.strs.size() : rf.nums.size());
        for (size_t k = 0; k < rf.nums.size(); k++) D.nums[k] = rf.nums[k];
        for (size_t k = 0; k < rf.strs.size(); k++) { D.refs[k] = -2; for (size_t r = 0; r < f->ref_names.size(); r++) if (f->ref_names[r] == rf.strs[k]) { D.refs[k] = (int32_t)r; break; } }
        if (rf.column == BAMSCAN_COL_END) RR.needs_end = 1;
      }
      if ((rc = s->d_keep[slot].ensure(8ull * n_rec + 64))) return rc;
      if ((rc = s->d_recoff2[slot].ensure(4ull * (n_rec + 1)))) return rc;
      uint32_t* d_keep = s->d_keep[slot].as<uint32_t>(); uint32_t* d_pos = d_keep + n_rec;
      if (RR.mode == 2) { rule_first_target_kernel<<<(n_rec + 255) / 256, 256, 0, cs>>>(U, d_recoff, n_rec, RR.ref, d_flags); s->st.kernel_launches++; }
      rule_keep_kernel<<<(n_rec + 255) / 256, 256, 0, cs>>>(U, d_recoff, n_rec, RR, d_keep, d_flags);
      rule_scan_kernel<<<1, 1024, 0, cs>>>(d_keep, d_pos, n_rec, d_flags);
      rule_compact_kernel<<<(n_rec + 255) / 256, 256, 0, cs>>>(d_recoff, d_pos, n_rec, s->d_recoff2[slot].as<uint32_t>());
      s->st.kernel_launches += 3;
      publish_kernel<<<1, 32, 0, cs>>>(d_flags, s->d_hflags, 16);
      CU_TRY(cudaEventRecord(s->ev_flags[slot], cs));
      CU_TRY(cudaEventSynchronize(s->ev_flags[slot]));
      CU_TRY(cudaGetLastError());
      n = s->h_flags[7];
      if (RR.mode == 2) { if (s->h_flags[5] != 0xffffffffu) s->tail_seen = true; if (s->h_flags[6] != 0xffffffffu) s->range_stop = true; }
      d_recoff = s->d_recoff2[slot].as<uint32_t>();
      if (n == 0) { CU_TRY(cudaEventRecord(s->ev_t[slot][3], cs)); goto timing; }
    }
    // ---- hand the rows to decode_slice(): one batch per slice of <= SLICE_BYTES inflated
    const uint32_t n_slices = (uint32_t)std::max<uint64_t>(1, (c.ubytes + SLICE_BYTES - 1) / SLICE_BYTES);
    s->cur.U = U_rows; s->cur.recoff = d_recoff; s->cur.n = n; s->cur.pos = 0; s->cur.cs = cs;
    s->cur.rows_per_slice = (n + n_slices - 1) / n_slices;
    // VCF FORMAT columns: at most FMT_SLICE_ELEMS elements (rows * samples) per slice, which keeps them below 2^31 and bounds the
    // per-element buffers
    if (s->n_format) s->cur.rows_per_slice = std::min<uint32_t>(s->cur.rows_per_slice, std::max<uint64_t>(1, FMT_SLICE_ELEMS / f->vcf_samples.size()));
    s->mean_record_bytes = (uint32_t)std::min<uint64_t>(0xffffffffull, (uint64_t)(data_hi - H) / std::max<uint32_t>(n_rec, 1));
    s->cur.long_records = (f->debug_flags & 2) || s->mean_record_bytes > 2048;
    s->cur.ubytes = c.ubytes / n_slices + (H / 4);
    CU_TRY(cudaEventRecord(s->ev_t[slot][3], cs));
  }
timing:
  CU_TRY(cudaEventRecord(s->ev_t[slot][4], cs));
  CU_TRY(cudaEventSynchronize(s->ev_t[slot][4]));
  {
    float a = 0, b = 0, d = 0;
    cudaEventElapsedTime(&a, s->ev_t[slot][0], s->ev_t[slot][1]);
    if (f->format == FMT_SAM) cudaEventElapsedTime(&a, s->ev_ing[slot][0], s->ev_ing[slot][1]);     // SAM: the ingest copy
    cudaEventElapsedTime(&b, s->ev_t[slot][1], s->ev_t[slot][2]);
    cudaEventElapsedTime(&d, s->ev_t[slot][2], s->ev_t[slot][3]);
    s->st.ms_inflate += a; s->st.ms_boundary += b; s->st.ms_decode += d;
    if (trace2) fprintf(stderr, "[bamscan chunk] phase %d: %.2f ms wall in this call ; gpu inflate %.2f boundary %.2f emit+rules %.2f ms\n", phase, wall_ms() - tw0, a, b, d);
  }
  return BAMSCAN_OK;
}

// H2D of chunk k (unless it was prefetched) and prefetch of chunk k + 1.
static int issue_chunk_h2d(BamScanStream* s, size_t k) {
  const int slot = (int)(k & 1);
  int rc;
  if (!s->have_h2d_ahead) { if ((rc = issue_h2d(s, s->chunks[k], slot))) return rc; }
  s->have_h2d_ahead = false;
  if (k + 1 < s->chunks.size()) { if ((rc = issue_h2d(s, s->chunks[k + 1], slot ^ 1))) return rc; s->have_h2d_ahead = true; }
  return BAMSCAN_OK;
}

// Queues the next chunk's inflate + boundary kernels on the other chunk stream.  Called as soon as the current chunk's
// boundaries (and so the carried tail) are known, i.e. BEFORE its rows are decoded: the two overlap on the GPU.
static int launch_next_chunk_early(BamScanStream* s) {
  if (!s->range_open || s->finished || s->launched_chunk >= 0) return BAMSCAN_OK;
  // By default the next inflate is queued once every row of this chunk is decoded.  debug_flags bit 5 queues it right behind
  // the chunk's FIRST decode slice, so that inflate and the remaining decode kernels share the SMs.  Measured (100 M reads,
  // device resident): the decode stage (66 ms) leaves the critical path but the co-running kernels take issue slots from the
  // latency-bound inflate kernel (15.9 -> 17.5 ms per launch): 456 -> 450 ms per scan.  Not worth a 10 % slower dominant kernel.
  if (!(s->f->debug_flags & 32) && s->cur.pos < s->cur.n) return BAMSCAN_OK;
  if (s->chunk_idx >= s->chunks.size()) return BAMSCAN_OK;          // extension chunks are planned when their turn comes
  const size_t k = s->chunk_idx;
  int rc = issue_chunk_h2d(s, k);
  if (rc) return rc;
  bool produced = false, owned_done = false; uint32_t new_carry = 0;
  rc = run_chunk(s, s->chunks[k], s->part->ranges[s->range_idx], (int)(k & 1), k == 0, &produced, &new_carry, &owned_done, 1);
  if (rc) return rc;
  s->launched_chunk = (int64_t)k;
  return BAMSCAN_OK;
}

// Advances the partition by one chunk.  Returns 1 when a chunk ran (a batch may be pending), 0 when the partition is exhausted.
static int advance(BamScanStream* s, bool* produced) {
  *produced = false;
  BamFile* f = s->f;
  for (;;) {
    if (s->cur.pos < s->cur.n) {   // rows of the current chunk still to decode
      int rc = decode_slice(s, produced);
      if (!rc) rc = launch_next_chunk_early(s);
      return rc ? rc : 1;
    }
    if (s->finished) { int frc = flush_slice(s); return frc ? frc : 0; }
    if (!s->range_open) {
      if (s->range_idx >= s->part->ranges.size()) { s->finished = true; int frc = flush_slice(s); return frc ? frc : 0; }
      const ScanRange& r = s->part->ranges[s->range_idx];
      if (r.region_mode < 0) { set_error("BAM region query failed: a region names a reference sequence that is not in the BAM header"); return BAMSCAN_ERR_INVALID; }
      s->tail_seen = false; s->range_stop = false;
      s->chunks.clear(); s->chunk_idx = 0; s->carry_len = 0; s->have_h2d_ahead = false; s->ext_blocks = 8; s->need_spec = !r.exact_start;
      s->fa_leading = f->format == FMT_FASTA && r.first_uoff == 0;
      plan_chunks(*f, r.block_begin, r.block_end, false, &s->chunks);
      s->range_open = true;
      if (s->chunks.empty()) { s->range_open = false; s->range_idx++; continue; }
    }
    const ScanRange& r = s->part->ranges[s->range_idx];
    if (s->chunk_idx >= s->chunks.size()) {
      // owned blocks exhausted: an incomplete tail record continues into the following blocks
      uint32_t last = s->chunks.back().b1;
      if (s->carry_len == 0 || last >= f->blocks.size()) {
        if (s->carry_len) {
          set_error("%s read error: unexpected EOF inside a record (%u trailing bytes)", format_name(f->format), s->carry_len);
          return BAMSCAN_ERR_FORMAT;
        }
        s->range_open = false; s->range_idx++;
        continue;
      }
      uint32_t e = std::min<uint32_t>((uint32_t)f->blocks.size(), last + s->ext_blocks);
      s->ext_blocks = std::min<uint32_t>(s->ext_blocks * 2, 4096);
      plan_chunks(*f, last, e, true, &s->chunks);
      s->have_h2d_ahead = false;
    }
    const size_t k = s->chunk_idx;
    const int slot = (int)(k & 1);
    int rc;
    const bool launched = s->launched_chunk == (int64_t)k;
    if (!launched && (rc = issue_chunk_h2d(s, k))) return rc;
    uint32_t new_carry = 0; bool owned_done = false;
    s->cur.n = s->cur.pos = 0;
    rc = run_chunk(s, s->chunks[k], r, slot, k == 0, produced, &new_carry, &owned_done, launched ? 2 : 0);
    s->launched_chunk = -1;
    if (rc) return rc;
    s->carry_len = new_carry;
    s->chunk_idx++;
    if (owned_done && s->chunks[k].extension) { s->carry_len = 0; s->range_open = false; s->range_idx++; }   // the tail record is complete
    else if (s->range_stop) { s->carry_len = 0; s->range_open = false; s->range_idx++; }                      // unmapped tail: another reference began
    // first slice now (its kernels get the whole GPU: decode_slice does not wait for them), then the next chunk's inflate on the
    // other stream -- a persistent kernel that fills the SMs as the decode CTAs drain and overlaps the remaining slices
    if (s->cur.pos < s->cur.n && (rc = decode_slice(s, produced))) return rc;
    if ((rc = launch_next_chunk_early(s))) return rc;
    return 1;
  }
}

// ---- Arrow export ---------------------------------------------------------------------------
struct NodePriv { BatchOwner* owner; std::vector<const void*> buffers; std::vector<ArrowArray> child_storage; std::vector<ArrowArray*> child_ptrs; };

static void release_array(ArrowArray* a) {
  if (!a || !a->release) return;
  NodePriv* p = static_cast<NodePriv*>(a->private_data);
  for (int64_t i = 0; i < a->n_children; i++) if (a->children[i] && a->children[i]->release) a->children[i]->release(a->children[i]);
  owner_unref(p->owner);
  delete p;
  a->release = nullptr;
}

static NodePriv* new_node(ArrowArray* a, BatchOwner* owner, int64_t length, int64_t null_count, int64_t offset, size_t n_buffers, size_t n_children) {
  NodePriv* p = new NodePriv();
  p->owner = owner; owner->refs.fetch_add(1);
  p->buffers.assign(n_buffers, nullptr);
  p->child_storage.resize(n_children); p->child_ptrs.resize(n_children);
  for (size_t i = 0; i < n_children; i++) { memset(&p->child_storage[i], 0, sizeof(ArrowArray)); p->child_ptrs[i] = &p->child_storage[i]; }
  a->length = length; a->null_count = null_count; a->offset = offset;
  a->n_buffers = (int64_t)n_buffers; a->n_children = (int64_t)n_children;
  a->buffers = p->buffers.data(); a->children = n_children ? p->child_ptrs.data() : nullptr;
  a->dictionary = nullptr; a->release = release_array; a->private_data = p;
  return p;
}

static int64_t count_nulls(const uint8_t* bm, uint64_t row0, uint64_t n) {
  int64_t set = 0;
  for (uint64_t i = row0; i < row0 + n;) {
    if ((i & 63) == 0 && i + 64 <= row0 + n) { uint64_t w; memcpy(&w, bm + i / 8, 8); set += __builtin_popcountll(w); i += 64; }
    else { set += (bm[i >> 3] >> (i & 7)) & 1; i++; }
  }
  return (int64_t)n - set;
}

static void export_batch(const BamScanStream* s, const ReadyBatch& rb, ArrowArray* out) {
  const bool on_device = rb.owner->dev != nullptr;     // device hand-off: same layout, device addresses, null counts unknown (-1)
  const uint8_t* H = on_device ? static_cast<const uint8_t*>(rb.owner->dev) : rb.owner->arena.p;
  const size_t n_out = s->out_to_dec.size();
  new_node(out, rb.owner, (int64_t)rb.nrows, 0, 0, 1, n_out);
  for (size_t i = 0; i < n_out; i++) {
    const ColLayout& L = rb.cols[s->out_to_dec[i]];
    ArrowArray* ch = out->children[i];
    int64_t nulls = L.has_validity ? (on_device ? -1 : count_nulls(H + L.validity_off, rb.row0, rb.nrows)) : 0;
    const void* validity = (L.has_validity && nulls) ? H + L.validity_off : nullptr;
    if (L.kind == HK_ListListInt32 || L.kind == HK_ListListFloat32) {
      // VCF FORMAT List<List<...>>: outer offsets; middle validity and offsets; leaf validity and values
      NodePriv* p = new_node(ch, rb.owner, (int64_t)rb.nrows, nulls, (int64_t)rb.row0, 2, 1);
      p->buffers[0] = validity; p->buffers[1] = H + L.offsets_off;
      const int64_t mnulls = on_device ? -1 : count_nulls(H + L.child_validity_off, 0, L.child_len);
      NodePriv* mp = new_node(ch->children[0], rb.owner, (int64_t)L.child_len, mnulls, 0, 2, 1);
      mp->buffers[0] = mnulls ? H + L.child_validity_off : nullptr; mp->buffers[1] = H + L.child_offsets_off;
      const int64_t lnulls = on_device ? -1 : count_nulls(H + L.leaf_validity_off, 0, L.leaf_len);
      NodePriv* lp = new_node(ch->children[0]->children[0], rb.owner, (int64_t)L.leaf_len, lnulls, 0, 2, 0);
      lp->buffers[0] = lnulls ? H + L.leaf_validity_off : nullptr; lp->buffers[1] = H + L.data_off;
    } else if (L.kind >= HK_ListInt8) {
      NodePriv* p = new_node(ch, rb.owner, (int64_t)rb.nrows, nulls, (int64_t)rb.row0, 2, 1);
      p->buffers[0] = validity; p->buffers[1] = H + L.offsets_off;
      // VCF lists have nullable elements (child validity) and List<Utf8> a child with offsets; the BAM tag lists have neither
      const bool utf8_items = L.kind == HK_ListUtf8;
      const int64_t cnulls = L.child_validity ? (on_device ? -1 : count_nulls(H + L.child_validity_off, 0, L.child_len)) : 0;
      NodePriv* cp = new_node(ch->children[0], rb.owner, (int64_t)L.child_len, cnulls, 0, utf8_items ? 3 : 2, 0);
      cp->buffers[0] = cnulls ? H + L.child_validity_off : nullptr;
      if (utf8_items) { cp->buffers[1] = H + L.child_offsets_off; cp->buffers[2] = H + L.data_off; }
      else cp->buffers[1] = H + L.data_off;
    } else if (is_var(L.kind)) {
      NodePriv* p = new_node(ch, rb.owner, (int64_t)rb.nrows, nulls, (int64_t)rb.row0, 3, 0);
      p->buffers[0] = validity; p->buffers[1] = H + L.offsets_off; p->buffers[2] = H + L.data_off;
    } else {
      NodePriv* p = new_node(ch, rb.owner, (int64_t)rb.nrows, nulls, (int64_t)rb.row0, 2, 0);
      p->buffers[0] = validity; p->buffers[1] = H + L.values_off;
    }
  }
}

// row: in the batch; row0: rows of the partition in front of the batch
static int decode_error_to_rc(uint32_t code, uint32_t row, uint64_t row0) {
  const unsigned long long prow = row0 + row;
  switch (code) {
    case DEC_ERR_FIELDS: set_error("BAM read error: record %u: fields exceed block_size", row); return BAMSCAN_ERR_FORMAT;
    case DEC_ERR_REF: set_error("BAM read error: record %u: reference sequence id out of range", row); return BAMSCAN_ERR_FORMAT;
    case DEC_ERR_CIGAR_OP: set_error("BAM read error: record %u: invalid CIGAR op", row); return BAMSCAN_ERR_FORMAT;
    case DEC_ERR_TAG_RANGE: set_error("tag value in record %u does not fit the column type", row); return BAMSCAN_ERR_SCHEMA;
    case DEC_ERR_TAG_TYPE: set_error("tag value type mismatch in record %u", row); return BAMSCAN_ERR_SCHEMA;
    case DEC_ERR_UNSUPPORTED_F2S: set_error("record %u: float tag into a Utf8 column is not supported by this build", row); return BAMSCAN_ERR_UNSUPPORTED;
    case DEC_ERR_QUAL: set_error("record %u: quality score in 95..222 (char::from(q + 33) is a two-byte UTF-8 sequence) is not supported by this build", row); return BAMSCAN_ERR_UNSUPPORTED;
    case DEC_ERR_NAME: set_error("record %u: non-ASCII read name is not supported by this build", row); return BAMSCAN_ERR_UNSUPPORTED;
    case FQ_ERR_NAME_PREFIX: set_error("FASTQ read error: record %u of the batch does not start with '@'", row); return BAMSCAN_ERR_FORMAT;
    case FQ_ERR_PLUS: set_error("FASTQ read error: record %u of the batch: third line does not start with '+'", row); return BAMSCAN_ERR_FORMAT;
    case FQ_ERR_UTF8: set_error("FASTQ record %u of the batch: non-ASCII byte (not supported by this build)", row); return BAMSCAN_ERR_UNSUPPORTED;
    case FA_ERR_NAME: set_error("FASTA read error: record %llu of the partition (0-based): empty name", prow); return BAMSCAN_ERR_FORMAT;
    case FA_ERR_UTF8: set_error("FASTA read error: record %llu of the partition (0-based): byte 0x80 or above", prow); return BAMSCAN_ERR_FORMAT;
    case vcf::VCF_ERR_FIELDS: set_error("VCF read error: record %llu of the partition (0-based): fewer than 8 fields", prow); return BAMSCAN_ERR_FORMAT;
    case vcf::VCF_ERR_HASH: set_error("VCF read error: record %llu of the partition (0-based): a '#' line or an empty line in the body", prow); return BAMSCAN_ERR_FORMAT;
    case vcf::VCF_ERR_POS: set_error("VCF read error: record %llu of the partition (0-based): POS is not an integer in [1, 2^31 - 1]", prow); return BAMSCAN_ERR_FORMAT;
    case vcf::VCF_ERR_CHROM: set_error("VCF read error: record %llu of the partition (0-based): empty CHROM", prow); return BAMSCAN_ERR_FORMAT;
    case vcf::VCF_ERR_REF: set_error("VCF read error: record %llu of the partition (0-based): empty REF", prow); return BAMSCAN_ERR_FORMAT;
    case vcf::VCF_ERR_END: set_error("VCF read error: record %llu of the partition (0-based): INFO END is below POS", prow); return BAMSCAN_ERR_FORMAT;
    case vcf::VCF_ERR_DUP: set_error("VCF read error: record %llu of the partition (0-based): an INFO key is given twice", prow); return BAMSCAN_ERR_FORMAT;
    case vcf::VCF_ERR_UTF8: set_error("VCF read error: record %llu of the partition (0-based): byte 0x80 or above in a text column", prow); return BAMSCAN_ERR_FORMAT;
    case vcf::VCF_ERR_QUAL: set_error("VCF read error: record %llu of the partition (0-based): QUAL is not '.' or a number", prow); return BAMSCAN_ERR_FORMAT;
    case vcf::VCF_ERR_VALUE: set_error("VCF read error: record %llu of the partition (0-based): an INFO value does not parse as its declared type", prow); return BAMSCAN_ERR_SCHEMA;
    case vcf::VCF_ERR_POS0: set_error("VCF read error: record %llu of the partition (0-based): POS 0 (a telomere) is not supported by this build", prow); return BAMSCAN_ERR_UNSUPPORTED;
    case vcf::VCF_ERR_LONG: set_error("VCF read error: record %llu of the partition (0-based): a line longer than %u bytes is not supported", prow, vcf::MAX_LINE); return BAMSCAN_ERR_UNSUPPORTED;
    case vcf::VCF_ERR_FMT_FIELDS: set_error("VCF read error: record %llu of the partition (0-based): the line does not have 9 + samples fields", prow); return BAMSCAN_ERR_FORMAT;
    case vcf::VCF_ERR_FMT_DUP: set_error("VCF read error: record %llu of the partition (0-based): a FORMAT key is given twice", prow); return BAMSCAN_ERR_FORMAT;
    case vcf::VCF_ERR_FMT_MANY: set_error("VCF read error: record %llu of the partition (0-based): a sample has more values than the FORMAT field has keys", prow); return BAMSCAN_ERR_FORMAT;
    case vcf::VCF_ERR_FMT_VALUE: set_error("VCF read error: record %llu of the partition (0-based): a FORMAT value does not parse as its declared type", prow); return BAMSCAN_ERR_SCHEMA;
    case FA_ERR_TOO_LONG: set_error("FASTA read error: record %llu of the partition (0-based) is larger than %llu bytes, which is not supported", prow, (unsigned long long)FA_MAX_RECORD); return BAMSCAN_ERR_UNSUPPORTED;
  }
  set_error("decode error %u at record %u", code, row);
  return BAMSCAN_ERR_FORMAT;
}

// waits for the pending batch's D2H and queues it (sliced to batch_rows) for hand-out
static int finalize_pending(BamScanStream* s) {
  NvtxRange nv("bamscan: wait for a batch's D2H");
  PendingBatch& P = s->pending;
  if (!P.valid) return BAMSCAN_OK;
  CU_TRY(cudaEventSynchronize(P.done));
  P.valid = false;
  const uint32_t* err = s->device_export ? s->h_flags + 514 : reinterpret_cast<const uint32_t*>(P.owner->arena.p + P.err_off);
  if (err[0]) { int rc = decode_error_to_rc(err[0], err[1], P.row0); owner_unref(P.owner); P.owner = nullptr; return rc; }
  s->ready.clear(); s->ready_pos = 0;
  uint64_t step = s->f->batch_rows > 0 ? (uint64_t)s->f->batch_rows : P.rows;
  for (uint64_t r0 = 0; r0 < P.rows; r0 += step) {
    ReadyBatch rb{P.owner, P.cols, P.rows, r0, std::min<uint64_t>(step, P.rows - r0)};
    P.owner->refs.fetch_add(1);
    s->ready.push_back(std::move(rb));
  }
  owner_unref(P.owner);   // the pending's own reference
  P.owner = nullptr;
  return BAMSCAN_OK;
}

}  // namespace bamscan

// =============================================================================================
extern "C" {

const char* bamscan_last_error(void) { return last_error_cstr(); }
const char* bamscan_version(void) { return "bamscan-b200 0.1 (sm_100a)"; }

static int bamscan_open_impl(const char* path, const char* index_path_or_null, const BamScanOptions* options, BamScanHandle** out, ScanFormat format = FMT_BAM);

// No C++ exception may cross the C ABI (a corrupt file can ask for absurd allocations): they become BAMSCAN_ERR_FORMAT.
#define BAMSCAN_GUARD(call)                                                                                          \
  try { return (call); }                                                                                             \
  catch (const std::bad_alloc&) { set_error("out of memory (corrupt or oversized input?)"); return BAMSCAN_ERR_FORMAT; } \
  catch (const std::exception& e) { set_error("internal error: %s", e.what()); return BAMSCAN_ERR_FORMAT; }           \
  catch (...) { set_error("internal error"); return BAMSCAN_ERR_FORMAT; }

int bamscan_open(const char* path, const char* index_path_or_null, const BamScanOptions* options, BamScanHandle** out) {
  BAMSCAN_GUARD(bamscan_open_impl(path, index_path_or_null, options, out))
}

static int bamscan_open_impl(const char* path, const char* index_path_or_null, const BamScanOptions* options, BamScanHandle** out, ScanFormat format) {
  if (!path || !out) { set_error("bamscan_open: null argument"); return BAMSCAN_ERR_INVALID; }
  if (format == FMT_BAM && is_sam_path(path)) format = FMT_SAM;
  BamScanOptions opt;
  memset(&opt, 0, sizeof opt);
  opt.coordinate_system_zero_based = 1; opt.infer_tag_types = 1; opt.infer_tag_sample_size = 100;
  if (options) memcpy(&opt, options, std::min<size_t>(sizeof opt, options->struct_size ? options->struct_size : sizeof opt));
  int ndev = 0;
  g_have_device = cudaGetDeviceCount(&ndev) == cudaSuccess && ndev > 0;
  if (!g_have_device) cudaGetLastError();   // planning-only mode: header, schema, filter classification and plans work; execute() does not
  else {
    if (opt.device_id < 0 || opt.device_id >= ndev) { set_error("device_id %d out of range (%d devices)", opt.device_id, ndev); return BAMSCAN_ERR_INVALID; }
    if (cudaSetDevice(opt.device_id) != cudaSuccess) { set_error("cudaSetDevice(%d) failed", opt.device_id); return BAMSCAN_ERR_CUDA; }
  }
  std::unique_ptr<BamScanHandle> h(new BamScanHandle());
  BamFile& f = h->file;
  f.path = path; f.device = opt.device_id; f.format = format;
  f.zero_based = opt.coordinate_system_zero_based != 0; f.binary_cigar = opt.binary_cigar != 0;
  f.has_tag_fields = opt.has_tag_fields != 0;
  for (int i = 0; i < opt.n_tag_fields && opt.tag_fields; i++) f.tag_fields.push_back(opt.tag_fields[i]);
  if (format == FMT_VCF && opt.has_format_fields)
    for (int i = 0; i < opt.n_format_fields && opt.format_fields; i++) f.format_fields.push_back(opt.format_fields[i] ? opt.format_fields[i] : "");
  f.batch_rows = opt.batch_rows;
  if (opt.chunk_inflated_bytes) f.chunk_bytes = std::min<uint64_t>(opt.chunk_inflated_bytes, 768ull << 20);   // an explicit size is also the slice size
  if (opt.segment_bytes) { f.seg_bytes = std::max<uint32_t>(256, opt.segment_bytes); f.seg_bytes_set = true; }
  f.skip_crc = opt.skip_crc != 0; f.debug_flags = opt.debug_flags; f.decode_all_tags = opt.decode_all_tag_fields != 0;
  int rc = load_file(&f);
  if (rc == BAMSCAN_ERR_IO || rc == BAMSCAN_ERR_CUDA || (format == FMT_SAM && rc)) { release_file(&f); return rc; }
  // a file whose header cannot be read still yields a provider with empty metadata (table_provider.rs:423-426);
  // scans on it fail later
  if (format == FMT_FASTQ) {
    // == determine_schema of bio-format-fastq/src/table_provider.rs:22-32
    if (rc) { release_file(&f); return rc; }
    f.fields = {FieldDef{"name", HK_Utf8, false, {}}, FieldDef{"description", HK_Utf8, true, {}}, FieldDef{"sequence", HK_Utf8, false, {}}, FieldDef{"quality_scores", HK_Utf8, false, {}}};
    *out = h.release();
    return BAMSCAN_OK;
  }
  if (format == FMT_VCF) {
    // VCF: the fixed columns and the INFO fields the header declares (info_fields travel as tag_fields); no metadata, no index
    if (rc) { release_file(&f); return rc; }
    if ((rc = build_vcf_schema(&f, &opt))) { release_file(&f); return rc; }
    *out = h.release();
    return BAMSCAN_OK;
  }
  if (format == FMT_FASTA) {
    // FASTA: name, description (NULL when empty), sequence; no metadata, as for FASTQ
    if (rc) { release_file(&f); return rc; }
    f.fields = {FieldDef{"name", HK_Utf8, false, {}}, FieldDef{"description", HK_Utf8, true, {}}, FieldDef{"sequence", HK_Utf8, false, {}}};
    *out = h.release();
    return BAMSCAN_OK;
  }
  if ((rc = build_schema(&f, &opt))) { release_file(&f); return rc; }
  if (format == FMT_SAM) { *out = h.release(); return BAMSCAN_OK; }     // SAM: no index (the reference discovers none for SAM paths)
  if (index_path_or_null) f.index_path = index_path_or_null; else f.index_path = discover_index(f.path);   // "" = no index
  if (!f.index_path.empty()) {
    f.bai.reset(new BaiIndex());
    if (load_bai(f.index_path, f.bai.get()) != BAMSCAN_OK) { f.bai.reset(); if (index_path_or_null) { release_file(&f); return BAMSCAN_ERR_IO; } f.index_path.clear(); }
  }
  *out = h.release();
  return BAMSCAN_OK;
}

int bamscan_open_fastq(const char* path, const BamScanOptions* options, BamScanHandle** out) {
  BAMSCAN_GUARD(bamscan_open_impl(path, nullptr, options, out, FMT_FASTQ))
}

int bamscan_open_fasta(const char* path, const BamScanOptions* options, BamScanHandle** out) {
  BAMSCAN_GUARD(bamscan_open_impl(path, nullptr, options, out, FMT_FASTA))
}

int bamscan_open_vcf(const char* path, const BamScanOptions* options, BamScanHandle** out) {
  BAMSCAN_GUARD(bamscan_open_impl(path, nullptr, options, out, FMT_VCF))
}

void bamscan_close(BamScanHandle* h) {
  if (!h) return;
  for (BamScanStream* s : h->idle_streams) stream_destroy(s, false);
  h->idle_streams.clear();
  if (h->file.data) { if (g_have_device) cudaSetDevice(h->file.device); release_file(&h->file); }
  delete h;
}

int bamscan_schema(BamScanHandle* h, struct ArrowSchema* out) {
  if (!h || !out) { set_error("null argument"); return BAMSCAN_ERR_INVALID; }
  return export_schema(h->file.fields, h->file.schema_metadata, out);
}

static int bamscan_describe_tags_impl(BamScanHandle* h, int32_t sample_size, char* buf, uint64_t cap, uint64_t* needed) {
  if (!h || !needed || (cap && !buf)) { set_error("null argument"); return BAMSCAN_ERR_INVALID; }
  if (h->file.format == FMT_FASTQ || h->file.format == FMT_FASTA || h->file.format == FMT_VCF) { set_error("describe is a BamTableProvider call"); return BAMSCAN_ERR_INVALID; }
  if (!h->file.header_ok) { set_error("BAM header could not be read: %s", h->file.path.c_str()); return BAMSCAN_ERR_FORMAT; }
  std::map<std::string, std::pair<char, int32_t>> found;
  infer_tag_types(h->file, {}, sample_size > 0 ? sample_size : 100, &found, true);
  static const char* kind_names[] = {"?", "Int32", "UInt32", "Float32", "Utf8", "Binary"};
  const auto& reg = known_tags();
  std::string out;
  for (auto& kv : found) {   // std::map: sorted by tag name, as describe() sorts them
    const int32_t k = kv.second.second;
    std::string ty;
    if (k >= HK_ListInt8) {
      static const char* el[] = {"Int8", "UInt8", "Int16", "UInt16", "Int32", "UInt32", "Float32"};
      ty = std::string("List<") + el[k - HK_ListInt8] + ">";
    } else ty = kind_names[k];
    auto r = reg.find(kv.first);
    const std::string desc = r != reg.end() ? r->second.description : std::string("Custom/unknown tag (") + kv.second.first + ")";
    out += kv.first; out += '\t'; out += kv.second.first; out += '\t'; out += ty; out += '\t'; out += desc; out += '\n';
  }
  *needed = out.size() + 1;
  if (cap < *needed) { set_error("buffer of %llu bytes is too small (%llu needed)", (unsigned long long)cap, (unsigned long long)*needed); return BAMSCAN_ERR_INVALID; }
  memcpy(buf, out.c_str(), out.size() + 1);
  return BAMSCAN_OK;
}
int bamscan_describe_tags(BamScanHandle* h, int32_t sample_size, char* buf, uint64_t cap, uint64_t* needed) {
  BAMSCAN_GUARD(bamscan_describe_tags_impl(h, sample_size, buf, cap, needed))
}

int bamscan_classify_filters(BamScanHandle* h, const BamScanFilter* filters, int32_t n_filters, uint8_t* out_pushdown) {
  if (!h || (n_filters && (!filters || !out_pushdown))) { set_error("null argument"); return BAMSCAN_ERR_INVALID; }
  if (h->file.format == FMT_FASTQ || h->file.format == FMT_FASTA || h->file.format == FMT_VCF) { for (int i = 0; i < n_filters; i++) out_pushdown[i] = 0; return BAMSCAN_OK; }   // the FASTQ, FASTA and VCF providers push no filter down
  return classify_filters(h->file, filters, n_filters, out_pushdown);
}

static int bamscan_plan_impl(BamScanHandle* h, const int32_t* projection, int32_t n_projection, const BamScanFilter* filters, int32_t n_filters,
                             int64_t limit_or_neg, int32_t target_partitions, int32_t partition_mode, BamScanPlan** out);
int bamscan_plan(BamScanHandle* h, const int32_t* projection, int32_t n_projection, const BamScanFilter* filters, int32_t n_filters,
                 int64_t limit_or_neg, int32_t target_partitions, int32_t partition_mode, BamScanPlan** out) {
  BAMSCAN_GUARD(bamscan_plan_impl(h, projection, n_projection, filters, n_filters, limit_or_neg, target_partitions, partition_mode, out))
}
static int bamscan_plan_impl(BamScanHandle* h, const int32_t* projection, int32_t n_projection, const BamScanFilter* filters, int32_t n_filters,
                             int64_t limit_or_neg, int32_t target_partitions, int32_t partition_mode, BamScanPlan** out) {
  (void)limit_or_neg;   // stored and never used by the reference either (physical_exec.rs:38,44)
  if (!h || !out) { set_error("null argument"); return BAMSCAN_ERR_INVALID; }
  Plan* p = nullptr;
  int rc = make_plan(&h->file, projection, n_projection, filters, n_filters, target_partitions, partition_mode, &p);
  if (rc) return rc;
  BamScanPlan* bp = new BamScanPlan();
  bp->plan = p; bp->handle = h;
  *out = bp;
  return BAMSCAN_OK;
}

int32_t bamscan_plan_num_partitions(const BamScanPlan* plan) { return plan && !plan->plan->empty_exec ? (int32_t)plan->plan->partitions.size() : 0; }

int bamscan_plan_schema(const BamScanPlan* plan, struct ArrowSchema* out) {
  if (!plan || !out) { set_error("null argument"); return BAMSCAN_ERR_INVALID; }
  return export_schema(plan->plan->out_fields, plan->plan->file->schema_metadata, out);
}

void bamscan_plan_free(BamScanPlan* plan) { if (plan) { delete plan->plan; delete plan; } }

int32_t bamscan_plan_num_ranges(const BamScanPlan* plan, int32_t partition) {
  if (!plan || partition < 0 || partition >= (int32_t)plan->plan->partitions.size()) return -1;
  return (int32_t)plan->plan->partitions[partition].ranges.size();
}

int32_t bamscan_plan_partition_regions(const BamScanPlan* plan, int32_t partition, struct BamScanAssignedRegion* out, int32_t cap) {
  if (!plan || partition < 0 || partition >= (int32_t)plan->plan->partitions.size()) return -1;
  const Partition& P = plan->plan->partitions[partition];
  const BamFile& f = *plan->plan->file;
  int32_t k = 0;
  for (const GenomicRegion& g : P.regions) {
    if (k < cap && out) {
      int ref = -1;
      for (size_t r = 0; r < f.ref_names.size(); r++) if (f.ref_names[r] == g.chrom) { ref = (int)r; break; }
      out[k].partition = partition; out[k].estimate_index = ref;
      out[k].has_start = g.has_start; out[k].start = g.start; out[k].has_end = g.has_end; out[k].end = g.end;
      out[k].unmapped_tail = g.unmapped_tail; out[k].partition_total_estimated_bytes = P.estimated_bytes;
    }
    k++;
  }
  return k;
}

int bamscan_plan_range_info(const BamScanPlan* plan, int32_t partition, int32_t range, uint64_t out[14]) {
  if (!plan || !out || partition < 0 || partition >= (int32_t)plan->plan->partitions.size()) { set_error("bad partition"); return BAMSCAN_ERR_INVALID; }
  const Partition& P = plan->plan->partitions[partition];
  if (range < 0 || range >= (int32_t)P.ranges.size()) { set_error("bad range"); return BAMSCAN_ERR_INVALID; }
  const ScanRange& r = P.ranges[range];
  const BamFile& f = *plan->plan->file;
  out[0] = r.block_begin; out[1] = r.block_end;
  out[2] = r.block_begin < f.blocks.size() ? f.blocks[r.block_begin].coff : f.size;
  out[3] = r.block_end < f.blocks.size() ? f.blocks[r.block_end].coff : f.size;
  out[4] = r.exact_start; out[5] = r.first_uoff; out[6] = r.stop_uoff;
  out[7] = (uint64_t)r.region_mode; out[8] = (uint64_t)(int64_t)r.region_ref; out[9] = r.region_start; out[10] = r.region_end;
  out[11] = P.estimated_bytes;
  auto to_voffset = [&](uint64_t uoff) -> uint64_t {
    if (uoff == ~0ull || uoff >= f.total_inflated) return uoff == ~0ull ? 0 : (uint64_t)f.size << 16;
    size_t lo = 0, hi = f.blocks.size();
    while (lo < hi) { size_t mid = (lo + hi) / 2; if (f.blocks[mid].uoff + f.blocks[mid].isize <= uoff) lo = mid + 1; else hi = mid; }
    return (f.blocks[lo].coff << 16) | (uoff - f.blocks[lo].uoff);
  };
  out[12] = to_voffset(r.first_uoff); out[13] = to_voffset(r.stop_uoff);   // virtual offsets (stop 0 = none)
  return BAMSCAN_OK;
}

static int make_stream(BamScanPlan* plan, int32_t partition, bool device_resident, BamScanStream** out, bool device_export = false) {
  if (!plan || !out) { set_error("null argument"); return BAMSCAN_ERR_INVALID; }
  if (partition < 0 || partition >= (int32_t)plan->plan->partitions.size()) { set_error("partition %d out of range", partition); return BAMSCAN_ERR_INVALID; }
  if (!g_have_device) { set_error("no CUDA device available: the BAM scan runs on the GPU only (libbamscan has no CPU path)"); return BAMSCAN_ERR_CUDA; }
  BamScanStream* s = nullptr;
  {
    std::lock_guard<std::mutex> lk(plan->handle->mu);
    if (!plan->handle->idle_streams.empty()) { s = plan->handle->idle_streams.back(); plan->handle->idle_streams.pop_back(); }
  }
  if (!s) s = new BamScanStream();
  s->plan = plan->plan; s->f = plan->plan->file; s->part = &plan->plan->partitions[partition]; s->handle = plan->handle;
  s->device_resident = device_resident; s->device_export = device_export;
  int rc = stream_init(s);
  if (rc) { stream_destroy(s, false); return rc; }
  *out = s;
  return BAMSCAN_OK;
}

int bamscan_execute(BamScanPlan* plan, int32_t partition, BamScanStream** out) { BAMSCAN_GUARD(make_stream(plan, partition, false, out)) }
int bamscan_execute_device(BamScanPlan* plan, int32_t partition, BamScanStream** out) { BAMSCAN_GUARD(make_stream(plan, partition, false, out, true)) }

int bamscan_next_device(BamScanStream* s, struct ArrowDeviceArray* out) {
  if (!s || !out) { set_error("null argument"); return BAMSCAN_ERR_INVALID; }
  if (!s->device_export) { set_error("bamscan_next_device needs a stream from bamscan_execute_device"); return BAMSCAN_ERR_INVALID; }
  memset(out, 0, sizeof *out);
  const int rc = bamscan_next(s, &out->array);
  if (rc != 1) return rc;
  BatchOwner* o = static_cast<NodePriv*>(out->array.private_data)->owner;
  out->device_id = s->f->device; out->device_type = ARROW_DEVICE_CUDA;
  out->sync_event = o->dev_ready ? &o->dev_ready : nullptr;
  return 1;
}

static int bamscan_next_impl(BamScanStream* s, struct ArrowArray* out);
int bamscan_next(BamScanStream* s, struct ArrowArray* out) { BAMSCAN_GUARD(bamscan_next_impl(s, out)) }
static int bamscan_next_impl(BamScanStream* s, struct ArrowArray* out) {
  if (!s || !out) { set_error("null argument"); return BAMSCAN_ERR_INVALID; }
  static const bool trace = getenv("BAMSCAN_TRACE") != nullptr;
  static thread_local double t_last_return = 0;
  const double t_enter = wall_ms();
  if (s->error) { set_error("stream is in an error state"); return s->error; }
  if (cudaSetDevice(s->f->device) != cudaSuccess) { set_error("cudaSetDevice failed"); return BAMSCAN_ERR_CUDA; }
  for (;;) {
    if (s->ready_pos < s->ready.size()) {
      export_batch(s, s->ready[s->ready_pos], out);
      owner_unref(s->ready[s->ready_pos].owner);   // the queue's reference; the exported nodes hold their own
      s->ready_pos++;
      t_last_return = wall_ms();
      return 1;
    }
    if (!s->finished) {
      // the batch produced by the previous chunk has had its D2H overlapped with nothing yet: keep it pending while
      // the next chunk is launched, then hand it out
      PendingBatch prev = s->pending;
      s->pending = PendingBatch();
      bool produced = false;
      const double t0 = wall_ms();
      int rc = advance(s, &produced);
      const double t1 = wall_ms();
      if (rc < 0) { s->error = rc; if (prev.valid) { cudaEventSynchronize(prev.done); owner_unref(prev.owner); cudaEventDestroy(prev.done); } return rc; }
      PendingBatch fresh = s->pending;
      s->pending = prev;
      if (prev.valid) {
        rc = finalize_pending(s);
        if (trace) fprintf(stderr, "[bamscan] outside %.2f ms | advance %.2f ms | wait+finalize d2h %.2f ms\n", t_last_return ? t_enter - t_last_return : 0.0, t1 - t0, wall_ms() - t1);
        if (prev.done) cudaEventDestroy(prev.done);
        s->pending = PendingBatch();
        if (rc) { s->error = rc; if (fresh.valid) { cudaEventSynchronize(fresh.done); owner_unref(fresh.owner); cudaEventDestroy(fresh.done); } return rc; }
      }
      s->pending = fresh;
      continue;
    }
    if (s->pending.valid) {
      cudaEvent_t ev = s->pending.done;
      int rc = finalize_pending(s);
      if (ev) cudaEventDestroy(ev);
      s->pending = PendingBatch();
      if (rc) { s->error = rc; return rc; }
      continue;
    }
    return 0;
  }
}

void bamscan_stream_free(BamScanStream* s) { stream_destroy(s); }

int bamscan_stream_stats(const BamScanStream* s, BamScanStats* out) {
  if (!s || !out) { set_error("null argument"); return BAMSCAN_ERR_INVALID; }
  *out = s->st;
  return BAMSCAN_OK;
}

int bamscan_run_device_resident(BamScanPlan* plan, int32_t partition, int32_t repeats, BamScanStats* stats) {
  if (!stats) { set_error("null argument"); return BAMSCAN_ERR_INVALID; }
  BamScanStream* s = nullptr;
  int rc = make_stream(plan, partition, true, &s);
  if (rc) return rc;
  BamFile* f = s->f;
  // stage the partition's compressed bytes in HBM (untimed)
  uint32_t bmin = 0xffffffffu, bmax = 0;
  for (auto& r : s->part->ranges) { bmin = std::min(bmin, r.block_begin); bmax = std::max(bmax, r.block_end); }
  if (bmin >= bmax) { memset(stats, 0, sizeof *stats); stream_destroy(s); return BAMSCAN_OK; }
  uint32_t bext = std::min<uint32_t>((uint32_t)f->blocks.size(), bmax + 8192);   // room for tail-record extension chunks
  uint64_t c0 = f->blocks[bmin].coff, c1 = f->blocks[bext - 1].coff + f->blocks[bext - 1].csize;
  if ((rc = s->d_comp_all_buf.ensure((size_t)(c1 - c0) + 1024))) { stream_destroy(s); return rc; }
  if (cudaMemcpy(s->d_comp_all_buf.p, f->data + c0, (size_t)(c1 - c0), cudaMemcpyHostToDevice) != cudaSuccess ||
      cudaMemset(s->d_comp_all_buf.as<uint8_t>() + (c1 - c0), 0, 1024) != cudaSuccess) { set_error("staging copy failed"); stream_destroy(s); return BAMSCAN_ERR_CUDA; }
  s->d_comp_all = s->d_comp_all_buf.as<uint8_t>(); s->comp_all_c0 = c0;
  cudaEvent_t e0, e1;
  cudaEventCreate(&e0); cudaEventCreate(&e1);
  double best_total = 0;
  BamScanStats acc{};
  for (int rep = 0; rep < std::max(1, repeats); rep++) {
    s->st = BamScanStats{}; s->st.first_record_uoff = ~0ull; s->range_idx = 0; s->range_open = false; s->finished = false; s->carry_len = 0; s->launched_chunk = -1; s->cur.n = s->cur.pos = 0;
    cudaEventRecord(e0, s->s_compute);
    bool produced;
    while ((rc = advance(s, &produced)) == 1) {}
    if (rc < 0) break;
    cudaEventRecord(e1, s->s_compute);
    cudaEventSynchronize(e1);
    float ms = 0; cudaEventElapsedTime(&ms, e0, e1);
    s->st.ms_total = ms;
    best_total += ms;
    acc = s->st;
  }
  cudaEventDestroy(e0); cudaEventDestroy(e1);
  if (rc >= 0) { acc.ms_total = best_total / std::max(1, repeats); *stats = acc; rc = BAMSCAN_OK; }
  stream_destroy(s);
  return rc;
}

int bamscan_check_partition_seams(const BamScanStats* stats, int32_t n) {
  if (!stats || n <= 0) { set_error("null argument"); return BAMSCAN_ERR_INVALID; }
  uint64_t expect = ~0ull;     // where the next partition that owns a record must start
  for (int32_t p = 0; p < n; p++) {
    const BamScanStats& S = stats[p];
    if (S.first_record_uoff != ~0ull && expect != ~0ull && S.first_record_uoff != expect) {
      set_error("block-range partition %d starts at inflated offset %llu but the chain of the partition before it lands at %llu: speculative record start rejected",
                p, (unsigned long long)S.first_record_uoff, (unsigned long long)expect);
      return BAMSCAN_ERR_FORMAT;
    }
    if (S.rows > 0 || S.end_chain_uoff) expect = S.end_chain_uoff;
  }
  return BAMSCAN_OK;
}

int bamscan_probe_pcie(int32_t device_id, uint64_t bytes, double* h2d_gbps, double* d2h_gbps, double* bidir_gbps) {
  if (cudaSetDevice(device_id) != cudaSuccess) { set_error("cudaSetDevice failed"); return BAMSCAN_ERR_CUDA; }
  void *h0 = nullptr, *h1 = nullptr, *d0 = nullptr, *d1 = nullptr;
  cudaStream_t s0, s1; cudaEvent_t e0, e1, e2;
  if (cudaHostAlloc(&h0, bytes, cudaHostAllocPortable) != cudaSuccess || cudaHostAlloc(&h1, bytes, cudaHostAllocPortable) != cudaSuccess ||
      cudaMalloc(&d0, bytes) != cudaSuccess || cudaMalloc(&d1, bytes) != cudaSuccess) { set_error("probe allocation failed"); return BAMSCAN_ERR_CUDA; }
  memset(h0, 1, bytes); memset(h1, 2, bytes);
  cudaStreamCreate(&s0); cudaStreamCreate(&s1); cudaEventCreate(&e0); cudaEventCreate(&e1); cudaEventCreate(&e2);
  float best_h2d = 1e30f, best_d2h = 1e30f, best_bi = 1e30f, ms;
  for (int rep = 0; rep < 3; rep++) {
    cudaEventRecord(e0, s0); cudaMemcpyAsync(d0, h0, bytes, cudaMemcpyHostToDevice, s0); cudaEventRecord(e1, s0); cudaEventSynchronize(e1);
    cudaEventElapsedTime(&ms, e0, e1); best_h2d = std::min(best_h2d, ms);
    cudaEventRecord(e0, s0); cudaMemcpyAsync(h1, d1, bytes, cudaMemcpyDeviceToHost, s0); cudaEventRecord(e1, s0); cudaEventSynchronize(e1);
    cudaEventElapsedTime(&ms, e0, e1); best_d2h = std::min(best_d2h, ms);
    cudaEventRecord(e0, s0); cudaStreamWaitEvent(s1, e0, 0);
    cudaMemcpyAsync(d0, h0, bytes, cudaMemcpyHostToDevice, s0); cudaMemcpyAsync(h1, d1, bytes, cudaMemcpyDeviceToHost, s1);
    cudaEventRecord(e2, s1); cudaStreamWaitEvent(s0, e2, 0); cudaEventRecord(e1, s0); cudaEventSynchronize(e1);
    cudaEventElapsedTime(&ms, e0, e1); best_bi = std::min(best_bi, ms);
  }
  *h2d_gbps = bytes / 1e6 / best_h2d; *d2h_gbps = bytes / 1e6 / best_d2h; *bidir_gbps = 2.0 * bytes / 1e6 / best_bi;
  cudaFreeHost(h0); cudaFreeHost(h1); cudaFree(d0); cudaFree(d1); cudaStreamDestroy(s0); cudaStreamDestroy(s1);
  cudaEventDestroy(e0); cudaEventDestroy(e1); cudaEventDestroy(e2);
  return BAMSCAN_OK;
}

int bamscan_bench_inflate(BamScanPlan* plan, int32_t partition, int32_t repeats, double* ms_per_launch, uint64_t* inflated_bytes, uint64_t* compressed_bytes) {
  BamScanStream* s = nullptr;
  int rc = make_stream(plan, partition, true, &s);
  if (rc) return rc;
  BamFile* f = s->f;
  if (f->format == FMT_SAM) { stream_destroy(s); set_error("a SAM scan has no inflate to benchmark"); return BAMSCAN_ERR_INVALID; }
  if (s->part->ranges.empty()) { stream_destroy(s); set_error("empty partition"); return BAMSCAN_ERR_INVALID; }
  const ScanRange& r = s->part->ranges[0];
  std::vector<ChunkPlan> chunks;
  {   // kernel-only benchmark: one full inflate wave, whatever the scan's chunk cap is (nothing is decoded here)
    const uint64_t saved = f->chunk_bytes;
    f->chunk_bytes = 0;
    plan_chunks(*f, r.block_begin, r.block_end, false, &chunks);
    f->chunk_bytes = saved;
  }
  const ChunkPlan& c = chunks[0];
  std::vector<BlockDesc> descs;
  uint32_t uoff = 0;
  for (uint32_t b = c.b0; b < c.b1; b++) {
    const BgzfBlock& B = f->blocks[b];
    if (B.isize) { BlockDesc d; d.cdata_off = (uint32_t)(B.coff - c.c0) + B.cdata_off; d.cdata_len = B.csize - B.cdata_off - 8; d.isize = B.isize; d.crc = B.crc; d.uoff = uoff; descs.push_back(d); }
    uoff += B.isize;
  }
  uint32_t nb = (uint32_t)descs.size();
  DeviceBuf comp, blk, infl, status, flags;
  auto fail = [&](int code) { comp.release(); blk.release(); infl.release(); status.release(); flags.release(); stream_destroy(s); return code; };
  if (comp.ensure((size_t)(c.c1 - c.c0) + 1024) || blk.ensure(sizeof(BlockDesc) * nb) || infl.ensure((size_t)c.ubytes + INFL_PAD) || status.ensure(4ull * nb) || flags.ensure(256)) return fail(BAMSCAN_ERR_CUDA);
  cudaMemcpy(comp.p, f->data + c.c0, (size_t)(c.c1 - c.c0), cudaMemcpyHostToDevice);
  cudaMemset(comp.as<uint8_t>() + (c.c1 - c.c0), 0, 1024);
  cudaMemcpy(blk.p, descs.data(), sizeof(BlockDesc) * nb, cudaMemcpyHostToDevice);
  cudaEvent_t e0, e1; cudaEventCreate(&e0); cudaEventCreate(&e1);
  float total = 0;
  const bool want_prof = getenv("BAMSCAN_ICTA_PROF") != nullptr;
  const size_t prof_n = (size_t)device_sms(f->device) * 2 * 16;
  if (want_prof) { cudaMalloc((void**)&g_icta_prof, prof_n * 8); }
  for (int rep = 0; rep < repeats + 1; rep++) {
    if (want_prof) cudaMemsetAsync(g_icta_prof, 0, prof_n * 8, s->s_compute);
    cudaMemsetAsync(flags.p, 0, 64, s->s_compute);
    cudaEventRecord(e0, s->s_compute);
    int nl = 0;
    launch_inflate(f, s->s_compute, comp.as<uint8_t>(), blk.as<BlockDesc>(), nb, infl.as<uint8_t>(), status.as<uint32_t>(), flags.as<uint32_t>() + 8, flags.as<uint32_t>() + 9, flags.as<uint32_t>() + 12, flags.as<uint32_t>() + 15, &s->d_sorted, &nl);
    cudaEventRecord(e1, s->s_compute);
    cudaEventSynchronize(e1);
    float ms = 0; cudaEventElapsedTime(&ms, e0, e1);
    if (rep > 0) total += ms;   // first launch is warm-up
  }
  uint32_t hflags[16];
  cudaMemcpy(hflags, flags.p, 64, cudaMemcpyDeviceToHost);
  if (want_prof) {   // last repetition: per-phase cycles of thread 0, summed over the CTAs, per member
    std::vector<unsigned long long> h(prof_n);
    cudaMemcpy(h.data(), g_icta_prof, prof_n * 8, cudaMemcpyDeviceToHost);
    cudaFree(g_icta_prof); g_icta_prof = nullptr;
    unsigned long long sum[16] = {};
    for (size_t i = 0; i < prof_n; i++) sum[i % 16] += h[i];
    static const char* names[] = {"ticket", "payload load", "block header", "tables", "count rounds", "scan+emit",
                                  "resolve", "crc", "store+status", "producer waits for window", "consumer waits for member"};
    const double m = (double)std::max<unsigned long long>(1, sum[13]);
    fprintf(stderr, "[icta prof] members %llu, count rounds/member %.2f, resolve batches/member %.2f; cycles per member:", sum[13], sum[12] / m, sum[11] / m);
    for (int k = 0; k < 11; k++) fprintf(stderr, " %s%s %.0f |", k < 6 || k == 9 ? "P " : "C ", names[k], sum[k] / m);
    fprintf(stderr, "\n");
  }
  cudaEventDestroy(e0); cudaEventDestroy(e1);
  if (cudaGetLastError() != cudaSuccess || hflags[9]) { set_error("inflate benchmark failed (flag %u)", hflags[9]); return fail(BAMSCAN_ERR_CRC); }
  *ms_per_launch = total / std::max(1, repeats); *inflated_bytes = c.ubytes; *compressed_bytes = c.c1 - c.c0;
  return fail(BAMSCAN_OK);
}

}  // extern "C"
