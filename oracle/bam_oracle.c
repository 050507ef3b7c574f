/*
 * oracle/bam_oracle.c -- CPU restatement of the reference's BAM -> Arrow scan.
 *
 * TEST INFRASTRUCTURE ONLY.  Nothing in the product path (datafusion-bio-formats_b200/) may link,
 * import or call this file; only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline /
 * --impl reference legs use it, and only as the checker / the timed CPU baseline.
 *
 * Parity pinning: the reference (Rust, noodles fork @42a3c016, libdeflater 1.25.2) cannot be
 * compiled in this environment (no cargo/rustc, un-vendored git dependencies).  This restatement
 * is pinned against the reference's own fixtures and test pins (tests/test_oracle_golden.py):
 * record counts 421/4277/20/14/10/2 (indexed_read_test.rs:76-77, indexed_read_large_test.rs:63,
 * tag_tests.rs), first/last record values, and the independent aggregate facts of SURVEY.md App. C.
 *
 * What it follows (file:line under /root/reference/datafusion):
 *   - BGZF framing + inflate + CRC32/ISIZE:       noodles-bgzf 0.49.0 io::Reader (call site
 *                                                 bio-format-bam/src/storage.rs:161-169); SAMv1 4.1
 *   - BAM header:                                 noodles-bam read_header (storage.rs:167)
 *   - record framing (block_size chain):          physical_exec.rs:409 (reader.read_record)
 *   - 12 core columns:                            physical_exec.rs:412-528
 *   - CIGAR text:                                 bio-format-core/src/alignment_utils.rs:667-701
 *   - tag columns and coercions:                  bio-format-core/src/sam_tag_io.rs:154-204, 658-1036
 *   - projection / batch assembly:                alignment_utils.rs:316-368, 432-451
 *   - batching (<= batch_size rows, tail batch):  physical_exec.rs:545-593
 *   - indexed keep rule / residual filters:       physical_exec.rs:1275-1344, record_filter.rs:57-283
 *
 * Inflate uses system zlib (raw, window -15) + zlib crc32; the reference uses libdeflate, which
 * is not installed here.  Any conformant inflater yields identical bytes (CRC32/ISIZE checked).
 */
#define _GNU_SOURCE
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <zlib.h>

#define ORC_API __attribute__((visibility("default")))

/* ------------------------------------------------------------------------------------------ */
/* column kinds (shared numbering with the python wrapper oracle/bam_oracle.py)                */
enum {
  K_Int32 = 1, K_UInt32 = 2, K_Float32 = 3, K_Utf8 = 4, K_Binary = 5,
  K_ListInt8 = 10, K_ListUInt8 = 11, K_ListInt16 = 12, K_ListUInt16 = 13,
  K_ListInt32 = 14, K_ListUInt32 = 15, K_ListFloat32 = 16
};

typedef struct { uint8_t *p; size_t len, cap; } Buf;

static int buf_reserve(Buf *b, size_t extra) {
  if (b->len + extra <= b->cap) return 0;
  size_t nc = b->cap ? b->cap * 2 : 4096;
  while (nc < b->len + extra) nc *= 2;
  uint8_t *np = (uint8_t *)realloc(b->p, nc);
  if (!np) return -1;
  b->p = np; b->cap = nc;
  return 0;
}
static inline void buf_put(Buf *b, const void *src, size_t n) {
  if (buf_reserve(b, n)) abort();
  memcpy(b->p + b->len, src, n); b->len += n;
}
static inline void buf_put_u8(Buf *b, uint8_t v) { if (buf_reserve(b, 1)) abort(); b->p[b->len++] = v; }
static inline void buf_put_i32(Buf *b, int32_t v) { buf_put(b, &v, 4); }

/* One output column under construction (Arrow layout: validity bitmap, i32 offsets, values).  */
typedef struct {
  int32_t kind;
  int64_t n;            /* rows appended */
  int64_t null_count;
  Buf validity;         /* bitmap, LSB-first */
  Buf offsets;          /* int32[n+1] for Utf8/Binary/List */
  Buf data;             /* values (fixed width), string bytes, or list child values */
} Col;

static void col_init(Col *c, int32_t kind) {
  memset(c, 0, sizeof *c);
  c->kind = kind;
  if (kind == K_Utf8 || kind == K_Binary || kind >= K_ListInt8) buf_put_i32(&c->offsets, 0);
}
static void col_reset(Col *c) {
  int32_t kind = c->kind;
  c->n = 0; c->null_count = 0; c->validity.len = 0; c->offsets.len = 0; c->data.len = 0;
  if (kind == K_Utf8 || kind == K_Binary || kind >= K_ListInt8) buf_put_i32(&c->offsets, 0);
}
static void col_free(Col *c) { free(c->validity.p); free(c->offsets.p); free(c->data.p); }

static inline void col_push_valid(Col *c, int valid) {
  int64_t i = c->n;
  if ((i & 7) == 0) buf_put_u8(&c->validity, 0);
  if (valid) c->validity.p[i >> 3] |= (uint8_t)(1u << (i & 7)); else c->null_count++;
  c->n++;
}
static inline void col_append_u32(Col *c, uint32_t v) { buf_put(&c->data, &v, 4); col_push_valid(c, 1); }
static inline void col_append_null_fixed(Col *c) { uint32_t z = 0; buf_put(&c->data, &z, 4); col_push_valid(c, 0); }
static inline void col_append_bytes(Col *c, const void *s, size_t n) {
  buf_put(&c->data, s, n);
  buf_put_i32(&c->offsets, (int32_t)c->data.len);
  col_push_valid(c, 1);
}
static inline void col_append_null_var(Col *c) {
  int32_t last; memcpy(&last, c->offsets.p + c->offsets.len - 4, 4);
  buf_put_i32(&c->offsets, last);
  col_push_valid(c, 0);
}
static inline int kind_elem_size(int32_t kind) {
  switch (kind) {
    case K_ListInt8: case K_ListUInt8: return 1;
    case K_ListInt16: case K_ListUInt16: return 2;
    default: return 4;
  }
}
static inline void col_list_close(Col *c) { /* offsets count list ELEMENTS */
  buf_put_i32(&c->offsets, (int32_t)(c->data.len / (size_t)kind_elem_size(c->kind)));
  col_push_valid(c, 1);
}
static void col_append_null(Col *c) {
  if (c->kind == K_Int32 || c->kind == K_UInt32 || c->kind == K_Float32) col_append_null_fixed(c);
  else col_append_null_var(c);
}

/* ------------------------------------------------------------------------------------------ */
/* BGZF streaming reader (continuous inflated byte stream, one block at a time)                */

typedef struct {
  const uint8_t *file; size_t size;
  size_t next_coff;        /* file offset of the next block to inflate */
  size_t cur_coff;         /* file offset of the block currently in buf */
  uint8_t buf[65536];
  uint32_t buf_len, buf_pos;
  int64_t inflated_bytes, blocks;
  int eof;
  char err[200];
} Bgzf;

static void bgzf_init(Bgzf *z, const uint8_t *file, size_t size, size_t coff) {
  z->file = file; z->size = size; z->next_coff = coff; z->cur_coff = coff;
  z->buf_len = z->buf_pos = 0; z->inflated_bytes = 0; z->blocks = 0; z->eof = 0; z->err[0] = 0;
}

/* Parses one BGZF member at `off`.  Returns total block size, or 0 on error. */
static uint32_t bgzf_block_size(const uint8_t *p, size_t avail, uint32_t *cdata_off) {
  if (avail < 18) return 0;
  if (p[0] != 0x1f || p[1] != 0x8b || p[2] != 8 || !(p[3] & 4)) return 0;
  uint32_t xlen = p[10] | (p[11] << 8);
  if (avail < 12 + xlen) return 0;
  uint32_t x = 0, bsize = 0; int found = 0;
  while (x + 4 <= xlen) {
    const uint8_t *sf = p + 12 + x;
    uint32_t slen = sf[2] | (sf[3] << 8);
    if (sf[0] == 'B' && sf[1] == 'C' && slen == 2 && x + 6 <= xlen) { bsize = sf[4] | (sf[5] << 8); found = 1; }
    x += 4 + slen;
  }
  if (!found) return 0;
  *cdata_off = 12 + xlen;
  return bsize + 1;
}

/* Loads the next non-empty block into buf.  Returns 1 ok, 0 clean EOF, -1 error. */
static int bgzf_next_block(Bgzf *z) {
  for (;;) {
    if (z->next_coff >= z->size) { z->eof = 1; return 0; }
    uint32_t cdata_off = 0;
    uint32_t total = bgzf_block_size(z->file + z->next_coff, z->size - z->next_coff, &cdata_off);
    if (total == 0 || z->next_coff + total > z->size || total < cdata_off + 8) {
      snprintf(z->err, sizeof z->err, "invalid BGZF block header at offset %zu", z->next_coff);
      return -1;
    }
    const uint8_t *blk = z->file + z->next_coff;
    uint32_t crc_expect, isize;
    memcpy(&crc_expect, blk + total - 8, 4); memcpy(&isize, blk + total - 4, 4);
    if (isize > 65536) { snprintf(z->err, sizeof z->err, "ISIZE > 64KiB at %zu", z->next_coff); return -1; }
    z_stream s; memset(&s, 0, sizeof s);
    if (inflateInit2(&s, -15) != Z_OK) { snprintf(z->err, sizeof z->err, "inflateInit2 failed"); return -1; }
    s.next_in = (Bytef *)(blk + cdata_off); s.avail_in = total - cdata_off - 8;
    s.next_out = z->buf; s.avail_out = sizeof z->buf;
    int rc = inflate(&s, Z_FINISH);
    size_t produced = s.total_out;
    inflateEnd(&s);
    if (rc != Z_STREAM_END || produced != isize) {
      snprintf(z->err, sizeof z->err, "inflate failed (rc=%d) or ISIZE mismatch at %zu", rc, z->next_coff);
      return -1;
    }
    if ((uint32_t)crc32(crc32(0L, Z_NULL, 0), z->buf, isize) != crc_expect) {
      snprintf(z->err, sizeof z->err, "CRC32 mismatch at %zu", z->next_coff);
      return -1;
    }
    z->cur_coff = z->next_coff; z->next_coff += total;
    z->buf_len = isize; z->buf_pos = 0; z->inflated_bytes += isize; z->blocks++;
    if (isize > 0) return 1;
  }
}

/* Reads exactly n bytes.  Returns n, 0 on clean EOF before the first byte, -1 on error/truncation. */
static int64_t bgzf_read_exact(Bgzf *z, uint8_t *dst, size_t n) {
  size_t got = 0;
  while (got < n) {
    if (z->buf_pos == z->buf_len) {
      int rc = bgzf_next_block(z);
      if (rc < 0) return -1;
      if (rc == 0) { if (got == 0) return 0; snprintf(z->err, sizeof z->err, "unexpected EOF inside a record"); return -1; }
    }
    size_t take = z->buf_len - z->buf_pos; if (take > n - got) take = n - got;
    memcpy(dst + got, z->buf + z->buf_pos, take); z->buf_pos += (uint32_t)take; got += take;
  }
  return (int64_t)n;
}

/* Makes sure the reader is positioned on a byte (loads the next block if the current one is
 * exhausted) so that (cur_coff, buf_pos) is the virtual position of the next byte.            */
static int bgzf_settle(Bgzf *z) {
  while (z->buf_pos == z->buf_len) { int rc = bgzf_next_block(z); if (rc <= 0) return rc; }
  return 1;
}

/* ------------------------------------------------------------------------------------------ */
/* scan arguments / result                                                                     */

typedef struct {
  char tag[2];
  int32_t kind;
} OrcTag;

typedef struct {
  int32_t op;      /* 0 EQ 1 NE 2 LT 3 LE 4 GT 5 GE 6 BETWEEN 7 NOT_BETWEEN 8 IN 9 NOT_IN */
  int32_t column;  /* 1 chrom 2 start 3 end 6 mapping_quality 4 flags (schema ids) */
  int32_t n_num;   double num[16];
  int32_t n_str;   const char *str[16];
} OrcFilter;

typedef struct {
  int32_t zero_based;
  int32_t binary_cigar;
  int32_t end_zero_span_mode;   /* 0: NULL (noodles bam::Record::alignment_end), 1: pos */
  int32_t n_tags; const OrcTag *tags;
  int32_t n_proj; const int32_t *proj;      /* n_proj < 0: no projection (all columns) */
  /* partition: records whose first byte lies in a block with start_coff <= coffset < end_coff */
  uint64_t start_voffset;                   /* virtual offset of first record; 0 = right after header */
  uint64_t end_coff;                        /* 0 = to EOF */
  int64_t max_records;                      /* 0 = unlimited */
  int32_t batch_rows;                       /* >0: timing mode, flush & drop every batch_rows rows */
  /* indexed-path row rules (physical_exec.rs:1275-1344); region_mode 0 = sequential path */
  int32_t region_mode;                      /* 1: mapped region, 2: per-ref unmapped tail, 3: "*" */
  int32_t region_ref;                       /* reference id the region is on */
  int64_t region_start, region_end;         /* 1-based closed, 0 = open */
  uint64_t stop_voffset;                    /* region_mode 1: stop once record voffset >= this (0 = none) */
  int32_t n_filters; const OrcFilter *filters;
} OrcArgs;

typedef struct {
  int64_t n_rows;
  int32_t n_cols;
  Col *cols;               /* in projection order */
  int32_t *col_ids;        /* schema index of each output column */
  int64_t inflated_bytes, blocks, batches, records_seen;
  uint64_t next_voffset;   /* virtual offset after the last owned record */
  char err[256];
} OrcResult;

typedef struct {
  uint8_t *file; size_t size;
  int32_t n_ref; char **ref_names; int32_t *ref_lens;
  char *text; int32_t l_text;
  uint64_t first_record_voffset;
  char err[256];
} OrcFile;

/* ------------------------------------------------------------------------------------------ */

ORC_API void orc_close(OrcFile *f) {
  if (!f) return;
  for (int i = 0; i < f->n_ref; i++) free(f->ref_names[i]);
  free(f->ref_names); free(f->ref_lens); free(f->text); free(f->file); free(f);
}

ORC_API OrcFile *orc_open(const char *path, char *errbuf, int errlen) {
  OrcFile *f = (OrcFile *)calloc(1, sizeof *f);
  FILE *fp = fopen(path, "rb");
  if (!fp) { snprintf(errbuf, errlen, "cannot open %s", path); free(f); return NULL; }
  fseek(fp, 0, SEEK_END); long sz = ftell(fp); fseek(fp, 0, SEEK_SET);
  f->file = (uint8_t *)malloc(sz > 0 ? (size_t)sz : 1); f->size = (size_t)sz;
  if (fread(f->file, 1, f->size, fp) != f->size) { snprintf(errbuf, errlen, "short read"); fclose(fp); orc_close(f); return NULL; }
  fclose(fp);
  Bgzf *z = (Bgzf *)malloc(sizeof *z);
  bgzf_init(z, f->file, f->size, 0);
  uint8_t hdr[8];
  if (bgzf_read_exact(z, hdr, 8) != 8 || memcmp(hdr, "BAM\1", 4) != 0) {
    snprintf(errbuf, errlen, "not a BAM file (%s)", z->err); free(z); orc_close(f); return NULL;
  }
  memcpy(&f->l_text, hdr + 4, 4);
  f->text = (char *)malloc((size_t)f->l_text + 1);
  if (f->l_text && bgzf_read_exact(z, (uint8_t *)f->text, (size_t)f->l_text) != f->l_text) goto bad;
  f->text[f->l_text] = 0;
  if (bgzf_read_exact(z, hdr, 4) != 4) goto bad;
  memcpy(&f->n_ref, hdr, 4);
  f->ref_names = (char **)calloc((size_t)f->n_ref + 1, sizeof(char *));
  f->ref_lens = (int32_t *)calloc((size_t)f->n_ref + 1, sizeof(int32_t));
  for (int i = 0; i < f->n_ref; i++) {
    int32_t l_name;
    if (bgzf_read_exact(z, hdr, 4) != 4) goto bad;
    memcpy(&l_name, hdr, 4);
    f->ref_names[i] = (char *)malloc((size_t)l_name + 1);
    if (bgzf_read_exact(z, (uint8_t *)f->ref_names[i], (size_t)l_name) != l_name) goto bad;
    f->ref_names[i][l_name] = 0;
    if (bgzf_read_exact(z, hdr, 4) != 4) goto bad;
    memcpy(&f->ref_lens[i], hdr, 4);
  }
  if (bgzf_settle(z) < 0) goto bad;
  f->first_record_voffset = z->eof ? ((uint64_t)z->next_coff << 16) : (((uint64_t)z->cur_coff << 16) | z->buf_pos);
  free(z);
  return f;
bad:
  snprintf(errbuf, errlen, "truncated BAM header (%s)", z->err);
  free(z); orc_close(f); return NULL;
}

ORC_API int32_t orc_n_ref(const OrcFile *f) { return f->n_ref; }
ORC_API const char *orc_ref_name(const OrcFile *f, int i) { return f->ref_names[i]; }
ORC_API int32_t orc_ref_len(const OrcFile *f, int i) { return f->ref_lens[i]; }
ORC_API const char *orc_header_text(const OrcFile *f) { return f->text; }
ORC_API int32_t orc_header_text_len(const OrcFile *f) { return f->l_text; }
ORC_API uint64_t orc_first_record_voffset(const OrcFile *f) { return f->first_record_voffset; }

/* ------------------------------------------------------------------------------------------ */
/* per-record helpers                                                                          */

static inline uint32_t rd_u32(const uint8_t *p) { uint32_t v; memcpy(&v, p, 4); return v; }
static inline int32_t rd_i32(const uint8_t *p) { int32_t v; memcpy(&v, p, 4); return v; }
static inline uint16_t rd_u16(const uint8_t *p) { uint16_t v; memcpy(&v, p, 2); return v; }

static const char CIGAR_OPS[] = "MIDNSHP=X";       /* alignment_utils.rs:667-679 */
static const char SEQ_CODES[] = "=ACMGRSVTWYHKDBN"; /* SAMv1 4.2 */

static int utf8_valid(const uint8_t *s, size_t n) {
  size_t i = 0;
  while (i < n) {
    uint8_t c = s[i];
    if (c < 0x80) { i++; continue; }
    int len; uint32_t cp;
    if ((c & 0xE0) == 0xC0) { len = 2; cp = c & 0x1F; }
    else if ((c & 0xF0) == 0xE0) { len = 3; cp = c & 0x0F; }
    else if ((c & 0xF8) == 0xF0) { len = 4; cp = c & 0x07; }
    else return 0;
    if (i + len > n) return 0;
    for (int k = 1; k < len; k++) { if ((s[i + k] & 0xC0) != 0x80) return 0; cp = (cp << 6) | (s[i + k] & 0x3F); }
    if ((len == 2 && cp < 0x80) || (len == 3 && cp < 0x800) || (len == 4 && cp < 0x10000)) return 0;
    if (cp > 0x10FFFF || (cp >= 0xD800 && cp <= 0xDFFF)) return 0;
    i += len;
  }
  return 1;
}

static size_t utf8_encode(uint32_t cp, uint8_t out[4]) {
  if (cp < 0x80) { out[0] = (uint8_t)cp; return 1; }
  if (cp < 0x800) { out[0] = 0xC0 | (cp >> 6); out[1] = 0x80 | (cp & 0x3F); return 2; }
  if (cp < 0x10000) { out[0] = 0xE0 | (cp >> 12); out[1] = 0x80 | ((cp >> 6) & 0x3F); out[2] = 0x80 | (cp & 0x3F); return 3; }
  out[0] = 0xF0 | (cp >> 18); out[1] = 0x80 | ((cp >> 12) & 0x3F); out[2] = 0x80 | ((cp >> 6) & 0x3F); out[3] = 0x80 | (cp & 0x3F);
  return 4;
}
static int is_char_cp(int64_t v) { return v >= 0 && v <= 0x10FFFF && !(v >= 0xD800 && v <= 0xDFFF); }

/* sam_tag_io.rs:698-741: integer value into the column's type. Returns 0 ok, -1 error. */
static int append_int_like(Col *c, int64_t v, char *err) {
  if (c->kind == K_Utf8) {
    if (is_char_cp(v)) { uint8_t u[4]; size_t n = utf8_encode((uint32_t)v, u); col_append_bytes(c, u, n); }
    else { char tmp[32]; int n = snprintf(tmp, sizeof tmp, "%lld", (long long)v); col_append_bytes(c, tmp, (size_t)n); }
    return 0;
  }
  if (c->kind == K_UInt32) {
    if (v < 0 || v > 0xFFFFFFFFLL) { snprintf(err, 256, "integer value %lld does not fit UInt32", (long long)v); return -1; }
    col_append_u32(c, (uint32_t)v); return 0;
  }
  if (c->kind == K_Int32) {
    if (v < INT32_MIN || v > INT32_MAX) { snprintf(err, 256, "integer value %lld does not fit Int32", (long long)v); return -1; }
    col_append_u32(c, (uint32_t)(int32_t)v); return 0;
  }
  snprintf(err, 256, "tag value type mismatch: integer into column kind %d", c->kind);
  return -1;
}

static int sub_size(uint8_t st) {
  switch (st) { case 'c': case 'C': return 1; case 's': case 'S': return 2; case 'i': case 'I': case 'f': return 4; default: return 0; }
}

/* sam_tag_io.rs:761-1036: B-array into List<T> with element-wise checked conversion. */
static int append_array(Col *c, uint8_t st, const uint8_t *p, int32_t count, char *err) {
  if (c->kind < K_ListInt8) { snprintf(err, 256, "tag value type mismatch: expected scalar column, got array"); return -1; }
  int es = sub_size(st);
  for (int32_t i = 0; i < count; i++) {
    const uint8_t *e = p + (size_t)i * es;
    int64_t iv = 0; float fv = 0; int is_f = 0;
    switch (st) {
      case 'c': iv = (int8_t)e[0]; break;
      case 'C': iv = e[0]; break;
      case 's': iv = (int16_t)rd_u16(e); break;
      case 'S': iv = rd_u16(e); break;
      case 'i': iv = rd_i32(e); break;
      case 'I': iv = rd_u32(e); break;
      case 'f': memcpy(&fv, e, 4); is_f = 1; break;
    }
    if (c->kind == K_ListFloat32) {
      float out = is_f ? fv : (float)iv;
      buf_put(&c->data, &out, 4);
      continue;
    }
    if (is_f) { snprintf(err, 256, "tag value type mismatch: float array into integer list"); return -1; }
    int64_t lo, hi;
    switch (c->kind) {
      case K_ListInt8: lo = -128; hi = 127; break;
      case K_ListUInt8: lo = 0; hi = 255; break;
      case K_ListInt16: lo = -32768; hi = 32767; break;
      case K_ListUInt16: lo = 0; hi = 65535; break;
      case K_ListInt32: lo = INT32_MIN; hi = INT32_MAX; break;
      default: lo = 0; hi = 0xFFFFFFFFLL; break;
    }
    if (iv < lo || iv > hi) { snprintf(err, 256, "array element %lld does not fit list kind %d", (long long)iv, c->kind); return -1; }
    switch (kind_elem_size(c->kind)) {
      case 1: { uint8_t o = (uint8_t)iv; buf_put(&c->data, &o, 1); break; }
      case 2: { uint16_t o = (uint16_t)iv; buf_put(&c->data, &o, 2); break; }
      default: { uint32_t o = (uint32_t)iv; buf_put(&c->data, &o, 4); break; }
    }
  }
  col_list_close(c);
  return 0;
}

/* "%.*e" text `s` (no sign) -> the decimal one unit above it in the last digit, with as many digits ("9.9e5" -> "1.0e6"). */
static void f32_next_up(const char *s, char *out, size_t cap) {
  char d[16]; int nd = 0; const char *p = s;
  for (; *p != 'e'; p++) if (*p != '.') d[nd++] = *p;
  int x = atoi(p + 1), i = nd - 1;
  while (i >= 0 && d[i] == '9') d[i--] = '0';
  if (i >= 0) d[i]++; else { d[0] = '1'; x++; }
  snprintf(out, cap, "%c.%.*se%d", d[0], nd - 1, d + 1, x);
}

/* Rust `f32::to_string()` (shortest digits inside the rounding interval, the closer of two; never exponent form): the
 * smallest precision whose correctly rounded "%.*e" reads back -- or, when that rounded down, the value one unit above it,
 * which can read back where the rounded one does not only at a power of two (the float below is half as far away as the
 * one above).  oracle/f32_exact.py is the exact reference. */
static size_t rust_f32_to_string(float v, char *out, size_t cap) {
  if (v != v) return (size_t)snprintf(out, cap, "NaN");
  if (v == 1.0f / 0.0f) return (size_t)snprintf(out, cap, "inf");
  if (v == -1.0f / 0.0f) return (size_t)snprintf(out, cap, "-inf");
  char tmp[64], alt[64]; int prec;
  const int minus = v < 0 || (v == 0 && 1.0f / v < 0);
  const float a = minus ? -v : v;
  for (prec = 1; prec <= 9; prec++) {
    snprintf(tmp, sizeof tmp, "%.*e", prec - 1, (double)a);
    if (strtof(tmp, NULL) == a) break;
    if (strtod(tmp, NULL) < (double)a) {
      f32_next_up(tmp, alt, sizeof alt);
      if (strtof(alt, NULL) == a) { memcpy(tmp, alt, sizeof tmp); break; }
    }
  }
  if (minus) { memmove(tmp + 1, tmp, strlen(tmp) + 1); tmp[0] = '-'; }
  /* tmp = d.ddddde[+-]XX -> expand to plain decimal */
  char digits[16]; int nd = 0; int neg = 0; const char *s = tmp;
  if (*s == '-') { neg = 1; s++; }
  for (; *s && *s != 'e'; s++) if (*s != '.') digits[nd++] = *s;
  int exp10 = atoi(s + 1);
  while (nd > 1 && digits[nd - 1] == '0') nd--;
  size_t o = 0;
  if (neg) out[o++] = '-';
  if (nd == 1 && digits[0] == '0') { out[o++] = '0'; out[o] = 0; return o; }
  if (exp10 < 0) { out[o++] = '0'; out[o++] = '.'; for (int i = 0; i < -exp10 - 1; i++) out[o++] = '0'; for (int i = 0; i < nd; i++) out[o++] = digits[i]; }
  else {
    for (int i = 0; i <= exp10; i++) out[o++] = i < nd ? digits[i] : '0';
    if (nd > exp10 + 1) { out[o++] = '.'; for (int i = exp10 + 1; i < nd; i++) out[o++] = digits[i]; }
  }
  out[o] = 0; (void)cap;
  return o;
}

/* Walks the aux region once, appending requested tags (sam_tag_io.rs:154-204). */
static int load_tags(const uint8_t *aux, size_t aux_len, const OrcArgs *a, Col **tag_cols, uint8_t *populated, char *err) {
  int nt = a->n_tags;
  memset(populated, 0, (size_t)nt);
  size_t i = 0;
  while (i + 3 <= aux_len) {
    const uint8_t *t = aux + i; uint8_t ty = t[2];
    const uint8_t *v = t + 3; size_t rem = aux_len - i - 3; size_t vlen;
    switch (ty) {
      case 'A': case 'c': case 'C': vlen = 1; break;
      case 's': case 'S': vlen = 2; break;
      case 'i': case 'I': case 'f': vlen = 4; break;
      case 'Z': case 'H': { const uint8_t *z = (const uint8_t *)memchr(v, 0, rem); if (!z) return 0; /* malformed: stop (warn + skip) */ vlen = (size_t)(z - v) + 1; break; }
      case 'B': { if (rem < 5) return 0; int es = sub_size(v[0]); if (!es) return 0; vlen = 5 + (size_t)rd_i32(v + 1) * es; break; }
      default: return 0; /* malformed field: noodles yields Err, the loader warns and skips */
    }
    if (vlen > rem) return 0;
    int idx = -1;
    for (int k = 0; k < nt; k++) if (a->tags[k].tag[0] == t[0] && a->tags[k].tag[1] == t[1]) idx = k; /* HashMap: last duplicate name wins */
    if (idx >= 0 && tag_cols[idx]) {
      Col *c = tag_cols[idx];
      populated[idx] = 1;
      int rc = 0;
      switch (ty) {
        case 'c': rc = append_int_like(c, (int8_t)v[0], err); break;
        case 'C': rc = append_int_like(c, v[0], err); break;
        case 's': rc = append_int_like(c, (int16_t)rd_u16(v), err); break;
        case 'S': rc = append_int_like(c, rd_u16(v), err); break;
        case 'i': rc = append_int_like(c, rd_i32(v), err); break;
        case 'I': rc = append_int_like(c, rd_u32(v), err); break;
        case 'f': {
          float fv; memcpy(&fv, v, 4);
          if (c->kind == K_Utf8) { char tmp[80]; size_t n = rust_f32_to_string(fv, tmp, sizeof tmp); col_append_bytes(c, tmp, n); }
          else if (c->kind == K_Float32) col_append_u32(c, rd_u32(v));
          else { snprintf(err, 256, "tag value type mismatch: float into column kind %d", c->kind); rc = -1; }
          break;
        }
        case 'Z': case 'H':
          if (c->kind != K_Utf8) { snprintf(err, 256, "tag value type mismatch: string into column kind %d", c->kind); rc = -1; }
          else if (utf8_valid(v, vlen - 1)) col_append_bytes(c, v, vlen - 1);
          else col_append_null(c);
          break;
        case 'A':
          if (c->kind == K_UInt32 || c->kind == K_Int32) col_append_u32(c, v[0]);
          else if (c->kind == K_Utf8) { uint8_t u[4]; size_t n = utf8_encode(v[0], u); col_append_bytes(c, u, n); }
          else { snprintf(err, 256, "tag value type mismatch: char into column kind %d", c->kind); rc = -1; }
          break;
        case 'B': rc = append_array(c, v[0], v + 5, rd_i32(v + 1), err); break;
      }
      if (rc) return rc;
    }
    i += 3 + vlen;
  }
  return 0;
}

/* record_filter.rs:57-283.  NULL accessor value => the filter passes.  */
static int eval_filters(const OrcArgs *a, const char *chrom, int has_start, uint32_t start, int has_end, uint32_t end,
                        uint32_t mapq, uint32_t flags) {
  for (int i = 0; i < a->n_filters; i++) {
    const OrcFilter *f = &a->filters[i];
    if (f->column == 1) { /* chrom: string = != IN NOT IN */
      if (!chrom) continue;
      int any = 0;
      for (int k = 0; k < f->n_str; k++) if (strcmp(chrom, f->str[k]) == 0) any = 1;
      int pass;
      switch (f->op) { case 0: case 8: pass = any; break; case 1: case 9: pass = !any; break; default: pass = 1; }
      if (!pass) return 0;
      continue;
    }
    double v; int has = 1;
    switch (f->column) {
      case 2: has = has_start; v = start; break;
      case 3: has = has_end; v = end; break;
      case 6: v = mapq; break;
      case 4: v = flags; break;
      default: has = 0; v = 0; break;
    }
    if (!has) continue;
    int pass = 1;
    switch (f->op) {
      case 0: pass = v == f->num[0]; break;
      case 1: pass = v != f->num[0]; break;
      case 2: pass = v < f->num[0]; break;
      case 3: pass = v <= f->num[0]; break;
      case 4: pass = v > f->num[0]; break;
      case 5: pass = v >= f->num[0]; break;
      case 6: pass = v >= f->num[0] && v <= f->num[1]; break;
      case 7: pass = !(v >= f->num[0] && v <= f->num[1]); break;
      case 8: case 9: { int any = 0; for (int k = 0; k < f->n_num; k++) if (v == f->num[k]) any = 1; pass = f->op == 8 ? any : !any; break; }
    }
    if (!pass) return 0;
  }
  return 1;
}

/* ------------------------------------------------------------------------------------------ */

ORC_API void orc_result_free(OrcResult *r) {
  if (!r) return;
  for (int i = 0; i < r->n_cols; i++) col_free(&r->cols[i]);
  free(r->cols); free(r->col_ids); free(r);
}

/* Scans one partition.  Mirrors the per-partition loop of physical_exec.rs:371-598 (sequential)
 * and, with region_mode != 0, the row rules of :1036-1356.                                       */
ORC_API OrcResult *orc_scan(const OrcFile *f, const OrcArgs *a) {
  OrcResult *r = (OrcResult *)calloc(1, sizeof *r);
  int n_schema = 12 + a->n_tags;
  /* ProjectionFlags (alignment_utils.rs:432-451) */
  int need[12]; int any_tag;
  if (a->n_proj < 0) { for (int i = 0; i < 12; i++) need[i] = 1; any_tag = 1; }
  else {
    for (int i = 0; i < 12; i++) need[i] = 0;
    any_tag = 0;
    for (int i = 0; i < a->n_proj; i++) { if (a->proj[i] < 12) need[a->proj[i]] = 1; else any_tag = 1; }
  }
  if (a->n_tags == 0) any_tag = 0;
  static const int32_t core_kinds[12] = { K_Utf8, K_Utf8, K_UInt32, K_UInt32, K_UInt32, K_Utf8, K_UInt32, K_Utf8, K_UInt32, K_Utf8, K_Utf8, K_Int32 };
  Col *all = (Col *)calloc((size_t)n_schema, sizeof(Col));
  uint8_t *built = (uint8_t *)calloc((size_t)n_schema, 1);
  for (int i = 0; i < 12; i++) if (need[i]) { col_init(&all[i], (i == 5 && a->binary_cigar) ? K_Binary : core_kinds[i]); built[i] = 1; }
  /* quirk (sam_tag_io.rs:33-76): when any tag column is projected, ALL tag_fields are decoded */
  Col **tag_cols = (Col **)calloc((size_t)a->n_tags + 1, sizeof(Col *));
  if (any_tag) for (int k = 0; k < a->n_tags; k++) { col_init(&all[12 + k], a->tags[k].kind); built[12 + k] = 1; tag_cols[k] = &all[12 + k]; }
  uint8_t *populated = (uint8_t *)calloc((size_t)a->n_tags + 1, 1);

  Bgzf *z = (Bgzf *)malloc(sizeof *z);
  uint64_t sv = a->start_voffset ? a->start_voffset : f->first_record_voffset;
  bgzf_init(z, f->file, f->size, (size_t)(sv >> 16));
  uint32_t skip = (uint32_t)(sv & 0xFFFF);
  size_t rec_cap = 1 << 16; uint8_t *rec = (uint8_t *)malloc(rec_cap);
  Buf tmp = {0};
  int64_t rows = 0, batch_rows = 0;
  int rc_err = 0, seen_target = 0;

  if (skip) { if (bgzf_settle(z) <= 0 || z->buf_len < skip) { snprintf(r->err, sizeof r->err, "bad start voffset"); rc_err = 1; } else z->buf_pos = skip; }

  while (!rc_err) {
    int st = bgzf_settle(z);
    if (st < 0) { snprintf(r->err, sizeof r->err, "BAM read error: %s", z->err); rc_err = 1; break; }
    if (st == 0) break;
    uint64_t rec_voff = ((uint64_t)z->cur_coff << 16) | z->buf_pos;
    if (a->end_coff && z->cur_coff >= a->end_coff) break;           /* ownership rule */
    if (a->stop_voffset && rec_voff >= a->stop_voffset) break;
    if (a->max_records && r->records_seen >= a->max_records) break;
    uint8_t bs4[4];
    int64_t g = bgzf_read_exact(z, bs4, 4);
    if (g == 0) break;
    if (g < 0) { snprintf(r->err, sizeof r->err, "BAM read error: %s", z->err); rc_err = 1; break; }
    uint32_t block_size = rd_u32(bs4);
    if (block_size < 32) { snprintf(r->err, sizeof r->err, "BAM read error: block_size %u < 32", block_size); rc_err = 1; break; }
    if (block_size > rec_cap) { while (rec_cap < block_size) rec_cap *= 2; rec = (uint8_t *)realloc(rec, rec_cap); }
    if (bgzf_read_exact(z, rec, block_size) != (int64_t)block_size) { snprintf(r->err, sizeof r->err, "BAM read error: %s", z->err[0] ? z->err : "truncated record"); rc_err = 1; break; }
    r->records_seen++;

    int32_t ref_id = rd_i32(rec), pos = rd_i32(rec + 4);
    uint32_t l_read_name = rec[8], mapq = rec[9];
    uint32_t n_cigar = rd_u16(rec + 12), flag = rd_u16(rec + 14);
    uint32_t l_seq = rd_u32(rec + 16);
    int32_t next_ref = rd_i32(rec + 20), next_pos = rd_i32(rec + 24), tlen = rd_i32(rec + 28);
    size_t o_name = 32, o_cigar = o_name + l_read_name, o_seq = o_cigar + 4 * (size_t)n_cigar;
    size_t o_qual = o_seq + ((size_t)l_seq + 1) / 2, o_aux = o_qual + l_seq;
    if (o_aux > block_size) { snprintf(r->err, sizeof r->err, "BAM read error: record fields exceed block_size"); rc_err = 1; break; }
    if (ref_id < -1 || ref_id >= f->n_ref || next_ref < -1 || next_ref >= f->n_ref) { snprintf(r->err, sizeof r->err, "BAM read error: reference id out of range"); rc_err = 1; break; }

    /* alignment span: sum of M/D/N/=/X lengths */
    uint64_t span = 0;
    for (uint32_t k = 0; k < n_cigar; k++) { uint32_t w = rd_u32(rec + o_cigar + 4 * k); uint32_t op = w & 15; if (op == 0 || op == 2 || op == 3 || op == 7 || op == 8) span += w >> 4; }
    int has_start = pos >= 0;
    uint32_t start1 = (uint32_t)pos + 1;                                    /* 1-based */
    int has_end = has_start && (span > 0 || a->end_zero_span_mode == 1);
    uint32_t end1 = (uint32_t)((uint64_t)start1 + span - 1);                  /* 1-based inclusive */
    if (has_start && span == 0 && a->end_zero_span_mode == 1) end1 = (uint32_t)pos; /* RecordBuf rule: start + 0 - 1 */

    if (a->region_mode == 1) {           /* physical_exec.rs:1275-1344 */
      if (!has_start) continue;
      if (ref_id != a->region_ref) continue;
      if (a->region_start && start1 < (uint64_t)a->region_start) continue;
      if (a->region_end && start1 > (uint64_t)a->region_end) continue;
      if (!eval_filters(a, ref_id >= 0 ? f->ref_names[ref_id] : NULL, has_start, a->zero_based ? start1 - 1 : start1, has_end, end1, mapq, flag)) continue;
    } else if (a->region_mode == 2) {    /* :1131-1258 per-reference unmapped tail: skip until the reference is seen, stop after it */
      if (ref_id != a->region_ref) { if (seen_target) break; continue; }
      seen_target = 1;
      if (has_start) continue;
      if (!eval_filters(a, f->ref_names[ref_id], 0, 0, 0, 0, mapq, flag)) continue;
    } else if (a->region_mode == 3) {    /* :1038-1129 "*" partition */
      if (ref_id != -1 || has_start) continue;
      if (!eval_filters(a, NULL, 0, 0, 0, 0, mapq, flag)) continue;
    }

    if (need[0]) { /* name: physical_exec.rs:413-418 */
      size_t nl = l_read_name ? l_read_name - 1 : 0;
      col_append_bytes(&all[0], rec + o_name, nl);
    }
    if (need[1]) { if (ref_id >= 0) col_append_bytes(&all[1], f->ref_names[ref_id], strlen(f->ref_names[ref_id])); else col_append_null(&all[1]); }
    if (need[2]) { if (has_start) col_append_u32(&all[2], a->zero_based ? start1 - 1 : start1); else col_append_null(&all[2]); }
    if (need[3]) { if (has_end) col_append_u32(&all[3], end1); else col_append_null(&all[3]); }
    if (need[4]) col_append_u32(&all[4], flag);
    if (need[5]) {
      if (a->binary_cigar) col_append_bytes(&all[5], rec + o_cigar, 4 * (size_t)n_cigar);
      else {
        tmp.len = 0;
        for (uint32_t k = 0; k < n_cigar; k++) {
          uint32_t w = rd_u32(rec + o_cigar + 4 * k); char t2[16];
          uint32_t op = w & 15; if (op > 8) { snprintf(r->err, sizeof r->err, "BAM read error: invalid CIGAR op %u", op); rc_err = 1; break; }
          int n = snprintf(t2, sizeof t2, "%u%c", w >> 4, CIGAR_OPS[op]);
          buf_put(&tmp, t2, (size_t)n);
        }
        if (rc_err) break;
        col_append_bytes(&all[5], tmp.p, tmp.len);
      }
    }
    if (need[6]) col_append_u32(&all[6], mapq);
    if (need[7]) { if (next_ref >= 0) col_append_bytes(&all[7], f->ref_names[next_ref], strlen(f->ref_names[next_ref])); else col_append_null(&all[7]); }
    if (need[8]) { if (next_pos >= 0) col_append_u32(&all[8], a->zero_based ? (uint32_t)next_pos : (uint32_t)next_pos + 1); else col_append_null(&all[8]); }
    if (need[9]) {
      tmp.len = 0; buf_reserve(&tmp, l_seq + 1);
      for (uint32_t k = 0; k < l_seq; k++) { uint8_t b = rec[o_seq + (k >> 1)]; tmp.p[k] = (uint8_t)SEQ_CODES[(k & 1) ? (b & 15) : (b >> 4)]; }
      col_append_bytes(&all[9], tmp.p, l_seq);
    }
    if (need[10]) {
      tmp.len = 0; buf_reserve(&tmp, 2 * (size_t)l_seq + 1);
      size_t o = 0;
      for (uint32_t k = 0; k < l_seq; k++) {  /* char::from(q + 33): code points >= 0x80 take 2 UTF-8 bytes (UNPINNED edge) */
        uint8_t q = (uint8_t)(rec[o_qual + k] + 33);
        if (q < 0x80) tmp.p[o++] = q; else { tmp.p[o++] = 0xC0 | (q >> 6); tmp.p[o++] = 0x80 | (q & 0x3F); }
      }
      col_append_bytes(&all[10], tmp.p, o);
    }
    if (need[11]) col_append_u32(&all[11], (uint32_t)tlen);
    if (any_tag) {
      if (load_tags(rec + o_aux, block_size - o_aux, a, tag_cols, populated, r->err)) { rc_err = 1; break; }
      for (int k = 0; k < a->n_tags; k++) if (!populated[k]) col_append_null(tag_cols[k]);
    }
    rows++; batch_rows++;
    if (a->batch_rows > 0 && batch_rows == a->batch_rows) { /* timing mode: yield + drop the batch */
      for (int i = 0; i < n_schema; i++) if (built[i]) col_reset(&all[i]);
      r->batches++; batch_rows = 0;
    }
  }
  if (a->batch_rows > 0 && batch_rows > 0) r->batches++;

  if (z->eof) r->next_voffset = (uint64_t)z->next_coff << 16;
  else r->next_voffset = ((uint64_t)z->cur_coff << 16) | z->buf_pos;
  r->inflated_bytes = z->inflated_bytes; r->blocks = z->blocks;
  r->n_rows = rows;

  /* batch assembly in projection order (alignment_utils.rs:316-368) */
  int n_out = a->n_proj < 0 ? n_schema : a->n_proj;
  r->cols = (Col *)calloc((size_t)n_out + 1, sizeof(Col));
  r->col_ids = (int32_t *)calloc((size_t)n_out + 1, sizeof(int32_t));
  r->n_cols = n_out;
  uint8_t *moved = (uint8_t *)calloc((size_t)n_schema, 1);
  for (int i = 0; i < n_out; i++) {
    int id = a->n_proj < 0 ? i : a->proj[i];
    r->col_ids[i] = id;
    if (id >= 0 && id < n_schema && built[id] && !moved[id]) { r->cols[i] = all[id]; moved[id] = 1; }
    else if (id >= 0 && id < n_schema && built[id]) { /* duplicate projection index: deep copy */
      Col *s = &r->cols[i - 1]; for (int j = 0; j < i; j++) if (r->col_ids[j] == id) s = &r->cols[j];
      Col *d = &r->cols[i]; memset(d, 0, sizeof *d); d->kind = s->kind; d->n = s->n; d->null_count = s->null_count;
      buf_put(&d->validity, s->validity.p, s->validity.len); buf_put(&d->offsets, s->offsets.p, s->offsets.len); buf_put(&d->data, s->data.p, s->data.len);
    } else col_init(&r->cols[i], K_Utf8);
  }
  for (int i = 0; i < n_schema; i++) if (built[i] && !moved[i]) col_free(&all[i]);
  free(moved); free(all); free(built); free(tag_cols); free(populated); free(rec); free(tmp.p); free(z);
  if (rc_err && !r->err[0]) snprintf(r->err, sizeof r->err, "scan failed");
  return r;
}

/* result accessors for ctypes */
ORC_API const char *orc_result_error(const OrcResult *r) { return r->err[0] ? r->err : NULL; }
ORC_API int64_t orc_result_rows(const OrcResult *r) { return r->n_rows; }
ORC_API int32_t orc_result_ncols(const OrcResult *r) { return r->n_cols; }
ORC_API int64_t orc_result_stat(const OrcResult *r, int which) {
  switch (which) { case 0: return r->inflated_bytes; case 1: return r->blocks; case 2: return r->batches; case 3: return r->records_seen; case 4: return (int64_t)r->next_voffset; }
  return -1;
}
ORC_API int32_t orc_col_kind(const OrcResult *r, int i) { return r->cols[i].kind; }
ORC_API int32_t orc_col_id(const OrcResult *r, int i) { return r->col_ids[i]; }
ORC_API int64_t orc_col_nulls(const OrcResult *r, int i) { return r->cols[i].null_count; }
ORC_API const uint8_t *orc_col_buf(const OrcResult *r, int i, int which, int64_t *len) {
  const Buf *b = which == 0 ? &r->cols[i].validity : which == 1 ? &r->cols[i].offsets : &r->cols[i].data;
  *len = (int64_t)b->len; return b->p;
}

/* Walks the whole record chain and returns the virtual offset of every `stride`-th record start
 * (used, untimed, to seed block-range partitions the way a BAI linear index would).             */
ORC_API int64_t orc_index_records(const OrcFile *f, int64_t stride, uint64_t *out_voff, uint64_t *out_index, int64_t cap, int64_t *n_records) {
  Bgzf *z = (Bgzf *)malloc(sizeof *z);
  bgzf_init(z, f->file, f->size, (size_t)(f->first_record_voffset >> 16));
  if (f->first_record_voffset & 0xFFFF) { bgzf_settle(z); z->buf_pos = (uint32_t)(f->first_record_voffset & 0xFFFF); }
  int64_t n = 0, k = 0; size_t last_block = (size_t)-1;
  for (;;) {
    if (bgzf_settle(z) <= 0) break;
    /* stride == 0: emit the first record start of every BGZF block */
    int emit = stride > 0 ? (n % stride == 0) : (z->cur_coff != last_block);
    if (emit && k < cap) { out_voff[k] = ((uint64_t)z->cur_coff << 16) | z->buf_pos; if (out_index) out_index[k] = (uint64_t)n; k++; }
    last_block = z->cur_coff;
    uint8_t bs4[4];
    if (bgzf_read_exact(z, bs4, 4) != 4) break;
    uint32_t bs = rd_u32(bs4);
    uint32_t left = bs;
    while (left) {  /* skip */
      if (z->buf_pos == z->buf_len && bgzf_next_block(z) <= 0) { left = 0; n--; break; }
      uint32_t take = z->buf_len - z->buf_pos; if (take > left) take = left;
      z->buf_pos += take; left -= take;
    }
    n++;
  }
  free(z);
  *n_records = n;
  return k;
}
