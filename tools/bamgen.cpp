// tools/bamgen.cpp -- the repo's own synthetic BAM writer (SURVEY.md 8(d) workloads).
//
// Deterministic for a given (mode, reads, seed) regardless of thread count.  Writes a standard
// BAM: BGZF members of 0xff00 payload bytes (records straddle block seams, as noodles' writer
// produces), zlib raw deflate at --level (default 6), 28-byte EOF marker; optional .bai.
//
//   bamgen --mode short|long --reads N --seed S --out file.bam [--threads T] [--level 6] [--bai]
//   bamgen --fasta genome|short --reads N --seed S --out file.fa.bgz [--threads T] [--level 6]   (BGZF FASTA, see write_fasta)
//          [--unmapped K] [--flush-header] [--sam]
//
// --sam: the same records (same header text, same reads for the same arguments) as plain SAM text instead of BGZF BAM, in
// `samtools view -h` layout; `f` values would be printed with 9 significant digits, which reads back as the same f32.
//
// short: 150 bp paired-end, coordinate-sorted, 25 GRCh38 contigs, tags NM:C MD:Z AS:C XS:C RG:Z MC:Z MQ:C
// long : ~10 kb lognormal single-end reads, ~1 CIGAR op / 8 bases, tags NM:i MD:Z MM:Z ML:B:C
#include <zlib.h>

#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <string>
#include <thread>
#include <vector>

static const char* kNames[25] = {"chr1","chr2","chr3","chr4","chr5","chr6","chr7","chr8","chr9","chr10","chr11","chr12","chr13",
  "chr14","chr15","chr16","chr17","chr18","chr19","chr20","chr21","chr22","chrX","chrY","chrM"};
static const int64_t kLens[25] = {248956422,242193529,198295559,190214555,181538259,170805979,159345973,145138636,138394717,
  133797422,135086622,133275309,114364328,107043718,101991189,90338345,83257441,80373285,58617616,64444167,46709983,50818468,
  156040895,57227415,16569};

struct Rng {  // xoshiro256** seeded by splitmix64
  uint64_t s[4];
  static uint64_t sm(uint64_t& x) { uint64_t z = (x += 0x9E3779B97F4A7C15ull); z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull; z = (z ^ (z >> 27)) * 0x94D049BB133111EBull; return z ^ (z >> 31); }
  explicit Rng(uint64_t seed) { for (auto& v : s) v = sm(seed); }
  static uint64_t rotl(uint64_t x, int k) { return (x << k) | (x >> (64 - k)); }
  uint64_t next() { uint64_t r = rotl(s[1] * 5, 7) * 9, t = s[1] << 17; s[2] ^= s[0]; s[3] ^= s[1]; s[1] ^= s[2]; s[0] ^= s[3]; s[2] ^= t; s[3] = rotl(s[3], 45); return r; }
  uint32_t below(uint32_t n) { return (uint32_t)(((next() >> 32) * (uint64_t)n) >> 32); }
  double uni() { return (double)(next() >> 11) * (1.0 / 9007199254740992.0); }
  double normal() { double u1 = uni(), u2 = uni(); if (u1 < 1e-300) u1 = 1e-300; return std::sqrt(-2.0 * std::log(u1)) * std::cos(6.283185307179586 * u2); }
};

static inline void put32(std::vector<uint8_t>& b, uint32_t v) { uint8_t t[4]; memcpy(t, &v, 4); b.insert(b.end(), t, t + 4); }
static inline void put16(std::vector<uint8_t>& b, uint16_t v) { uint8_t t[2]; memcpy(t, &v, 2); b.insert(b.end(), t, t + 2); }

static int reg2bin(int64_t beg, int64_t end) {  // SAMv1 5.3
  --end;
  if (beg >> 14 == end >> 14) return (int)(((1 << 15) - 1) / 7 + (beg >> 14));
  if (beg >> 17 == end >> 17) return (int)(((1 << 12) - 1) / 7 + (beg >> 17));
  if (beg >> 20 == end >> 20) return (int)(((1 << 9) - 1) / 7 + (beg >> 20));
  if (beg >> 23 == end >> 23) return (int)(((1 << 6) - 1) / 7 + (beg >> 23));
  if (beg >> 26 == end >> 26) return (int)(((1 << 3) - 1) / 7 + (beg >> 26));
  return 0;
}

struct RecMeta { int32_t ref; int32_t beg, end; uint64_t off; uint32_t len; };  // off = offset in chunk bytes
struct Chunk { std::vector<uint8_t> bytes; std::vector<RecMeta> recs; };

struct Cigar { std::vector<uint32_t> ops; int span = 0; std::string text; };
static const char kOps[] = "MIDNSHP=X";
static void cig_push(Cigar& c, uint32_t len, int op) {
  c.ops.push_back(len << 4 | (uint32_t)op);
  if (op == 0 || op == 2 || op == 3 || op == 7 || op == 8) c.span += (int)len;
  c.text += std::to_string(len); c.text += kOps[op];
}
static Cigar short_cigar(Rng& r) {
  Cigar c; uint32_t u = r.below(100);
  if (u < 85) cig_push(c, 150, 0);
  else if (u < 95) { uint32_t k = 1 + r.below(50); if (r.below(2)) { cig_push(c, k, 4); cig_push(c, 150 - k, 0); } else { cig_push(c, 150 - k, 0); cig_push(c, k, 4); } }
  else { uint32_t b = 1 + r.below(5), a = 20 + r.below(100); if (r.below(2)) { cig_push(c, a, 0); cig_push(c, b, 1); cig_push(c, 150 - a - b, 0); } else { cig_push(c, a, 0); cig_push(c, b, 2); cig_push(c, 150 - a, 0); } }
  return c;
}

static void gen_seq(Rng& r, std::vector<uint8_t>& out, int l_seq) {
  static const uint8_t code[4] = {1, 2, 4, 8};
  int nb = (l_seq + 1) / 2; size_t base = out.size(); out.resize(base + nb);
  uint64_t bits = 0; int have = 0;
  for (int i = 0; i < nb; i++) {
    if (have < 4) { bits = r.next(); have = 64; }
    uint8_t hi = code[bits & 3], lo = code[(bits >> 2) & 3]; bits >>= 4; have -= 4;
    out[base + i] = (uint8_t)(hi << 4 | lo);
  }
  int nN = 0; double lam = l_seq * 0.001;           // 0.1 % N
  while (r.uni() < lam / (nN + 1) && nN < 8) nN++;
  for (int k = 0; k < nN; k++) { int p = (int)r.below((uint32_t)l_seq); uint8_t& b = out[base + p / 2]; b = (p & 1) ? (uint8_t)((b & 0xF0) | 15) : (uint8_t)((b & 0x0F) | 0xF0); }
  if (l_seq & 1) out[base + nb - 1] &= 0xF0;
}
static void gen_qual_binned(Rng& r, std::vector<uint8_t>& out, int l_seq) {
  size_t base = out.size(); out.resize(base + l_seq);
  for (int i = 0; i < l_seq; i += 8) {
    uint64_t v = r.next();
    for (int k = 0; k < 8 && i + k < l_seq; k++) { uint8_t t = (uint8_t)(v >> (8 * k)); out[base + i + k] = t < 5 ? 2 : t < 18 ? 11 : t < 51 ? 25 : 37; }
  }
}

static void aux_Z(std::vector<uint8_t>& b, const char* tag, const std::string& s) { b.push_back(tag[0]); b.push_back(tag[1]); b.push_back('Z'); b.insert(b.end(), s.begin(), s.end()); b.push_back(0); }
static void aux_C(std::vector<uint8_t>& b, const char* tag, uint8_t v) { b.push_back(tag[0]); b.push_back(tag[1]); b.push_back('C'); b.push_back(v); }

struct ShortRead { int64_t g; int32_t ref, pos; Cigar cig; uint16_t flag; uint8_t mapq; int frag; int which; };

struct Genome { int64_t cum[26]; int64_t total; Genome() { cum[0] = 0; for (int i = 0; i < 25; i++) cum[i + 1] = cum[i] + kLens[i]; total = cum[25]; }
  void locate(int64_t g, int32_t& ref, int32_t& pos) const { int r = (int)(std::upper_bound(cum, cum + 26, g) - cum) - 1; if (r > 24) r = 24; ref = r; pos = (int32_t)(g - cum[r]); } };

static void emit_record(Chunk& ch, int32_t ref, int32_t pos, uint8_t mapq, uint16_t flag, const Cigar& cig, int l_seq,
                        int32_t nref, int32_t npos, int32_t tlen, const std::string& name,
                        const std::vector<uint8_t>& seq, const std::vector<uint8_t>& qual, const std::vector<uint8_t>& aux) {
  std::vector<uint8_t>& b = ch.bytes; size_t start = b.size();
  uint32_t bs = 32 + (uint32_t)name.size() + 1 + 4 * (uint32_t)cig.ops.size() + (uint32_t)seq.size() + (uint32_t)qual.size() + (uint32_t)aux.size();
  int endpos = pos + (cig.span > 0 ? cig.span : 1);
  put32(b, bs); put32(b, (uint32_t)ref); put32(b, (uint32_t)pos);
  b.push_back((uint8_t)(name.size() + 1)); b.push_back(mapq); put16(b, (uint16_t)(ref >= 0 ? reg2bin(pos, endpos) : 4680));
  put16(b, (uint16_t)cig.ops.size()); put16(b, flag); put32(b, (uint32_t)l_seq);
  put32(b, (uint32_t)nref); put32(b, (uint32_t)npos); put32(b, (uint32_t)tlen);
  b.insert(b.end(), name.begin(), name.end()); b.push_back(0);
  for (uint32_t w : cig.ops) put32(b, w);
  b.insert(b.end(), seq.begin(), seq.end()); b.insert(b.end(), qual.begin(), qual.end()); b.insert(b.end(), aux.begin(), aux.end());
  ch.recs.push_back({ref, pos, endpos, (uint64_t)start, (uint32_t)(b.size() - start)});
}

static std::string md_for(Rng& r, int span, int nm) {
  if (nm == 0) return std::to_string(span);
  std::string s; int left = span; static const char B[] = "ACGT";
  for (int k = 0; k < nm && left > 1; k++) { int a = (int)r.below((uint32_t)left); s += std::to_string(a); s += B[r.below(4)]; left -= a + 1; }
  s += std::to_string(left < 0 ? 0 : left); return s;
}

// chunk c of the short-read workload: fragments [f0, f1) of F
static void gen_short_chunk(uint64_t seed, int64_t c, int64_t f0, int64_t f1, int64_t F, const Genome& G, Chunk& out) {
  Rng r(seed * 0x100000001B3ull + (uint64_t)c * 2654435761ull + 17);
  int64_t n = f1 - f0;
  int64_t g_lo = (int64_t)((__int128)G.total * f0 / F), g_hi = (int64_t)((__int128)G.total * f1 / F);
  std::vector<ShortRead> reads; reads.reserve((size_t)n * 2);
  std::vector<std::string> names((size_t)n);
  for (int64_t i = 0; i < n; i++) {
    int64_t g = (int64_t)((__int128)G.total * (f0 + i) / F) + (int64_t)r.below((uint32_t)std::max<int64_t>(1, G.total / F));
    if (g >= g_hi) g = g_hi - 1;
    if (g < g_lo) g = g_lo;
    int32_t ref, pos; G.locate(g, ref, pos);
    int64_t clen = kLens[ref];
    if (pos > clen - 160) { pos = (int32_t)std::max<int64_t>(0, clen - 160); g = G.cum[ref] + pos; }
    int insert = (int)std::lround(400 + 50 * r.normal()); if (insert < 160) insert = 160; if (insert > 800) insert = 800;
    int64_t mpos = pos + insert - 150;
    if (mpos > clen - 156) mpos = clen - 156;
    if (G.cum[ref] + mpos >= g_hi) mpos = g_hi - 1 - G.cum[ref];
    if (mpos < pos) mpos = pos;
    bool fwd_first = r.below(2) == 0; bool dup = r.below(100) == 0;
    ShortRead a, b;
    a.g = g; a.ref = ref; a.pos = pos; a.cig = short_cigar(r); a.flag = (uint16_t)((fwd_first ? 99 : 83) | (dup ? 0x400 : 0)); a.frag = (int)i; a.which = 0;
    b.g = G.cum[ref] + mpos; b.ref = ref; b.pos = (int32_t)mpos; b.cig = short_cigar(r); b.flag = (uint16_t)((fwd_first ? 147 : 163) | (dup ? 0x400 : 0)); b.frag = (int)i; b.which = 1;
    a.mapq = r.below(100) < 85 ? 60 : (uint8_t)r.below(60); b.mapq = r.below(100) < 85 ? 60 : (uint8_t)r.below(60);
    char nm[64]; int tile = 1101 + (int)r.below(1578); int pad = (int)r.below(9);
    int len = snprintf(nm, sizeof nm, "A%05u:%03u:HSYN%cDSX%c:%u:%d:%u:%u", 836u + r.below(64), 100 + r.below(900), 'A' + (int)r.below(26), '2' + (int)r.below(6), 1 + r.below(4), tile, 1000 + r.below(31000), 1000 + r.below(36000));
    std::string name(nm, (size_t)len);
    while ((int)name.size() < 28 + pad && name.size() < 36) name += (char)('0' + r.below(10));
    if (name.size() > 36) name.resize(36);
    names[(size_t)i] = name;
    reads.push_back(std::move(a)); reads.push_back(std::move(b));
  }
  std::vector<uint32_t> order(reads.size());
  for (uint32_t k = 0; k < order.size(); k++) order[k] = k;
  std::stable_sort(order.begin(), order.end(), [&](uint32_t x, uint32_t y) { return reads[x].g < reads[y].g; });
  std::vector<uint8_t> seq, qual, aux;
  out.bytes.reserve(reads.size() * 350);
  for (uint32_t k : order) {
    const ShortRead& me = reads[k]; const ShortRead& mate = reads[k ^ 1u];
    seq.clear(); qual.clear(); aux.clear();
    gen_seq(r, seq, 150); gen_qual_binned(r, qual, 150);
    int nmv = r.below(100) < 70 ? 0 : 1 + (int)r.below(5);
    aux_C(aux, "NM", (uint8_t)nmv); aux_Z(aux, "MD", md_for(r, me.cig.span, nmv));
    aux_C(aux, "AS", (uint8_t)std::max(0, 150 - 5 * nmv - (int)r.below(4))); aux_C(aux, "XS", (uint8_t)r.below(100));
    aux_Z(aux, "RG", "rg1"); aux_Z(aux, "MC", mate.cig.text); aux_C(aux, "MQ", mate.mapq);
    int32_t lo = std::min(me.pos, mate.pos), hi = std::max(me.pos + me.cig.span, mate.pos + mate.cig.span);
    int32_t tlen = hi - lo; bool leftmost = me.pos < mate.pos || (me.pos == mate.pos && me.which == 0);
    emit_record(out, me.ref, me.pos, me.mapq, me.flag, me.cig, 150, mate.ref, mate.pos, leftmost ? tlen : -tlen, names[(size_t)me.frag], seq, qual, aux);
  }
}

// chunk of the long-read workload: reads [i0, i1) of N
static void gen_long_chunk(uint64_t seed, int64_t c, int64_t i0, int64_t i1, int64_t N, const Genome& G, Chunk& out) {
  Rng r(seed * 0x100000001B3ull + (uint64_t)c * 2654435761ull + 99);
  std::vector<uint8_t> seq, qual, aux;
  static const uint16_t flags[4] = {0, 16, 256, 2048};
  const double mu = std::log(10000.0) - 0.125;   // lognormal with mean 10 kb, sigma 0.5
  for (int64_t i = i0; i < i1; i++) {
    int64_t g = (int64_t)((__int128)G.total * i / N) + (int64_t)r.below((uint32_t)std::max<int64_t>(1, G.total / N));
    int64_t g_next = (int64_t)((__int128)G.total * (i + 1) / N); if (g >= g_next) g = g_next - 1;
    int32_t ref, pos; G.locate(g, ref, pos);
    int l = (int)std::lround(std::exp(mu + 0.5 * r.normal())); if (l < 1000) l = 1000; if (l > 100000) l = 100000;
    if (kLens[ref] < 300000) l = std::min(l, 4000);
    if (pos > kLens[ref] - 2 * (int64_t)l - 10) pos = (int32_t)std::max<int64_t>(0, kLens[ref] - 2 * (int64_t)l - 10);
    Cigar cig; int q = 0, nm = 0; std::string md; int md_run = 0; static const char B[] = "ACGT";
    while (q < l && cig.ops.size() < 65000) {
      int run = 1 + (int)r.below(15); if (run > l - q) run = l - q;
      uint32_t u = r.below(100);
      if (u < 55) { cig_push(cig, (uint32_t)run, 7); q += run; md_run += run; }                       // =
      else if (u < 70) { cig_push(cig, (uint32_t)run, 0); q += run; md_run += run; }                  // M
      else if (u < 80) { int k = std::min(run, 3); cig_push(cig, (uint32_t)k, 8); q += k; nm += k; for (int t = 0; t < k; t++) { md += std::to_string(md_run); md += B[r.below(4)]; md_run = 0; } }   // X
      else if (u < 90) { int k = std::min(run, 4); cig_push(cig, (uint32_t)k, 1); q += k; nm += k; }  // I
      else { int k = std::min(run, 4); cig_push(cig, (uint32_t)k, 2); nm += k; md += std::to_string(md_run); md += '^'; for (int t = 0; t < k; t++) md += B[r.below(4)]; md_run = 0; }  // D
    }
    if (q < l) { cig_push(cig, (uint32_t)(l - q), 0); md_run += l - q; }
    md += std::to_string(md_run);
    seq.clear(); qual.clear(); aux.clear();
    gen_seq(r, seq, l);
    qual.resize((size_t)l); for (int k = 0; k < l; k++) qual[(size_t)k] = (uint8_t)(1 + r.below(50));
    aux.push_back('N'); aux.push_back('M'); aux.push_back('i'); put32(aux, (uint32_t)nm);
    aux_Z(aux, "MD", md);
    int nmod = l / 10; std::string mm = "C+m?";
    for (int k = 0; k < nmod; k++) { mm += ','; mm += std::to_string(r.below(12)); }
    mm += ';'; aux_Z(aux, "MM", mm);
    aux.push_back('M'); aux.push_back('L'); aux.push_back('B'); aux.push_back('C'); put32(aux, (uint32_t)nmod);
    for (int k = 0; k < nmod; k++) aux.push_back((uint8_t)r.below(256));
    char nmbuf[64]; int nl = snprintf(nmbuf, sizeof nmbuf, "%08x-%04x-%04x-%04x-%012llx", (uint32_t)r.next(), (uint32_t)r.below(65536), (uint32_t)r.below(65536), (uint32_t)r.below(65536), (unsigned long long)(r.next() & 0xFFFFFFFFFFFFull));
    uint8_t mapq = r.below(100) < 85 ? 60 : (uint8_t)r.below(60);
    emit_record(out, ref, pos, mapq, flags[r.below(4)], cig, l, -1, -1, 0, std::string(nmbuf, (size_t)nl), seq, qual, aux);
  }
}

// One BAM record (block_size first) -> one SAM line, '\n' included.
static void render_sam(const uint8_t* p, std::string& o) {
  auto r32 = [](const uint8_t* q) { uint32_t v; memcpy(&v, q, 4); return v; };
  auto r16 = [](const uint8_t* q) { uint16_t v; memcpy(&v, q, 2); return v; };
  const uint32_t bs = r32(p); const uint8_t* b = p + 4;
  const int32_t ref = (int32_t)r32(b), pos = (int32_t)r32(b + 4), nref = (int32_t)r32(b + 20), npos = (int32_t)r32(b + 24), tlen = (int32_t)r32(b + 28);
  const uint32_t l_name = b[8], mapq = b[9], n_cig = r16(b + 12), flag = r16(b + 14), l_seq = r32(b + 16);
  size_t k = 32;
  char t[64];
  o.append((const char*)b + k, l_name - 1); k += l_name;
  o += '\t'; o += std::to_string(flag); o += '\t'; o += ref >= 0 ? kNames[ref] : "*";
  o += '\t'; o += std::to_string(pos + 1); o += '\t'; o += std::to_string(mapq); o += '\t';
  if (!n_cig) o += '*';
  for (uint32_t c = 0; c < n_cig; c++, k += 4) { const uint32_t w = r32(b + k); o += std::to_string(w >> 4); o += "MIDNSHP=X"[w & 15]; }
  o += '\t'; o += nref < 0 ? "*" : nref == ref ? "=" : kNames[nref];
  o += '\t'; o += std::to_string(npos + 1); o += '\t'; o += std::to_string(tlen); o += '\t';
  if (!l_seq) o += '*';
  for (uint32_t i = 0; i < l_seq; i++) o += "=ACMGRSVTWYHKDBN"[(b[k + i / 2] >> ((i & 1) ? 0 : 4)) & 15];
  k += (l_seq + 1) / 2;
  o += '\t';
  bool missing = true;
  for (uint32_t i = 0; i < l_seq; i++) missing &= b[k + i] == 0xff;
  if (!l_seq || missing) o += '*'; else for (uint32_t i = 0; i < l_seq; i++) o += (char)(b[k + i] + 33);
  k += l_seq;
  while (k + 3 <= bs) {
    o += '\t'; o.append((const char*)b + k, 2); const char ty = (char)b[k + 2]; k += 3;
    switch (ty) {
      case 'A': o += ":A:"; o += (char)b[k]; k += 1; break;
      case 'c': o += ":i:"; o += std::to_string((int8_t)b[k]); k += 1; break;
      case 'C': o += ":i:"; o += std::to_string(b[k]); k += 1; break;
      case 's': o += ":i:"; o += std::to_string((int16_t)r16(b + k)); k += 2; break;
      case 'S': o += ":i:"; o += std::to_string(r16(b + k)); k += 2; break;
      case 'i': o += ":i:"; o += std::to_string((int32_t)r32(b + k)); k += 4; break;
      case 'I': o += ":i:"; o += std::to_string(r32(b + k)); k += 4; break;
      case 'f': { float f; memcpy(&f, b + k, 4); snprintf(t, sizeof t, ":f:%.9g", f); o += t; k += 4; break; }
      case 'Z': case 'H': { o += ':'; o += ty; o += ':'; const size_t n = strlen((const char*)b + k); o.append((const char*)b + k, n); k += n + 1; break; }
      default: {   // 'B'
        const char st = (char)b[k]; const uint32_t cnt = r32(b + k + 1); k += 5;
        o += ":B:"; o += st;
        for (uint32_t e = 0; e < cnt; e++) {
          o += ',';
          switch (st) {
            case 'c': o += std::to_string((int8_t)b[k]); k += 1; break;
            case 'C': o += std::to_string(b[k]); k += 1; break;
            case 's': o += std::to_string((int16_t)r16(b + k)); k += 2; break;
            case 'S': o += std::to_string(r16(b + k)); k += 2; break;
            case 'i': o += std::to_string((int32_t)r32(b + k)); k += 4; break;
            case 'I': o += std::to_string(r32(b + k)); k += 4; break;
            default: { float f; memcpy(&f, b + k, 4); snprintf(t, sizeof t, "%.9g", f); o += t; k += 4; }
          }
        }
      }
    }
  }
  o += '\n';
}

// ------------------------------------------------------------------------------------------
struct BaiRef { std::map<uint32_t, std::vector<std::pair<uint64_t, uint64_t>>> bins; std::vector<uint64_t> lin; uint64_t beg = ~0ull, end = 0, n_mapped = 0, n_unmapped = 0; };

static size_t deflate_block(const uint8_t* src, size_t n, int level, uint8_t* dst /* >= 65536+64 */) {
  static const uint8_t hdr[12] = {0x1f, 0x8b, 8, 4, 0, 0, 0, 0, 0, 0xff, 6, 0};
  memcpy(dst, hdr, 12); dst[12] = 'B'; dst[13] = 'C'; dst[14] = 2; dst[15] = 0;
  z_stream s; memset(&s, 0, sizeof s);
  deflateInit2(&s, level, Z_DEFLATED, -15, 8, Z_DEFAULT_STRATEGY);
  s.next_in = (Bytef*)src; s.avail_in = (uInt)n; s.next_out = dst + 18; s.avail_out = 65536 + 64 - 18 - 8;
  int rc = deflate(&s, Z_FINISH); size_t clen = s.total_out; deflateEnd(&s);
  if (rc != Z_STREAM_END) { fprintf(stderr, "deflate failed\n"); exit(2); }
  size_t total = 18 + clen + 8; uint16_t bsize = (uint16_t)(total - 1); memcpy(dst + 16, &bsize, 2);
  uint32_t crc = (uint32_t)crc32(crc32(0, nullptr, 0), src, (uInt)n), isz = (uint32_t)n;
  memcpy(dst + 18 + clen, &crc, 4); memcpy(dst + 18 + clen + 4, &isz, 4);
  return total;
}

// BGZF FASTA of one of two shapes, members of exactly 0xff00 inflated bytes + the EOF marker.
//   genome: the 25 records of kNames / kLens (about 3.1 Gb), 60-column lines, runs of lower case (soft-masked) and of N;
//   short:  N records of 300 residues, even records on one line, odd ones wrapped at 60 columns.
static int write_fasta(const std::string& shape, const std::string& out, int64_t N, uint64_t seed, int threads, int level) {
  const bool genome = shape == "genome";
  if (!genome && shape != "short") { fprintf(stderr, "--fasta genome|short\n"); return 1; }
  const int64_t units = genome ? 25 : N, per = genome ? 1 : 65536, n_pieces = (units + per - 1) / per;
  std::vector<std::string> piece((size_t)n_pieces);
  std::vector<std::thread> th;
  for (int t = 0; t < threads; t++) th.emplace_back([&, t]() {
    for (int64_t c = t; c < n_pieces; c += threads) {
      Rng r(seed * 1000003ull + (uint64_t)c);
      std::string& o = piece[(size_t)c];
      for (int64_t u = c * per; u < std::min(units, (c + 1) * per); u++) {
        const int64_t len = genome ? kLens[u] : 300;
        o += genome ? std::string(">") + kNames[u] + " synthetic chromosome " + std::to_string(u + 1) + " len=" + std::to_string(len) + "\n"
                    : ">seq" + std::to_string(u) + ((u % 3) ? " sample=" + std::to_string(r.below(1000)) : std::string()) + "\n";
        const int64_t width = (genome || (u & 1)) ? 60 : len;
        o.reserve(o.size() + (size_t)(len + len / 60 + 2));
        int64_t run = 0; char kind = 'U';                // U upper, l lower, N
        for (int64_t i = 0; i < len; i += width) {
          const int64_t w = std::min(width, len - i);
          for (int64_t k = 0; k < w; k++) {
            if (run == 0) { const uint32_t x = r.below(100); kind = x < 70 ? 'U' : x < 95 ? 'l' : 'N'; run = 1 + r.below(kind == 'N' ? 2000 : 400); }
            run--;
            static const char up[4] = {'A', 'C', 'G', 'T'}, lo[4] = {'a', 'c', 'g', 't'};
            o += kind == 'N' ? 'N' : kind == 'U' ? up[r.next() >> 62] : lo[r.next() >> 62];
          }
          o += '\n';
        }
      }
    } });
  for (auto& x : th) x.join();
  FILE* fp = fopen(out.c_str(), "wb"); if (!fp) { perror("open"); return 1; }
  const size_t P = 0xff00;
  std::string pend;
  uint64_t inflated = 0, compressed = 0, blocks = 0;
  auto flush = [&](bool final) {
    const size_t nb = pend.size() / P, tail = pend.size() - nb * P, total = nb + ((final && tail) ? 1 : 0);
    std::vector<std::vector<uint8_t>> comp(total);
    std::vector<std::thread> ft;
    for (int t = 0; t < threads; t++) ft.emplace_back([&, t]() {
      std::vector<uint8_t> tmp(65536 + 64);
      for (size_t b = (size_t)t; b < total; b += (size_t)threads) { const size_t c = deflate_block((const uint8_t*)pend.data() + b * P, b < nb ? P : tail, level, tmp.data()); comp[b].assign(tmp.begin(), tmp.begin() + (long)c); } });
    for (auto& x : ft) x.join();
    for (auto& cb : comp) { if (fwrite(cb.data(), 1, cb.size(), fp) != cb.size()) { perror("write"); exit(2); } compressed += cb.size(); blocks++; }
    const size_t used = std::min(pend.size(), total * P);
    inflated += used; pend.erase(0, used);
  };
  for (auto& x : piece) { pend += x; std::string().swap(x); if (pend.size() >= (256u << 20)) flush(false); }
  flush(true);
  static const uint8_t eof_marker[28] = {0x1f, 0x8b, 8, 4, 0, 0, 0, 0, 0, 0xff, 6, 0, 0x42, 0x43, 2, 0, 0x1b, 0, 3, 0, 0, 0, 0, 0, 0, 0, 0, 0};
  fwrite(eof_marker, 1, 28, fp); fclose(fp);
  printf("{\"fasta\": \"%s\", \"records\": %lld, \"seed\": %llu, \"compressed_bytes\": %llu, \"inflated_bytes\": %llu, \"blocks\": %llu, \"level\": %d}\n",
         shape.c_str(), (long long)units, (unsigned long long)seed, (unsigned long long)(compressed + 28), (unsigned long long)inflated, (unsigned long long)blocks + 1, level);
  return 0;
}

int main(int argc, char** argv) {
  std::string mode = "short", out; int64_t N = 1000000; uint64_t seed = 1; int threads = (int)std::thread::hardware_concurrency(); int level = 6; bool bai = false; int64_t n_unmapped = 0; bool sam = false; std::string fasta;
  for (int i = 1; i < argc; i++) {
    std::string a = argv[i];
    auto nxt = [&]() { if (i + 1 >= argc) { fprintf(stderr, "missing value for %s\n", a.c_str()); exit(1); } return std::string(argv[++i]); };
    if (a == "--mode") mode = nxt(); else if (a == "--reads") N = atoll(nxt().c_str()); else if (a == "--seed") seed = strtoull(nxt().c_str(), 0, 10);
    else if (a == "--out") out = nxt(); else if (a == "--threads") threads = atoi(nxt().c_str()); else if (a == "--level") level = atoi(nxt().c_str());
    else if (a == "--bai") bai = true; else if (a == "--unmapped") n_unmapped = atoll(nxt().c_str()); else if (a == "--sam") sam = true;
    else if (a == "--fasta") fasta = nxt();
    else { fprintf(stderr, "unknown arg %s\n", a.c_str()); return 1; }
  }
  if (out.empty() || N <= 0) { fprintf(stderr, "usage: bamgen --mode short|long --reads N --seed S --out f.bam [--threads T] [--level L] [--bai] [--unmapped K] [--sam]\n"); return 1; }
  if (sam && bai) { fprintf(stderr, "--bai needs BAM output\n"); return 1; }
  if (threads < 1) threads = 1;
  if (!fasta.empty()) return write_fasta(fasta, out, N, seed, threads, level);
  bool is_long = mode == "long";
  if (!is_long && (N & 1)) N++;
  Genome G;
  FILE* fp = fopen(out.c_str(), "wb"); if (!fp) { perror("open"); return 1; }

  std::string text = "@HD\tVN:1.6\tSO:coordinate\n";
  for (int i = 0; i < 25; i++) text += std::string("@SQ\tSN:") + kNames[i] + "\tLN:" + std::to_string(kLens[i]) + "\n";
  text += "@RG\tID:rg1\tSM:sample1\tPL:ILLUMINA\tLB:lib1\tPU:unit1\n";
  text += "@PG\tID:bamgen\tPN:bamgen\tVN:1.0\tCL:bamgen --mode " + mode + " --reads " + std::to_string(N) + " --seed " + std::to_string(seed) + "\n";
  if (sam) {
    // the same records as text, rendered in parallel per chunk, written in order
    if (fwrite(text.data(), 1, text.size(), fp) != text.size()) { perror("write"); return 2; }
    const int64_t units = is_long ? N : N / 2, per_chunk = is_long ? 512 : 16384, n_chunks = (units + per_chunk - 1) / per_chunk, group = (int64_t)threads * 2;
    for (int64_t c0 = 0; c0 < n_chunks; c0 += group) {
      const int64_t c1 = std::min(n_chunks, c0 + group);
      std::vector<std::string> txt((size_t)(c1 - c0));
      std::vector<std::thread> th;
      for (int t = 0; t < threads; t++) th.emplace_back([&, t]() {
        for (int64_t c = c0 + t; c < c1; c += threads) {
          Chunk ch;
          const int64_t u0 = c * per_chunk, u1 = std::min(units, u0 + per_chunk);
          if (is_long) gen_long_chunk(seed, c, u0, u1, units, G, ch); else gen_short_chunk(seed, c, u0, u1, units, G, ch);
          std::string& o = txt[(size_t)(c - c0)];
          o.reserve(ch.bytes.size() * 2);
          for (auto& r : ch.recs) render_sam(ch.bytes.data() + r.off, o);
        } });
      for (auto& t : th) t.join();
      for (auto& o : txt) if (fwrite(o.data(), 1, o.size(), fp) != o.size()) { perror("write"); return 2; }
    }
    if (n_unmapped > 0) { fprintf(stderr, "--unmapped needs BAM output\n"); return 1; }
    fclose(fp);
    return 0;
  }
  std::vector<uint8_t> pend;     // inflated stream bytes not yet written; pend[0] is at absolute offset pend_abs
  uint64_t pend_abs = 0;
  pend.insert(pend.end(), {'B', 'A', 'M', 1}); put32(pend, (uint32_t)text.size()); pend.insert(pend.end(), text.begin(), text.end());
  put32(pend, 25);
  for (int i = 0; i < 25; i++) { put32(pend, (uint32_t)strlen(kNames[i]) + 1); pend.insert(pend.end(), kNames[i], kNames[i] + strlen(kNames[i]) + 1); put32(pend, (uint32_t)kLens[i]); }

  const size_t P = 0xff00;        // every block but the last carries exactly P payload bytes
  std::vector<uint64_t> block_coff;   // compressed offset of block b; block_coff[n_blocks] = end of file so far
  block_coff.push_back(0);
  uint64_t n_records = 0, n_no_coor = 0;
  std::vector<BaiRef> bref(25);
  struct PendRec { int32_t ref, beg, end; uint64_t abs; uint32_t len; };
  std::vector<PendRec> prec; size_t prec_head = 0;

  auto voff = [&](uint64_t abs) { size_t b = (size_t)(abs / P); return (block_coff[b] << 16) | (abs % P); };
  auto index_ready = [&](uint64_t written_abs) {
    while (prec_head < prec.size() && prec[prec_head].abs + prec[prec_head].len <= written_abs) {
      const PendRec& p = prec[prec_head++];
      if (p.ref < 0) { n_no_coor++; continue; }
      uint64_t v0 = voff(p.abs), v1 = voff(p.abs + p.len);
      BaiRef& R = bref[(size_t)p.ref];
      auto& ch = R.bins[(uint32_t)reg2bin(p.beg, p.end)];
      if (!ch.empty() && (ch.back().second == v0 || ch.back().second >> 16 == v0 >> 16)) ch.back().second = v1; else ch.push_back({v0, v1});
      size_t w0 = (size_t)(p.beg >> 14), w1 = (size_t)((p.end - 1) >> 14);
      if (R.lin.size() <= w1) R.lin.resize(w1 + 1, 0);
      for (size_t w = w0; w <= w1; w++) if (R.lin[w] == 0) R.lin[w] = v0;
      R.beg = std::min(R.beg, v0); R.end = std::max(R.end, v1); R.n_mapped++;
    }
    if (prec_head > (1u << 20)) { prec.erase(prec.begin(), prec.begin() + (long)prec_head); prec_head = 0; }
  };
  auto flush_blocks = [&](bool final) {
    size_t nb = pend.size() / P, tail = pend.size() - nb * P;
    size_t total_blocks = nb + ((final && tail) ? 1 : 0);
    if (!total_blocks) return;
    std::vector<std::vector<uint8_t>> comp(total_blocks);
    std::vector<std::thread> th;
    for (int t = 0; t < threads; t++) th.emplace_back([&, t]() {
      std::vector<uint8_t> tmp(65536 + 64);
      for (size_t b = (size_t)t; b < total_blocks; b += (size_t)threads) {
        size_t c = deflate_block(pend.data() + b * P, b < nb ? P : tail, level, tmp.data());
        comp[b].assign(tmp.begin(), tmp.begin() + (long)c);
      } });
    for (auto& t : th) t.join();
    for (size_t b = 0; b < total_blocks; b++) { if (fwrite(comp[b].data(), 1, comp[b].size(), fp) != comp[b].size()) { perror("write"); exit(2); } block_coff.push_back(block_coff.back() + comp[b].size()); }
    size_t consumed = std::min(pend.size(), total_blocks * P);
    pend_abs += consumed;
    pend.erase(pend.begin(), pend.begin() + (long)consumed);
    if (bai) index_ready(pend_abs);
  };

  const int64_t units = is_long ? N : N / 2;
  const int64_t per_chunk = is_long ? 512 : 16384;
  const int64_t n_chunks = (units + per_chunk - 1) / per_chunk;
  const int64_t group = (int64_t)threads * 2;
  for (int64_t c0 = 0; c0 < n_chunks; c0 += group) {
    int64_t c1 = std::min(n_chunks, c0 + group);
    std::vector<Chunk> chunks((size_t)(c1 - c0));
    std::vector<std::thread> th;
    for (int t = 0; t < threads; t++) th.emplace_back([&, t]() {
      for (int64_t c = c0 + t; c < c1; c += threads) {
        int64_t u0 = c * per_chunk, u1 = std::min(units, u0 + per_chunk);
        if (is_long) gen_long_chunk(seed, c, u0, u1, units, G, chunks[(size_t)(c - c0)]);
        else gen_short_chunk(seed, c, u0, u1, units, G, chunks[(size_t)(c - c0)]);
      } });
    for (auto& t : th) t.join();
    for (auto& ch : chunks) {
      uint64_t base = pend_abs + pend.size();
      pend.insert(pend.end(), ch.bytes.begin(), ch.bytes.end());
      n_records += ch.recs.size();
      if (bai) for (auto& r : ch.recs) prec.push_back({r.ref, r.beg, r.end, base + r.off, r.len});
    }
    flush_blocks(false);
  }
  if (n_unmapped > 0) {   // unplaced unmapped tail (refID -1, pos -1)
    Rng r(seed ^ 0xABCDEF); Chunk ch; std::vector<uint8_t> seq, qual, aux; Cigar none;
    for (int64_t i = 0; i < n_unmapped; i++) {
      seq.clear(); qual.clear(); aux.clear(); gen_seq(r, seq, 150); gen_qual_binned(r, qual, 150); aux_Z(aux, "RG", "rg1");
      char nm[48]; int nl = snprintf(nm, sizeof nm, "UNMAPPED:%lld:%u", (long long)i, r.below(100000));
      emit_record(ch, -1, -1, 0, (uint16_t)((i & 1) ? 141 : 77), none, 150, -1, -1, 0, std::string(nm, (size_t)nl), seq, qual, aux);
    }
    uint64_t base = pend_abs + pend.size();
    pend.insert(pend.end(), ch.bytes.begin(), ch.bytes.end()); n_records += ch.recs.size();
    if (bai) for (auto& rr : ch.recs) prec.push_back({-1, -1, 0, base + rr.off, rr.len});
  }
  flush_blocks(true);
  uint64_t inflated_total = pend_abs;
  static const uint8_t eof_marker[28] = {0x1f, 0x8b, 8, 4, 0, 0, 0, 0, 0, 0xff, 6, 0, 0x42, 0x43, 2, 0, 0x1b, 0, 3, 0, 0, 0, 0, 0, 0, 0, 0, 0};
  fwrite(eof_marker, 1, 28, fp); fclose(fp);
  uint64_t comp_total = block_coff.back() + 28;

  if (bai) {
    FILE* fi = fopen((out + ".bai").c_str(), "wb"); if (!fi) { perror("bai"); return 1; }
    auto w32 = [&](uint32_t v) { fwrite(&v, 4, 1, fi); }; auto w64 = [&](uint64_t v) { fwrite(&v, 8, 1, fi); };
    fwrite("BAI\1", 1, 4, fi); w32(25);
    for (auto& R : bref) {
      bool any = R.n_mapped > 0;
      w32((uint32_t)R.bins.size() + (any ? 1 : 0));
      for (auto& kv : R.bins) { w32(kv.first); w32((uint32_t)kv.second.size()); for (auto& c : kv.second) { w64(c.first); w64(c.second); } }
      if (any) { w32(37450); w32(2); w64(R.beg); w64(R.end); w64(R.n_mapped); w64(R.n_unmapped); }
      for (long l = (long)R.lin.size() - 2; l >= 0; --l) if (R.lin[(size_t)l] == 0) R.lin[(size_t)l] = R.lin[(size_t)l + 1];
      w32((uint32_t)R.lin.size()); for (uint64_t v : R.lin) w64(v);
    }
    w64(n_no_coor); fclose(fi);
  }
  printf("{\"mode\": \"%s\", \"reads\": %llu, \"seed\": %llu, \"compressed_bytes\": %llu, \"inflated_bytes\": %llu, \"blocks\": %llu, \"level\": %d}\n",
         mode.c_str(), (unsigned long long)n_records, (unsigned long long)seed, (unsigned long long)comp_total, (unsigned long long)inflated_total,
         (unsigned long long)(block_coff.size() - 1), level);
  return 0;
}
