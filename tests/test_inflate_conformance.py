"""DEFLATE conformance of the three inflate kernels (CTA-per-member, warp-per-member, lane-group) and of the host model.

Real BGZF writers (libdeflate, igzip, htsjdk, `bgzip -l`, this project's GPU writer) make streams zlib's default strategy
never does: mixed block types, long codes, empty blocks, 50 KB payloads.  tests/deflate_craft.py builds such members
piece by piece, and zlib judges each one (it must reproduce a valid member and reject an invalid one).  The corpus:

  valid   BAM members re-encoded in rotating shapes (mixed block types, ~64 blocks per member, XLEN variants, 1-byte and
          empty members, output offsets at every residue mod 16); BAM members with extreme codes (15-bit codes, distance
          second-level tables exactly at the CTA kernel's limit and over it, a single 1-bit distance code, an empty
          distance code, HLIT 286 / HDIST 30, HCLEN 4, a repeat run crossing from lit/len into distance lengths); FASTQ
          members with 50 KB Huffman payloads, match extremes and match counts around the resolver's batch size.
  invalid one member breaking one validity rule each; CRC and ISIZE are what a lenient decoder would output, so that
          the CRC check is not what catches them.

A canonical lit/len code over at most 286 symbols needs at most n_long + 124 < 512 second-level entries with a 10-bit
root (every length class adds at most one partly filled root prefix), so only the distance table (8-bit root, 128
entries) can make the CTA kernel refuse a member: the refused members here are distance-code ones.
"""
import random
import re
import struct
import subprocess
import zlib
from pathlib import Path

import pyarrow as pa
import pytest

import deflate_craft as D
from conftest import ROOT, gen_bam

LIST_CAP = 3136      # Cfg::LIST_CAP in kernels_inflate_cta.cuh: matches the CTA kernel resolves per batch
R_LL, R_D, SUB_LL, SUB_D = 10, 8, 512, 128   # inflate_cta_core.h: root bits and second-level entries of the CTA kernel's LUTs
KERNELS = [16, 4, 8, 0]                      # debug_flags: CTA-per-member, warp-per-member, lane-group, default path
KERNEL_IDS = ["cta_per_member", "warp_per_member", "lane_group", "default"]


def _inflate_all(raw: bytes) -> bytes:
    out, off = [], 0
    while off < len(raw):
        xlen, = struct.unpack_from("<H", raw, off + 10)
        bsize, = struct.unpack_from("<H", raw, off + 16)
        out.append(zlib.decompress(raw[off + 12 + xlen:off + bsize + 1 - 8], -15))
        off += bsize + 1
    return b"".join(out)


def _plain(data: bytes) -> D.Member:
    c = zlib.compressobj(6, zlib.DEFLATED, -15)
    payload = c.compress(data) + c.flush()
    return D.Member(D.bgzf_member(payload, data), data, True, "zlib")


def _write(path: Path, members) -> Path:
    path.write_bytes(b"".join(m.raw for m in members) + D.EOF_MEMBER)
    return path


# ---------------- valid shapes ----------------
def _mixed(data):
    """V1: stored -> fixed -> dynamic -> empty stored -> dynamic (final); matches reach into earlier blocks."""
    n = len(data)
    a, b, c = n // 10, n * 3 // 10, n * 6 // 10
    f = D.Deflate().stored(data[:a]).fixed(D.tokenize(data, a, b)).dynamic(D.tokenize(data, b, c)).stored(b"")
    return D.member(f.dynamic(D.tokenize(data, c), final=True), "mixed")


def _headers(data):
    """V2: ~64 small dynamic blocks, EOB-only dynamic and fixed blocks, sync-flush style empty stored blocks."""
    f, n = D.Deflate(), len(data)
    step = max(1, n // 56)
    for k, i in enumerate(range(0, n, step)):
        f.dynamic(D.tokenize(data, i, min(n, i + step)))
        if k % 8 == 3:
            f.dynamic([]).fixed([]).stored(b"")
    return D.member(f.dynamic([], final=True), "headers")


def _xlen(data, k):
    """V7: the payload at every offset mod 16 (an extra subfield of 4 + k bytes before or after BC)."""
    f = D.Deflate().dynamic(D.tokenize(data), final=True)
    sf = D.subfield(4 + k)
    return D.member(f, f"xlen{k}", extra_before=sf if k % 2 else b"", extra_after=b"" if k % 2 else sf)


def _tiny(data):
    return D.member(D.Deflate().fixed(list(data), final=True), "tiny")


def _empty_members():
    """V7: valid empty members (a fixed block with only EOB = `03 00`, and an empty stored block)."""
    return [D.member(D.Deflate().fixed([], final=True), "empty fixed"), D.member(D.Deflate().stored(b"", final=True), "empty stored")]


def _shaped_bam(stream: bytes):
    members, pos, k = [], 0, 0
    sizes = [1] * 16 + [65536, 40000, 777, 23456, 65536, 5000, 12345, 3, 65536, 30001, 1, 60000]
    while pos < len(stream):
        n = sizes[k % len(sizes)]
        data = stream[pos:pos + n]
        kind = k % 4 if k >= 16 else 4
        members.append(_mixed(data) if kind == 0 else _headers(data) if kind == 1 else _xlen(data, k % 16) if kind == 2 else
                       D.member(D.Deflate().dynamic(D.tokenize(data), final=True), "dynamic") if kind == 3 else _tiny(data))
        if k % 5 == 2:
            members += _empty_members()
        pos += len(data)
        k += 1
    return members


def _used(tokens):
    fl, fd = D.Deflate.freqs(tokens)
    return [s for s in range(286) if fl[s]], [s for s in range(30) if fd[s]], fl, fd


def _tail(used, freq, n, lens, spare_order):
    """Assigns the long lengths `lens` to the least frequent used symbols first (so that the data decodes through the
    second level), then to unused ones."""
    order = sorted(used, key=lambda s: (freq[s], s)) + [s for s in spare_order if s not in used]
    return dict(zip(order, lens))


def _codes_member(data, shape):
    """V4 shapes; returns (member, refused by the CTA kernel)."""
    if shape == 2:                                   # a single distance code of length 1: every match has distance 1
        toks = D.tokenize(data, dist=1)
        _, ud, _, _ = _used(toks)
        assert ud == [0]
        return D.member(D.Deflate().dynamic(toks, d=[1], final=True), "one 1-bit distance code"), False
    if shape == 3:                                   # empty distance code (HDIST = 1, length 0), literal-only block
        return D.member(D.Deflate().dynamic(D.tokenize(data, literal_only=True), d=[0], hdist=1, final=True), "empty distance code"), False
    if shape == 5:                                   # HCLEN = 4 (8 code-length codes: 16 17 18 0 8 7 9 6), lengths 8 and 9 only
        toks = D.tokenize(data, literal_only=True)
        ll = [8] * 254 + [9] * 4
        f = D.Deflate().dynamic(toks, ll=ll, d=[0], hlit=258, hdist=1, hclen=8, final=True)
        return D.member(f, "HCLEN 4"), False
    toks = D.tokenize(data)
    ul, ud, fl, fd = _used(toks)
    if shape in (0, 1):                              # 15-bit lit/len codes; distance second level at the limit / just over it
        ll = D.fill_lengths(286, _tail(ul, fl, 286, [11, 12, 13, 14, 15, 15], range(285, -1, -1)), ul, R_LL)
        dl = D.fill_lengths(30, _tail(ud, fd, 30, ([9] if shape == 0 else [9, 9, 9]) + [10, 11, 12, 13, 14, 15, 15], range(29, -1, -1)), ud, R_D)
        assert D.sub_usage(dl, R_D) == (SUB_D if shape == 0 else SUB_D + 2) and D.sub_usage(ll, R_LL) <= SUB_LL
        return D.member(D.Deflate().dynamic(toks, ll=ll, d=dl, final=True), f"distance sub-table {D.sub_usage(dl, R_D)}"), shape == 1
    # shape 4: HLIT 286, HDIST 30, and a repeat run of 9s that crosses from the lit/len lengths into the distance lengths
    ll = D.fill_lengths(286, {s: 9 for s in range(281, 286)}, [s for s in ul if s < 281], R_LL)
    dl = D.fill_lengths(30, {s: 9 for s in range(4)}, [s for s in ud if s >= 4], R_D)
    f = D.Deflate().dynamic(toks, ll=ll, d=dl, hlit=286, hdist=30, final=True)
    i, crossed = 0, False
    for s, xv, _ in f.ops:
        run = xv + 3 if s == 16 else xv + 3 if s == 17 else xv + 11 if s == 18 else 1
        crossed |= s == 16 and i < 286 < i + run
        i += run
    assert crossed and i == 316
    return D.member(f, "HLIT 286 / HDIST 30"), False


def _codes_bam(stream: bytes):
    """The first member carries the header as zlib writes it; then V4 shapes in turn, a refused member every sixth."""
    members, refused, pos, k = [_plain(stream[:65280])], 0, 65280, 0
    while pos < len(stream):
        data = stream[pos:pos + 65280]
        m, r = _codes_member(data, k % 6)
        m.refused = r
        members.append(m)
        refused += r
        pos += len(data)
        k += 1
    return members, refused


def _random_records(rng, n_bytes, alphabet, name="r"):
    out, i = [], 0
    while sum(map(len, out)) < n_bytes:
        L = rng.randint(50, 300)
        out.append(f"@{name}{i}\n".encode() + bytes(rng.choice(alphabet) for _ in range(L)) + b"\n+\n" + bytes(rng.choice(alphabet) for _ in range(L)) + b"\n")
        i += 1
    return b"".join(out)


def _exact_records(rng, n, alphabet, name):
    """Whole FASTQ records of exactly n bytes in all (random ones, then a filler record)."""
    recs = b""
    while True:
        nxt = _random_records(rng, 1, alphabet, f"{name}{len(recs)}_")
        if len(recs) + len(nxt) > n - 64:
            return recs + _filler(n - len(recs), name)
        recs += nxt


def _filler(n, tag):
    """A FASTQ record of exactly n bytes (n >= 12)."""
    k = (n - 6 - len(tag)) // 2
    name = tag + "x" * ((n - 6 - len(tag)) % 2)
    rec = f"@{name}\n".encode() + b"C" * k + b"\n+\n" + b"#" * k + b"\n"
    assert len(rec) == n
    return rec


def _fastq_members(rng):
    """FASTQ text and its members (V3, V5, V6, repeat-code maxima)."""
    printable = bytes(range(33, 127))
    pieces, members = [], []

    def add(m):
        members.append(m)
        pieces.append(m.data)

    # V3: ISIZE 65536, one literal-only dynamic block of > 48 KB payload
    text = _exact_records(rng, 65536, printable, "big")
    add(D.member(D.Deflate().dynamic(D.tokenize(text, literal_only=True), final=True), "big literal block"))
    # V3: a dynamic block header inside the last 1 KB in front of the first reload point of the 24 KB payload buffer
    text = _exact_records(rng, 65536, printable, "reload")
    n = 29000
    for _ in range(4):
        f = D.Deflate().dynamic(D.tokenize(text, 0, n, literal_only=True))
        n += int((23900 - f.bw.bitpos / 8) * 8 / 6.6)
    f = D.Deflate().dynamic(D.tokenize(text, 0, n, literal_only=True)).dynamic(D.tokenize(text, n, literal_only=True), final=True)
    add(D.member(f, "header before reload"))
    # V5: periods 1..17 with len >> dist, lengths 3 and 258 (as 285 and as 284 + 31), chains of matches
    recs = b"".join(f"@p{p}\n".encode() + (bytes(rng.choice(b"ACGT") for _ in range(p)) * (700 // p + 1))[:700] + b"\n+\n" + b"I" * 700 + b"\n" for p in range(1, 18))
    toks = D.tokenize(recs, 0, 4000, max_len=3) + D.tokenize(recs, 4000)
    k = 0
    for i, t in enumerate(toks):
        if not isinstance(t, int) and t[0] == 258:
            k += 1
            if k % 2:
                toks[i] = (258, t[1], "284")
    assert k >= 4 and any(not isinstance(t, int) and t[0] == 3 for t in toks)
    add(D.member(D.Deflate().dynamic(toks[:len(toks) // 2]).fixed(toks[len(toks) // 2:], final=True), "match extremes"))
    # V5: distance exactly 32768, and a distance equal to the bytes produced so far (the match reads member byte 0)
    r0 = _random_records(rng, 10, b"ACGT", "first")
    r2 = b"@far\n" + bytes(rng.choice(b"ACGT") for _ in range(150)) + b"\n+\n" + b"F" * 150 + b"\n"
    text = r0 + _filler(1000, "a") + r0 + _filler(2000, "b") + r2
    q = len(text) - len(r2)
    text += _filler(32768 - len(r2), "c") + r2
    p0 = len(r0) + 1000
    toks = (D.tokenize(text, 0, p0) + D.tokenize(text, p0, p0 + len(r0), dist=p0) + D.tokenize(text, p0 + len(r0), q + 32768)
            + D.tokenize(text, q + 32768, dist=32768))
    assert any(not isinstance(t, int) and t[1] == p0 for t in toks) and any(not isinstance(t, int) and t[1] == 32768 for t in toks)
    add(D.member(D.Deflate().dynamic(toks, final=True), "distance 32768 / to byte 0"))
    # code-length repeat codes at their maxima: 16 x 6, 17 x 10 (bytes 0-9), 18 x 138 (bytes above 'Z')
    text = _random_records(rng, 20000, b"ACGTNIJKLMOPQRSUVWXYZ0123456789", "R")
    toks = D.tokenize(text)
    ul = _used(toks)[0]
    ll = D.fill_lengths(286, {s: 6 for s in range(ord("I"), ord("Q"))}, [s for s in ul if not ord("I") <= s < ord("Q")], R_LL)
    f = D.Deflate().dynamic(toks, ll=ll, final=True)
    assert {(16, 3, 2), (17, 7, 3), (18, 127, 7)} <= set(f.ops), f.ops
    add(D.member(f, "repeat maxima"))
    # V6: members with LIST_CAP - 1, LIST_CAP, LIST_CAP + 1, 2 LIST_CAP + 1 matches, and a 65 536-byte member of length-3
    # matches only (after the first record's literals: 21 829, the most a FASTQ member whose lines average >= 8 bytes holds)
    rec = b"@r\n" + b"A" * 20 + b"\n+\n" + b"I" * 20 + b"\n"
    sizes = [3 * m + 3 * len(rec) for m in (LIST_CAP - 1, LIST_CAP, LIST_CAP + 1, 2 * LIST_CAP + 1)] + [65536]
    text = rec * (sum(sizes) // len(rec) + 1)
    text = text[:sum(sizes) // len(rec) * len(rec) + len(rec)]
    pos, counts = 0, []
    for m_cnt, n in zip((LIST_CAP - 1, LIST_CAP, LIST_CAP + 1, 2 * LIST_CAP + 1, None), sizes):
        toks = D.tokenize(text[pos:pos + n], max_len=3, max_matches=m_cnt)
        counts.append(sum(1 for t in toks if not isinstance(t, int)))
        add(D.member(D.Deflate().dynamic(toks, final=True), f"{counts[-1]} matches"))
        pos += n
    assert counts[:4] == [LIST_CAP - 1, LIST_CAP, LIST_CAP + 1, 2 * LIST_CAP + 1] and counts[4] >= (65536 - len(rec)) // 3, counts
    while pos < len(text):
        add(_plain(text[pos:pos + 65280]))
        pos += 65280
    return members


# ---------------- invalid shapes ----------------
def _invalid_members(chunk: bytes):
    """{label: member}: one validity rule broken per member; CRC / ISIZE as a lenient decoder would output."""
    toks = D.tokenize(chunk)
    ul, ud, fl, fd = _used(toks)
    ll, dl = D.huffman_lengths(fl, 15), D.huffman_lengths(fd, 15)
    out = {}

    def bad(label, f, **kw):
        out[label] = D.member(f, label, valid=False, **kw)

    def mod(lengths, k, top=15):                     # over-subscribed (k = -1: one code a bit shorter) / incomplete (+1: longer)
        L = list(lengths)
        s = max((i for i, v in enumerate(L) if (v and v < top if k > 0 else v > 1)), key=lambda i: (L[i], i))
        L[s] += k
        return L

    bad("btype3", D.Deflate().raw_bits(0b111, 3).raw_bits(0, 16), crc=0, isize=100)
    bad("stored len nlen", D.Deflate().stored(chunk[:500], final=True, nlen=0x1234))
    bad("stored len past payload", D.Deflate().stored(chunk[:100], final=True, length=3000), isize=100)
    bad("hlit 287", D.Deflate().dynamic(toks, ll=ll, d=dl, hlit=287, final=True))
    bad("hlit 288", D.Deflate().dynamic(toks, ll=ll, d=dl, hlit=288, final=True))
    bad("hdist 31", D.Deflate().dynamic(toks, ll=ll, d=dl, hdist=31, final=True))
    bad("hdist 32", D.Deflate().dynamic(toks, ll=ll, d=dl, hdist=32, final=True))
    bad("over-subscribed lit/len", D.Deflate().dynamic(toks, ll=mod(ll, -1), d=dl, final=True))
    bad("over-subscribed distance", D.Deflate().dynamic(toks, ll=ll, d=mod(dl, -1), final=True))
    bad("incomplete lit/len", D.Deflate().dynamic(toks, ll=mod(ll, 1), d=dl, final=True))
    bad("incomplete distance", D.Deflate().dynamic(toks, ll=ll, d=mod(dl, 1), final=True))
    ops = D.rle_code_lengths((ll + [0] * 286)[:max(257, max(i for i, v in enumerate(ll) if v) + 1)] + dl[:max(i for i, v in enumerate(dl) if v) + 1])
    fp = [0] * 19
    for s, _, _ in ops:
        fp[s] += 1
    pre = D.huffman_lengths(fp, 7)
    assert sum(1 for v in pre if v) >= 2
    bad("over-subscribed precode", D.Deflate().dynamic(toks, ll=ll, d=dl, pre=mod(pre, -1), final=True))
    bad("incomplete precode", D.Deflate().dynamic(toks, ll=ll, d=dl, pre=mod(pre, 1, top=7), final=True))
    bad("code 16 first", D.Deflate().dynamic(toks, ll=ll, d=dl, ops=[(16, 0, 2)] + ops[1:], final=True))
    bad("run past hlit+hdist", D.Deflate().dynamic(toks, ll=ll, d=dl, ops=ops[:-1] + [(18, 127, 7)], final=True))
    no_eob = list(ll)
    no_eob[256] = 0
    bad("no end-of-block code", D.Deflate().dynamic([t for t in toks if isinstance(t, int)][:50], ll=no_eob, d=dl, final=True))
    lit = list(chunk[:40])
    lit2 = list(chunk[40:80])                        # (a lenient decoder that drops the bad symbol outputs chunk[:80])
    bad("fixed symbol 286", D.Deflate().fixed(lit + [("ll", 286)] + lit2, final=True))
    bad("fixed symbol 287", D.Deflate().fixed(lit + [("ll", 287)] + lit2, final=True))
    bad("fixed distance 30", D.Deflate().fixed(lit + [("ll", 257), ("d", 30)] + lit2, final=True))
    bad("fixed distance 31", D.Deflate().fixed(lit + [("ll", 257), ("d", 31)] + lit2, final=True))
    bad("distance past member start (first token)", D.Deflate().fixed([(3, 1)] + lit, final=True))
    bad("distance past member start (mid-member)", D.Deflate().dynamic(lit + [(10, 41)] + lit, final=True))
    last = max(i for i, t in enumerate(toks) if not isinstance(t, int))
    f = D.Deflate().dynamic(toks[:last + 1], final=True)       # ends with a match; ISIZE ends inside it
    bad("match past ISIZE", f, crc=zlib.crc32(f.data[:-2]) & 0xffffffff, isize=len(f.data) - 2)
    bad("ISIZE larger than output", D.Deflate().dynamic(toks, final=True), isize=len(chunk) + 7)
    bad("no final block", D.Deflate().dynamic(toks[:len(toks) // 2]).stored(b""))
    out["empty member CRC != 0"] = D.member(D.Deflate().fixed([], final=True), "empty crc", valid=False, crc=0x12345678)
    f = D.Deflate().fixed(lit, final=True)
    out["empty member with bytes"] = D.member(f, "empty with bytes", valid=False, crc=zlib.crc32(f.data) & 0xffffffff, isize=0)
    return out


@pytest.fixture(scope="session")
def corpus(tmp_path_factory):
    d = tmp_path_factory.mktemp("conformance")
    src = gen_bam(d, "short", 3000, seed=21)
    stream = _inflate_all(src.read_bytes())
    shaped = _shaped_bam(stream)
    codes_src = gen_bam(d, "short", 6000, seed=22)
    codes_stream = _inflate_all(codes_src.read_bytes())
    codes, refused = _codes_bam(codes_stream)
    fq = _fastq_members(random.Random(5))
    small = gen_bam(d, "short", 300, seed=23)
    small_stream = _inflate_all(small.read_bytes())
    cut = len(small_stream) // 2
    invalid = {}
    for i, (label, m) in enumerate(_invalid_members(small_stream[cut:cut + 6000]).items()):
        # the stream goes on behind what a lenient decoder would output (trusting ISIZE), so that the record chain stays
        # intact wherever that output is the original bytes: then only the inflate checks can catch the member
        isize, = struct.unpack_from("<I", m.raw, len(m.raw) - 4)
        rest = cut + min(isize, len(m.data))
        invalid[label] = _write(d / f"invalid_{i:02d}.bam", [_plain(small_stream[:cut]), m, _plain(small_stream[rest:])])
    return {
        "src": src, "small": small,
        "valid": {"shaped": _write(d / "shaped.bam", shaped), "codes": _write(d / "codes.bam", codes), "fastq": _write(d / "crafted.fastq.bgz", fq)},
        "members": {"shaped": shaped, "codes": codes, "fastq": fq},
        "refused": refused, "invalid": invalid,
    }


@pytest.fixture(scope="session")
def inflate_sim(tmp_path_factory):
    exe = tmp_path_factory.mktemp("isim") / "inflate_sim"
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-o", str(exe), str(ROOT / "tools" / "inflate_sim.cpp"), "-lz"])
    return exe


def _oracle_table(path):
    if str(path).endswith(".bam"):
        from oracle.bam_oracle import OracleBam
        return pa.Table.from_batches([OracleBam(str(path)).scan()])
    from oracle.fastq_oracle import OracleFastq
    return pa.Table.from_batches([OracleFastq(path).scan()])


# ---------------- CPU ----------------
def test_builder_checks_every_member_with_zlib(corpus):
    members = [m for ms in corpus["members"].values() for m in ms]
    for m in members:
        m.check()
    assert sum(m.refused for m in corpus["members"]["codes"]) == corpus["refused"] > 0
    for path in corpus["invalid"].values():
        with pytest.raises(zlib.error):
            _gunzip_strict(path.read_bytes())


def _gunzip_strict(raw):
    while raw:
        d = zlib.decompressobj(31)
        d.decompress(raw)
        if not d.eof:
            raise zlib.error("truncated member")
        raw = d.unused_data


def test_corpus_shapes_are_in_the_files(corpus):
    """The shapes are asserted from the files themselves: payload sizes, ISIZE, payload offsets and output offsets."""
    def members_of(path):
        raw, off, out = path.read_bytes(), 0, []
        while off < len(raw):
            xlen, = struct.unpack_from("<H", raw, off + 10)
            x, bsize = 0, None
            while x + 4 <= xlen:
                slen, = struct.unpack_from("<H", raw, off + 12 + x + 2)
                if raw[off + 12 + x:off + 14 + x] == b"BC":
                    bsize, = struct.unpack_from("<H", raw, off + 12 + x + 4)
                x += 4 + slen
            isize, = struct.unpack_from("<I", raw, off + bsize + 1 - 4)
            out.append((off + 12 + xlen, bsize + 1 - 20 - xlen, isize))
            off += bsize + 1
        return out
    fq = members_of(corpus["valid"]["fastq"])
    assert fq[0][2] == 65536 and fq[0][1] > 48 * 1024                    # one literal-only block: several buffer reloads
    assert fq[1][2] == 65536 and fq[1][1] > 48 * 1024
    hdr = corpus["members"]["fastq"][1]
    shaped = members_of(corpus["valid"]["shaped"])
    assert {p % 16 for p, _, _ in shaped} == set(range(16))
    uoffs, u = set(), 0
    for _, _, isize in shaped:
        uoffs.add(u % 16)
        u += isize
    assert uoffs == set(range(16))
    assert sum(1 for _, _, isize in shaped if isize == 0) >= 4 and sum(1 for _, _, isize in shaped if isize == 1) >= 10
    assert hdr.label == "header before reload"


def test_reencoded_bam_equals_source_through_the_oracle(corpus):
    want = _oracle_table(corpus["src"])
    for name in ("shaped",):
        assert _oracle_table(corpus["valid"][name]).equals(want), name
    codes_src = gen_bam(corpus["src"].parent, "short", 6000, seed=22)
    assert _oracle_table(corpus["valid"]["codes"]).equals(_oracle_table(codes_src))
    assert _oracle_table(corpus["valid"]["fastq"]).num_rows > 2000           # the crafted FASTQ text is whole records


def test_oracle_rejects_every_invalid_file(corpus):
    for label, path in corpus["invalid"].items():
        with pytest.raises((RuntimeError, OSError)):
            _oracle_table(path)


def _sim(exe, path, span):
    r = subprocess.run([str(exe), str(path), "--span-bytes", str(span), "--resolve", "6", "--list-cap", str(LIST_CAP)], capture_output=True, text=True)
    m = re.search(r"members=(\d+) bad=(\d+) refused\(sub-table\)=(\d+)", r.stdout)
    assert m, r.stdout + r.stderr
    return r.returncode, [int(x) for x in m.groups()], r.stdout + r.stderr


@pytest.mark.parametrize("span", [2048, 24576])
@pytest.mark.parametrize("name", ["shaped", "codes", "fastq"])
def test_host_model_on_valid_files(corpus, inflate_sim, name, span):
    rc, (members, bad, refused), log = _sim(inflate_sim, corpus["valid"][name], span)
    assert rc == 0 and bad == 0 and members > 0, log
    assert refused == (corpus["refused"] if name == "codes" else 0), log


def test_host_model_rejects_what_zlib_rejects(corpus, inflate_sim):
    """The model (the CTA kernel's algorithm) must not accept a member zlib rejects; it did accept incomplete codes."""
    failed = []
    for label, path in corpus["invalid"].items():
        rc, (members, bad, _), log = _sim(inflate_sim, path, 24576)
        if bad:
            failed.append(label)
    assert not failed


# ---------------- GPU ----------------
def _scan(path, flags, **kw):
    import bamscan
    if str(path).endswith(".bam"):
        p = bamscan.BamTableProvider(str(path), None, True, None, False, True, 100, None, index_path="", debug_flags=flags, **kw)
        return p, p.scan(None, [], None)
    p = bamscan.FastqTableProvider(str(path), debug_flags=flags)
    return p, p.scan()


def _assert_tables_equal(got, want, ctx):
    assert got.num_rows == want.num_rows, f"{ctx}: rows {got.num_rows} != {want.num_rows}"
    assert got.schema.names == want.schema.names, ctx
    for name in want.schema.names:
        g, w = got[name].combine_chunks(), want[name].combine_chunks()
        assert g.type == w.type, f"{ctx}: column {name} type {g.type} != {w.type}"
        if not g.equals(w):
            for i in range(len(w)):
                if g[i] != w[i]:
                    raise AssertionError(f"{ctx}: column {name} row {i}: got {g[i]!r} want {w[i]!r}")
            raise AssertionError(f"{ctx}: column {name} differs (null masks?)")


@pytest.mark.gpu
@pytest.mark.parametrize("flags", KERNELS, ids=KERNEL_IDS)
@pytest.mark.parametrize("name", ["shaped", "codes", "fastq"])
def test_gpu_valid_files_equal_the_oracle(corpus, name, flags):
    path = corpus["valid"][name]
    p, plan = _scan(path, flags)
    got = plan.collect()
    _assert_tables_equal(got, _oracle_table(path), f"{name} flags={flags}")
    if name == "codes" and flags in (0, 16):
        assert plan.last_stats["inflate_retries"] == corpus["refused"]
    elif str(path).endswith(".bam"):
        assert plan.last_stats["inflate_retries"] == 0
    p.close()


@pytest.mark.gpu
@pytest.mark.parametrize("flags", KERNELS, ids=KERNEL_IDS)
def test_gpu_rejects_every_invalid_file(corpus, flags):
    import bamscan
    accepted = []
    for label, path in corpus["invalid"].items():
        p = None
        try:
            p, plan = _scan(path, flags)
            t = plan.collect()
            accepted.append(f"{label}: {t.num_rows} rows")
        except bamscan.BamScanError:
            pass
        finally:
            if p is not None:
                p.close()
    assert not accepted, accepted


@pytest.mark.gpu
@pytest.mark.parametrize("chunk", [0, 1 << 20], ids=["one_chunk", "multi_chunk"])
@pytest.mark.parametrize("nparts", [2, 3, 8])
def test_gpu_refused_members_keep_partition_seams(corpus, nparts, chunk):
    """Members the CTA kernel refuses (redone by the warp kernel) must not disturb the seam evidence of block-range
    partitions: every partition after the first that has rows starts where the chain of the one before it landed."""
    import bamscan
    path = corpus["valid"]["codes"]
    kw = {"chunk_inflated_bytes": chunk} if chunk else {}
    p1 = bamscan.BamTableProvider(str(path), None, True, None, False, True, 100, None, index_path="", **kw)
    plan1 = p1.scan(None, [], None)
    want = plan1.collect()
    p = bamscan.BamTableProvider(str(path), None, True, None, False, True, 100, None, index_path="", **kw)
    plan = p.scan(None, [], None, target_partitions=nparts, partition_mode="block_range")
    assert plan.output_partition_count() == nparts
    batches, stats = [], []
    for part in range(nparts):
        batches += list(plan.execute(part))
        stats.append(plan.last_stats)
    for part in range(1, nparts):
        if stats[part]["rows"]:
            assert stats[part]["first_record_uoff"] != 2 ** 64 - 1, f"partition {part}: no first record offset ({stats[part]})"
            assert stats[part]["first_record_uoff"] == stats[part - 1]["end_chain_uoff"], f"partition {part}: {stats[part - 1]} -> {stats[part]}"
    bamscan.check_partition_seams(stats)
    _assert_tables_equal(pa.Table.from_batches(batches, schema=want.schema), want, f"{nparts} partitions")
    assert plan1.last_stats["inflate_retries"] == corpus["refused"]
    assert sum(s["inflate_retries"] for s in stats) >= corpus["refused"]       # (extension chunks may inflate members twice)
    p.close()
    p1.close()
