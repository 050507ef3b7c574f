"""DEFLATE (RFC 1951) streams and BGZF members built piece by piece, for the inflate conformance tests.

Plain Python: a bit writer, canonical codes from given lengths, stored / fixed / dynamic block emitters over a token list
(literal bytes and (length, distance) matches), a greedy LZ77 tokenizer with a few knobs and a BGZF member writer.
zlib stays the judge of validity: `Member.check()` asserts that a member built as valid inflates (gzip, CRC and ISIZE
checked) to exactly the bytes the tokens describe, and that a member built as invalid makes zlib raise.
"""
import heapq
import struct
import zlib

CLC_ORDER = [16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15]
LBASE = [3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 15, 17, 19, 23, 27, 31, 35, 43, 51, 59, 67, 83, 99, 115, 131, 163, 195, 227, 258]
LEXT = [0, 0, 0, 0, 0, 0, 0, 0, 1, 1, 1, 1, 2, 2, 2, 2, 3, 3, 3, 3, 4, 4, 4, 4, 5, 5, 5, 5, 0]
DBASE = [1, 2, 3, 4, 5, 7, 9, 13, 17, 25, 33, 49, 65, 97, 129, 193, 257, 385, 513, 769, 1025, 1537, 2049, 3073, 4097, 6145,
         8193, 12289, 16385, 24577]
DEXT = [0, 0, 0, 0, 1, 1, 2, 2, 3, 3, 4, 4, 5, 5, 6, 6, 7, 7, 8, 8, 9, 9, 10, 10, 11, 11, 12, 12, 13, 13]
FIXED_LL = [8] * 144 + [9] * 112 + [7] * 24 + [8] * 8
FIXED_D = [5] * 32


def len_code(n, long_258=False):
    """(symbol, extra value, extra bits) of match length n; long_258 writes 258 as symbol 284 + 31 (zlib accepts it)."""
    if n == 258 and long_258:
        return 284, 31, 5
    s = max(i for i in range(29) if LBASE[i] <= n)
    return 257 + s, n - LBASE[s], LEXT[s]


def dist_code(d):
    s = max(i for i in range(30) if DBASE[i] <= d)
    return s, d - DBASE[s], DEXT[s]


def canonical(lengths):
    """Canonical codes (RFC 1951 3.2.2) of the given lengths; None for length 0."""
    bl = [0] * 16
    for L in lengths:
        bl[L] += 1
    bl[0] = 0
    nxt, code = [0] * 16, 0
    for b in range(1, 16):
        code = (code + bl[b - 1]) << 1
        nxt[b] = code
    out = []
    for L in lengths:
        out.append(None if L == 0 else nxt[L])
        if L:
            nxt[L] += 1
    return out


def kraft_left(lengths, maxbits=15):
    """Code space the lengths leave unused, in units of 2^-maxbits (0: complete, < 0: over-subscribed)."""
    return (1 << maxbits) - sum(1 << (maxbits - L) for L in lengths if L)


def sub_usage(lengths, rbits):
    """Second-level LUT entries the CTA inflate kernel needs for this code with an `rbits`-bit root (lut_sub_warp)."""
    widest = {}
    for L, c in zip(lengths, canonical(lengths)):
        if L > rbits:
            q = c >> (L - rbits)
            widest[q] = max(widest.get(q, 0), L - rbits)
    return sum(1 << b for b in widest.values())


def huffman_lengths(freqs, maxbits):
    """Length-limited Huffman code lengths of `freqs` (frequencies are flattened until the limit holds); a lone symbol
    gets a partner so that the code is complete."""
    f = list(freqs)
    used = [i for i, v in enumerate(f) if v]
    if not used:
        return [0] * len(f)
    if len(used) == 1:
        other = 0 if used[0] != 0 else 1
        f[other] = 1
        used = sorted([used[0], other])
    while True:
        heap = [(f[i], i, (i,)) for i in used]
        heapq.heapify(heap)
        depth = [0] * len(f)
        k = len(f)
        while len(heap) > 1:
            a, b = heapq.heappop(heap), heapq.heappop(heap)
            for s in a[2] + b[2]:
                depth[s] += 1
            heapq.heappush(heap, (a[0] + b[0], k, a[2] + b[2]))
            k += 1
        if max(depth) <= maxbits:
            return depth
        f = [(v + 1) // 2 if v else 0 for v in f]


def fill_lengths(n, fixed, need, maxlen):
    """Lengths of an n-symbol code: `fixed` {symbol: length} as given, every symbol of `need` (and more when the space
    requires it) at <= maxlen bits, so that the code is exactly complete."""
    lengths = [0] * n
    for s, L in fixed.items():
        lengths[s] = L
    left = kraft_left(lengths)
    assert left % (1 << (15 - maxlen)) == 0, "the fixed codes must leave whole maxlen-bit slots"
    D = left >> (15 - maxlen)                        # free space in maxlen-bit slots
    units = {s: 1 for s in need if s not in fixed}
    D -= len(units)
    assert D >= 0, "more symbols needed than the code space holds"
    spare = iter(s for s in range(n) if s not in fixed and s not in units)
    while D > 0:
        cand = [s for s, u in units.items() if u <= D and 2 * u <= 1 << (maxlen - 1)]
        if cand:
            s = max(cand, key=lambda x: (units[x], -x))
            D -= units[s]
            units[s] *= 2
        else:
            units[next(spare)] = 1
            D -= 1
    for s, u in units.items():
        lengths[s] = maxlen - (u.bit_length() - 1)
    assert kraft_left(lengths) == 0
    return lengths


class BitWriter:
    def __init__(self):
        self.out = bytearray()
        self.acc = 0
        self.n = 0

    def bits(self, v, n):
        self.acc |= (v & ((1 << n) - 1)) << self.n
        self.n += n
        while self.n >= 8:
            self.out.append(self.acc & 0xff)
            self.acc >>= 8
            self.n -= 8

    def huff(self, code, length):
        if not length:                           # a symbol without a code (crafted invalid streams): nothing to write
            return
        self.bits(int(format(code, f"0{length}b")[::-1], 2), length)

    def align(self):
        if self.n % 8:
            self.bits(0, 8 - self.n % 8)

    @property
    def bitpos(self):
        return len(self.out) * 8 + self.n

    def getvalue(self):
        return bytes(self.out) + (bytes([self.acc & 0xff]) if self.n else b"")


def rle_code_lengths(lengths, max16=6, max17=10, max18=138):
    """Code-length symbols (symbol, extra value, extra bits) for `lengths` (lit/len then distance, one sequence: a run
    may cross from one into the other).  Runs are taken as long as the caps allow."""
    ops, i, n = [], 0, len(lengths)
    while i < n:
        v = lengths[i]
        run = 1
        while i + run < n and lengths[i + run] == v:
            run += 1
        if v == 0 and run >= 3:
            r = min(run, max18 if run >= 11 else max17)
            ops.append((18, r - 11, 7) if r >= 11 else (17, r - 3, 3))
            i += r
            continue
        ops.append((v, 0, 0))
        i += 1
        run -= 1
        while v and run >= 3:
            r = min(run, max16)
            ops.append((16, r - 3, 2))
            i += r
            run -= r
    return ops


def expand(tokens, history=b""):
    """The bytes `tokens` produce after `history` (history + output).  A distance beyond the output (invalid streams)
    reads zeros, as a lenient decoder with a zeroed window would."""
    out = bytearray(history)
    for t in tokens:
        if isinstance(t, int):
            out.append(t)
        else:
            L, d = t[0], t[1]
            for _ in range(L):
                out.append(out[-d] if d <= len(out) else 0)
    return bytes(out)


def tokenize(data, start=0, end=None, max_dist=32768, max_len=258, dist=None, min_len=3, max_matches=None, literal_only=False):
    """Greedy LZ77 over data[start:end], matches may reach back into data[:start] (max_dist).  dist: use exactly this
    distance (a match wherever data repeats at that distance); max_matches: literals once that many matches are made."""
    end = len(data) if end is None else end
    toks, i, table, made = [], start, {}, 0
    lo = max(0, start - max_dist)
    for j in range(lo, max(lo, start - 2)):
        table.setdefault(data[j:j + 3], []).append(j)
    while i < end:
        best_l, best_d = 0, 0
        if not literal_only and (max_matches is None or made < max_matches) and i + min_len <= end:
            cands = [i - dist] if dist is not None and i - dist >= 0 else ([] if dist is not None else table.get(data[i:i + 3], [])[-64:])
            for j in reversed(cands):
                d = i - j
                if d > max_dist or d < 1:
                    continue
                L = 0
                while L < max_len and i + L < end and data[j + L] == data[i + L]:
                    L += 1
                if L > best_l:
                    best_l, best_d = L, d
                    if L == max_len:
                        break
        step = best_l if best_l >= min_len else 1
        if best_l >= min_len:
            toks.append((best_l, best_d))
            made += 1
        else:
            toks.append(data[i])
        for k in range(i, i + step):
            if k + 3 <= len(data):
                table.setdefault(data[k:k + 3], []).append(k)
        i += step
    return toks


class Deflate:
    """A raw DEFLATE stream being written; `data` is what a decoder must produce."""

    def __init__(self):
        self.bw = BitWriter()
        self.data = b""
        self.block_bits = []      # bit offset of every block header

    def _start(self, final, btype):
        self.block_bits.append(self.bw.bitpos)
        self.bw.bits(1 if final else 0, 1)
        self.bw.bits(btype, 2)

    def stored(self, payload, final=False, nlen=None, length=None):
        self._start(final, 0)
        self.bw.align()
        n = len(payload) if length is None else length
        self.bw.bits(n, 16)
        self.bw.bits((~n & 0xffff) if nlen is None else nlen, 16)
        for b in payload:
            self.bw.bits(b, 8)
        self.data += payload
        return self

    def _tokens(self, tokens, ll_codes, ll_len, d_codes, d_len):
        bw = self.bw
        for t in tokens:
            if isinstance(t, int):
                bw.huff(ll_codes[t], ll_len[t])
            elif t[0] == "ll":                    # a bare lit/len symbol (crafted invalid streams)
                bw.huff(ll_codes[t[1]], ll_len[t[1]])
            elif t[0] == "d":                     # a bare distance symbol
                bw.huff(d_codes[t[1]], d_len[t[1]])
            else:
                L, d = t[0], t[1]
                s, xv, xb = len_code(L, long_258=len(t) > 2 and t[2] == "284")
                bw.huff(ll_codes[s], ll_len[s])
                bw.bits(xv, xb)
                s, xv, xb = dist_code(d)
                bw.huff(d_codes[s], d_len[s])
                bw.bits(xv, xb)
        bw.huff(ll_codes[256], ll_len[256])
        self.data = expand([t for t in tokens if isinstance(t, int) or isinstance(t[0], int)], self.data)

    def fixed(self, tokens, final=False):
        self._start(final, 1)
        self._tokens(tokens, canonical(FIXED_LL), FIXED_LL, canonical(FIXED_D), FIXED_D)
        return self

    @staticmethod
    def freqs(tokens):
        fl, fd = [0] * 286, [0] * 30
        fl[256] = 1
        for t in tokens:
            if isinstance(t, int):
                fl[t] += 1
            elif isinstance(t[0], int):
                fl[len_code(t[0], len(t) > 2 and t[2] == "284")[0]] += 1
                fd[dist_code(t[1])[0]] += 1
        return fl, fd

    def dynamic(self, tokens, final=False, ll=None, d=None, pre=None, hlit=None, hdist=None, hclen=None, ops=None, rle=None):
        """ll / d / pre: code lengths (default: length-limited Huffman of the token frequencies); hlit / hdist / hclen:
        the alphabet sizes written (default: up to the last used length, at least 257 / 1 / 4); ops: the code-length
        symbols (default rle_code_lengths(..., **rle))."""
        fl, fd = self.freqs(tokens)
        ll = list(ll) if ll is not None else huffman_lengths(fl, 15)
        if d is None:
            d = huffman_lengths(fd, 15) if any(fd) else [0]
        d = list(d)
        n_ll = hlit or max(257, max(i for i, L in enumerate(ll) if L) + 1)
        n_d = hdist or max(1, max([i for i, L in enumerate(d) if L], default=0) + 1)
        ll = (ll + [0] * 288)[:n_ll]
        d = (d + [0] * 32)[:n_d]
        ops = ops if ops is not None else rle_code_lengths(ll + d, **(rle or {}))
        fp = [0] * 19
        for s, _, _ in ops:
            fp[s] += 1
        pre = list(pre) if pre is not None else huffman_lengths(fp, 7)
        n_clc = hclen or max(4, max(i for i, s in enumerate(CLC_ORDER) if pre[s]) + 1)
        self._start(final, 2)
        bw = self.bw
        bw.bits(n_ll - 257, 5)
        bw.bits(n_d - 1, 5)
        bw.bits(n_clc - 4, 4)
        for i in range(n_clc):
            bw.bits(pre[CLC_ORDER[i]], 3)
        pc = canonical(pre)
        for s, xv, xb in ops:
            bw.huff(pc[s], pre[s])
            bw.bits(xv, xb)
        self.ops, self.ll, self.d = ops, ll, d
        self._tokens(tokens, canonical(ll + [0] * (288 - len(ll))), ll + [0] * (288 - len(ll)), canonical(d + [0] * (32 - len(d))), d + [0] * (32 - len(d)))
        return self

    def raw_bits(self, v, n):
        self.bw.bits(v, n)
        return self

    def payload(self):
        return self.bw.getvalue()


def bgzf_member(payload, data, crc=None, isize=None, extra_before=b"", extra_after=b""):
    """One BGZF member around a raw DEFLATE payload: BC subfield with extra subfields (whole subfields) around it."""
    xfield = extra_before + b"BC\x02\x00" + b"\0\0" + extra_after
    hdr = b"\x1f\x8b\x08\x04\0\0\0\0\0\xff" + struct.pack("<H", len(xfield))
    bsize = len(hdr) + len(xfield) + len(payload) + 8 - 1
    assert bsize < 65536
    k = len(extra_before) + 4
    xfield = xfield[:k] + struct.pack("<H", bsize) + xfield[k + 2:]
    crc = zlib.crc32(data) & 0xffffffff if crc is None else crc
    isize = len(data) if isize is None else isize
    return hdr + xfield + payload + struct.pack("<II", crc, isize)


def subfield(n):
    """An extra-field subfield of n bytes (n >= 4) that is not BC."""
    assert n >= 4
    return b"XY" + struct.pack("<H", n - 4) + bytes(range(n - 4))


class Member:
    """A BGZF member and what it must do: `valid` members inflate to `data`; invalid ones make zlib raise."""

    def __init__(self, raw, data, valid, label, refused=False):
        self.raw, self.data, self.valid, self.label, self.refused = raw, data, valid, label, refused

    def check(self):
        if self.valid:
            d = zlib.decompressobj(31)
            out = d.decompress(self.raw)
            assert d.eof and not d.unused_data and out == self.data, f"{self.label}: zlib does not reproduce the data"
        else:
            try:
                d = zlib.decompressobj(31)
                d.decompress(self.raw)
                if not d.eof:
                    raise zlib.error("truncated")
            except zlib.error:
                return
            raise AssertionError(f"{self.label}: built as invalid but zlib accepts it")


def member(dfl, label="", valid=True, refused=False, **kw):
    m = Member(bgzf_member(dfl.payload(), dfl.data, **kw), dfl.data, valid, label, refused)
    m.check()
    return m


EOF_MEMBER = bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000")
