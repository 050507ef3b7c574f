"""CPU oracle of the plain-SAM scan: a restatement of noodles-sam's RecordBuf parsing (one record per line) and of the SAM loop
of BamTableProvider.

Each line is parsed and validated in Python and transcoded to a BAM record (the same narrowing of `i` values to the smallest
BAM integer type, f32 values correctly rounded from their decimal text).  The records go into a BGZF BAM in a temporary
directory, which OracleBam (bam_oracle.c) scans with end_zero_span_mode = 1: RecordBuf's end of a placed read whose CIGAR
spans no reference base is start + 0 - 1, not NULL -- except at POS 1, where that is 0 and Position::new gives None, so the
end of those rows is set back to NULL here.  Then RecordBuf's second difference: QUAL '*' with a non-empty SEQ gives an
empty quality string (the BAM path renders the 0xFF fill as spaces).
"""
import os
import re
import struct
import tempfile
from fractions import Fraction

import pyarrow as pa

from oracle.bam_oracle import OracleBam
from oracle.bam_write_oracle import bam_header_bytes, bgzf_member

_BASES = {c: i for i, c in enumerate("=ACMGRSVTWYHKDBN")}
_OPS = "MIDNSHP=X"
_RANGES = {"c": (-128, 127), "C": (0, 255), "s": (-32768, 32767), "S": (0, 65535), "i": (-2 ** 31, 2 ** 31 - 1), "I": (0, 2 ** 32 - 1)}
_FMT = {"c": "b", "C": "B", "s": "h", "S": "H", "i": "i", "I": "I", "f": "f"}
_FLOAT = re.compile(r"[+-]?(\d+\.?\d*|\.\d+)([eE][+-]?\d+)?\Z")
_INT = re.compile(r"[+-]?\d+\Z")
_UINT = re.compile(r"\+?\d+\Z")


class SamError(ValueError):
    def __init__(self, record, what):
        super().__init__(f"record {record}: {what}")
        self.record, self.what = record, what


def f32_from_text(s: str) -> int:
    """Rust's f32::from_str, exactly (fractions.Fraction): the bit pattern of the nearest f32, ties to even."""
    low = s.lower().lstrip("+-")
    sign = 0x80000000 if s.startswith("-") else 0
    if low in ("inf", "infinity"):
        return sign | 0x7F800000
    if low == "nan":
        return sign | 0x7FC00000
    if not _FLOAT.match(s):
        raise ValueError(s)
    v = abs(Fraction(s.lstrip("+")))
    if v == 0:
        return sign
    best, lo, hi = None, 0, 0x7F800000        # smallest bits whose upper halfway point is >= v (ties to even)
    def value(b):
        e, m = b >> 23, b & 0x7FFFFF
        return Fraction(m if e == 0 else m | 0x800000) * Fraction(2) ** ((e if e else 1) - 150)
    while lo < hi:
        mid = (lo + hi) // 2
        if (value(mid) + value(mid + 1)) / 2 < v if mid + 1 < 0x7F800000 else \
                (value(mid) + Fraction(2) ** 128) / 2 < v:
            lo = mid + 1
        else:
            hi = mid
    b = lo
    if b < 0x7F800000 and (b & 1) and v == (value(b) + (value(b + 1) if b + 1 < 0x7F800000 else Fraction(2) ** 128)) / 2:
        b += 1                                 # a tie goes to the even neighbour
    return sign | b


def _int(s, signed, lo, hi, rec, what):
    if not (_INT if signed else _UINT).match(s) or not lo <= int(s) <= hi:
        raise SamError(rec, what)
    return int(s)


def _narrow(v):
    for t in ("CSI" if v >= 0 else "csi"):
        lo, hi = _RANGES[t]
        if lo <= v <= hi:
            return t
    return None


def _aux(field, rec):
    if len(field) < 5 or field[2] != ":" or field[4] != ":" or not re.match(r"[A-Za-z][A-Za-z0-9]\Z", field[:2]):
        raise SamError(rec, "malformed aux field")
    tag, ty, val = field[:2], field[3], field[5:]
    out = tag.encode()
    if ty == "A":
        if len(val) != 1 or not "!" <= val <= "~":
            raise SamError(rec, "malformed aux field")
        return tag, out + b"A" + val.encode()
    if ty == "i":
        if not _INT.match(val):
            raise SamError(rec, "malformed aux field")
        t = _narrow(int(val))
        if t is None:
            raise SamError(rec, "aux value out of range for its type")
        return tag, out + t.encode() + struct.pack("<" + _FMT[t], int(val))
    if ty == "f":
        try:
            return tag, out + b"f" + struct.pack("<I", f32_from_text(val))
        except ValueError:
            raise SamError(rec, "malformed aux field")
    if ty == "Z":
        if any(not " " <= c <= "~" for c in val):
            raise SamError(rec, "malformed aux field")
        return tag, out + b"Z" + val.encode() + b"\0"
    if ty == "H":
        if len(val) % 2 or not re.match(r"[0-9A-Fa-f]*\Z", val):
            raise SamError(rec, "malformed aux field")
        return tag, out + b"H" + val.encode() + b"\0"
    if ty == "B":
        if not val or val[0] not in _FMT:
            raise SamError(rec, "malformed aux field")
        st, parts = val[0], val[1:]
        if parts and parts[0] != ",":
            raise SamError(rec, "malformed aux field")
        elems = parts[1:].split(",") if parts else []
        body = b""
        for e in elems:
            if st == "f":
                try:
                    body += struct.pack("<I", f32_from_text(e))
                except ValueError:
                    raise SamError(rec, "malformed aux field")
            else:
                if not _INT.match(e):
                    raise SamError(rec, "malformed aux field")
                lo, hi = _RANGES[st]
                if not lo <= int(e) <= hi:
                    raise SamError(rec, "aux value out of range for its type")
                body += struct.pack("<" + _FMT[st], int(e))
        return tag, out + b"B" + st.encode() + struct.pack("<i", len(elems)) + body
    raise SamError(rec, "malformed aux field")


def parse_sam(data: bytes):
    """-> (header_text, ref_names, ref_lens, header_ok, [BAM record bytes], {record index whose QUAL is '*' with a SEQ},
    {record index of a read at POS 1 whose CIGAR spans no reference base})"""
    lines = data.split(b"\n")
    if lines and lines[-1] == b"":
        lines.pop()                                   # the final newline ends the last line; it does not start another
    k = 0
    while k < len(lines) and lines[k].startswith(b"@"):
        k += 1
    header = b"".join(ln + b"\n" for ln in lines[:k]).decode()
    names, lens, ok = [], [], True
    for ln in header.split("\n"):
        ln = ln.rstrip("\r")
        if not ln.startswith("@SQ\t"):
            continue
        kv = {}
        for tok in ln.split("\t")[1:]:
            if tok[2:3] == ":":
                kv[tok[:2]] = tok[3:]
        ln_v = kv.get("LN", "")
        if not kv.get("SN") or not (ln_v.isdigit() and len(ln_v) <= 10 and 1 <= int(ln_v) <= 2 ** 31 - 1) or kv["SN"] in names:
            ok = False
            break
        names.append(kv["SN"]); lens.append(int(ln_v))
    if not ok:
        names, lens = [], []
    ref_id = {n: i for i, n in enumerate(names)}
    recs, no_qual, end_null = [], set(), set()
    for rec, raw in enumerate(lines[k:]):
        line = raw.decode("latin-1")
        if line.endswith("\r"):
            line = line[:-1]
        f = line.split("\t")
        if len(f) < 11:
            raise SamError(rec, "fewer than 11 fields")
        qname, flag, rname, pos, mapq, cigar, rnext, pnext, tlen, seq, qual = f[:11]
        if not 1 <= len(qname) <= 254 or any(not ("!" <= c <= "~") or c == "@" for c in qname):
            raise SamError(rec, "invalid QNAME")
        flag = _int(flag, False, 0, 65535, rec, "invalid FLAG")
        if rname != "*" and rname not in ref_id:
            raise SamError(rec, "RNAME is not a reference sequence of the header")
        ref = ref_id.get(rname, -1)
        pos = _int(pos, False, 0, 2 ** 31, rec, "invalid POS")
        mapq = _int(mapq, False, 0, 255, rec, "invalid MAPQ")
        ops = []
        if cigar != "*":
            if not re.match(r"(\d+[MIDNSHP=X])+\Z", cigar):
                raise SamError(rec, "invalid CIGAR")
            for n, op in re.findall(r"(\d+)([MIDNSHP=X])", cigar):
                if int(n) >= 1 << 28:
                    raise SamError(rec, "invalid CIGAR")
                ops.append((int(n) << 4) | _OPS.index(op))
            if len(ops) > 65535:
                raise SamError(rec, "CIGAR with more than 65535 operations is not supported")
        if rnext == "=":
            nref = ref
        elif rnext == "*":
            nref = -1
        elif rnext in ref_id:
            nref = ref_id[rnext]
        else:
            raise SamError(rec, "RNEXT is not a reference sequence of the header")
        pnext = _int(pnext, False, 0, 2 ** 31, rec, "invalid PNEXT")
        tlen = _int(tlen, True, -2 ** 31, 2 ** 31 - 1, rec, "invalid TLEN")
        if seq != "*" and not re.match(r"[A-Za-z=.]+\Z", seq):
            raise SamError(rec, "invalid SEQ")
        seq = "" if seq == "*" else seq
        if qual == "*":
            q = b"\xff" * len(seq)
            if seq:
                no_qual.add(rec)
        else:
            if len(qual) != len(seq):
                raise SamError(rec, "QUAL length differs from SEQ length")
            if any(not "!" <= c <= "~" for c in qual):
                raise SamError(rec, "invalid QUAL")
            q = bytes(ord(c) - 33 for c in qual)
        aux, seen = b"", set()
        for field in f[11:]:
            tag, b = _aux(field, rec)
            if tag in seen:
                raise SamError(rec, "duplicate aux tag")
            seen.add(tag)
            aux += b
        if pos == 1 and sum(o >> 4 for o in ops if (o & 15) in (0, 2, 3, 7, 8)) == 0:
            end_null.add(rec)            # RecordBuf::alignment_end: Position::new(1 + 0 - 1) is None
        packed = bytearray((len(seq) + 1) // 2)
        for i, c in enumerate(seq.upper()):
            packed[i >> 1] |= _BASES.get(c, 15) << (4 if i % 2 == 0 else 0)
        body = struct.pack("<iiBBHHHiiii", ref, pos - 1, len(qname) + 1, mapq, 4680, len(ops), flag, len(seq), nref, pnext - 1, tlen)
        body += qname.encode() + b"\0" + struct.pack(f"<{len(ops)}I", *ops) + bytes(packed) + q + aux
        recs.append(struct.pack("<i", len(body)) + body)
    return header, names, lens, ok, recs, no_qual, end_null


class OracleSam:
    """CPU restatement of BamTableProvider over a plain SAM file; same constructor arguments and scan() as OracleBam."""

    def __init__(self, path, zero_based=True, tag_fields=None, binary_cigar=False, infer_tag_types=True,
                 infer_tag_sample_size=100, tag_type_hints=None):
        header, names, lens, ok, recs, self.no_qual, self.end_null = parse_sam(open(path, "rb").read())
        self._dir = tempfile.TemporaryDirectory()
        bam = os.path.join(self._dir.name, "t.bam")
        stream = bam_header_bytes(header if ok else "", names, lens) + b"".join(recs)
        with open(bam, "wb") as fh:
            for i in range(0, len(stream), 0xff00):
                fh.write(bgzf_member(stream[i:i + 0xff00]))
            fh.write(bgzf_member(b""))
        self.bam = OracleBam(bam, zero_based, tag_fields, binary_cigar, infer_tag_types, infer_tag_sample_size, tag_type_hints,
                             end_zero_span_mode=1)
        self.schema = self.bam.schema
        self.n_records = len(recs)

    def scan(self, projection=None) -> pa.RecordBatch:
        b = self.bam.scan(projection)
        if "quality_scores" in b.schema.names and self.no_qual:
            i = b.schema.get_field_index("quality_scores")
            q = b.column(i).to_pylist()
            for r in self.no_qual:
                q[r] = ""
            b = b.set_column(i, b.schema.field(i), pa.array(q, pa.utf8()))
        if "end" in b.schema.names and self.end_null:
            i = b.schema.get_field_index("end")
            e = b.column(i).to_pylist()
            for r in self.end_null:
                e[r] = None
            b = b.set_column(i, b.schema.field(i), pa.array(e, pa.uint32()))
        return b

    def close(self):
        self.bam.close()
        self._dir.cleanup()
