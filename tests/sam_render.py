"""BAM -> SAM text in `samtools view -h` layout: the header text, then one tab-separated line per record.  Used by the SAM
tests to turn every golden BAM into a SAM of the same records.

`f` values (scalar and `B:f` elements) are printed as the shortest decimal that reads back as the same f32, so the SAM
holds exactly the BAM's values.  When the header text has no @SQ lines, they are made from the binary reference list."""
import gzip
import struct

import numpy as np

_BASES = "=ACMGRSVTWYHKDBN"
_OPS = "MIDNSHP=X"
_B_FMT = {"c": "b", "C": "B", "s": "h", "S": "H", "i": "i", "I": "I", "f": "f"}


def _f32(v) -> str:
    return str(np.float32(v))


def read_bam(data: bytes):
    """-> (header_text, ref_names, ref_lens, [record bytes without block_size])"""
    u = gzip.decompress(data)
    assert u[:4] == b"BAM\1"
    l_text = struct.unpack_from("<i", u, 4)[0]
    text = u[8:8 + l_text].rstrip(b"\0").decode()
    p = 8 + l_text
    n_ref = struct.unpack_from("<i", u, p)[0]; p += 4
    names, lens = [], []
    for _ in range(n_ref):
        ln = struct.unpack_from("<i", u, p)[0]
        names.append(u[p + 4:p + 4 + ln].rstrip(b"\0").decode()); lens.append(struct.unpack_from("<i", u, p + 4 + ln)[0])
        p += 8 + ln
    recs = []
    while p + 4 <= len(u):
        bs = struct.unpack_from("<i", u, p)[0]
        recs.append(u[p + 4:p + 4 + bs]); p += 4 + bs
    return text, names, lens, recs


def render_record(rec: bytes, names) -> str:
    ref, pos, l_name, mapq, _bin, n_cig, flag, l_seq, nref, npos, tlen = struct.unpack_from("<iiBBHHHiiii", rec, 0)
    o = 32
    qname = rec[o:o + l_name - 1].decode(); o += l_name
    cig = "".join(f"{w >> 4}{_OPS[w & 15]}" for w in struct.unpack_from(f"<{n_cig}I", rec, o)) or "*"; o += 4 * n_cig
    seq = "".join(_BASES[(rec[o + i // 2] >> (4 if i % 2 == 0 else 0)) & 15] for i in range(l_seq)) or "*"; o += (l_seq + 1) // 2
    q = rec[o:o + l_seq]; o += l_seq
    qual = "*" if l_seq == 0 or all(b == 0xFF for b in q) else "".join(chr(b + 33) for b in q)
    rname = names[ref] if ref >= 0 else "*"
    rnext = "*" if nref < 0 else ("=" if nref == ref else names[nref])
    fields = [qname, str(flag), rname, str(pos + 1), str(mapq), cig, rnext, str(npos + 1), str(tlen), seq, qual]
    while o + 3 <= len(rec):
        tag, ty = rec[o:o + 2].decode(), chr(rec[o + 2]); o += 3
        if ty == "A":
            fields.append(f"{tag}:A:{chr(rec[o])}"); o += 1
        elif ty in "cCsSiI":
            fmt = _B_FMT[ty]; v = struct.unpack_from("<" + fmt, rec, o)[0]; o += struct.calcsize(fmt)
            fields.append(f"{tag}:i:{v}")
        elif ty == "f":
            fields.append(f"{tag}:f:{_f32(struct.unpack_from('<f', rec, o)[0])}"); o += 4
        elif ty in "ZH":
            e = rec.index(b"\0", o)
            fields.append(f"{tag}:{ty}:{rec[o:e].decode()}"); o = e + 1
        elif ty == "B":
            st = chr(rec[o]); cnt = struct.unpack_from("<i", rec, o + 1)[0]; o += 5
            vals = struct.unpack_from(f"<{cnt}{_B_FMT[st]}", rec, o); o += cnt * struct.calcsize(_B_FMT[st])
            fields.append(f"{tag}:B:{st}" + "".join("," + (_f32(v) if st == "f" else str(v)) for v in vals))
        else:
            raise ValueError(f"aux type {ty!r}")
    return "\t".join(fields)


def bam_to_sam(data: bytes) -> bytes:
    text, names, lens, recs = read_bam(data)
    lines = [ln for ln in text.split("\n") if ln]
    if not any(ln.startswith("@SQ\t") for ln in lines):
        sq = [f"@SQ\tSN:{n}\tLN:{l}" for n, l in zip(names, lens)]
        at = 1 if lines and lines[0].startswith("@HD") else 0
        lines[at:at] = sq
    out = lines + [render_record(r, names) for r in recs]
    return ("\n".join(out) + "\n").encode()
