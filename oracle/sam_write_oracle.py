"""CPU restatement of the SAM write path -- TEST INFRASTRUCTURE ONLY (nothing under datafusion-bio-formats_b200/ imports it).

In the reference a `.sam` target is batch_to_alignment_records -> noodles RecordBuf -> noodles-sam's writer.  The first half is
the BAM write oracle's: every row goes through bam_write_oracle.encode_record, so the SAM writer accepts and refuses exactly the
rows the BAM writer does (shared refusals are re-raised with the row number).  The line is then rendered from that record:

  QNAME   the record's name (NULL / "*" -> '*')            FLAG   decimal
  RNAME   the resolved reference's name, '*' for none     POS    1-based, 0 when missing
  MAPQ    decimal                                         CIGAR  the parsed operations ('010M' -> '10M'), '*' for none
  RNEXT   '*' for none, '=' for the record's own reference, else the name;  PNEXT as POS;  TLEN decimal
  SEQ     the row's own string, as given (no case folding), '*' when NULL / "" / "*"
  QUAL    the BAM score max(0, c - 33) + 33 (characters below '!' become '!'), '*' when NULL / "" / "*"
  tags    tag_fields order, NULL -> no field: c C s S i I -> TG:i:<decimal>; f -> TG:f:<Rust f32 Display>; Z as given; H upper-
          cased; A one character; B:x -> TG:B:x,v1,v2... (TG:B:x when empty); unknown letters: strings as Z

noodles-sam's writer is not vendored, so these text rules are this project's (DESIGN 3.9, unpinned).  Guiding rule: a row is
refused when its line would not read back as the same row.  The SAM-only refusals, one per row, the first in this order:
  invalid QNAME (outside SAMv1 [!-?A-~]{1,254}; "" included), invalid SEQ (outside [A-Za-z=.]), invalid QUAL (a character
  above '~'), invalid Z tag value (outside [ !-~]), invalid A tag value (outside [!-~]).
"""
from __future__ import annotations

import struct
from fractions import Fraction

import pyarrow as pa

from oracle import bam_write_oracle as W

_OPS = "MIDNSHP=X"
SAM_RULES = ["invalid QNAME", "invalid SEQ", "invalid QUAL", "invalid Z tag value", "invalid A tag value"]


class WriteError(Exception):
    """A refused row: `shared` when the BAM writer refuses it too (its message then is the BAM oracle's)."""

    def __init__(self, row, what, shared):
        super().__init__(f"row {row}: {what}")
        self.row, self.what, self.shared = row, what, shared


# ---------------------------------------------------------------------------------------------------------------------
# f32 text: oracle/bam_oracle.c::rust_f32_to_string -- the smallest precision N <= 9 whose correctly rounded "%.{N-1}e" reads
# back as the same f32, or, when that rounded down, whose value one unit above reads back (possible only at a power of two,
# where the float below is half as far away as the one above), written in plain positional notation.  The exact reference
# is oracle/f32_exact.py.

def _f32_value(bits: int) -> Fraction:
    e, m = (bits >> 23) & 0xff, bits & 0x7fffff
    return Fraction(m if e == 0 else m | 0x800000) * Fraction(2) ** ((e if e else 1) - 150)


def _reads_back(text: str, bits: int) -> bool:
    """Does the decimal `text` (no sign) round to the positive finite f32 `bits` (round half to even)?"""
    r, v = Fraction(text), _f32_value(bits)
    if r == v:
        return True
    up = ((_f32_value(bits + 1) if bits + 1 < 0x7f800000 else Fraction(2) ** 128) - v) / 2
    down = (v - _f32_value(bits - 1)) / 2 if bits > 0 else up
    gap = up if r > v else down
    return abs(r - v) < gap or (abs(r - v) == gap and bits % 2 == 0)


def _next_up(t: str) -> str:
    """The "d.ddde+x" decimal one unit above `t` in its last digit, with as many digits ("9.9e+05" -> "1.0e+06")."""
    mant, exp10 = t.split("e")
    digits = mant.replace(".", "")
    up, x = str(int(digits) + 1), int(exp10)
    if len(up) > len(digits):
        up, x = up[:-1], x + 1
    return f"{up[0]}.{up[1:]}e{x}" if len(up) > 1 else f"{up}e{x}"


def f32_text(bits: int) -> str:
    bits &= 0xffffffff
    sign, mag = bits >> 31, bits & 0x7fffffff
    if mag > 0x7f800000:
        return "NaN"
    if mag == 0x7f800000:
        return "-inf" if sign else "inf"
    if mag == 0:
        return "-0" if sign else "0"
    x = float(_f32_value(mag))                        # exact: every f32 is a double
    for prec in range(1, 10):
        t = f"{x:.{prec - 1}e}"
        if _reads_back(t, mag):
            break
        if Fraction(t) < x:
            t = _next_up(t)
            if _reads_back(t, mag):
                break
    mant, exp10 = t.split("e")
    digits, exp10 = mant.replace(".", "").rstrip("0") or "0", int(exp10)
    if exp10 < 0:
        body = "0." + "0" * (-exp10 - 1) + digits
    else:
        body = "".join(digits[i] if i < len(digits) else "0" for i in range(exp10 + 1))
        if len(digits) > exp10 + 1:
            body += "." + digits[exp10 + 1:]
    return ("-" if sign else "") + body


def _f32_bits(value) -> int:
    """The f32 the BAM writer stores (a Float64 is narrowed, round to nearest even)."""
    return struct.unpack("<I", struct.pack("<f", value))[0]


# ---------------------------------------------------------------------------------------------------------------------
# lines

def _qname_ok(b: bytes) -> bool:
    return 1 <= len(b) <= 254 and all(0x21 <= c <= 0x7e and c != 0x40 for c in b)


def _seq_ok(b: bytes) -> bool:
    return all(0x41 <= c <= 0x5a or 0x61 <= c <= 0x7a or c in b"=." for c in b)


def _tag_text(tag, value, arrow_type, spec, fail):
    """TG:x:value of one non-NULL tag (None when the BAM writer drops it); SAM-only failures go to `fail`."""
    t, sub = W.parse_sam_tag_type(spec)
    if t in "cCsSiI":
        return f"{tag}:i:{value}"
    if t == "f":
        return f"{tag}:f:{f32_text(_f32_bits(value))}"
    if t == "H":
        return f"{tag}:H:{value.upper()}"
    if t == "A":
        c = value.encode()[0] if isinstance(value, str) else value
        if not 0x21 <= c <= 0x7e:
            fail.add(4)
        return f"{tag}:A:{chr(c)}"
    if t == "B":
        st = sub or W._ARROW_SUBTYPE.get(arrow_type.value_type)
        elems = "".join("," + (f32_text(_f32_bits(v)) if st == "f" else str(v)) for v in value)
        return f"{tag}:B:{st}{elems}"
    if t == "Z" or pa.types.is_string(arrow_type):       # (unknown letters: strings as Z, anything else dropped)
        if any(not 0x20 <= c <= 0x7e for c in value.encode()):
            fail.add(3)
        return f"{tag}:Z:{value}"
    return None


def render_row(r: int, row: dict, ref_names, ref_map: dict, tags, zero_based: bool) -> bytes:
    """One SAM line (with its '\\n') from a row of python values; `tags` is [(name, value_or_None, arrow_type, spec)]."""
    try:
        rec = W.encode_record(row, ref_map, tags, zero_based)
    except W.WriteError as e:
        raise WriteError(r, str(e), True) from None
    ref, pos, l_name, mapq, _bin, n_cig, flag, l_seq, nref, npos, tlen = struct.unpack_from("<iiBBHHHiiii", rec, 4)
    name = rec[36:36 + l_name - 1]
    ops = struct.unpack_from(f"<{n_cig}I", rec, 36 + l_name)
    fail = set()
    if row["name"] is not None and not _qname_ok(row["name"].encode()):
        fail.add(0)
    seq = b"" if row["sequence"] in (None, "", "*") else row["sequence"].encode()
    if not _seq_ok(seq):
        fail.add(1)
    qual = b"" if row["quality_scores"] in (None, "", "*") else row["quality_scores"].encode()
    if any(c > 0x7e for c in qual):
        fail.add(2)
    aux = [_tag_text(n, v, t, s, fail) for n, v, t, s in tags if v is not None]
    if fail:
        raise WriteError(r, SAM_RULES[min(fail)], False)
    fields = [name.decode(), str(flag), ref_names[ref] if ref >= 0 else "*", str(pos + 1), str(mapq),
              "".join(f"{o >> 4}{_OPS[o & 15]}" for o in ops) or "*",
              "*" if nref < 0 else ("=" if nref == ref else ref_names[nref]), str(npos + 1), str(tlen),
              seq.decode() if l_seq else "*", "".join(chr(max(c, 33)) for c in qual) if qual else "*"]
    return ("\t".join(fields + [a for a in aux if a is not None]) + "\n").encode()


def render_batch(batch: pa.RecordBatch, ref_names, tag_fields, zero_based: bool = True) -> bytes:
    """The SAM lines of one batch (header not included); raises WriteError for the first refused row."""
    if batch.num_rows == 0:
        return b""
    for c in W.REQUIRED:
        if batch.schema.get_field_index(c) < 0:
            raise W.WriteError(f"Required column '{c}' not found in batch")
    ref_map = {n: i for i, n in enumerate(ref_names)}          # a later duplicate wins
    cols = {c: batch.column(batch.schema.get_field_index(c)).to_pylist() for c in W.REQUIRED}
    tcols = [(n, batch.column(i).to_pylist(), batch.schema.field(i).type, spec) for n, i, spec in W.tag_columns(batch.schema, tag_fields)]
    return b"".join(render_row(r, {c: cols[c][r] for c in W.REQUIRED}, ref_names, ref_map,
                               [(n, v[r], t, s) for n, v, t, s in tcols], zero_based) for r in range(batch.num_rows))


def sam_text(batches, schema: pa.Schema, tag_fields, zero_based: bool = True, overrides=None) -> bytes:
    """The whole file: build_bam_header's text, then every batch's lines in arrival order."""
    text, names, _lens = W.build_bam_header(schema, overrides)
    return text.encode() + b"".join(render_batch(b, names, tag_fields, zero_based) for b in batches)


def write_sam(path, batches, schema: pa.Schema, tag_fields, zero_based: bool = True, overrides=None) -> int:
    """== SamWriteExec::execute; returns the row count."""
    batches = list(batches)
    data = sam_text(batches, schema, tag_fields, zero_based, overrides)
    with open(path, "wb") as f:
        f.write(data)
    return sum(b.num_rows for b in batches)
