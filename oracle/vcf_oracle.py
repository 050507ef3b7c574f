"""CPU restatement of the VCF scan -- TEST INFRASTRUCTURE ONLY (nothing under datafusion-bio-formats_b200/ imports it; only
tests/ may).

The reference's VCF provider (bio-format-vcf) is not vendored here and no reference VCF fixture exists, so every rule below is this
project's own statement of the format (DESIGN 3.11), unpinned.  Where the reference may well differ, that is said: the type of
`qual` (Float32 here, as BCF stores it), `alt` and `filter` kept as the text of the column (not split into lists), and the field
metadata key names (bio.vcf.info.number / type / description).

Header (read at open):
- the first line starts with "##fileformat=VCF"; the header ends with the "#CHROM\\tPOS\\tID\\tREF\\tALT\\tQUAL\\tFILTER\\tINFO" line
  (sample names behind it are ignored); a missing #CHROM line or an INFO ID declared twice is a format error;
- ##INFO=<ID=..,Number=..,Type=..,Description=".."> lines decide the INFO columns; quoted values may hold ',' '=' '>' and \\" \\\\.

Schema: chrom Utf8, start UInt32 (POS - 1, or POS when not zero-based), end UInt32 (INFO END if present, else POS + len(REF) - 1),
id Utf8?, ref Utf8, alt Utf8?, qual Float32?, filter Utf8?, then one column per selected INFO field: Type=Flag -> Boolean (not
null); Number=1 -> Int32 / Float32 / Utf8 (Integer / Float / String or Character); any other Number -> List of those (nullable
elements).  info_fields None selects every ##INFO field in header order; a list selects those IDs in that order.  Schema errors,
naming the field: an undeclared ID, an ID selected twice, an ID equal to a fixed column's name, an unknown Type, Number=0 on a type
other than Flag.  At most 112 INFO columns can be projected in one scan (more is unsupported, at execute).

Records (one per line behind the header; one trailing '\\r' per line is dropped; FORMAT and sample columns are skipped):
- format errors: fewer than 8 fields; a '#' line or an empty line; POS not an integer in [1, 2^31 - 1]; an empty CHROM or REF;
  QUAL neither '.' nor a number; END below POS; a looked-up INFO key (a projected one, or END) given twice in one record; a byte of
  0x80 or above in a projected Utf8 column;
- schema errors: a value of a projected INFO column (or END) that does not parse as its type: an empty numeric element, a Flag
  with '=value', a non-Flag key without '=', a ',' in a Number=1 value.  Values of unprojected INFO columns are not checked;
- unsupported: POS 0; a line longer than 16 MiB;
- INFO is '.' or ';'-separated key[=value] pairs (empty pairs are skipped); a value '.' is NULL, a list element '.' a NULL element;
  Integers lie in the i32 range ([+-]digits); Floats follow f32_parse.h (oracle/sam_oracle.py::f32_from_text); strings are kept as given.
"""
import struct
from functools import lru_cache

import pyarrow as pa

from oracle.sam_oracle import f32_from_text

FIXED = ["chrom", "start", "end", "id", "ref", "alt", "qual", "filter"]
FIXED_SCHEMA = [pa.field("chrom", pa.string(), False), pa.field("start", pa.uint32(), False), pa.field("end", pa.uint32(), False),
                pa.field("id", pa.string(), True), pa.field("ref", pa.string(), False), pa.field("alt", pa.string(), True),
                pa.field("qual", pa.float32(), True), pa.field("filter", pa.string(), True)]
MAX_LINE = 16 << 20
CHROM_LINE = b"#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO"


class VcfError(ValueError):
    """kind: "format", "schema" or "unsupported"; record: 0-based record number (None for header / open errors)."""

    def __init__(self, kind, why, record=None):
        super().__init__(f"{kind}: record {record}: {why}" if record is not None else f"{kind}: {why}")
        self.kind = kind
        self.record = record


def _info_line(line: bytes) -> dict:
    s = line.decode("latin-1")[len("##INFO=<"):]
    out, k = {}, 0
    while True:
        eq = s.find("=", k)
        if eq < 0:
            raise VcfError("format", "malformed ##INFO line")
        key, k, val = s[k:eq], eq + 1, ""
        if k < len(s) and s[k] == '"':
            k += 1
            while k < len(s) and s[k] != '"':
                if s[k] == "\\" and k + 1 < len(s):
                    k += 1
                val += s[k]
                k += 1
            if k >= len(s):
                raise VcfError("format", "malformed ##INFO line")
            k += 1
        else:
            while k < len(s) and s[k] not in ",>":
                val += s[k]
                k += 1
        out[key] = val
        if k >= len(s):
            raise VcfError("format", "malformed ##INFO line")
        if s[k] == ">":
            if k + 1 != len(s) or not out.get("ID") or "Number" not in out or "Type" not in out:
                raise VcfError("format", "malformed ##INFO line")
            return out
        if s[k] != ",":
            raise VcfError("format", "malformed ##INFO line")
        k += 1


def parse_header(text: bytes):
    """-> (list of INFO dicts in header order, offset of the first record)."""
    pos, infos, first = 0, [], True
    while True:
        if pos >= len(text):
            raise VcfError("format", "no #CHROM line")
        nl = text.find(b"\n", pos)
        end = len(text) if nl < 0 else nl
        line, pos = text[pos:end], end + 1 if nl >= 0 else len(text)
        if line.endswith(b"\r"):
            line = line[:-1]
        if first and not line.startswith(b"##fileformat=VCF"):
            raise VcfError("format", "not a VCF file")
        first = False
        if line.startswith(b"##"):
            if line.startswith(b"##INFO=<"):
                d = _info_line(line)
                if any(o["ID"] == d["ID"] for o in infos):
                    raise VcfError("format", f"INFO {d['ID']} declared twice")
                infos.append(d)
            continue
        if not line.startswith(CHROM_LINE) or (len(line) > len(CHROM_LINE) and line[len(CHROM_LINE):len(CHROM_LINE) + 1] != b"\t"):
            raise VcfError("format", "no #CHROM line")
        return infos, pos


_SCALAR = {"Integer": pa.int32(), "Float": pa.float32(), "String": pa.string(), "Character": pa.string()}


def schema(infos, info_fields=None) -> pa.Schema:
    by_id = {d["ID"]: d for d in infos}
    if info_fields is None:
        sel = list(infos)
    else:
        sel = []
        for i in info_fields:
            if i not in by_id:
                raise VcfError("schema", f"INFO field '{i}' is not declared")
            if by_id[i] in sel:
                raise VcfError("schema", f"INFO field '{i}' is selected twice")
            sel.append(by_id[i])
    fields = list(FIXED_SCHEMA)
    for d in sel:
        if d["ID"] in FIXED:
            raise VcfError("schema", f"INFO field '{d['ID']}' has the name of a fixed column")
        if d["Type"] == "Flag":
            typ, nullable = pa.bool_(), False
        elif d["Type"] in _SCALAR:
            if d["Number"] == "0":
                raise VcfError("schema", f"INFO field '{d['ID']}': Number=0 on Type={d['Type']}")
            typ, nullable = _SCALAR[d["Type"]], True
            if d["Number"] != "1":
                typ = pa.list_(typ)
        else:
            raise VcfError("schema", f"INFO field '{d['ID']}' has the unknown Type {d['Type']}")
        md = {"bio.vcf.info.number": d["Number"], "bio.vcf.info.type": d["Type"], "bio.vcf.info.description": d.get("Description", "")}
        fields.append(pa.field(d["ID"], typ, nullable, metadata=md))
    return pa.schema(fields)


def _i32(v: bytes):
    s = v[1:] if v[:1] in (b"+", b"-") else v
    if not s or not s.isdigit():
        return None
    x = int(v)
    return x if -2**31 <= x < 2**31 else None


@lru_cache(maxsize=1 << 16)
def _f32(v: bytes):
    try:
        return struct.unpack("<f", struct.pack("<I", f32_from_text(v.decode("latin-1"))))[0]
    except Exception:
        return None


def _value(typ, v: bytes, r):
    """One INFO value of a non-Flag column -> a Python value (None for '.')."""
    if v == b".":
        return None
    if pa.types.is_list(typ):
        out = []
        for e in v.split(b","):
            out.append(None if e == b"." else _value(typ.value_type, e, r))
        return out
    if pa.types.is_string(typ):
        if b"," in v:
            raise VcfError("schema", "',' in a Number=1 value", r)
        return v
    x = _i32(v) if pa.types.is_int32(typ) else _f32(v)
    if x is None:
        raise VcfError("schema", "value does not parse as its type", r)
    return x


def _text(b: bytes, r):
    if not b.isascii():
        raise VcfError("format", "byte 0x80 or above", r)
    return b.decode()


def scan_text(text: bytes, info_fields=None, projection=None, zero_based=True) -> pa.Table:
    """The inflated VCF text -> the scan's rows (projection: schema indices, None = all)."""
    infos, pos = parse_header(text)
    sc = schema(infos, info_fields)
    idx = list(range(len(sc))) if projection is None else list(projection)
    names = [sc.field(i).name for i in idx]
    body = text[pos:]
    lines = body.split(b"\n")
    if lines and lines[-1] == b"":
        lines.pop()
    cols = {n: [] for n in names}
    info_types = {sc.field(i).name: sc.field(i).type for i in range(8, len(sc))}
    looked_up = {n for n in names if n in info_types} | {"END"}
    for r, raw in enumerate(lines):
        if len(raw) + 1 > MAX_LINE:
            raise VcfError("unsupported", "line longer than 16 MiB", r)
        line = raw[:-1] if raw.endswith(b"\r") else raw
        if not line or line.startswith(b"#"):
            raise VcfError("format", "'#' or empty line", r)
        f = line.split(b"\t")
        if len(f) < 8:
            raise VcfError("format", "fewer than 8 fields", r)
        if not f[0]:
            raise VcfError("format", "empty CHROM", r)
        if not f[1].isdigit() or len(f[1]) > 10 or int(f[1]) > 2**31 - 1:
            raise VcfError("format", "bad POS", r)
        p = int(f[1])
        if p == 0:
            raise VcfError("unsupported", "POS 0", r)
        if not f[3]:
            raise VcfError("format", "empty REF", r)
        qual = None
        if f[5] != b".":
            qual = _f32(f[5])
            if qual is None:
                raise VcfError("format", "bad QUAL", r)
        info = {}
        if f[7] not in (b".", b""):
            for tok in f[7].split(b";"):
                if not tok:
                    continue
                k, eq, v = tok.partition(b"=")
                k = k.decode("latin-1")
                if k not in looked_up:
                    continue
                if k in info:
                    raise VcfError("format", f"INFO key {k} twice", r)
                info[k] = v if eq else None          # None: no '='
        end = p + len(f[3]) - 1
        if "END" in info:
            v = info["END"]
            if v is None:
                raise VcfError("schema", "END without a value", r)
            if v != b".":
                e = _i32(v)
                if e is None:
                    raise VcfError("schema", "END is not an integer", r)
                if e < p:
                    raise VcfError("format", "END below POS", r)
                end = e
        fixed = {"chrom": f[0], "start": p - 1 if zero_based else p, "end": end, "id": None if f[2] == b"." else f[2],
                 "ref": f[3], "alt": None if f[4] == b"." else f[4], "qual": qual, "filter": None if f[6] == b"." else f[6]}
        for n in names:
            if n in fixed:
                v = fixed[n]
            else:
                typ, present = info_types[n], n in info
                if pa.types.is_boolean(typ):
                    if present and info[n] is not None:
                        raise VcfError("schema", "Flag with a value", r)
                    v = present
                elif not present:
                    v = None
                elif info[n] is None:
                    raise VcfError("schema", "key without '='", r)
                else:
                    v = _value(typ, info[n], r)
            cols[n].append(v)
    out_fields = [sc.field(i) for i in idx]
    arrays = []
    for fld in out_fields:
        vals = cols[fld.name]
        t = fld.type
        if pa.types.is_string(t):
            vals = [None if v is None else _text(v, r) for r, v in enumerate(vals)]
        elif pa.types.is_list(t) and pa.types.is_string(t.value_type):
            vals = [None if v is None else [None if e is None else _text(e, r) for e in v] for r, v in enumerate(vals)]
        arrays.append(pa.array(vals, t))
    if not out_fields:
        return pa.Table.from_batches([pa.RecordBatch.from_struct_array(pa.array([{}] * len(lines), pa.struct([])))])
    return pa.Table.from_arrays(arrays, schema=pa.schema(out_fields))
