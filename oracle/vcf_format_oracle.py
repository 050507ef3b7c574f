"""CPU restatement of the VCF scan's FORMAT columns -- TEST INFRASTRUCTURE ONLY (nothing under datafusion-bio-formats_b200/ imports
it; only tests/ may).  It extends oracle/vcf_oracle.py, whose rules for the header, the fixed columns and INFO hold unchanged.

As there, every rule is this project's own statement of the format (DESIGN 3.11a), unpinned.  Where the reference may well differ:
the column names (format_<ID>), the nested types, and GT kept as text (not allele indices and a phased flag).

format_fields is a list of FORMAT IDs.  None, the default, and [] select none -- unlike info_fields, where None selects all -- and
then the header, schema and records are read exactly as oracle/vcf_oracle.py reads them.

Header, read only when format_fields is non-empty:
- ##FORMAT=<ID,Number,Type,Description> lines parse as ##INFO lines do; a malformed one or an ID declared twice is a format error;
- the sample names are the #CHROM fields behind FORMAT; fields behind INFO whose first one is not FORMAT are a format error.

Schema: behind the INFO columns, in format_fields order, one non-nullable column format_<ID> per ID holding one element per sample
(header sample order).  Number=1 -> List<Int32 / Float32 / Utf8> (Integer / Float / String or Character) with nullable elements;
Integer or Float with any other Number -> List<List<Int32 / Float32>>, middle lists and leaves nullable.  Field metadata
bio.vcf.format.{number,type,description}; schema metadata bio.vcf.samples = json.dumps(sample names, ensure_ascii=False).
Refused at open, in this order: more than 16 IDs (unsupported); no samples (schema); then per ID in order: undeclared, selected
twice, Type=Flag, an unknown Type, Number=0 (schema); String / Character with Number other than 1 (unsupported); format_<ID>
equal to an existing column name (schema).

Records, checked only when a FORMAT column is projected:
- a line must have exactly 9 + S fields (format error);
- the FORMAT field is a ':'-separated key list ('.' or empty: no keys) whose order may differ per line; a projected key given twice
  is a format error (other keys are not compared);
- a sample is ':'-separated values matched to the keys by position; a lone '.' has no values; missing trailing values, a '.'
  value and keys the line does not list give NULL (for nested columns a NULL middle list); more values than keys is a format
  error;
- inside a nested value ',' separates leaves and '.' is a NULL leaf;
- values parse as INFO values do; one that does not (an empty number, a ',' in a Number=1 value) is a schema error; a byte of
  0x80 or above in a projected text value is a format error;
- GT is a String: kept as written, only a lone '.' is NULL.
The scan fails at the first record with an error; when a record breaks a rule of oracle/vcf_oracle.py and a FORMAT rule, the
former is reported.
"""
import json
from functools import lru_cache

import pyarrow as pa

from oracle import vcf_oracle as V
from oracle.vcf_oracle import VcfError

MAX_FORMAT = 16
_SCALAR = {"Integer": pa.int32(), "Float": pa.float32(), "String": pa.string(), "Character": pa.string()}


def _format_line(line: bytes) -> dict:
    """One ##FORMAT=<...> line, parsed by the ##INFO line rules."""
    try:
        return V._info_line(b"##INFO=<" + line[len(b"##FORMAT=<"):])
    except VcfError:
        raise VcfError("format", "malformed ##FORMAT line") from None


def parse_format_header(text: bytes):
    """-> (list of FORMAT dicts in header order, sample names).  Read only when format_fields is non-empty."""
    pos, formats = 0, []
    while pos < len(text):
        nl = text.find(b"\n", pos)
        end = len(text) if nl < 0 else nl
        line, pos = text[pos:end], end + 1 if nl >= 0 else len(text)
        if line.endswith(b"\r"):
            line = line[:-1]
        if line.startswith(b"##FORMAT=<"):
            d = _format_line(line)
            if any(o["ID"] == d["ID"] for o in formats):
                raise VcfError("format", f"FORMAT {d['ID']} declared twice")
            formats.append(d)
        elif not line.startswith(b"##"):
            extra = line.split(b"\t")[8:]
            if extra and extra[0] != b"FORMAT":
                raise VcfError("format", "the first field behind INFO is not FORMAT")
            return formats, [x.decode("utf-8", "surrogateescape") for x in extra[1:]]
    raise VcfError("format", "no #CHROM line")


def schema(infos, info_fields=None, format_fields=None, format_header=None) -> pa.Schema:
    """oracle/vcf_oracle.py's schema, then the FORMAT columns (format_header: parse_format_header's result)."""
    base = V.schema(infos, info_fields)
    if not format_fields:
        return base
    formats, samples = format_header
    if len(format_fields) > MAX_FORMAT:
        raise VcfError("unsupported", f"more than {MAX_FORMAT} FORMAT fields")
    if not samples:
        raise VcfError("schema", "FORMAT fields selected but the header has no samples")
    fields = list(base)
    by_id = {d["ID"]: d for d in formats}
    for i, fid in enumerate(format_fields):
        if fid not in by_id:
            raise VcfError("schema", f"FORMAT field '{fid}' is not declared")
        if fid in format_fields[:i]:
            raise VcfError("schema", f"FORMAT field '{fid}' is selected twice")
        d = by_id[fid]
        if d["Type"] == "Flag":
            raise VcfError("schema", f"FORMAT field '{fid}' has Type=Flag")
        if d["Type"] not in _SCALAR:
            raise VcfError("schema", f"FORMAT field '{fid}' has the unknown Type {d['Type']}")
        if d["Number"] == "0":
            raise VcfError("schema", f"FORMAT field '{fid}' has Number=0")
        typ = _SCALAR[d["Type"]]
        if d["Number"] != "1":
            if pa.types.is_string(typ):
                raise VcfError("unsupported", f"FORMAT field '{fid}': Type={d['Type']} with Number={d['Number']}")
            typ = pa.list_(typ)
        name = "format_" + fid
        if any(f.name == name for f in fields):
            raise VcfError("schema", f"FORMAT field '{fid}': a column named {name} exists")
        md = {"bio.vcf.format.number": d["Number"], "bio.vcf.format.type": d["Type"], "bio.vcf.format.description": d.get("Description", "")}
        fields.append(pa.field(name, pa.list_(typ), False, metadata=md))
    return pa.schema(fields, metadata={"bio.vcf.samples": json.dumps(samples, ensure_ascii=False)})


def _format_value(typ, v: bytes):
    """One FORMAT value of an element -> a Python value (None for '.')."""
    if v == b".":
        return None
    if pa.types.is_list(typ):
        return [None if e == b"." else _format_value(typ.value_type, e) for e in v.split(b",")]
    if b"," in v:
        raise VcfError("schema", "',' in a Number=1 value")
    if pa.types.is_string(typ):
        if not v.isascii():
            raise VcfError("format", "byte 0x80 or above")
        return v.decode()
    x = V._i32(v) if pa.types.is_int32(typ) else V._f32(v)
    if x is None:
        raise VcfError("schema", "FORMAT value does not parse as its type")
    return x


@lru_cache(maxsize=1 << 16)
def _sample(smp: bytes, at: tuple, types: tuple, n_keys: int) -> tuple:
    """One sample -> its element per FORMAT column (at: each column's key index in the line's FORMAT field, or None)."""
    vals = [] if smp == b"." else smp.split(b":")
    if len(vals) > n_keys:
        raise VcfError("format", "more values than keys")
    return tuple(None if k is None or k >= len(vals) else _format_value(t, vals[k]) for k, t in zip(at, types))


def _format_row(f, n_samples, ids, types, r):
    """One record's FORMAT columns: a list per column of one element per sample (ids, types: per column)."""
    if len(f) != 9 + n_samples:
        raise VcfError("format", "not 9 + samples fields", r)
    keys = [] if f[8] in (b".", b"") else f[8].split(b":")
    at = [None] * len(ids)
    for k, key in enumerate(keys):
        for c, fid in enumerate(ids):
            if key == fid:
                if at[c] is not None:
                    raise VcfError("format", "FORMAT key given twice", r)
                at[c] = k
    try:
        per_sample = [_sample(smp, tuple(at), types, len(keys)) for smp in f[9:]]
    except VcfError as e:
        raise VcfError(e.kind, str(e).split(": ", 1)[1], r) from None
    return [[ps[c] for ps in per_sample] for c in range(len(ids))]


def scan_text(text: bytes, info_fields=None, projection=None, zero_based=True, format_fields=None) -> pa.Table:
    """The inflated VCF text -> the scan's rows (projection: schema indices, None = all; no index twice)."""
    if not format_fields:
        return V.scan_text(text, info_fields, projection, zero_based)
    infos, pos = V.parse_header(text)
    fh = parse_format_header(text)
    sc = schema(infos, info_fields, format_fields, fh)
    info_end = len(sc) - len(format_fields)
    idx = list(range(len(sc))) if projection is None else list(projection)
    base_idx = [i for i in idx if i < info_end]
    fmt_idx = [i for i in idx if i >= info_end]
    base, base_err = None, None
    try:
        base = V.scan_text(text, info_fields, base_idx, zero_based)
    except VcfError as e:
        base_err = e
    fmt_cols = {}
    if fmt_idx:
        lines = text[pos:].split(b"\n")
        if lines and lines[-1] == b"":
            lines.pop()
        ids = [sc.field(i).name[len("format_"):].encode() for i in fmt_idx]
        types = tuple(sc.field(i).type.value_type for i in fmt_idx)
        vals = [[] for _ in fmt_idx]
        stop = len(lines) if base_err is None or base_err.record is None else base_err.record
        for r in range(min(stop + 1, len(lines))):
            raw = lines[r]
            line = raw[:-1] if raw.endswith(b"\r") else raw
            try:
                row = _format_row(line.split(b"\t"), len(fh[1]), ids, types, r)
            except VcfError:
                if r < stop:
                    raise
                break          # the same record breaks a rule of oracle/vcf_oracle.py: that error is reported
            for c in range(len(fmt_idx)):
                vals[c].append(row[c])
        if base_err is None:
            fmt_cols = {i: pa.array(vals[c], sc.field(i).type) for c, i in enumerate(fmt_idx)}
    if base_err is not None:
        raise base_err
    if not idx:
        return base
    arrays = [base.column(base_idx.index(i)) if i < info_end else fmt_cols[i] for i in idx]
    return pa.Table.from_arrays(arrays, schema=pa.schema([sc.field(i) for i in idx], metadata=sc.metadata))
