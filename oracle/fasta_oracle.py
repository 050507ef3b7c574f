"""CPU restatement of the FASTA scan -- TEST INFRASTRUCTURE ONLY (nothing under datafusion-bio-formats_b200/ imports it; only
tests/ may).

The reference's FASTA provider (bio-format-fasta) is not vendored here and no reference fixture exists, so every rule below is
this project's own statement of the format (DESIGN 3.10), unpinned:

- a record starts with a '>' at the start of a line; its definition is the rest of that line without one trailing '\\r', split at
  its first space or tab into name and description (an empty description is NULL, an empty name is an error);
- its sequence is every following line up to the next line that starts with '>' or the end of the text, each without its '\\n'
  and one trailing '\\r', joined with nothing in between; blank lines add nothing, bytes are kept as given; no sequence line: "";
- an unterminated last line is a line;
- refused: bytes other than whitespace (space, tab, '\\n', '\\r', form feed) in front of the first '>', and any byte of 0x80 or
  above in a column (the scan checks the projected columns);
- a record of more than 1 GiB of text (definition line and line breaks included) is refused as unsupported.
"""
import pyarrow as pa

SCHEMA = pa.schema([pa.field("name", pa.string(), False), pa.field("description", pa.string(), True),
                    pa.field("sequence", pa.string(), False)])
MAX_RECORD = 1 << 30
_SPACE = b" \t\n\r\f"


class FastaError(ValueError):
    """`unsupported` is True for a record over MAX_RECORD (BAMSCAN_ERR_UNSUPPORTED), else a format error; `record` is 0-based."""

    def __init__(self, record, why, unsupported=False):
        super().__init__(f"record {record}: {why}")
        self.record = record
        self.unsupported = unsupported


def _strip(line: bytes) -> bytes:
    return line[:-1] if line.endswith(b"\r") else line


def parse_records(text: bytes):
    """-> list of (name, description or None, sequence) byte strings."""
    lines = text.split(b"\n")
    if lines and lines[-1] == b"":
        lines.pop()                       # the text ended with a newline
    recs, cur, seq, size = [], None, [], 0
    for ln in lines:
        if ln.startswith(b">"):
            if cur is not None:
                recs.append((cur, seq, size))
            cur, seq, size = ln, [], len(ln) + 1
            continue
        if cur is None:
            if ln.strip(_SPACE):
                raise FastaError(0, "bytes other than whitespace in front of the first '>'")
            continue
        seq.append(_strip(ln))
        size += len(ln) + 1
    if cur is not None:
        recs.append((cur, seq, size))
    out = []
    for i, (d, seq, size) in enumerate(recs):
        if size > MAX_RECORD:
            raise FastaError(i, "record larger than 1 GiB", unsupported=True)
        d = _strip(d)[1:]
        k = next((j for j, b in enumerate(d) if b in (0x20, 0x09)), len(d))
        name, desc, s = d[:k], d[k + 1:], b"".join(seq)
        if not name:
            raise FastaError(i, "empty name")
        if any(b >= 0x80 for b in name + desc) or max(s, default=0) >= 0x80:
            raise FastaError(i, "byte 0x80 or above")
        out.append((name, desc if desc else None, s))
    return out


def to_batch(recs, projection=None) -> pa.RecordBatch:
    cols = [pa.array([r[0].decode() for r in recs], pa.string()),
            pa.array([None if r[1] is None else r[1].decode() for r in recs], pa.string()),
            pa.array([r[2].decode() for r in recs], pa.string())]
    idx = list(range(3)) if projection is None else list(projection)
    if not idx:
        return pa.RecordBatch.from_struct_array(pa.array([{}] * len(recs), pa.struct([])))
    return pa.RecordBatch.from_arrays([cols[i] for i in idx], schema=pa.schema([SCHEMA.field(i) for i in idx]))


def scan_text(text: bytes, projection=None) -> pa.RecordBatch:
    """The inflated FASTA text -> the scan's rows as one pyarrow.RecordBatch."""
    return to_batch(parse_records(text), projection)
