"""CPU restatement of the FASTQ write path -- TEST INFRASTRUCTURE ONLY (nothing under datafusion-bio-formats_b200/ imports it).

A row is written as '@' + name, then ' ' + description when the description is non-NULL and non-empty, then '\\n', the
sequence, "\\n+\\n", the quality scores and '\\n'.  This is the layout of the reference's two FASTQ fixtures (bare '+' lines,
one space in front of the description, LF line ends, a final newline): re-rendering the rows the read oracle gets from them
gives their inflated bytes exactly (tests/test_fastq_write_oracle.py).  The reference's FASTQ writer is not vendored; the
refusals below are this project's rules, chosen so that the file reads back as the same rows (DESIGN 3.8):
  * a NULL name, sequence or quality_scores;
  * a '\\n' or '\\r' in any field (the reader splits lines there and drops one '\\r' in front of a '\\n');
  * a space or tab in the name (the reader splits the definition line at the first one).
Sequence and quality lengths are not compared; bytes are written as given.  Columns are looked up by name; description is
optional and every other column is ignored.
"""
import pyarrow as pa

from oracle.bam_write_oracle import BGZF_BLOCK, BGZF_EOF, bgzf_member


class WriteError(Exception):
    pass


def render_record(row: int, name, desc, seq, qual) -> bytes:
    """One record from str / bytes / None fields; raises WriteError("row N: ...") on the refusal rules, checked in this order."""
    def b(v):
        return v.encode() if isinstance(v, str) else v
    name, desc, seq, qual = b(name), b(desc), b(seq), b(qual)
    for v, what in ((name, "name"), (seq, "sequence"), (qual, "quality_scores")):
        if v is None:
            raise WriteError(f"row {row}: {what} is NULL")
    if b"\n" in name or b"\r" in name:
        raise WriteError(f"row {row}: line break in name")
    if b" " in name or b"\t" in name:
        raise WriteError(f"row {row}: space or tab in name")
    for v, what in ((desc or b"", "description"), (seq, "sequence"), (qual, "quality_scores")):
        if b"\n" in v or b"\r" in v:
            raise WriteError(f"row {row}: line break in {what}")
    head = b"@" + name + (b" " + desc if desc else b"")
    return head + b"\n" + seq + b"\n+\n" + qual + b"\n"


def render_batch(batch: pa.RecordBatch) -> bytes:
    """The FASTQ text of a batch (columns by name: name, sequence, quality_scores required, description optional)."""
    names = batch.schema.names
    for c in ("name", "sequence", "quality_scores"):
        if c not in names:
            raise WriteError(f"Required column '{c}' not found in batch")

    def col(c):
        return batch.column(names.index(c)).to_pylist()
    n, s, q = col("name"), col("sequence"), col("quality_scores")
    d = col("description") if "description" in names else [None] * batch.num_rows
    return b"".join(render_record(r, n[r], d[r], s[r], q[r]) for r in range(batch.num_rows))


def bgzf_bytes(text: bytes, level: int = 6) -> bytes:
    """`text` as 0xff00-byte BGZF members followed by the EOF marker (an empty text: the EOF marker alone)."""
    return b"".join(bgzf_member(text[i:i + BGZF_BLOCK], level) for i in range(0, len(text), BGZF_BLOCK)) + BGZF_EOF


def write_fastq(path, batches, compression: int = 0) -> int:
    """The file FastqWriteExec writes, up to the DEFLATE bytes: compression 0 (zlib level 6) / 1 (level 0) BGZF, 2 plain text.
    Returns the row count."""
    batches = list(batches)
    text = b"".join(render_batch(b) for b in batches)
    with open(path, "wb") as f:
        f.write(text if compression == 2 else bgzf_bytes(text, 6 if compression == 0 else 0))
    return sum(b.num_rows for b in batches)
