"""GPU: the single-CTA scans (kernels_scan.cuh) at their 1024-element step boundaries, through the public API.  The scan CTA takes
1024 elements per step and carries the running total into the next step; a wrong carry only shows on inputs that take a second
step.

- Newline and record-start scans: a FASTQ or FASTA file of 4096-byte BGZF members, scanned with chunk_inflated_bytes = k x 4096,
  gives chunks of exactly k members; the first chunk carries nothing in, so its newline scan (and FASTA's '>' scan) runs over
  exactly k tiles of FQ_TILE = 4096 bytes.
- Member offsets of the writer: one FASTQ batch of exactly k x 0xff00 bytes of text is one slice, compressed by one deflate launch
  of k members, whose sizes are scanned into the members' file offsets; nothing is left for the final flush."""
import numpy as np
import pyarrow as pa
import pytest

from conftest import make_fastq_text, write_bgzf
from oracle import fasta_oracle as FA
from oracle import fastq_oracle as FQ
from oracle import fastq_write_oracle as FW
from oracle.bam_write_oracle import BGZF_BLOCK, BGZF_EOF, inflate_bgzf

pytestmark = pytest.mark.gpu

TILE = 4096
STEPS = [1023, 1024, 1025, 2049]             # tiles (members) per scan: one step short, exact, one over, three steps


def _scan(cls, path, chunk):
    p = cls(str(path), chunk_inflated_bytes=chunk)
    try:
        plan = p.scan()
        return pa.Table.from_batches(list(plan.execute(0)), schema=plan.schema()), plan.last_stats
    finally:
        p.close()


def _assert_equal(got: pa.Table, want: pa.Table, what):
    assert got.num_rows == want.num_rows, f"{what}: {got.num_rows} rows, want {want.num_rows}"
    for name in want.schema.names:
        assert got[name].combine_chunks().equals(want[name].combine_chunks()), f"{what}: column {name} differs"


@pytest.fixture(scope="module")
def fastq_4k(tmp_path_factory):
    text = make_fastq_text(45000, 31)
    assert len(text) > (max(STEPS) + 64) * TILE
    path = tmp_path_factory.mktemp("edges") / "m4k.fastq.bgz"
    write_bgzf(path, text, block=TILE, level=1)
    return path, pa.Table.from_batches([FQ.OracleFastq(path).scan()]), -(-len(text) // TILE)


@pytest.fixture(scope="module")
def fasta_4k(tmp_path_factory):
    rng = np.random.default_rng(32)
    parts = []
    for i in range(60000):
        seq = np.frombuffer(b"ACGTNacgt", np.uint8)[rng.integers(0, 9, int(rng.integers(0, 300)))].tobytes()
        parts.append(b">r%d%s\n" % (i, b" d%d" % i if i % 3 else b"") + b"".join(seq[k:k + 60] + b"\n" for k in range(0, len(seq), 60)))
    text = b"".join(parts)
    assert len(text) > (max(STEPS) + 64) * TILE
    path = tmp_path_factory.mktemp("edges") / "m4k.fa.bgz"
    write_bgzf(path, text, block=TILE, level=1)
    return path, pa.Table.from_batches([FA.scan_text(text)]), -(-len(text) // TILE)


@pytest.mark.parametrize("k", STEPS)
def test_fastq_newline_scan_at_step_boundaries(fastq_4k, k):
    import bamscan
    path, want, members = fastq_4k
    got, st = _scan(bamscan.FastqTableProvider, path, k * TILE)
    assert st["chunks"] == -(-members // k), st            # k members per chunk: the first chunk's scan has k tiles
    _assert_equal(got, want, f"FASTQ, {k} tiles")


@pytest.mark.parametrize("k", STEPS)
def test_fasta_newline_and_record_start_scans_at_step_boundaries(fasta_4k, k):
    import bamscan
    path, want, members = fasta_4k
    got, st = _scan(bamscan.FastaTableProvider, path, k * TILE)
    assert st["chunks"] == -(-members // k), st
    _assert_equal(got, want, f"FASTA, {k} tiles")


@pytest.fixture(scope="module")
def fastq_rows():
    """Records of exactly 255 bytes (9-byte name, 120 bases, 120 qualities): 256 of them fill one 0xff00-byte BGZF member."""
    n = 256 * max(STEPS)
    rng = np.random.default_rng(33)
    seq = np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, (n, 120))]
    qual = rng.integers(33, 74, (n, 120), dtype=np.uint8)
    return pa.RecordBatch.from_arrays([pa.array([f"r{i:08d}" for i in range(n)], pa.string()), pa.nulls(n, pa.string()),
                                       pa.array([r.tobytes().decode() for r in seq], pa.string()),
                                       pa.array([r.tobytes().decode() for r in qual], pa.string())], schema=FQ.SCHEMA)


@pytest.mark.parametrize("k", STEPS)
def test_fastq_write_member_offsets_at_step_boundaries(fastq_rows, k, tmp_path):
    import bamscan
    batch = fastq_rows.slice(0, 256 * k)
    text = FW.render_batch(batch)
    assert len(text) == k * BGZF_BLOCK
    out = tmp_path / "o.fastq.bgz"
    ex = bamscan.FastqWriteExec(str(out), FQ.SCHEMA)
    assert ex.execute([batch]) == batch.num_rows
    assert ex.stats["members"] == k, ex.stats
    data = out.read_bytes()
    stream, sizes = inflate_bgzf(data)                          # strict: member headers, BSIZE chain, CRC-32, ISIZE
    assert data.endswith(BGZF_EOF) and sizes == [BGZF_BLOCK] * k + [0]
    assert stream == text
    got, _ = _scan(bamscan.FastqTableProvider, out, 0)
    _assert_equal(got, pa.Table.from_batches([batch]), f"FASTQ write, {k} members")
