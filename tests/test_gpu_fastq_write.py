"""GPU: the FASTQ write path (bamscan_fastq_writer_open + bamscan_writer_*) against oracle/fastq_write_oracle.py.  The written
file passes a strict BGZF reader (BSIZE chain, CRC-32, ISIZE, 0xff00-byte members, EOF marker), its inflated text equals the
oracle's byte for byte, and the GPU FASTQ scan reads it back to the rows that went in."""
import random

import pyarrow as pa
import pytest

from conftest import GOLDEN, make_fastq_text, write_bgzf
from oracle import fastq_oracle as R
from oracle import fastq_write_oracle as FW
from oracle.bam_write_oracle import BGZF_BLOCK, BGZF_EOF, bgzf_member, inflate_bgzf
from test_fastq_write_oracle import REFUSALS, _batch, _random_rows, refusal_batch

pytestmark = pytest.mark.gpu
FQ = GOLDEN / "fastq"


def gpu_write(path, batches, schema, compression=None):
    import bamscan
    ex = bamscan.FastqWriteExec(str(path), schema, compression)
    n = ex.execute(batches)
    return n, ex.stats


def check_bgzf(path, want_text):
    data = open(path, "rb").read()
    stream, sizes = inflate_bgzf(data)                          # strict: member headers, BSIZE chain, CRC-32, ISIZE
    assert data.endswith(BGZF_EOF) and sizes[-1] == 0
    assert all(s == BGZF_BLOCK for s in sizes[:-2]) and (len(sizes) == 1 or 0 < sizes[-2] <= BGZF_BLOCK)
    assert len(stream) == len(want_text)
    if stream != want_text:
        i = next(k for k in range(len(want_text)) if stream[k] != want_text[k])
        raise AssertionError(f"inflated text differs from the oracle at byte {i}: {stream[i:i+24]!r} vs {want_text[i:i+24]!r}")
    return len(data)


def scan_table(path, **kw):
    import bamscan
    p = bamscan.FastqTableProvider(str(path), **kw)
    t = p.scan().collect()
    p.close()
    return t


def assert_rows(got: pa.Table, want, what=""):
    want = pa.Table.from_batches(want) if isinstance(want, list) else want
    assert got.num_rows == want.num_rows, f"{what}: {got.num_rows} rows, want {want.num_rows}"
    for name in ("name", "description", "sequence", "quality_scores"):
        assert got[name].combine_chunks().equals(want[name].combine_chunks().cast(pa.string())), f"{what}: column {name} differs"


@pytest.mark.parametrize("name", ["sample.fastq.bgz", "example.fastq.bgz"])
def test_fixture_scan_write_is_byte_exact_and_reads_back(name, tmp_path):
    import bamscan
    text = R.gunzip_members((FQ / name).read_bytes())
    p = bamscan.FastqTableProvider(str(FQ / name))
    schema = p.schema()
    batches = list(p.scan().execute(0))
    orig = pa.Table.from_batches(batches, schema=schema)
    for comp in (0, 1):
        out = tmp_path / f"o{comp}.fastq.bgz"
        n, st = gpu_write(out, batches, schema, comp)
        assert n == orig.num_rows == st["rows"] and st["bam_bytes"] == len(text) and st["members"] == (len(text) + BGZF_BLOCK - 1) // BGZF_BLOCK
        size = check_bgzf(out, text)
        assert (size > len(text)) == (comp == 1)
        assert_rows(scan_table(out), orig, f"{name} compression {comp}")
    out = tmp_path / "o.fastq"
    n, st = gpu_write(out, batches, schema)                       # plain by extension
    assert out.read_bytes() == text and st["members"] == 0 and st["ms_deflate"] == 0 and st["compressed_bytes"] == len(text)
    p.close()


def _synthetic(tmp_path):
    """60 k reads of the scan tests' generator (descriptions with spaces / tabs / none, quality lines starting with '@' / '+')
    plus 200 long reads of 10-100 kb."""
    recs = R.parse_records(make_fastq_text(60000, 23))
    rng = random.Random(9)
    for i in range(200):
        L = rng.randint(10000, 100000)
        recs.append((f"long{i}".encode(), rng.choice([None, b"len=%d" % L]), "".join(rng.choices("ACGT", k=L)).encode(),
                     "".join(rng.choices("#+5?@FI", k=L)).encode()))
    rows = [(n.decode(), None if d is None else d.decode(), s.decode(), q.decode()) for n, d, s, q in recs]
    return _batch(rows)


def test_synthetic_sliced_batches_long_reads_and_partitions(tmp_path):
    import bamscan
    b = _synthetic(tmp_path)
    n = b.num_rows
    cuts = [0, 1, 17, 17 + 8192, n // 3, n // 3, 60000, n - 7, n]        # empty and sliced batches (array offset != 0); long reads last
    parts = [b.slice(x, y - x) for x, y in zip(cuts, cuts[1:])]
    text = FW.render_batch(b)
    out = tmp_path / "syn.fastq.bgz"
    rows, st = gpu_write(out, parts, b.schema)
    assert rows == n and st["batches"] == len(parts)
    size = check_bgzf(out, text)
    z6 = sum(len(bgzf_member(text[i:i + BGZF_BLOCK])) for i in range(0, len(text), BGZF_BLOCK))
    assert size < 1.6 * z6 and size < 0.8 * len(text), (size, z6, len(text))
    want = pa.Table.from_batches([b])
    p = bamscan.FastqTableProvider(str(out))
    for tp in (1, 2, 4, 8):
        plan = p.scan(None, None, None, target_partitions=tp, partition_mode="block_range")
        got, stats = [], []
        for i in range(plan.output_partition_count()):
            got += list(plan.execute(i))
            stats.append(plan.last_stats)
        assert_rows(pa.Table.from_batches(got, schema=plan.schema()), want, f"{tp} partitions")
        if len(stats) > 1:
            bamscan.check_partition_seams(stats)
    p.close()


def test_seeded_random_rows_against_the_oracle(tmp_path):
    rows = _random_rows(random.Random(20261020), 6000)
    for with_desc in (True, False):
        b = _batch(rows, with_desc)
        text = FW.render_batch(b)
        for comp in (0, 2):
            out = tmp_path / f"rnd{int(with_desc)}{comp}.fastq.bgz"
            gpu_write(out, [b.slice(0, 2222), b.slice(2222)], b.schema, comp)
            if comp == 2:
                assert out.read_bytes() == text
            else:
                check_bgzf(out, text)


@pytest.mark.parametrize("change,msg", REFUSALS, ids=[m.replace(" ", "_") + f"_{i}" for i, (_c, m) in enumerate(REFUSALS)])
def test_each_refusal_rule(change, msg, tmp_path):
    import bamscan
    b = refusal_batch(change, bad_row=37, n=100)
    with pytest.raises(FW.WriteError, match=f"row 37: {msg}"):
        FW.render_batch(b)
    with pytest.raises(bamscan.BamScanError, match=f"row 37: {msg}") as e:
        gpu_write(tmp_path / "bad.fastq.bgz", [b], b.schema)
    assert e.value.code == -2
    # the row number is the row within the batch, the same for a sliced batch
    with pytest.raises(bamscan.BamScanError, match=f"row 30: {msg}"):
        gpu_write(tmp_path / "bad2.fastq", [b.slice(7)], b.schema)


def test_device_batches_are_written_in_place(tmp_path):
    import bamscan
    src = tmp_path / "src.fastq.bgz"
    write_bgzf(src, make_fastq_text(30000, 4))
    p = bamscan.FastqTableProvider(str(src), chunk_inflated_bytes=1 << 20)     # several device batches
    host = list(p.scan().execute(0))
    out_h, out_d = tmp_path / "h.fastq.bgz", tmp_path / "d.fastq.bgz"
    gpu_write(out_h, host, p.schema())
    ex = bamscan.FastqWriteExec(str(out_d), p.schema())
    n = ex.execute(p.scan().execute_device(0))
    assert n == 30000 and ex.stats["arrow_bytes"] == 0 and ex.stats["batches"] > 1
    text = FW.render_batch(pa.Table.from_batches(host).combine_chunks().to_batches()[0])
    check_bgzf(out_h, text)
    check_bgzf(out_d, text)
    # insert_into on a provider made for writing, and on the scanned provider's own file
    pw = bamscan.FastqTableProvider.new_for_write(str(tmp_path / "w.fastq"))
    assert pw.insert_into(host) == 30000 and (tmp_path / "w.fastq").read_bytes() == text
    with pytest.raises(NotImplementedError):
        pw.insert_into(host, "append")
    p.close()
    own = tmp_path / "own.fastq.bgz"
    own.write_bytes(src.read_bytes())
    po = bamscan.FastqTableProvider(str(own))
    keep = [b.slice(0, b.num_rows // 2) for b in po.scan().execute(0)]
    assert po.insert_into(keep) == sum(b.num_rows for b in keep)
    po.close()
    check_bgzf(own, FW.render_batch(pa.Table.from_batches(keep).combine_chunks().to_batches()[0]))


def test_bam_scan_batches_write_as_fastq(tmp_path):
    """A BAM scan's batch: extra columns are ignored, there is no description column, bases are written as stored."""
    import bamscan
    for name in ("multi_chrom.bam", "nanopore_custom_tags.bam"):
        p = bamscan.BamTableProvider(str(GOLDEN / name), None, True, ["NM"], index_path="")
        batches = list(p.scan(None, [], None).execute(0))
        text = FW.render_batch(pa.Table.from_batches(batches).combine_chunks().to_batches()[0])
        out = tmp_path / f"{name}.fastq.bgz"
        n, _st = gpu_write(out, batches, p.schema())
        assert n == sum(b.num_rows for b in batches)
        check_bgzf(out, text)
        p.close()


def test_edge_files(tmp_path):
    import bamscan
    s = bamscan.FASTQ_SCHEMA
    n, st = gpu_write(tmp_path / "none.fastq.bgz", [], s)                    # zero rows: the EOF marker alone
    assert n == 0 and (tmp_path / "none.fastq.bgz").read_bytes() == BGZF_EOF and st["members"] == 0
    gpu_write(tmp_path / "none.fastq", [pa.RecordBatch.from_pylist([], schema=s)], s)
    assert (tmp_path / "none.fastq").read_bytes() == b""
    one = pa.RecordBatch.from_pylist([dict(name="r", description="d e", sequence="ACGT", quality_scores="IIII")], schema=s)
    gpu_write(tmp_path / "one.fastq.bgz", [one], s)
    check_bgzf(tmp_path / "one.fastq.bgz", b"@r d e\nACGT\n+\nIIII\n")
    # high-entropy qualities and names; stored members (compression 1) carry the same text
    rng = random.Random(5)
    rows = [dict(name="".join(chr(rng.randint(33, 126)) for _ in range(30)), description=None,
                 sequence="".join(rng.choices("ACGTN", k=250)), quality_scores="".join(chr(rng.randint(33, 126)) for _ in range(250)))
            for _ in range(3000)]
    b = pa.RecordBatch.from_pylist(rows, schema=s)
    text = FW.render_batch(b)
    for comp in (0, 1):
        out = tmp_path / f"hi{comp}.fastq.bgz"
        _n, st = gpu_write(out, [b], s, comp)
        size = check_bgzf(out, text)
        assert (size > len(text)) == (comp == 1), (comp, size, len(text))
