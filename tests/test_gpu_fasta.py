"""GPU: the BGZF-FASTA scan against oracle/fasta_oracle.py -- edge files, many short records, records far larger than a chunk
and than a decode slice, projections, block-range partitions with the seam check, device batches, the inflate kernels, refusals."""
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pyarrow as pa
import pytest

from conftest import build_bamgen
from oracle.bam_write_oracle import inflate_bgzf
from oracle.fasta_oracle import SCHEMA, scan_text
from oracle.fastq_write_oracle import BGZF_BLOCK, BGZF_EOF, bgzf_bytes, bgzf_member

pytestmark = pytest.mark.gpu

EDGE = (b"\n \n>w60 wrapped at sixty\n" + b"".join(b"ACGTN" * 12 + b"\n" for _ in range(7)) + b"ACG\n"
        b">w80\t tab then space\n" + b"".join(b"acgtNNNNac" * 8 + b"\n" for _ in range(5)) +
        b">one line > kept * and -\n" + b"ACGT*-acgt" * 40 + b"\n"
        b">crlf x\r\n" + b"AC\r\nGT\r\n\r\n" +
        b">blank\n\n\nAC\n\n\nGT\n\n" +
        b">empty1\n>empty2 \n>cr\rinside\nA\rC\n" +
        b">lower\ngattacagattaca\n>last no final newline\nACGT\nAC")


def _bgzf_parallel(text: bytes, level=1) -> bytes:
    """bgzf_bytes with the members compressed on a thread pool (zlib releases the GIL)."""
    with ThreadPoolExecutor(16) as ex:
        members = list(ex.map(lambda i: bgzf_member(text[i:i + BGZF_BLOCK], level), range(0, len(text), BGZF_BLOCK)))
    return b"".join(members) + BGZF_EOF


def _write(tmp_path, name, text, level=1):
    p = tmp_path / name
    p.write_bytes(_bgzf_parallel(text, level) if len(text) > (8 << 20) else bgzf_bytes(text, level))
    return p


def _table(batches, schema):
    return pa.Table.from_batches(list(batches), schema=schema)


def _scan(path, projection=None, **kw):
    import bamscan
    p = bamscan.FastaTableProvider(str(path), **kw)
    try:
        plan = p.scan(projection)
        return _table(plan.execute(0), plan.schema())
    finally:
        p.close()


def _want(text, projection=None):
    return pa.Table.from_batches([scan_text(text, projection)])


@pytest.fixture(scope="module")
def edge(tmp_path_factory):
    path = _write(tmp_path_factory.mktemp("fa"), "edge.fa.bgz", EDGE)
    return path, _want(EDGE)


@pytest.fixture(scope="module")
def mixed(tmp_path_factory):
    """~150 MB: short records, one-line and wrapped, and ten records of 3-24 MB (one of 20 MiB), so that block ranges fall inside
    records and 4 MiB chunks carry records longer than the engine's fixed carry room (16 MiB)."""
    rng = np.random.default_rng(7)
    parts = []
    for i in range(40000):
        n = int(rng.integers(0, 700)) if i % 4000 else (20 << 20) if i == 8000 else int(rng.integers(3, 24)) << 20
        seq = np.frombuffer(b"ACGTacgtNN", np.uint8)[rng.integers(0, 10, n)].tobytes()
        w = (60, 80, 1 << 30)[i % 3]
        parts.append(b">r%d%s\n" % (i, b" d%d" % i if i % 5 else b"") + b"".join(seq[k:k + w] + b"\n" for k in range(0, n, w)))
    text = b"".join(parts)
    path = _write(tmp_path_factory.mktemp("fa"), "mixed.fa.bgz", text)
    return path, _want(text)


def test_edge_file_every_rule(edge):
    path, want = edge
    got = _scan(path)
    assert got.equals(want), (got.to_pydict(), want.to_pydict())
    assert got.num_rows == 10


@pytest.mark.parametrize("flags", [4, 8, 16], ids=["warp_per_member", "lane_group", "cta_per_member"])
def test_inflate_kernel_overrides(edge, mixed, flags):
    for path, want in (edge, mixed):
        assert _scan(path, debug_flags=flags).equals(want)


@pytest.mark.parametrize("proj", [[0], [1], [2], [2, 0], [1, 1, 2], []])
def test_projections(mixed, proj):
    import bamscan
    path, want = mixed
    p = bamscan.FastaTableProvider(str(path))
    plan = p.scan(proj)
    batches = list(plan.execute(0))
    if not proj:
        assert sum(b.num_rows for b in batches) == want.num_rows
    else:
        got = _table(batches, plan.schema())
        assert got.equals(pa.Table.from_arrays([want.column(i) for i in proj], schema=pa.schema([SCHEMA.field(i) for i in proj])))
    p.close()


@pytest.mark.parametrize("partitions", [1, 2, 4, 8])
def test_block_range_partitions(mixed, partitions):
    """The partitions concatenate to the sequential scan and pass the seam check; small chunks carry records across chunks."""
    import bamscan
    path, want = mixed
    for chunk in (0, 4 << 20):
        p = bamscan.FastaTableProvider(str(path), chunk_inflated_bytes=chunk)
        plan = p.scan(None, None, None, target_partitions=partitions)
        assert plan.output_partition_count() == partitions
        got = plan.collect()
        assert got.equals(want), (partitions, chunk)
        p.close()


def test_limit_is_not_applied_by_the_scan(mixed):
    import bamscan
    path, want = mixed
    p = bamscan.FastaTableProvider(str(path))
    assert p.scan(None, None, 5).collect().equals(want)
    p.close()


def test_device_batches_equal_host_batches(mixed):
    import bamscan
    path, want = mixed
    p = bamscan.FastaTableProvider(str(path), chunk_inflated_bytes=16 << 20)
    plan = p.scan([2, 1, 0])
    host = list(plan.execute(0))
    dev = [d.to_host() for d in plan.execute_device(0)]
    assert len(host) == len(dev) > 1
    for a, b in zip(host, dev):
        assert a.equals(b)
    p.close()


def test_many_short_records(tmp_path):
    """1 M records of 300 residues (bamgen --fasta short: one-line and wrapped at 60), in one chunk and in small chunks."""
    import subprocess
    path = tmp_path / "short.fa.bgz"
    subprocess.check_call([str(build_bamgen()), "--fasta", "short", "--reads", "1000000", "--seed", "5", "--out", str(path)],
                          stdout=subprocess.DEVNULL)
    text, _ = inflate_bgzf(path.read_bytes())
    want = _want(text)
    assert want.num_rows == 1000000
    for chunk in (0, 32 << 20):
        assert _scan(path, chunk_inflated_bytes=chunk).equals(want), chunk


def _big_text():
    """Records of 20 MB, 800 MB (more than a decode slice), 600 MB on one line and 300 MB, then two small ones: 1.7 GB of text,
    more than one default chunk; the 300 MB record straddles the first chunk boundary.  -> (text, expected table)."""
    rng = np.random.default_rng(11)
    alphabet = np.frombuffer(b"ACGTacgtN", np.uint8)
    spec = [(b"r20", b"twenty", 20_000_000, 60), (b"r800", None, 800_000_000, 80), (b"r600", b"one line", 600_000_000, 0),
            (b"r300", b"x", 300_000_000, 60), (b"tail1", None, 10, 60), (b"tail2", b"t", 0, 60)]
    parts, names, descs, seqs = [], [], [], []
    for name, desc, n, width in spec:
        seq = alphabet[rng.integers(0, 9, n, dtype=np.uint8)]
        parts.append(b">" + name + (b" " + desc if desc else b"") + b"\n")
        if width and n:
            full = n // width
            body = np.concatenate([seq[:full * width].reshape(full, width), np.full((full, 1), 10, np.uint8)], axis=1).ravel()
            parts += [body.tobytes(), seq[full * width:].tobytes() + (b"\n" if n % width else b"")]
        elif n:
            parts += [seq.tobytes(), b"\n"]
        names.append(name.decode()); descs.append(desc.decode() if desc else None); seqs.append(seq)
    offs = np.zeros(len(seqs) + 1, np.int64)
    offs[1:] = np.cumsum([len(s) for s in seqs])
    seq_arr = pa.Array.from_buffers(pa.large_string(), len(seqs), [None, pa.py_buffer(offs.tobytes()), pa.py_buffer(np.concatenate(seqs).tobytes())])
    want = pa.table([pa.array(names, pa.string()), pa.array(descs, pa.string()), seq_arr], schema=pa.schema([
        SCHEMA.field(0), SCHEMA.field(1), pa.field("sequence", pa.large_string(), False)]))
    return b"".join(parts), want


@pytest.fixture(scope="module")
def big(tmp_path_factory):
    text, want = _big_text()
    path = _write(tmp_path_factory.mktemp("fa"), "big.fa.bgz", text)
    return path, want


def _seq_rows(col: pa.ChunkedArray):
    """The values of a (large) string column as memoryviews, row by row: one column of all rows is more than 2 GiB."""
    for ch in col.chunks:
        wide = pa.types.is_large_string(ch.type)
        offs = np.frombuffer(ch.buffers()[1], np.int64 if wide else np.int32)[ch.offset:ch.offset + len(ch) + 1]
        data = memoryview(ch.buffers()[2]) if ch.buffers()[2] is not None else memoryview(b"")
        for j in range(len(ch)):
            yield data[offs[j]:offs[j + 1]]


def _equal_large(got: pa.Table, want: pa.Table):
    assert got.schema.equals(SCHEMA) and got.num_rows == want.num_rows
    assert got.column(0).equals(want.column(0)) and got.column(1).equals(want.column(1))
    rows = list(zip(_seq_rows(got.column(2)), _seq_rows(want.column(2))))
    assert len(rows) == want.num_rows
    for k, (g, w) in enumerate(rows):
        assert g == w, f"sequence of row {k} differs"


@pytest.mark.parametrize("chunk", [0, 64 << 20], ids=["default_chunks", "64MiB_chunks"])
def test_records_far_larger_than_a_chunk(big, chunk):
    path, want = big
    got = _scan(path, chunk_inflated_bytes=chunk)
    _equal_large(got, want)
    if chunk == 0:
        import bamscan
        p = bamscan.FastaTableProvider(str(path))
        plan = p.scan([0])
        assert plan.collect().num_rows == 6 and plan.last_stats["chunks"] >= 2      # the 300 MB record crosses a default chunk boundary
        p.close()


def test_big_records_over_partitions(big):
    import bamscan
    path, want = big
    p = bamscan.FastaTableProvider(str(path), chunk_inflated_bytes=256 << 20)
    plan = p.scan([0, 1], None, None, target_partitions=8)
    got = plan.collect()                                                   # (collect runs the seam check)
    assert got.column(0).equals(want.column(0)) and got.column(1).equals(want.column(1))
    p.close()


@pytest.mark.parametrize("case", ["leading", "empty_name", "utf8_name", "utf8_desc", "utf8_seq"])
def test_malformed_files_name_the_record(tmp_path, case):
    import bamscan
    good = b"".join(b">r%d\nACGT\n" % i for i in range(5000))
    bad = {"leading": b"junk\n" + good, "empty_name": good + b">\nAC\n" + good, "utf8_name": good + b">n\xc3\xa9\nAC\n" + good,
           "utf8_desc": good + b">n d\x80\nAC\n" + good, "utf8_seq": good + b">n\nA\xffC\n" + good}[case]
    path = _write(tmp_path, "bad.fa.bgz", bad)
    with pytest.raises(bamscan.BamScanError) as e:
        _scan(path)
    assert e.value.code == -2, e.value
    assert ("record 0 " if case == "leading" else "record 5000 ") in str(e.value), e.value


@pytest.mark.parametrize("chunk", [0, 256 << 20])
def test_record_over_one_gib_is_refused(tmp_path_factory, chunk):
    import bamscan
    d = tmp_path_factory.getbasetemp() / "gib"
    path = d / "gib.fa.bgz"
    if not path.exists():
        d.mkdir(exist_ok=True)
        line = b"A" * 99 + b"\n"
        text = b">small\nAC\n>huge\n" + line * ((1 << 30) // 100 + 1)
        path.write_bytes(_bgzf_parallel(text, 1))
    with pytest.raises(bamscan.BamScanError) as e:
        _scan(path, chunk_inflated_bytes=chunk)
    assert e.value.code == -5 and "record 1 " in str(e.value), e.value
