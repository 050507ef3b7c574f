"""GPU: plain SAM through BamTableProvider (kernels_sam.cuh -> the BAM decode stage), bit-exact against oracle/sam_oracle.py
and, outside the two documented cells (end of a zero-span placed read, QUAL '*'), against the GPU scan of the BAM the SAM was
rendered from."""
import gzip

import pyarrow as pa
import pytest

import sam_render
from conftest import GOLDEN, gen_bam

pytestmark = pytest.mark.gpu

FIXTURES = ["multi_chrom.bam", "bam_with_tags.bam", "10x_pbmc_tags.bam", "nanopore_custom_tags.bam", "no_coor_only.bam"]


def _provider(path, **kw):
    import bamscan
    return bamscan.BamTableProvider(str(path), None, kw.pop("zero_based", True), kw.pop("tag_fields", None), kw.pop("binary_cigar", False),
                                    True, 100, None, **kw)


def _oracle(path, **kw):
    from oracle.sam_oracle import OracleSam
    return OracleSam(str(path), kw.get("zero_based", True), kw.get("tag_fields"), kw.get("binary_cigar", False))


def _render(tmp_path, bam, name="t.sam"):
    p = tmp_path / name
    p.write_bytes(sam_render.bam_to_sam(bam.read_bytes()))
    return p


def _equal(got: pa.Table, want: pa.RecordBatch, ctx):
    want = pa.Table.from_batches([want])
    assert got.num_rows == want.num_rows, f"{ctx}: rows {got.num_rows} != {want.num_rows}"
    assert got.schema.names == want.schema.names, ctx
    for n in want.schema.names:
        g, w = got[n].combine_chunks(), want[n].combine_chunks()
        if not g.equals(w):
            bad = next(i for i in range(len(w)) if g[i] != w[i] or g[i].is_valid != w[i].is_valid)
            raise AssertionError(f"{ctx}: column {n} row {bad}: got {g[bad]!r} want {w[bad]!r}")


def _all_tags(bam):
    p = _provider(bam, index_path="")
    return [r for r, c in zip(p.describe()["column_name"].to_pylist(), p.describe()["category"].to_pylist()) if c == "tag"]


@pytest.mark.parametrize("fixture", FIXTURES)
@pytest.mark.parametrize("zero_based", [True, False])
@pytest.mark.parametrize("binary_cigar", [False, True])
def test_golden_fixture_rendered_to_sam(tmp_path, fixture, zero_based, binary_cigar):
    from oracle.bam_oracle import schema_equal
    bam = GOLDEN / fixture
    sam = _render(tmp_path, bam)
    for tags in (None, _all_tags(bam)):
        kw = dict(zero_based=zero_based, tag_fields=tags, binary_cigar=binary_cigar)
        prov, orc = _provider(sam, **kw), _oracle(sam, **kw)
        assert schema_equal(prov.schema(), orc.schema)
        bam_prov = _provider(bam, index_path="", **kw)
        assert schema_equal(prov.schema(), bam_prov.schema())
        n = len(prov.schema())
        bam_full = bam_prov.scan(None, [], None).collect()
        for proj in (None, [3, 0, 1], list(range(12, n)) or [11], []):
            ctx = f"{fixture} tags={tags} proj={proj}"
            got = prov.scan(proj, [], None).collect()
            if proj == []:
                assert sum(b.num_rows for b in got) == orc.n_records, ctx
                continue
            _equal(got, orc.scan(proj), ctx)
            for name in got.schema.names:
                g, w = got[name].to_pylist(), bam_full[name].to_pylist()
                if name == "end":   # RecordBuf: a placed read whose CIGAR spans nothing ends at start - 1 (1-based), BAM: NULL
                    w = [x if x is not None or s is None or s - (0 if zero_based else 1) == 0 else s - (0 if zero_based else 1) for x, s in zip(w, bam_full["start"].to_pylist())]
                assert g == w, f"{ctx}: {name} differs from the BAM scan"


EDGE = (b"@HD\tVN:1.6\tSO:unsorted\n@SQ\tSN:chrA\tLN:1000\n@SQ\tSN:chrB\tLN:2000\n@CO\tedge cases\n"
        b"r1\t99\tchrA\t100\t255\t5S10M2I3D4N1=1X\t=\t200\t-160\tACGTNACGTNACGTNACGT\t!\"#$%&'()*+,-./0123\tNM:i:5\tXS:i:-2\tXU:i:4000000000\tXI:i:-70000\tXF:f:1.5\tXA:A:q\tMD:Z:10A5\tXH:H:1aE0\tXB:B:S,7,65535\tXE:B:c\tXG:B:f,0.1,-1e-45,3.4028235e38\r\n"
        b"*\t4\t*\t0\t0\t*\t*\t0\t0\t*\t*\n"
        b"r3\t16\tchrB\t+1\t60\t268435455M\tchrA\t6\t+160\tAC\t!I\r\n"
        b"placed_no_cigar\t133\tchrA\t6\t3\t*\tchrA\t6\t0\tac\t\"#\n"
        b"no_qual\t0\tchrB\t8\t20\t40M\t*\t0\t0\t" + b"ACGT" * 10 + b"\t*\tXX:f:16777217\tXY:f:inf\tXZ:f:7.006492321624087e-46\n"
        b"pos1\t0\tchrA\t1\t0\t*\t*\t0\t0\tA\tI\n"                # zero span at POS 1: start + 0 - 1 = 0 is no position -> NULL
        b"last\t0\tchrA\t1\t0\t2M1D\t*\t0\t0\tAC\tII")       # no final newline


def test_edge_sam(tmp_path):
    p = tmp_path / "edge.SAM"                 # the extension is matched in any case
    p.write_bytes(EDGE)
    tags = ["NM", "XS", "XU", "XI", "XF", "XA", "MD", "XH", "XB", "XE", "XG", "XX", "XY", "XZ"]
    for zero_based in (True, False):
        prov = _provider(p, tag_fields=tags, zero_based=zero_based)
        got = prov.scan(None, [], None).collect()
        _equal(got, _oracle(p, tag_fields=tags, zero_based=zero_based).scan(), "edge")
        rows = got.to_pylist()
        assert [r["name"] for r in rows] == ["r1", "*", "r3", "placed_no_cigar", "no_qual", "pos1", "last"]
        assert rows[1]["mapping_quality"] == 0 and rows[0]["mapping_quality"] == 255 and rows[0]["template_length"] == -160
        off = 0 if zero_based else 1
        assert rows[3]["start"] == 5 + off and rows[3]["end"] == 5                   # zero span: end = start + 0 - 1 (1-based)
        assert rows[4]["quality_scores"] == "" and rows[4]["sequence"] == "ACGT" * 10
        assert rows[3]["sequence"] == "AC" and rows[2]["quality_scores"] == "!I" and rows[2]["template_length"] == 160
        assert rows[0]["XU"] == 4000000000 and rows[0]["XS"] == -2 and rows[0]["XE"] == [] and rows[0]["XH"] == "1aE0"
        assert rows[4]["XX"] == 16777216.0 and rows[4]["XY"] == float("inf")
        assert rows[5]["start"] == off and rows[5]["end"] is None
        assert rows[6]["end"] == 3 and rows[6]["quality_scores"] == "II"
    s = {f.name: f.type for f in _provider(p, tag_fields=tags).schema()}
    assert s["XU"] == pa.uint32() and s["XS"] == pa.int32() and s["NM"] == pa.int32() and s["XB"] == pa.list_(pa.uint16())


@pytest.mark.parametrize("mode,reads", [("short", 60000), ("long", 400)])
def test_synthetic_reads_small_chunks(tmp_path, mode, reads):
    bam = gen_bam(tmp_path, mode=mode, reads=reads, seed=3)
    sam = _render(tmp_path, bam)
    want = _oracle(sam).scan()
    chunk = 1 << 20 if mode == "short" else 3 << 16                   # lines cross chunk boundaries and are carried
    for flags in (0, 2):                                              # bit 1: the long-record kernels
        got = _provider(sam, chunk_inflated_bytes=chunk, debug_flags=flags).scan(None, [], None).collect()
        _equal(got, want, f"{mode} flags={flags}")
        for n in (2, 3, 8):
            prov = _provider(sam, chunk_inflated_bytes=chunk, debug_flags=flags)
            plan = prov.scan(None, [], None, target_partitions=n, partition_mode="block_range")
            assert plan.output_partition_count() == n
            _equal(plan.collect(), want, f"{mode} {n} partitions")        # collect() checks the seams


def test_long_lines_over_64k(tmp_path):
    seq = "ACGT" * 20000
    text = ("@SQ\tSN:c\tLN:100000\n" + "".join(f"q{i}\t0\tc\t{i + 1}\t9\t{len(seq)}M\t*\t0\t0\t{seq}\t{'I' * len(seq)}\tMD:Z:{len(seq)}\n" for i in range(6))).encode()
    p = tmp_path / "long.sam"
    p.write_bytes(text)
    want = _oracle(p, tag_fields=["MD"]).scan()
    for chunk in (0, 1 << 16):
        _equal(_provider(p, tag_fields=["MD"], chunk_inflated_bytes=chunk).scan(None, [], None).collect(), want, f"chunk {chunk}")
    plan = _provider(p, tag_fields=["MD"], chunk_inflated_bytes=1 << 16).scan(None, [], None, target_partitions=3, partition_mode="block_range")
    _equal(plan.collect(), want, "3 partitions")


def test_device_handoff_and_device_resident(tmp_path):
    sam = _render(tmp_path, GOLDEN / "bam_with_tags.bam")
    prov = _provider(sam, tag_fields=["NM", "MD"])
    plan = prov.scan(None, [], None)
    got = pa.Table.from_batches([b.to_host() for b in plan.execute_device(0)])
    _equal(got, _oracle(sam, tag_fields=["NM", "MD"]).scan(), "device hand-off")
    st = plan.run_device_resident(0, 2)
    assert st["rows"] == 14 and st["compressed_bytes"] == st["inflated_bytes"] > 0


BAD = [   # (record line 0 replaced by, code, what) -- record 1 is always fine
    ("a\t0\tchrA\t1\t0\t*\t*\t0\t0\t*", -2, "fewer than 11 fields"),
    ("a\t70000\tchrA\t1\t0\t*\t*\t0\t0\t*\t*", -2, "FLAG"),
    ("a\t0\tchrZ\t1\t0\t*\t*\t0\t0\t*\t*", -2, "RNAME"),
    ("a\t0\tchrA\t-1\t0\t*\t*\t0\t0\t*\t*", -2, "POS"),
    ("a\t0\tchrA\t1\t256\t*\t*\t0\t0\t*\t*", -2, "MAPQ"),
    ("a\t0\tchrA\t1\t0\t4M3\t*\t0\t0\t*\t*", -2, "CIGAR"),
    ("a\t0\tchrA\t1\t0\t" + "1M" * 65536 + "\t*\t0\t0\t*\t*", -5, "65535"),
    ("a\t0\tchrA\t1\t0\t*\tchrQ\t0\t0\t*\t*", -2, "RNEXT"),
    ("a\t0\tchrA\t1\t0\t*\t*\t0\t3000000000\t*\t*", -2, "TLEN"),
    ("a\t0\tchrA\t1\t0\t*\t*\t0\t0\tAC1\tIII", -2, "SEQ"),
    ("a\t0\tchrA\t1\t0\t*\t*\t0\t0\tACG\tII", -2, "QUAL length"),
    ("a\t0\tchrA\t1\t0\t*\t*\t0\t0\t*\t*\tNM:i:x", -2, "malformed aux"),
    ("a\t0\tchrA\t1\t0\t*\t*\t0\t0\t*\t*\tNM:i:1\tNM:i:2", -2, "duplicate"),
    ("a\t0\tchrA\t1\t0\t*\t*\t0\t0\t*\t*\tXB:B:c,1,200", -2, "out of range"),
    ("a\t0\tchrA\t1\t0\t*\t*\t0\t0\t*\t*\tXI:i:4294967296", -2, "out of range"),
    ("n" * 255 + "\t0\tchrA\t1\t0\t*\t*\t0\t0\t*\t*", -2, "QNAME"),
    ("a\t0\tchrA\t1\t0\t*\t*\t2147483649\t0\t*\t*", -2, "PNEXT"),
    ("a\t0\tchrA\t1\t0\t*\t*\t0\t0\tAC\tI\x7f", -2, "invalid QUAL"),
    ("a\t0\tchrA\t1\t0\t*\t*\t0\t0\t*\t*\tXZ:Z:caf\xe9", -2, "malformed aux"),
    ("a\t0\tchrA\t1\t0\t*\t*\t0\t0\t*\t*\tXA:A:ab", -2, "malformed aux"),
    ("a\t0\tchrA\t1\t0\t*\t*\t0\t0\t*\t*\tXH:H:ABC", -2, "malformed aux"),
    ("a\t0\tchrA\t1\t0\t*\t*\t0\t0\t*\t*\t1X:i:1", -2, "malformed aux"),
    ("a\t0\tchrA\t1\t0\t*\t*\t0\t0\t*\t*\tXB:B:c,x", -2, "malformed aux"),
    ("", -2, "fewer than 11 fields"),
]


@pytest.mark.parametrize("line,code,what", BAD, ids=[b[2] + str(i) for i, b in enumerate(BAD)])
def test_malformed_line_refused(tmp_path, line, code, what):
    import bamscan
    good = "ok\t0\tchrA\t5\t0\t2M\t*\t0\t0\tAC\tII"
    p = tmp_path / "bad.sam"
    p.write_text("@SQ\tSN:chrA\tLN:100\n" + good + "\n" + line + "\n" + good + "\n")
    plan = _provider(p).scan(None, [], None)
    rows = []
    with pytest.raises(bamscan.BamScanError) as ei:
        for b in plan.execute(0):
            rows.append(b.num_rows)
    assert ei.value.code == code and "record 1 " in str(ei.value) and what in str(ei.value), str(ei.value)
    assert rows == []


def test_gzip_sam_refused(tmp_path):
    import bamscan
    p = tmp_path / "z.sam"
    p.write_bytes(gzip.compress(EDGE))
    with pytest.raises(bamscan.BamScanError) as ei:
        _provider(p)
    assert ei.value.code == -5


def test_try_new_with_inferred_schema_on_sam(tmp_path):
    import bamscan
    sam = _render(tmp_path, GOLDEN / "nanopore_custom_tags.bam")
    tags = _all_tags(GOLDEN / "nanopore_custom_tags.bam")
    prov = bamscan.BamTableProvider.try_new_with_inferred_schema(str(sam), None, True, tags, 50)
    bam = bamscan.BamTableProvider.try_new_with_inferred_schema(str(GOLDEN / "nanopore_custom_tags.bam"), None, True, tags, 50, index_path="")
    from oracle.bam_oracle import schema_equal
    assert schema_equal(prov.schema(), bam.schema())
    want = _oracle(sam, tag_fields=tags).scan()
    _equal(prov.scan(None, [], None).collect(), want, "inferred schema")
