"""GPU: VCF FORMAT columns against oracle/vcf_format_oracle.py -- the edge file, projections, genotype inputs on both lane paths, small
chunks, block-range partitions, device batches, the inflate kernels, the column caps, slice cuts, runtime refusals."""
import pyarrow as pa
import pytest

from oracle.vcf_format_oracle import scan_text
from oracle.vcf_oracle import VcfError
from vcf_format_inputs import ALL, EDGE_FMT, FIVE, FORMAT_HEADER, format_text
from vcf_inputs import CHROM, HEADER, bgzf_parallel

pytestmark = pytest.mark.gpu


def _write(d, name, text):
    p = d / name
    p.write_bytes(bgzf_parallel(text))
    return p


def _scan(path, projection=None, format_fields=None, info_fields=None, target_partitions=1, **kw):
    import bamscan
    v = bamscan.VcfTableProvider(str(path), info_fields, format_fields=format_fields, **kw)
    try:
        plan = v.scan(projection, target_partitions=target_partitions)
        return plan.collect(), plan
    finally:
        v.close()


def _same(got, want):
    assert got.schema.equals(want.schema, check_metadata=True), (got.schema, want.schema)
    assert got.equals(want), [n for n in want.column_names if not got[n].equals(want[n])]


@pytest.fixture(scope="module")
def edge(tmp_path_factory):
    return _write(tmp_path_factory.mktemp("vcff"), "edge.vcf.gz", EDGE_FMT)


@pytest.fixture(scope="module")
def wide(tmp_path_factory):
    text = format_text(2000)
    return _write(tmp_path_factory.mktemp("vcff"), "wide.vcf.gz", text), scan_text(text, format_fields=FIVE)


@pytest.fixture(scope="module")
def short(tmp_path_factory):
    text = format_text(200000, n_samples=3, seed=5)
    return _write(tmp_path_factory.mktemp("vcff"), "short.vcf.gz", text), scan_text(text, format_fields=FIVE)


@pytest.mark.parametrize("zero_based", [True, False])
def test_edge_file_every_rule(edge, zero_based):
    got, _ = _scan(edge, format_fields=ALL, coordinate_system_zero_based=zero_based)
    _same(got, scan_text(EDGE_FMT, format_fields=ALL, zero_based=zero_based))


def test_edge_every_single_column(edge):
    want = scan_text(EDGE_FMT, format_fields=ALL)
    for i in range(want.num_columns):
        got, _ = _scan(edge, [i], format_fields=ALL)
        _same(got, scan_text(EDGE_FMT, format_fields=ALL, projection=[i]))


def test_format_fields_subsets_and_reorders(edge):
    for sel in (["GT"], ["PL", "GT"], ["HQ", "AD", "FT", "DP"], ["GL"], FIVE[::-1], ALL[::-1]):
        got, _ = _scan(edge, format_fields=sel)
        _same(got, scan_text(EDGE_FMT, format_fields=sel))
    got, _ = _scan(edge, [20, 0, 19], format_fields=["AD", "GT"])
    _same(got, scan_text(EDGE_FMT, format_fields=["AD", "GT"], projection=[20, 0, 19]))


def test_no_format_column_projected(edge, wide):
    """format_fields given but no FORMAT column projected: the scan of the same columns without format_fields"""
    for path in (edge, wide[0]):
        a, pa_ = _scan(path, list(range(12)), format_fields=FIVE)
        b, pb = _scan(path, list(range(12)))
        assert a.equals(b)
        assert pa_.last_stats["kernel_launches"] == pb.last_stats["kernel_launches"]
        assert pa_.last_stats["arrow_bytes"] == pb.last_stats["arrow_bytes"]


def test_wide_lines_32_lanes(wide):
    path, want = wide
    got, plan = _scan(path, format_fields=FIVE)
    _same(got, want)
    got, _ = _scan(path, format_fields=FIVE, debug_flags=2)
    _same(got, want)


def test_short_lines_8_lanes_many_batches(short):
    path, want = short
    got, plan = _scan(path, format_fields=FIVE, batch_rows=7000)
    _same(got, want)
    assert plan.last_stats["batches"] >= 1 and len(got[0].chunks) > 20


@pytest.mark.parametrize("which", ["wide", "short"])
def test_small_chunks(request, which):
    path, want = request.getfixturevalue(which)
    got, plan = _scan(path, format_fields=FIVE, chunk_inflated_bytes=1 << 20)
    assert plan.last_stats["chunks"] > 1
    _same(got, want)


@pytest.mark.parametrize("n", [1, 2, 4, 8])
def test_block_range_partitions(wide, short, edge, n):
    for path, want in (wide, short, (edge, scan_text(EDGE_FMT, format_fields=FIVE))):
        got, plan = _scan(path, format_fields=FIVE, target_partitions=n)     # collect() checks the seams
        assert plan.output_partition_count() == n
        _same(got, want)


def test_device_batches_equal_host(edge, short):
    import bamscan
    for path in (edge, short[0]):
        v = bamscan.VcfTableProvider(str(path), format_fields=ALL if path == edge else FIVE)
        plan = v.scan(None)
        host = plan.collect()
        dev = pa.Table.from_batches([b.to_host() for b in plan.execute_device(0)], schema=plan.schema())
        assert dev.equals(host)
        v.close()


@pytest.mark.parametrize("flags", [4, 8, 16], ids=["warp_per_member", "lane_group", "cta_per_member"])
def test_inflate_kernel_overrides(edge, short, flags):
    _same(_scan(edge, format_fields=ALL, debug_flags=flags)[0], scan_text(EDGE_FMT, format_fields=ALL))
    _same(_scan(short[0], format_fields=FIVE, debug_flags=flags)[0], short[1])


def test_112_info_and_16_format_columns(tmp_path):
    head = b"##fileformat=VCFv4.3\n" + b"".join(b"##INFO=<ID=I%d,Number=1,Type=Integer,Description=\"x\">\n" % i for i in range(112))
    head += b"".join(b"##FORMAT=<ID=F%d,Number=%s,Type=%s,Description=\"y\">\n" % (i, b"1" if i % 2 else b"2", [b"Integer", b"Float", b"String"][i % 3] if i % 2 else b"Integer") for i in range(16))
    keys = b":".join(b"F%d" % i for i in range(15, -1, -1))
    body = b"".join(b"1\t%d\t.\tA\tT\t.\t.\t" % (r + 1) + b";".join(b"I%d=%d" % (i, r * i) for i in range(0, 112, 1 + r % 3)) + b"\t" + keys
                    + b"".join(b"\t" + b":".join((b"%d" % (r + i + j)) if i % 2 else b"%d,%d" % (i, j) for i in range(15, -1, -1)) for j in range(3)) + b"\n"
                    for r in range(70))
    text = head + CHROM + b"\tFORMAT\ta\tb\tc\n" + body
    path = _write(tmp_path, "caps.vcf.gz", text)
    sel = [f"F{i}" for i in range(16)]
    got, _ = _scan(path, format_fields=sel)
    _same(got, scan_text(text, format_fields=sel))


def test_slice_cut_by_many_samples(tmp_path):
    """At most 2^24 elements (rows x samples) per decode slice: 40 000 samples cut 500 lines into two slices"""
    s = 40000
    fmt = b"##FORMAT=<ID=GT,Number=1,Type=String,Description=\"g\">\n"
    row = b"\t".join([b"0", b"1", b"."] * (s // 3) + [b"0"] * (s % 3))
    text = HEADER + fmt + CHROM + b"\tFORMAT\t" + b"\t".join(b"s%d" % k for k in range(s)) + b"\n" + b"".join(b"1\t%d\t.\tA\tT\t.\t.\t.\tGT\t%s\n" % (r + 1, row) for r in range(500))
    path = _write(tmp_path, "many.vcf.gz", text)
    got, plan = _scan(path, [0, 1, 20], format_fields=["GT"])
    assert plan.last_stats["batches"] >= 2
    _same(got, scan_text(text, format_fields=["GT"], projection=[0, 1, 20]))


OK_LINE = b"1\t10\t.\tA\tT\t1\tPASS\t.\tGT:DP:AD\t0|1:3:1,2\t.\n"
REFUSALS = {
    "too_few_fields": (b"1\t10\t.\tA\tT\t1\tPASS\t.\tGT:DP\t0|1\n", -2),
    "no_format_field": (b"1\t10\t.\tA\tT\t1\tPASS\t.\n", -2),
    "too_many_fields": (b"1\t10\t.\tA\tT\t1\tPASS\t.\tGT\t0\t1\t2\n", -2),
    "dup_key": (b"1\t10\t.\tA\tT\t1\tPASS\t.\tGT:DP:GT\t0:1:0\t.\n", -2),
    "more_values": (b"1\t10\t.\tA\tT\t1\tPASS\t.\tGT:DP\t0:1:2\t.\n", -2),
    "no_keys_but_values": (b"1\t10\t.\tA\tT\t1\tPASS\t.\t.\t0\t.\n", -2),
    "non_ascii": (b"1\t10\t.\tA\tT\t1\tPASS\t.\tGT\t0\xc3\xa9\t.\n", -2),
    "int_value": (b"1\t10\t.\tA\tT\t1\tPASS\t.\tDP\t1.5\t.\n", -7),
    "empty_int": (b"1\t10\t.\tA\tT\t1\tPASS\t.\tGT:DP\t0:\t.\n", -7),
    "empty_leaf": (b"1\t10\t.\tA\tT\t1\tPASS\t.\tAD\t1,,2\t.\n", -7),
    "comma_in_number1": (b"1\t10\t.\tA\tT\t1\tPASS\t.\tGT\t0,1\t.\n", -7),
    "int_range": (b"1\t10\t.\tA\tT\t1\tPASS\t.\tDP\t2147483648\t.\n", -7),
}


@pytest.mark.parametrize("case", sorted(REFUSALS))
def test_refusals(tmp_path, case):
    import bamscan
    bad, code = REFUSALS[case]
    text = HEADER + FORMAT_HEADER + CHROM + b"\tFORMAT\tA\tB\n" + OK_LINE * 3 + bad + OK_LINE
    with pytest.raises(VcfError) as oe:
        scan_text(text, format_fields=["GT", "DP", "AD"])
    assert oe.value.record == 3 and {"format": -2, "schema": -7, "unsupported": -5}[oe.value.kind] == code
    path = _write(tmp_path, case + ".vcf.gz", text)
    with pytest.raises(bamscan.BamScanError) as e:
        _scan(path, format_fields=["GT", "DP", "AD"])
    assert e.value.code == code, str(e.value)
    assert "record 3 " in str(e.value), str(e.value)
    _scan(path)     # the same file without FORMAT columns scans
