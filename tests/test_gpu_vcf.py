"""GPU: the BGZF-VCF scan against oracle/vcf_oracle.py -- an edge file, sites-only and genotype inputs, projections, small chunks,
block-range partitions with the seam check, device batches, the inflate kernels, refusals."""
import pyarrow as pa
import pytest

from oracle.vcf_oracle import scan_text
from vcf_inputs import CHROM, EDGE, HEADER, bgzf_parallel, genotypes_text, sites_text

pytestmark = pytest.mark.gpu


def _write(d, name, text):
    p = d / name
    p.write_bytes(bgzf_parallel(text))
    return p


def _scan(path, projection=None, info_fields=None, target_partitions=1, **kw):
    import bamscan
    v = bamscan.VcfTableProvider(str(path), info_fields, **kw)
    try:
        plan = v.scan(projection, target_partitions=target_partitions)
        t = plan.collect()
        return t, plan
    finally:
        v.close()


@pytest.fixture(scope="module")
def edge(tmp_path_factory):
    return _write(tmp_path_factory.mktemp("vcf"), "edge.vcf.gz", EDGE), EDGE


@pytest.fixture(scope="module")
def sites(tmp_path_factory):
    text = sites_text(1000000)
    return _write(tmp_path_factory.mktemp("vcf"), "sites.vcf.gz", text), scan_text(text)


@pytest.fixture(scope="module")
def genotypes(tmp_path_factory):
    text = genotypes_text(20000)
    return _write(tmp_path_factory.mktemp("vcf"), "gt.vcf.gz", text), scan_text(text)


def test_edge_file_every_rule(edge):
    path, text = edge
    got, _ = _scan(path)
    want = scan_text(text)
    assert got.schema.equals(want.schema, check_metadata=True)
    assert got.equals(want), (got.to_pydict(), want.to_pydict())
    got1, _ = _scan(path, coordinate_system_zero_based=False)
    assert got1.equals(scan_text(text, zero_based=False))


def test_edge_every_single_column_and_empty_projection(edge):
    path, text = edge
    want = scan_text(text)
    for i in range(want.num_columns):
        got, _ = _scan(path, [i])
        assert got.equals(scan_text(text, projection=[i])), want.schema.field(i).name
    got, _ = _scan(path, [])
    assert sum(b.num_rows for b in got) == want.num_rows


def test_info_fields_subsets_and_reorders(edge):
    path, text = edge
    for sel in (["CSQ"], ["MQ", "DB", "AF"], [], ["END", "SVTYPE"], ["GL", "AC", "NS", "TC", "H2"]):
        got, _ = _scan(path, info_fields=sel)
        assert got.equals(scan_text(text, info_fields=sel)), sel
    got, _ = _scan(path, [2, 9, 0], info_fields=["CSQ", "DP"])
    assert got.equals(scan_text(text, info_fields=["CSQ", "DP"], projection=[2, 9, 0]))


@pytest.mark.parametrize("which", ["sites", "genotypes"])
def test_inputs_at_test_size(request, which):
    path, want = request.getfixturevalue(which)
    got, plan = _scan(path)
    assert got.equals(want)
    assert plan.last_stats["rows"] == want.num_rows


@pytest.mark.parametrize("which", ["sites", "genotypes"])
def test_small_chunks(request, which):
    path, want = request.getfixturevalue(which)
    got, plan = _scan(path, chunk_inflated_bytes=64 << 20)
    assert plan.last_stats["chunks"] > 1
    assert got.equals(want)


@pytest.mark.parametrize("n", [1, 2, 4, 8])
def test_block_range_partitions(sites, genotypes, edge, n):
    for path, want in (sites, genotypes, (edge[0], scan_text(edge[1]))):
        got, plan = _scan(path, target_partitions=n)     # collect() checks the seams (bamscan_check_partition_seams)
        assert plan.output_partition_count() == n
        assert got.equals(want)


def test_sites_projection_subset(sites):
    path, want = sites
    got, _ = _scan(path, [0, 2, 11, 6, 7])
    assert got.equals(want.select([0, 2, 11, 6, 7]))


def test_device_batches_equal_host(sites, edge):
    import bamscan
    for path in (edge[0], sites[0]):
        v = bamscan.VcfTableProvider(str(path))
        plan = v.scan(None)
        host = plan.collect()
        dev = pa.Table.from_batches([b.to_host() for b in plan.execute_device(0)], schema=plan.schema())
        assert dev.equals(host)
        v.close()


@pytest.mark.parametrize("flags", [4, 8, 16], ids=["warp_per_member", "lane_group", "cta_per_member"])
def test_inflate_kernel_overrides(edge, genotypes, flags):
    path, text = edge
    assert _scan(path, debug_flags=flags)[0].equals(scan_text(text))
    assert _scan(genotypes[0], debug_flags=flags)[0].equals(genotypes[1])


def test_wide_groups(edge, sites):
    """debug_flags bit 1 forces 32 lanes per line (the long-line path); the sites CSQ values (0.5-2 kB) span several 512-byte
    windows of a 32-lane group"""
    path, text = edge
    assert _scan(path, debug_flags=2)[0].equals(scan_text(text))
    got, _ = _scan(sites[0], debug_flags=2)
    assert got.equals(sites[1])


def _many_info(n_info, n_rows=70):
    head = b"##fileformat=VCFv4.3\n" + b"".join(b"##INFO=<ID=I%d,Number=1,Type=Integer,Description=\"x\">\n" % i for i in range(n_info))
    body = b"".join(b"1\t%d\t.\tA\tT\t.\t.\t" % (r + 1) + b";".join(b"I%d=%d" % (i, r * i) for i in range(0, n_info, 1 + r % 3)) + b"\n"
                    for r in range(n_rows))
    return head + CHROM + b"\n" + body


def test_info_column_cap(tmp_path):
    """At most 112 projected INFO columns (vcf::MAX_INFO), counted without the fixed columns"""
    import bamscan
    text = _many_info(130)
    path = _write(tmp_path, "wide.vcf.gz", text)
    for proj in (list(range(8, 8 + 113)), [0] + list(range(8, 8 + 113)), None):
        with pytest.raises(bamscan.BamScanError) as e:
            _scan(path, proj)
        assert e.value.code == -5 and "INFO columns" in str(e.value), str(e.value)
    for proj in (list(range(8, 8 + 112)), list(range(0, 8 + 112)), list(range(18, 130))):
        got, _ = _scan(path, proj)
        assert got.equals(scan_text(text, projection=proj))
    got, _ = _scan(path, info_fields=[f"I{i}" for i in range(129, 17, -1)])
    assert got.equals(scan_text(text, info_fields=[f"I{i}" for i in range(129, 17, -1)]))


BODY_OK = b"1\t10\t.\tA\tT\t1\tPASS\tDP=1\n"
REFUSALS = {
    "fields": (b"1\t10\t.\tA\tT\t1\tPASS\n", -2),
    "hash_line": (b"#1\t10\t.\tA\tT\t1\tPASS\t.\n", -2),
    "empty_line": (b"\n", -2),
    "pos_text": (b"1\tx10\t.\tA\tT\t1\tPASS\t.\n", -2),
    "pos_big": (b"1\t2147483648\t.\tA\tT\t1\tPASS\t.\n", -2),
    "empty_chrom": (b"\t10\t.\tA\tT\t1\tPASS\t.\n", -2),
    "empty_ref": (b"1\t10\t.\t\tT\t1\tPASS\t.\n", -2),
    "end_below_pos": (b"1\t10\t.\tA\tT\t1\tPASS\tEND=9\n", -2),
    "dup_key": (b"1\t10\t.\tA\tT\t1\tPASS\tDP=1;DP=2\n", -2),
    "non_ascii": (b"1\t10\t.\tA\tT\t1\tPASS\tSVTYPE=D\xc3\xa9L\n", -2),
    "qual": (b"1\t10\t.\tA\tT\tq\tPASS\t.\n", -2),
    "int_value": (b"1\t10\t.\tA\tT\t1\tPASS\tDP=1.5\n", -7),
    "empty_numeric_element": (b"1\t10\t.\tA\tT\t1\tPASS\tAC=1,,2\n", -7),
    "flag_with_value": (b"1\t10\t.\tA\tT\t1\tPASS\tDB=1\n", -7),
    "key_without_value": (b"1\t10\t.\tA\tT\t1\tPASS\tDP\n", -7),
    "comma_in_number1": (b"1\t10\t.\tA\tT\t1\tPASS\tSVTYPE=A,B\n", -7),
    "int_range": (b"1\t10\t.\tA\tT\t1\tPASS\tDP=2147483648\n", -7),
    "pos0": (b"1\t0\t.\tA\tT\t1\tPASS\t.\n", -5),
}


@pytest.mark.parametrize("case", sorted(REFUSALS))
def test_refusals(tmp_path, case):
    import bamscan
    bad, code = REFUSALS[case]
    text = HEADER + CHROM + b"\n" + BODY_OK * 3 + bad + BODY_OK
    from oracle.vcf_oracle import VcfError
    with pytest.raises(VcfError) as oe:
        scan_text(text)
    assert oe.value.record == 3 and {"format": -2, "schema": -7, "unsupported": -5}[oe.value.kind] == code
    path = _write(tmp_path, case + ".vcf.gz", text)
    with pytest.raises(bamscan.BamScanError) as e:
        _scan(path)
    assert e.value.code == code, str(e.value)
    assert "record 3 " in str(e.value), str(e.value)


def test_unprojected_values_are_not_checked(tmp_path):
    text = HEADER + CHROM + b"\n" + b"1\t10\t.\tA\tT\t1\tPASS\tDP=x;DB=1\n"
    path = _write(tmp_path, "u.vcf.gz", text)
    got, _ = _scan(path, info_fields=["AF"])
    assert got.equals(scan_text(text, info_fields=["AF"]))


def test_line_over_16_mib_is_unsupported(tmp_path):
    import bamscan
    text = HEADER + CHROM + b"\n" + BODY_OK + b"1\t10\t.\tA\tT\t1\tPASS\tSVTYPE=" + b"A" * (17 << 20) + b"\n" + BODY_OK
    path = _write(tmp_path, "long.vcf.gz", text)
    with pytest.raises(bamscan.BamScanError) as e:
        _scan(path)
    assert e.value.code == -5, str(e.value)
