"""CPU: the VCF oracle rule by rule, and the VCF entry of the C ABI (open, schema, classify, plans, range info) without a GPU."""
import gzip
import subprocess

import pyarrow as pa
import pytest

from conftest import ROOT
from oracle.vcf_oracle import VcfError, parse_header, scan_text, schema
from vcf_inputs import CHROM, EDGE, HEADER, bgzf_parallel, sites_text

H = HEADER + CHROM + b"\n"


def _gpu_present() -> bool:
    try:
        import torch
        return torch.cuda.is_available()
    except Exception:
        return False


def _rows(body, **kw):
    return scan_text(H + body, **kw).to_pylist()


def _err(text, **kw):
    with pytest.raises(VcfError) as e:
        scan_text(text, **kw)
    return e.value


def test_fixed_columns():
    r = _rows(b"chr1\t10\trs1\tAC\tA,<DEL>\t9.5\tq10;s50\t.\n")[0]
    assert (r["chrom"], r["start"], r["end"], r["id"], r["ref"], r["alt"], r["qual"], r["filter"]) == \
        ("chr1", 9, 11, "rs1", "AC", "A,<DEL>", 9.5, "q10;s50")
    assert _rows(b"1\t10\t.\tA\tT\t.\t.\t.\n", zero_based=False)[0]["start"] == 10


def test_dots_are_null():
    r = _rows(b"1\t10\t.\tA\t.\t.\t.\t.\n")[0]
    assert r["id"] is None and r["alt"] is None and r["qual"] is None and r["filter"] is None and r["DP"] is None


def test_end_from_info_or_ref():
    assert _rows(b"1\t10\t.\tACG\tT\t.\t.\tEND=50\n")[0]["end"] == 50
    assert _rows(b"1\t10\t.\tACG\tT\t.\t.\tEND=.\n")[0]["end"] == 12
    assert _rows(b"1\t10\t.\tACG\tT\t.\t.\tDP=1\n", info_fields=[])[0]["end"] == 12


def test_crlf_and_unterminated_last_line():
    assert len(_rows(b"1\t10\t.\tA\tT\t.\t.\tDP=1\r\n2\t5\t.\tA\tT\t.\t.\tDP=2")) == 2
    assert _rows(b"1\t10\t.\tA\tT\t.\t.\tSVTYPE=DEL\r\n")[0]["SVTYPE"] == "DEL"


def test_samples_are_skipped():
    r = _rows(b"1\t10\t.\tA\tT\t.\t.\tDP=3\tGT\t0|1\t1|1\n")[0]
    assert r["DP"] == 3 and len(r) == 8 + 12


def test_info_types():
    r = _rows(b"1\t10\t.\tA\tT\t.\t.\tDP=-3;AF=0.5,.;DB;CSQ=a|b,.,;AC=1,.;GL=1e-3;NS=1,2,3;TC=x;MQ=+1.5;XX=1;UNK\n")[0]
    assert r["DP"] == -3 and r["AF"] == [0.5, None] and r["DB"] is True and r["H2"] is False
    assert r["CSQ"] == ["a|b", None, ""] and r["AC"] == [1, None] and r["NS"] == [1, 2, 3] and r["TC"] == "x" and r["MQ"] == 1.5
    assert abs(r["GL"][0] - 1e-3) < 1e-9


def test_empty_tokens_and_empty_info():
    assert _rows(b"1\t10\t.\tA\tT\t.\t.\t;;DP=2;;\n")[0]["DP"] == 2
    assert _rows(b"1\t10\t.\tA\tT\t.\t.\t\n")[0]["DP"] is None


def test_header_info_parse():
    infos, pos = parse_header(H)
    assert pos == len(H)
    dp = infos[0]
    assert dp["ID"] == "DP" and dp["Number"] == "1" and dp["Type"] == "Integer" and dp["Description"] == 'Total depth, as in "DP=">'
    sc = schema(infos)
    assert sc.names[:8] == ["chrom", "start", "end", "id", "ref", "alt", "qual", "filter"]
    assert sc.field("DP").type == pa.int32() and sc.field("AF").type == pa.list_(pa.float32()) and sc.field("DB").type == pa.bool_()
    assert not sc.field("DB").nullable and sc.field("CSQ").type == pa.list_(pa.string()) and sc.field("TC").type == pa.string()
    assert sc.field("AF").metadata == {b"bio.vcf.info.number": b"A", b"bio.vcf.info.type": b"Float", b"bio.vcf.info.description": b"Allele frequency"}
    assert schema(infos, ["MQ", "DB"]).names[8:] == ["MQ", "DB"]


@pytest.mark.parametrize("bad", [b"##fileformat=VCFv4.3\n##INFO=<ID=start,Number=1,Type=Integer,Description=\"x\">\n",
                                 b"##fileformat=VCFv4.3\n##INFO=<ID=Z,Number=0,Type=Integer,Description=\"x\">\n",
                                 b"##fileformat=VCFv4.3\n##INFO=<ID=Z,Number=1,Type=Blob,Description=\"x\">\n"])
def test_schema_errors(bad):
    assert _err(bad + CHROM + b"\n").kind == "schema"
    assert _err(H, info_fields=["NOPE"]).kind == "schema"
    assert _err(H, info_fields=["DP", "AF", "DP"]).kind == "schema"


@pytest.mark.parametrize("text", [b"##fileformat=VCFv4.3\n1\t2\n", b"##fileformat=BAM\n" + CHROM + b"\n",
                                  HEADER + b"##INFO=<ID=DP,Number=1,Type=Integer,Description=\"again\">\n" + CHROM + b"\n"])
def test_header_format_errors(text):
    assert _err(text).kind == "format"


@pytest.mark.parametrize("body,kind", [
    (b"1\t10\t.\tA\tT\t1\tPASS\n", "format"), (b"#x\n", "format"), (b"\n", "format"), (b"1\tx\t.\tA\tT\t.\t.\t.\n", "format"),
    (b"1\t2147483648\t.\tA\tT\t.\t.\t.\n", "format"), (b"\t1\t.\tA\tT\t.\t.\t.\n", "format"), (b"1\t1\t.\t\tT\t.\t.\t.\n", "format"),
    (b"1\t10\t.\tA\tT\t.\t.\tEND=9\n", "format"), (b"1\t10\t.\tA\tT\t.\t.\tDP=1;DP=1\n", "format"), (b"1\t1\t.\tA\tT\tx\t.\t.\n", "format"),
    (b"1\t1\t.\tA\tT\t.\t.\tSVTYPE=\xff\n", "format"), (b"1\t1\t.\tA\tT\t.\t.\tDP=a\n", "schema"), (b"1\t1\t.\tA\tT\t.\t.\tAC=1,\n", "schema"),
    (b"1\t1\t.\tA\tT\t.\t.\tDB=1\n", "schema"), (b"1\t1\t.\tA\tT\t.\t.\tDP\n", "schema"), (b"1\t1\t.\tA\tT\t.\t.\tTC=a,b\n", "schema"),
    (b"1\t1\t.\tA\tT\t.\t.\tEND\n", "schema"), (b"1\t0\t.\tA\tT\t.\t.\t.\n", "unsupported")])
def test_record_refusals(body, kind):
    e = _err(H + b"1\t5\t.\tA\tT\t.\t.\t.\n" + body)
    assert e.kind == kind and e.record == 1


def test_unprojected_values_not_checked_but_end_always_read():
    assert _rows(b"1\t1\t.\tA\tT\t.\t.\tDP=a;DP=b\n", info_fields=["AF"])[0]["AF"] is None
    assert _err(H + b"1\t10\t.\tA\tT\t.\t.\tEND=2\n", info_fields=[]).kind == "format"


def test_edge_file_parses():
    assert scan_text(EDGE).num_rows == 7


# ---- the C ABI without a GPU ----

def _provider(path, **kw):
    import bamscan
    return bamscan.VcfTableProvider(str(path), **kw)


@pytest.fixture(scope="module")
def vcf_file(tmp_path_factory):
    p = tmp_path_factory.mktemp("vcf") / "sites.vcf.gz"
    p.write_bytes(bgzf_parallel(sites_text(3000, n_extra=2, csq_lo=50, csq_hi=200)))
    return p


def test_open_schema_matches_oracle(vcf_file):
    v = _provider(vcf_file)
    text = gzip.decompress(vcf_file.read_bytes())
    want = schema(parse_header(text)[0])
    assert v.schema().equals(want, check_metadata=True)
    assert v.schema().metadata is None
    sel = _provider(vcf_file, info_fields=["CSQ", "DB"]).schema()
    assert sel.names == want.names[:8] + ["CSQ", "DB"]


@pytest.mark.parametrize("sel,name", [(["NOPE"], "NOPE"), (["DP", "CSQ", "DP"], "DP")])
def test_open_schema_error(vcf_file, sel, name):
    import bamscan
    with pytest.raises(bamscan.BamScanError) as e:
        _provider(vcf_file, info_fields=sel)
    assert e.value.code == -7 and f"'{name}'" in str(e.value)


def test_open_refuses_plain_and_gzip(tmp_path, vcf_file):
    import bamscan
    text = gzip.decompress(vcf_file.read_bytes())
    for name, data in (("plain.vcf", text), ("gz.vcf.gz", gzip.compress(text))):
        p = tmp_path / name
        p.write_bytes(data)
        with pytest.raises(bamscan.BamScanError) as e:
            _provider(p)
        assert e.value.code == -2


def test_open_refuses_other_bgzf(tmp_path):
    import bamscan
    p = tmp_path / "x.fa.gz"
    p.write_bytes(bgzf_parallel(b">r\nACGT\n"))
    with pytest.raises(bamscan.BamScanError) as e:
        _provider(p)
    assert e.value.code == -2


def test_classify_all_unsupported(vcf_file):
    v = _provider(vcf_file)
    assert v.supports_filters_pushdown([("chrom", "=", "1"), ("start", ">", 5)]) == ["Unsupported", "Unsupported"]


@pytest.mark.parametrize("n", [1, 2, 4, 8])
def test_block_ranges_cover_every_member_once(vcf_file, n):
    v = _provider(vcf_file)
    text = gzip.decompress(vcf_file.read_bytes())
    first = parse_header(text)[1]
    plan = v.scan(None, target_partitions=n)
    assert plan.output_partition_count() == n
    ranges = [r for p in range(n) for r in plan.partition_ranges(p)]
    assert ranges[0]["first_uoff"] == first and ranges[0]["exact_start"] == 1
    owned_begin = [ranges[0]["block_begin"]] + [r["block_begin"] + 1 for r in ranges[1:]]   # later ranges inflate the member in front
    for a, b, r in zip(owned_begin, owned_begin[1:] + [None], ranges):
        if b is not None:
            assert r["block_end"] == b
    assert ranges[-1]["stop_uoff"] == 2**64 - 1


def test_execute_without_gpu_is_a_cuda_error(vcf_file):
    import bamscan
    if _gpu_present():
        pytest.skip("a GPU is present")
    v = _provider(vcf_file)
    with pytest.raises(bamscan.BamScanError) as e:
        list(v.scan().execute(0))
    assert e.value.code == -4


def test_cpp_provider_builds_and_plans(tmp_path, vcf_file):
    """include/bamscan.hpp's VcfTableProvider compiles with -Wall -Werror against the library and plans without a GPU."""
    lib = ROOT / "datafusion-bio-formats_b200"
    exe = tmp_path / "vcf_cpp_check"
    r = subprocess.run(["g++", "-std=c++17", "-O1", "-Wall", "-Werror", f"-I{ROOT / 'include'}", "-o", str(exe),
                        str(ROOT / "tests" / "native" / "vcf_cpp_check.cpp"), str(lib / "libbamscan.so"), f"-Wl,-rpath,{lib}"],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    r = subprocess.run([str(exe), str(vcf_file)], capture_output=True, text=True)
    assert r.returncode == 0 and "vcf cpp check ok" in r.stdout, r.stdout + r.stderr
