"""CPU: the VCF FORMAT rules of oracle/vcf_format_oracle.py, one test per rule, and the provider's schema and open refusals (the C ABI
without a GPU), checked against the oracle."""
import gzip

import pyarrow as pa
import pytest

from oracle.vcf_format_oracle import parse_format_header, scan_text, schema
from oracle.vcf_oracle import VcfError, parse_header
from vcf_format_inputs import ALL, EDGE_FMT, FIVE, FORMAT_HEADER
from vcf_inputs import CHROM, HEADER, bgzf_parallel

HEAD = HEADER + FORMAT_HEADER + CHROM + b"\tFORMAT\tA\tB\n"


def _rows(body, sel):
    return scan_text(HEAD + body, format_fields=sel).select([f"format_{s}" for s in sel]).to_pylist()


def test_header_format_parse():
    formats, samples = parse_format_header(EDGE_FMT)
    assert [d["ID"] for d in formats] == ALL
    assert formats[2] == {"ID": "AD", "Number": "R", "Type": "Integer", "Description": 'Allelic depths, "ref,alt"'}
    assert samples == ["NA1", 'NA"2', "S 3"]
    assert parse_format_header(HEADER + CHROM + b"\n") == ([], [])


@pytest.mark.parametrize("text", [HEADER + b"##FORMAT=<ID=GT,Number=1>\n" + CHROM + b"\tFORMAT\tA\n",
                                  HEADER + FORMAT_HEADER + b"##FORMAT=<ID=GT,Number=1,Type=String>\n" + CHROM + b"\tFORMAT\tA\n",
                                  HEADER + FORMAT_HEADER + CHROM + b"\tA\tB\n"])
def test_header_format_errors_only_with_format_fields(text):
    with pytest.raises(VcfError) as e:
        scan_text(text, format_fields=["GT"])
    assert e.value.kind == "format"
    scan_text(text)                  # without format_fields the header reads as before
    scan_text(text, format_fields=[])


def test_schema_types_names_metadata():
    sc = schema(parse_header(EDGE_FMT)[0], None, ALL, parse_format_header(EDGE_FMT))
    fmt = [sc.field(i) for i in range(len(sc) - len(ALL), len(sc))]
    assert [f.name for f in fmt] == [f"format_{i}" for i in ALL]
    assert [f.type for f in fmt] == [pa.list_(pa.string()), pa.list_(pa.int32()), pa.list_(pa.list_(pa.int32())), pa.list_(pa.int32()),
                                     pa.list_(pa.list_(pa.int32())), pa.list_(pa.list_(pa.float32())), pa.list_(pa.float32()), pa.list_(pa.string())]
    assert not any(f.nullable for f in fmt)
    assert fmt[2].metadata == {b"bio.vcf.format.number": b"R", b"bio.vcf.format.type": b"Integer",
                               b"bio.vcf.format.description": b'Allelic depths, "ref,alt"'}
    assert sc.metadata == {b"bio.vcf.samples": b'["NA1", "NA\\"2", "S 3"]'}
    assert schema(parse_header(EDGE_FMT)[0]).metadata is None


OPEN_REFUSALS = {
    "undeclared": (FORMAT_HEADER, ["GT", "NOPE"], "schema"),
    "twice": (FORMAT_HEADER, ["DP", "GT", "DP"], "schema"),
    "flag": (b"##FORMAT=<ID=FL,Number=0,Type=Flag,Description=\"f\">\n", ["FL"], "schema"),
    "number0": (b"##FORMAT=<ID=Z,Number=0,Type=Integer,Description=\"z\">\n", ["Z"], "schema"),
    "unknown_type": (b"##FORMAT=<ID=U,Number=1,Type=Blob,Description=\"u\">\n", ["U"], "schema"),
    "name_taken": (b"##INFO=<ID=format_DP,Number=1,Type=Integer,Description=\"i\">\n" + FORMAT_HEADER, ["DP"], "schema"),
    "string_number2": (b"##FORMAT=<ID=S2,Number=2,Type=String,Description=\"s\">\n", ["S2"], "unsupported"),
    "more_than_16": (b"".join(b"##FORMAT=<ID=F%d,Number=1,Type=Integer,Description=\"f\">\n" % i for i in range(17)), [f"F{i}" for i in range(17)], "unsupported"),
}


@pytest.mark.parametrize("case", sorted(OPEN_REFUSALS))
def test_open_refusals_oracle(case):
    extra, sel, kind = OPEN_REFUSALS[case]
    text = HEADER + extra + CHROM + b"\tFORMAT\tA\n"
    with pytest.raises(VcfError) as e:
        scan_text(text, format_fields=sel)
    assert e.value.kind == kind and e.value.record is None


def test_no_samples_refused():
    with pytest.raises(VcfError) as e:
        scan_text(HEADER + FORMAT_HEADER + CHROM + b"\tFORMAT\n", format_fields=["GT"])
    assert e.value.kind == "schema"


def test_format_order_per_line():
    assert _rows(b"1\t1\t.\tA\tT\t.\t.\t.\tGT:DP\t0|1:5\t1|1:6\n1\t2\t.\tA\tT\t.\t.\t.\tDP:GT\t7:0/0\t8:./.\n", ["DP", "GT"]) == [
        {"format_DP": [5, 6], "format_GT": ["0|1", "1|1"]}, {"format_DP": [7, 8], "format_GT": ["0/0", "./."]}]


def test_trailing_values_dropped_and_lone_dot():
    assert _rows(b"1\t1\t.\tA\tT\t.\t.\t.\tGT:DP:AD\t0|1\t.\n", ["GT", "DP", "AD"]) == [
        {"format_GT": ["0|1", None], "format_DP": [None, None], "format_AD": [None, None]}]


def test_absent_key_is_null_for_every_sample():
    assert _rows(b"1\t1\t.\tA\tT\t.\t.\t.\tGT\t0\t1\n1\t2\t.\tA\tT\t.\t.\t.\t.\t.\t.\n", ["DP", "GT"]) == [
        {"format_DP": [None, None], "format_GT": ["0", "1"]}, {"format_DP": [None, None], "format_GT": [None, None]}]


def test_nested_nulls():
    assert _rows(b"1\t1\t.\tA\tT\t.\t.\t.\tAD:GL\t.:1,.,-2\t3,.:.\n", ["AD", "GL"]) == [
        {"format_AD": [None, [3, None]], "format_GL": [[1.0, None, -2.0], None]}]


def test_unprojected_keys_not_compared():
    assert _rows(b"1\t1\t.\tA\tT\t.\t.\t.\tXX:GT:XX\tx:0:y\t::\n", ["GT"]) == [{"format_GT": ["0", ""]}]


RECORD_REFUSALS = {
    "fields": (b"1\t1\t.\tA\tT\t.\t.\t.\tGT\t0\n", "format"),
    "dup_key": (b"1\t1\t.\tA\tT\t.\t.\t.\tGT:GT\t0:1\t.\n", "format"),
    "more_values": (b"1\t1\t.\tA\tT\t.\t.\t.\tGT\t0:1\t.\n", "format"),
    "non_ascii": (b"1\t1\t.\tA\tT\t.\t.\t.\tGT\t\xff\t.\n", "format"),
    "bad_int": (b"1\t1\t.\tA\tT\t.\t.\t.\tDP\tx\t.\n", "schema"),
    "empty_int": (b"1\t1\t.\tA\tT\t.\t.\t.\tDP\t\t.\n", "schema"),
    "comma_number1": (b"1\t1\t.\tA\tT\t.\t.\t.\tGT\t0,1\t.\n", "schema"),
}


@pytest.mark.parametrize("case", sorted(RECORD_REFUSALS))
def test_record_refusals(case):
    body, kind = RECORD_REFUSALS[case]
    with pytest.raises(VcfError) as e:
        scan_text(HEAD + body, format_fields=["GT", "DP"])
    assert e.value.kind == kind and e.value.record == 0
    scan_text(HEAD + body)               # without FORMAT columns the line is not looked at
    scan_text(HEAD + body, format_fields=["GT", "DP"], projection=[0, 1])


# ---- the C ABI without a GPU ----

@pytest.fixture(scope="module")
def edge_file(tmp_path_factory):
    p = tmp_path_factory.mktemp("vcff") / "edge.vcf.gz"
    p.write_bytes(bgzf_parallel(EDGE_FMT))
    return p


def test_open_schema_matches_oracle(edge_file):
    import bamscan
    for sel in (ALL, FIVE[::-1], ["PL"], [], None):
        v = bamscan.VcfTableProvider(str(edge_file), format_fields=sel)
        want = scan_text(EDGE_FMT, format_fields=sel).schema
        assert v.schema().equals(want, check_metadata=True), sel
        v.close()


@pytest.mark.parametrize("case", sorted(OPEN_REFUSALS))
def test_open_refusals_provider(tmp_path, case):
    import bamscan
    extra, sel, kind = OPEN_REFUSALS[case]
    p = tmp_path / "r.vcf.gz"
    p.write_bytes(bgzf_parallel(HEADER + extra + CHROM + b"\tFORMAT\tA\n"))
    with pytest.raises(bamscan.BamScanError) as e:
        bamscan.VcfTableProvider(str(p), format_fields=sel)
    assert e.value.code == {"schema": -7, "unsupported": -5}[kind], str(e.value)
    if kind == "schema" and case != "name_taken":
        assert f"'{sel[-1] if case != 'twice' else 'DP'}'" in str(e.value) or case == "flag", str(e.value)
    bamscan.VcfTableProvider(str(p)).close()


def test_open_header_errors_provider(tmp_path):
    import bamscan
    for i, text in enumerate((HEADER + b"##FORMAT=<ID=GT,Number=1>\n" + CHROM + b"\tFORMAT\tA\n", HEADER + FORMAT_HEADER + CHROM + b"\tA\tB\n",
                              HEADER + FORMAT_HEADER + FORMAT_HEADER + CHROM + b"\tFORMAT\tA\n")):
        p = tmp_path / f"h{i}.vcf.gz"
        p.write_bytes(bgzf_parallel(text))
        with pytest.raises(bamscan.BamScanError) as e:
            bamscan.VcfTableProvider(str(p), format_fields=["GT"])
        assert e.value.code == -2, str(e.value)
        bamscan.VcfTableProvider(str(p)).close()
        bamscan.VcfTableProvider(str(p), format_fields=[]).close()
    p = tmp_path / "ns.vcf.gz"
    p.write_bytes(bgzf_parallel(HEADER + FORMAT_HEADER + CHROM + b"\tFORMAT\n"))
    with pytest.raises(bamscan.BamScanError) as e:
        bamscan.VcfTableProvider(str(p), format_fields=["GT"])
    assert e.value.code == -7
    assert gzip.decompress(p.read_bytes()).endswith(b"FORMAT\n")


def test_cpp_provider_format_schema(tmp_path, edge_file):
    """include/bamscan.hpp's VcfTableProvider with format_fields compiles with -Wall -Werror and gives the nested schema."""
    import subprocess
    from conftest import ROOT
    lib = ROOT / "datafusion-bio-formats_b200"
    exe = tmp_path / "vcf_format_cpp_check"
    r = subprocess.run(["g++", "-std=c++17", "-O1", "-Wall", "-Werror", f"-I{ROOT / 'include'}", "-o", str(exe),
                        str(ROOT / "tests" / "native" / "vcf_format_cpp_check.cpp"), str(lib / "libbamscan.so"), f"-Wl,-rpath,{lib}"],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    r = subprocess.run([str(exe), str(edge_file)], capture_output=True, text=True)
    assert r.returncode == 0 and "vcf format cpp check ok" in r.stdout, r.stdout + r.stderr
