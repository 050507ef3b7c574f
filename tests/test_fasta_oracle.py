"""CPU: the FASTA oracle rule by rule, and the FASTA entry of the C ABI (open, schema, plans, range info) without a GPU."""
import gzip
import subprocess

import pyarrow as pa
import pytest

from conftest import ROOT
from oracle.bam_write_oracle import inflate_bgzf
from oracle.fasta_oracle import SCHEMA, FastaError, parse_records, scan_text
from oracle.fastq_write_oracle import bgzf_bytes


def _gpu_present() -> bool:
    try:
        import torch
        return torch.cuda.is_available()
    except Exception:
        return False


def test_definition_line_split():
    """Name up to the first space or tab, the rest is the description (tabs and '>' kept); an empty description is NULL."""
    r = parse_records(b">a desc with  spaces\nAC\n>b\tx>y\tz\nG\n>c \nT\n>d\n")
    assert r == [(b"a", b"desc with  spaces", b"AC"), (b"b", b"x>y\tz", b"G"), (b"c", None, b"T"), (b"d", None, b"")]


def test_wrapped_lines_are_joined():
    seq = b"ACGTN" * 37
    wrapped = b"".join(seq[i:i + 60] + b"\n" for i in range(0, len(seq), 60))
    assert parse_records(b">r\n" + wrapped) == [(b"r", None, seq)]
    assert parse_records(b">r\n" + seq + b"\n") == [(b"r", None, seq)]


def test_crlf_and_one_trailing_cr_per_line():
    assert parse_records(b">r d\r\nAC\r\nGT\r\n") == [(b"r", b"d", b"ACGT")]
    assert parse_records(b">r\nA\r\r\nC\rG\n") == [(b"r", None, b"A\rC\rG")]


def test_blank_lines_add_nothing():
    assert parse_records(b"\n\n>r\n\nAC\n\n\nGT\n\n>s\n\n") == [(b"r", None, b"ACGT"), (b"s", None, b"")]


def test_unterminated_last_line_is_a_line():
    assert parse_records(b">r\nAC\nGT") == [(b"r", None, b"ACGT")]
    assert parse_records(b">r x") == [(b"r", b"x", b"")]


def test_bytes_kept_as_given():
    assert parse_records(b">r\nacgtNNNN*-ACGT\n") == [(b"r", None, b"acgtNNNN*-ACGT")]


def test_only_line_starts_begin_records():
    assert parse_records(b">r\nAC>GT\n >x\n") == [(b"r", None, b"AC>GT >x")]


def test_empty_and_whitespace_only_texts():
    assert parse_records(b"") == [] and parse_records(b" \n\t\r\n\f\n") == []


def test_refusal_leading_bytes():
    with pytest.raises(FastaError) as e:
        parse_records(b"\n  \nx\n>r\nAC\n")
    assert e.value.record == 0 and not e.value.unsupported
    with pytest.raises(FastaError):
        parse_records(b" >r\nAC\n")


def test_refusal_empty_name():
    with pytest.raises(FastaError) as e:
        parse_records(b">a\nAC\n> desc\nGT\n")
    assert e.value.record == 1 and not e.value.unsupported
    with pytest.raises(FastaError):
        parse_records(b">a\n>\r\n")


@pytest.mark.parametrize("where", ["name", "desc", "seq"])
def test_refusal_non_ascii(where):
    bad = {"name": b">a\nA\n>b\xc3\xa9\nC\n", "desc": b">a\nA\n>b d\x80\nC\n", "seq": b">a\nA\n>b\nC\xffG\n"}[where]
    with pytest.raises(FastaError) as e:
        parse_records(bad)
    assert e.value.record == 1 and not e.value.unsupported


def test_refusal_record_over_one_gib(monkeypatch):
    """The limit counts the record's whole text: definition line and line breaks included (shown here with a small limit)."""
    import oracle.fasta_oracle as F
    assert F.MAX_RECORD == 1 << 30
    monkeypatch.setattr(F, "MAX_RECORD", 16)
    assert parse_records(b">a\nC\n>b\nACGTACG\nACGT\n") == [(b"a", None, b"C"), (b"b", None, b"ACGTACGACGT")]   # 16 bytes
    with pytest.raises(FastaError) as e:
        parse_records(b">a\nC\n>b\nACGTACG\r\nACGT\n")
    assert e.value.record == 1 and e.value.unsupported


def test_batches_and_projections():
    b = scan_text(b">a x\nAC\n>b\nG\n")
    assert b.schema.equals(SCHEMA) and b.num_rows == 2
    assert b.column(1).to_pylist() == ["x", None]
    assert scan_text(b">a x\nAC\n", [2, 0]).schema.names == ["sequence", "name"]
    assert scan_text(b">a x\nAC\n>b\n", []).num_rows == 2


def test_bgzf_round_trip_of_the_test_writer():
    text = b"".join(b">r%d\n%s\n" % (i, b"ACGT" * i) for i in range(5000))
    stream, sizes = inflate_bgzf(bgzf_bytes(text, 1))
    assert stream == text and max(sizes) == 0xff00 and sizes[-1] == 0


def _write(tmp_path, name, text):
    p = tmp_path / name
    p.write_bytes(bgzf_bytes(text, 1))
    return p


def test_abi_opens_and_plans_without_gpu(tmp_path):
    import bamscan
    text = b"".join(b">chr%d desc\n%s\n" % (i, b"ACGTACGTNN" * 3000) for i in range(60))
    path = _write(tmp_path, "g.fa.bgz", text)
    p = bamscan.FastaTableProvider(str(path))
    assert p.schema().equals(SCHEMA) and not p.schema().metadata
    assert p.supports_filters_pushdown([("name", "=", ["x"])]) == ["Unsupported"]
    with pytest.raises(bamscan.BamScanError):
        p.describe()
    plan = p.scan([2, 0], None, 10)
    assert plan.output_partition_count() == 1 and plan.schema().names == ["sequence", "name"]
    r = plan.partition_ranges(0)
    assert len(r) == 1 and r[0]["block_begin"] == 0 and r[0]["first_uoff"] == 0 and r[0]["exact_start"]
    n_blocks = len(inflate_bgzf(path.read_bytes())[1])
    plan = p.scan(None, None, None, target_partitions=4)
    assert plan.output_partition_count() == 4
    ranges = [plan.partition_ranges(i)[0] for i in range(4)]
    assert ranges[0]["block_begin"] == 0 and ranges[-1]["block_end"] == n_blocks
    for a, b in zip(ranges, ranges[1:]):
        # a range owns from its first member on, and also inflates the member in front of it (owned by the range before)
        assert b["block_begin"] == a["block_end"] - 1 and b["exact_start"]
        assert b["first_uoff"] == a["block_end"] * 0xff00 == a["stop_uoff"]
    if not _gpu_present():
        with pytest.raises(bamscan.BamScanError) as e:
            list(plan.execute(0))
        assert e.value.code == -4
    p.close()


def test_plain_and_gzip_fasta_refused(tmp_path):
    import bamscan
    text = b">r\nACGT\n"
    plain = tmp_path / "plain.fa"
    plain.write_bytes(text)
    gz = tmp_path / "plain.fa.gz"
    gz.write_bytes(gzip.compress(text))
    for p in (plain, gz):
        with pytest.raises(bamscan.BamScanError) as e:
            bamscan.FastaTableProvider(str(p))
        assert e.value.code == -2, (p, e.value)
    with pytest.raises(bamscan.BamScanError):
        bamscan.FastaTableProvider(str(plain), object_storage_options={})


def test_cpp_fasta_provider_compiles_and_plans(tmp_path):
    """include/bamscan.hpp's FastaTableProvider compiles with -Wall -Werror against the library and plans without a GPU."""
    lib = ROOT / "datafusion-bio-formats_b200"
    exe = tmp_path / "fasta_cpp_check"
    r = subprocess.run(["g++", "-std=c++17", "-O1", "-Wall", "-Werror", f"-I{ROOT / 'include'}", "-o", str(exe),
                        str(ROOT / "tests" / "native" / "fasta_cpp_check.cpp"), str(lib / "libbamscan.so"), f"-Wl,-rpath,{lib}"],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    path = _write(tmp_path, "c.fa.bgz", b"".join(b">s%d\n%s\n" % (i, b"ACGT" * 9000) for i in range(20)))
    r = subprocess.run([str(exe), str(path)], capture_output=True, text=True)
    assert r.returncode == 0 and "fasta cpp check ok" in r.stdout, r.stdout + r.stderr
