"""CPU: the FASTQ write-path oracle (oracle/fastq_write_oracle.py) pinned on the reference's FASTQ fixtures -- re-rendering the
rows the read oracle gets from them reproduces their inflated bytes exactly -- plus render -> parse round trips, every refusal
rule, the host-side schema checks of bamscan_fastq_writer_open and the C++ mirror."""
import random
import subprocess
from pathlib import Path

import pyarrow as pa
import pytest

from conftest import GOLDEN, ROOT
from oracle import fastq_oracle as R
from oracle import fastq_write_oracle as FW
from oracle.bam_write_oracle import inflate_bgzf

FQ = GOLDEN / "fastq"


def _gpu_present():
    try:
        import torch
        return torch.cuda.is_available()
    except ImportError:
        return False


def _batch(rows, with_desc=True):
    cols = {"name": [r[0] for r in rows], "sequence": [r[2] for r in rows], "quality_scores": [r[3] for r in rows]}
    if with_desc:
        cols["description"] = [r[1] for r in rows]
    order = ["name", "description", "sequence", "quality_scores"] if with_desc else ["name", "sequence", "quality_scores"]
    return pa.RecordBatch.from_arrays([pa.array(cols[c], pa.string()) for c in order], names=order)


def _as_bytes(rows):
    def b(v):
        return None if v is None else v.encode()
    return [(b(n), b(d) if d else None, b(s), b(q)) for n, d, s, q in rows]


@pytest.mark.parametrize("name", ["sample.fastq.bgz", "example.fastq.bgz"])
def test_rendering_the_fixture_rows_gives_the_fixture_bytes(name):
    o = R.OracleFastq(FQ / name)
    text = R.gunzip_members((FQ / name).read_bytes())
    assert FW.render_batch(o.scan()) == text
    # the fixture layout the writer follows: bare '+' lines, single-space separators, no tab, no CR, a final newline
    assert b"\t" not in text and b"\r" not in text and text.endswith(b"\n")
    assert all(ln == b"+" for ln in text.split(b"\n")[2::4])


def test_round_trip_on_synthetic_text():
    from conftest import make_fastq_text
    recs = R.parse_records(make_fastq_text(3000, 11))
    # the synthetic text separates some descriptions with a tab; written back they get one space and parse to the same rows
    rows = [(n.decode(), None if d is None else d.decode(), s.decode(), q.decode()) for n, d, s, q in recs]
    text = FW.render_batch(_batch(rows))
    assert R.parse_records(text) == recs


def _random_rows(rng, n):
    alphabet = "ACGTNacgtn.-*"
    descs = [None, "", " ", "x", "a b\tc", "HSQ:1:2/1", "ünïcödé ☃", "  lead", "+plus", "@at"]
    rows = []
    for i in range(n):
        L = rng.choice([0, 1, 2, 3, 4, 5, 7, 8, 31, 101, 300])
        name = rng.choice(["", "r", f"read{i}", "ü" * rng.randint(1, 9), "@x", "+y", "a/1"])
        seq = "".join(rng.choice(alphabet) for _ in range(L))
        qual = "".join(chr(rng.randint(33, 126)) for _ in range(rng.choice([L, L, rng.randint(0, 20)])))
        rows.append((name, rng.choice(descs), seq, qual))
    return rows


def test_round_trip_on_seeded_random_rows():
    rng = random.Random(20261020)
    rows = _random_rows(rng, 4000)
    recs = R.parse_records(FW.render_batch(_batch(rows)))
    assert recs == _as_bytes(rows)
    # without a description column every description reads back NULL
    recs = R.parse_records(FW.render_batch(_batch(rows, with_desc=False)))
    assert recs == [(n, None, s, q) for n, _d, s, q in _as_bytes(rows)]


REFUSALS = [
    (dict(name=None), "name is NULL"), (dict(sequence=None), "sequence is NULL"), (dict(quality_scores=None), "quality_scores is NULL"),
    (dict(name="a\nb"), "line break in name"), (dict(name="a\r"), "line break in name"), (dict(name="a b"), "space or tab in name"),
    (dict(name="\tb"), "space or tab in name"), (dict(description="x\ny"), "line break in description"),
    (dict(description="\r"), "line break in description"), (dict(sequence="AC\nGT"), "line break in sequence"),
    (dict(sequence="ACGT\r"), "line break in sequence"), (dict(quality_scores="II\nII"), "line break in quality_scores"),
    (dict(quality_scores="\rIII"), "line break in quality_scores"),
]


def refusal_batch(change, bad_row=3, n=8):
    rows = [dict(name=f"r{i}", description="d", sequence="ACGT", quality_scores="IIII") for i in range(n)]
    rows[bad_row].update(change)
    return _batch([(r["name"], r["description"], r["sequence"], r["quality_scores"]) for r in rows])


@pytest.mark.parametrize("change,msg", REFUSALS, ids=[m.replace(" ", "_") + f"_{i}" for i, (_c, m) in enumerate(REFUSALS)])
def test_each_refusal_rule(change, msg):
    with pytest.raises(FW.WriteError, match=f"row 3: {msg}"):
        FW.render_batch(refusal_batch(change))


def test_accepted_corners():
    """Empty fields, unequal sequence / quality lengths, spaces and tabs inside a description, lower case: all written as given."""
    rows = [("", None, "", ""), ("n", "", "acgt", "I"), ("n2", "a\tb c", "ACGT", "IIIIII")]
    assert FW.render_batch(_batch(rows)) == b"@\n\n+\n\n@n\nacgt\n+\nI\n@n2 a\tb c\nACGT\n+\nIIIIII\n"


def test_write_fastq_files(tmp_path):
    rows = _random_rows(random.Random(3), 2500)
    b = _batch(rows)
    text = FW.render_batch(b)
    assert len(text) > 2 * 0xff00
    for comp in (0, 1):
        p = tmp_path / f"o{comp}.fastq.bgz"
        assert FW.write_fastq(p, [b.slice(0, 1000), b.slice(1000)], comp) == 2500
        stream, sizes = inflate_bgzf(p.read_bytes())
        assert stream == text and sizes[-1] == 0 and all(s == 0xff00 for s in sizes[:-2])
    p = tmp_path / "o.fastq"
    FW.write_fastq(p, [b], 2)
    assert p.read_bytes() == text
    FW.write_fastq(tmp_path / "e.fastq.bgz", [], 0)
    assert inflate_bgzf((tmp_path / "e.fastq.bgz").read_bytes()) == (b"", [0])


def test_compression_follows_the_extension():
    import bamscan
    for path, want in (("a.fastq.bgz", 0), ("a.FQ.BGZF", 0), ("a.fastq.gz", 0), ("a.fastq", 2), ("a.fq", 2), ("a.txt", 2)):
        assert bamscan.fastq_compression_for(path) == want, path
        assert bamscan.FastqWriteExec(path, bamscan.FASTQ_SCHEMA).compression == want
    assert bamscan.FastqWriteExec("a.fastq", bamscan.FASTQ_SCHEMA, 1).compression == 1
    pw = bamscan.FastqTableProvider.new_for_write("x.fastq.bgz")
    assert pw.schema().equals(bamscan.FASTQ_SCHEMA) and pw.schema().equals(R.SCHEMA)


def test_fastq_writer_validates_the_schema_and_refuses_without_gpu(tmp_path):
    """Columns by name, Utf8 only, checked on the host before the device is touched; no CPU path behind it."""
    import bamscan
    out = tmp_path / "o.fastq.bgz"
    no_seq = pa.schema([f for f in R.SCHEMA if f.name != "sequence"])
    with pytest.raises(bamscan.BamScanError, match="Required column 'sequence' not found") as e:
        bamscan.FastqWriteExec(str(out), no_seq).execute([])
    assert e.value.code == -7
    for col in ("name", "description", "quality_scores"):
        wrong = pa.schema([pa.field(col, pa.binary()) if f.name == col else f for f in R.SCHEMA])
        with pytest.raises(bamscan.BamScanError, match=f"Column '{col}' must be Utf8") as e:
            bamscan.FastqWriteExec(str(out), wrong).execute([])
        assert e.value.code == -7
    with pytest.raises(bamscan.BamScanError, match="compression 3") as e:
        bamscan.FastqWriteExec(str(out), R.SCHEMA, 3).execute([])
    assert e.value.code == -6
    assert not out.exists()
    if _gpu_present():
        return
    # description is optional and extra columns are ignored: such schemas pass the checks and reach the device check
    from oracle.bam_oracle import OracleBam
    bam_schema = OracleBam(str(GOLDEN / "multi_chrom.bam"), tag_fields=["NM"]).schema
    for schema in (R.SCHEMA, pa.schema([f for f in R.SCHEMA if f.name != "description"]), bam_schema):
        for comp in (None, 0, 1, 2):
            with pytest.raises(bamscan.BamScanError, match="no CPU path") as e:
                bamscan.FastqWriteExec(str(out), schema, comp).execute([])
            assert e.value.code == -4 and not out.exists()
    with pytest.raises(bamscan.BamScanError, match="no CPU path"):
        bamscan.FastqTableProvider.new_for_write(str(tmp_path / "p.fastq")).insert_into([])
    assert not (tmp_path / "p.fastq").exists()
    with pytest.raises(NotImplementedError):
        bamscan.FastqTableProvider.new_for_write(str(out)).insert_into([], "append")


CPP_CHECK = r"""
#include <cstdio>
#include "bamscan.hpp"

static ArrowSchema field(const char* name, const char* fmt) { ArrowSchema s{}; s.format = fmt; s.name = name; return s; }

int main(int argc, char** argv) {
  ArrowSchema name = field("name", "u"), seq = field("sequence", "u"), qual = field("quality_scores", "u"), extra = field("flags", "I");
  ArrowSchema* full[4] = {&name, &seq, &qual, &extra};
  ArrowSchema* partial[2] = {&name, &qual};
  ArrowSchema st = field("", "+s");
  st.n_children = 2; st.children = partial;
  try { bamscan_cpp::FastqWriteExec w(argv[1], &st); return 1; }
  catch (const bamscan_cpp::Error& e) { std::printf("partial %d %s\n", e.code, e.what()); }
  st.n_children = 4; st.children = full;
  try {
    bamscan_cpp::FastqWriteExec w(argv[1], &st, 2);
    std::printf("opened %llu\n", (unsigned long long)w.finish());
  } catch (const bamscan_cpp::Error& e) { std::printf("full %d %s\n", e.code, e.what()); }
  return 0;
}
"""


def test_cpp_fastq_writer_compiles_and_checks_the_schema(tmp_path):
    """include/bamscan.hpp's FastqWriteExec compiles with -Wall against the library; the schema check runs on the host."""
    lib = ROOT / "datafusion-bio-formats_b200"
    src = tmp_path / "fq_write.cpp"
    src.write_text(CPP_CHECK)
    exe = tmp_path / "fq_write"
    r = subprocess.run(["g++", "-std=c++17", "-O1", "-Wall", "-Werror", f"-I{ROOT / 'include'}", "-o", str(exe), str(src),
                        str(lib / "libbamscan.so"), f"-Wl,-rpath,{lib}"], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    out = tmp_path / "o.fastq"
    r = subprocess.run([str(exe), str(out)], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "partial -7 Required column 'sequence' not found" in r.stdout, r.stdout
    if _gpu_present():
        assert "opened 0" in r.stdout and out.read_bytes() == b""
    else:
        assert "full -4" in r.stdout and not out.exists()
