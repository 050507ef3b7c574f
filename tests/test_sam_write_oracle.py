"""CPU: the SAM write-path oracle (oracle/sam_write_oracle.py) pinned against an independent renderer (tests/sam_render.py) on the
reference's fixtures, read back through the SAM scan oracle against the BAM write + scan of the same batches, every refusal rule
and the accepted corners, the float text against the C oracle's rule, and the host-side checks of bamscan_sam_writer_open."""
import random
import struct
import subprocess

import numpy as np
import pyarrow as pa
import pytest

from conftest import GOLDEN, ROOT, make_edge_bam
from oracle import bam_write_oracle as W
from oracle import sam_write_oracle as SW
from oracle.bam_oracle import OracleBam
from oracle.sam_oracle import OracleSam
from sam_render import read_bam, render_record

FIXTURES = ["multi_chrom.bam", "bam_with_tags.bam", "10x_pbmc_tags.bam", "nanopore_custom_tags.bam", "multi_chrom_large.bam", "no_coor_only.bam"]


def _gpu_present():
    try:
        import torch
        return torch.cuda.is_available()
    except ImportError:
        return False


def _aux_letters(recs):
    """{tag: (letter, subtype)} over every record's aux fields, tags in order of first appearance."""
    out = {}
    for rec in recs:
        l_name, n_cig, l_seq = rec[8], struct.unpack_from("<H", rec, 12)[0], struct.unpack_from("<i", rec, 16)[0]
        p = 32 + l_name + 4 * n_cig + (l_seq + 1) // 2 + l_seq
        while p < len(rec):
            tag, t = rec[p:p + 2].decode(), chr(rec[p + 2]); p += 3
            sub = None
            if t in "cCA": p += 1
            elif t in "sS": p += 2
            elif t in "iIf": p += 4
            elif t in "ZH": p = rec.index(b"\0", p) + 1
            else:
                sub = chr(rec[p]); n = struct.unpack_from("<I", rec, p + 1)[0]
                p += 5 + n * {"c": 1, "C": 1, "s": 2, "S": 2, "i": 4, "I": 4, "f": 4}[sub]
            out.setdefault(tag, (t, sub))
    return out


def fixture_batch(name, zero_based=True):
    """The fixture's rows with all of its tags, in file order, typed with the file's own letters (integers by column type: SAM
    text writes every integer letter as `i`).  A tag the scan reads into a column of another kind than its letter (an integer
    tag the registry declares as a string) is left out: its SAM text cannot be the file's.  -> (batch, schema, tags, records)"""
    _text, _names, _lens, recs = read_bam((GOLDEN / name).read_bytes())
    letters = _aux_letters(recs)
    o = OracleBam(str(GOLDEN / name), zero_based=zero_based, tag_fields=list(letters))
    letters = {t: v for t, v in letters.items() if not (v[0] in "cCsSiI" and o.schema.field(t).type == pa.string())}
    tags = list(letters)
    o = OracleBam(str(GOLDEN / name), zero_based=zero_based, tag_fields=tags)
    batch = o.scan(None)
    fields = list(o.schema)[:12]
    for tag, (t, sub) in letters.items():
        f = o.schema.field(tag)
        spec = f"B:{sub}" if t == "B" else ("I" if f.type == pa.uint32() else "i") if t in "cCsSiI" else t
        fields.append(pa.field(tag, f.type, True, {"bio.bam.tag.tag": tag, "bio.bam.tag.type": spec}))
    schema = pa.schema(fields, metadata=o.schema.metadata)
    b = pa.RecordBatch.from_arrays([batch.column(batch.schema.get_field_index(f.name)) for f in fields], schema=schema)
    return b, schema, tags, recs


def _f32(text):
    return np.array([np.float32(text)]).view(np.uint32)[0]


def assert_same_line(got: str, want: str, what, tags):
    g, w = got.split("\t"), want.split("\t")
    assert g[:11] == w[:11], f"{what}: core fields {g[:11]} vs {w[:11]}"
    ga, wa = {f[:2]: f for f in g[11:]}, {f[:2]: f for f in w[11:] if f[:2] in tags}
    assert sorted(ga) == sorted(wa), what
    for tag, wf in wa.items():
        gf = ga[tag]
        if wf[3] == "f" or wf.startswith(tag + ":B:f"):
            gv, wv = gf.split(":", 2)[2].split(","), wf.split(":", 2)[2].split(",")
            assert gf[:5] == wf[:5] and len(gv) == len(wv) and [_f32(x) for x in gv[1 if wf[3] == "B" else 0:]] == \
                [_f32(x) for x in wv[1 if wf[3] == "B" else 0:]], f"{what}: {gf} vs {wf}"
        else:
            assert gf == wf, f"{what}: {gf} vs {wf}"


@pytest.mark.parametrize("name", FIXTURES)
def test_fixture_lines_equal_the_independent_renderer(name):
    """Every oracle line equals sam_render.render_record of the fixture's own record bytes, field by field (f values as f32).
    One allowed difference: a record without qualities scans as ' ' x n, which the writers take as scores 0 ('!')."""
    b, schema, tags, recs = fixture_batch(name)
    text, names, _lens = W.build_bam_header(schema)
    lines = SW.render_batch(b, names, tags, True).decode().split("\n")
    assert lines[-1] == "" and len(lines) - 1 == len(recs) == b.num_rows
    for i, (line, rec) in enumerate(zip(lines, recs)):
        want = render_record(rec, names).split("\t")
        if want[10] == "*" and want[9] != "*":
            want[10] = "!" * len(want[9])
        assert_same_line(line, "\t".join(want), f"{name} record {i}", tags)
    assert SW.sam_text([b], schema, tags).startswith(text.encode())


def _no_qual_rows(batch):
    return {i for i, (s, q) in enumerate(zip(batch.column(batch.schema.get_field_index("sequence")).to_pylist(),
                                             batch.column(batch.schema.get_field_index("quality_scores")).to_pylist()))
            if s not in (None, "", "*") and q in (None, "", "*")}


def assert_round_trip(sam_batch, bam_batch, no_qual, what):
    """The SAM scan of the SAM file equals the BAM scan of the BAM file, except (1) `end` of placed reads whose CIGAR spans no
    reference base and (2) "" against ' ' x n for rows that had a sequence and no qualities."""
    assert sam_batch.schema.names == bam_batch.schema.names and sam_batch.num_rows == bam_batch.num_rows, what
    cig = bam_batch.column(bam_batch.schema.get_field_index("cigar")).to_pylist()
    start = bam_batch.column(bam_batch.schema.get_field_index("start")).to_pylist()
    for name in bam_batch.schema.names:
        g = sam_batch.column(sam_batch.schema.get_field_index(name)).to_pylist()
        w = bam_batch.column(bam_batch.schema.get_field_index(name)).to_pylist()
        for r, (x, y) in enumerate(zip(g, w)):
            if x == y or (isinstance(x, float) and isinstance(y, float) and np.isnan(x) and np.isnan(y)):
                continue
            if name == "end" and start[r] is not None and W.parse_cigar(cig[r]) is not None and \
                    sum(o >> 4 for o in W.parse_cigar(cig[r]) if (o & 15) in (0, 2, 3, 7, 8)) == 0:
                continue
            if name == "quality_scores" and r in no_qual and x == "" and y == " " * len(y):
                continue
            if isinstance(x, list) and isinstance(y, list) and len(x) == len(y) and \
                    all(a == c or (np.isnan(a) and np.isnan(c)) for a, c in zip(x, y)):
                continue
            raise AssertionError(f"{what}: column {name} row {r}: {x!r} vs {y!r}")


@pytest.mark.parametrize("name", FIXTURES)
def test_round_trip_equals_the_bam_round_trip(name, tmp_path):
    b, schema, tags, _recs = fixture_batch(name)
    for zb in (True, False):
        sam, bam = tmp_path / f"o{int(zb)}.sam", tmp_path / f"o{int(zb)}.bam"
        assert SW.write_sam(sam, [b], schema, tags, zb) == b.num_rows
        W.write_bam(bam, [b], schema, tags, zb)
        assert_round_trip(OracleSam(sam, zb, tags).scan(None), OracleBam(str(bam), zb, tags).scan(None), _no_qual_rows(b), f"{name} zero_based={zb}")


def test_edge_bam_round_trip(tmp_path):
    src = tmp_path / "edge.bam"
    make_edge_bam(src, missing_qual=True)
    tags = ["NM", "MD", "XS", "XF", "XB", "XA", "XI", "XU"]
    o = OracleBam(str(src), tag_fields=tags)
    b = o.scan(None)
    SW.write_sam(tmp_path / "o.sam", [b], o.schema, tags)
    W.write_bam(tmp_path / "o.bam", [b], o.schema, tags)
    assert_round_trip(OracleSam(tmp_path / "o.sam", True, tags).scan(None), OracleBam(str(tmp_path / "o.bam"), True, tags).scan(None),
                      _no_qual_rows(b), "edge")
    text = (tmp_path / "o.sam").read_bytes().decode()
    assert text.startswith(W.build_bam_header(o.schema)[0])


# ---- rules ----------------------------------------------------------------------------------------------------------------

def tf(name, typ, spec):
    return pa.field(name, typ, True, {"bio.bam.tag.tag": name, "bio.bam.tag.type": spec})


RULE_TAGS = [tf("Xi", pa.int32(), "i"), tf("Xf", pa.float32(), "f"), tf("Xd", pa.float64(), "f"), tf("XZ", pa.string(), "Z"),
             tf("XH", pa.string(), "H"), tf("XA", pa.string(), "A"), tf("Xa", pa.int32(), "A"), tf("XB", pa.list_(pa.uint8()), "B:C"),
             tf("XF", pa.list_(pa.float32()), "B:f"), tf("Xs", pa.list_(pa.int32()), "B:s"), tf("Xq", pa.string(), "q")]
RULE_TAG_NAMES = [f.name for f in RULE_TAGS]


def rule_schema():
    core = [pa.field("name", pa.string()), pa.field("chrom", pa.string()), pa.field("start", pa.uint32()), pa.field("end", pa.uint32()),
            pa.field("flags", pa.uint32(), False), pa.field("cigar", pa.string(), False), pa.field("mapping_quality", pa.uint32(), False),
            pa.field("mate_chrom", pa.string()), pa.field("mate_start", pa.uint32()), pa.field("sequence", pa.string(), False),
            pa.field("quality_scores", pa.string(), False), pa.field("template_length", pa.int32(), False)]
    md = {"bio.bam.reference_sequences": '[{"name":"chr1","length":249250621},{"name":"chr2","length":1000}]'}
    return pa.schema(core + RULE_TAGS, metadata=md)


def row(**kw):
    d = dict(name="r", chrom="chr1", start=99, end=None, flags=0, cigar="4M", mapping_quality=60, mate_chrom=None, mate_start=None,
             sequence="ACGT", quality_scores="IIII", template_length=0)
    d.update(kw)
    return d


def one_line(zero_based=True, **kw):
    return SW.render_batch(pa.RecordBatch.from_pylist([row(**kw)], schema=rule_schema()), ["chr1", "chr2"], RULE_TAG_NAMES, zero_based).decode()


# (change to row 3, GPU error code, message): shared rules first (the BAM writer's reasons), then the SAM-only ones
REFUSALS = [
    (dict(flags=65536), -2, "16-bit SAM flags", True), (dict(cigar="10M5"), -2, "CIGAR", True), (dict(cigar="M"), -2, "CIGAR", True),
    (dict(quality_scores="III"), -2, "length mismatch", True), (dict(name="n" * 255), -2, "longer than 254", True),
    (dict(start=2**31), -2, "position does not fit", True), (dict(Xi=None, XB=[1, 2], Xs=[40000]), -7, "fit", True),
    (dict(XH="abc"), -7, "hex", True), (dict(XA="ab"), -7, "single ASCII byte|Character tags", True), (dict(Xd=1e39), -7, "fit", True),
    (dict(name=""), -2, "invalid QNAME", False), (dict(name="a b"), -2, "invalid QNAME", False), (dict(name="a\tb"), -2, "invalid QNAME", False),
    (dict(name="@r"), -2, "invalid QNAME", False), (dict(name="ü"), -2, "invalid QNAME", False),
    (dict(sequence="AC-T"), -2, "invalid SEQ", False), (dict(sequence="ACG ", quality_scores="IIII"), -2, "invalid SEQ", False),
    (dict(quality_scores="II\x7fI"), -2, "invalid QUAL", False), (dict(quality_scores="IIIé"[:4]), -2, "invalid QUAL|length mismatch", None),
    (dict(XZ="a\tb"), -2, "invalid Z tag value", False), (dict(XZ="x\ny"), -2, "invalid Z tag value", False),
    (dict(Xq="é"), -2, "invalid Z tag value", False), (dict(XA=" "), -2, "invalid A tag value", False),
    (dict(Xa=127), -2, "invalid A tag value", False), (dict(Xa=32), -2, "invalid A tag value", False),
]


def refusal_batch(change, bad_row=3, n=8):
    rows = [row(name=f"r{i}") for i in range(n)]
    rows[bad_row].update(change)
    return pa.RecordBatch.from_pylist(rows, schema=rule_schema())


REFUSAL_IDS = [f"{i}_{m.split('|')[0].replace(' ', '_')}" for i, (_c, _e, m, _s) in enumerate(REFUSALS)]


@pytest.mark.parametrize("change,code,msg,shared", REFUSALS, ids=REFUSAL_IDS)
def test_each_refusal_rule(change, code, msg, shared):
    with pytest.raises(SW.WriteError, match=f"row 3: .*({msg})") as e:
        SW.render_batch(refusal_batch(change), ["chr1", "chr2"], RULE_TAG_NAMES)
    if shared is not None:
        assert e.value.shared == shared
    if shared:                                                       # the BAM writer refuses the same row
        with pytest.raises(W.WriteError):
            W.encode_batch(refusal_batch(change), ["chr1", "chr2"], RULE_TAG_NAMES, True)
    elif shared is False:
        W.encode_batch(refusal_batch(change), ["chr1", "chr2"], RULE_TAG_NAMES, True)


def test_accepted_corners():
    f = one_line().rstrip("\n").split("\t")
    assert f == ["r", "0", "chr1", "100", "60", "4M", "*", "0", "0", "ACGT", "IIII"]
    assert one_line(zero_based=False).split("\t")[3] == "99"
    # '*' / NULL / "" fields, unknown references, position 0, '=' mates
    f = one_line(name=None, chrom="chrNope", start=None, cigar="*", sequence="*", quality_scores="*", mate_chrom="=", mate_start=0).split("\t")
    assert f[:11] == ["*", "0", "*", "0", "60", "*", "*", "1", "0", "*", "*\n"]
    f = one_line(name="*", cigar="", sequence="", quality_scores=None, mate_chrom="chr1", mate_start=5, zero_based=False).split("\t")
    assert f[:11] == ["*", "0", "chr1", "99", "60", "*", "=", "5", "0", "*", "*\n"]
    assert one_line(start=0, zero_based=False).split("\t")[3] == "0"
    assert one_line(mate_chrom="chr2", mate_start=7).split("\t")[6:8] == ["chr2", "8"]
    assert one_line(mate_chrom="chrNope", mate_start=7).split("\t")[6] == "*"
    # CIGAR from its operations, lower-case and '.' bases as given, qualities below '!' as '!', NULL MAPQ-like values
    f = one_line(cigar="010M0002I", sequence="ac.=N" * 2 + "gg", quality_scores=" !\"~" * 3, mapping_quality=300, template_length=-2**31,
                 flags=65535).split("\t")
    assert f[1] == "65535" and f[4] == "44" and f[5] == "10M2I" and f[8] == "-2147483648" and f[9] == "ac.=Nac.=Ngg" and f[10] == "!!\"~" * 3 + "\n"
    f = one_line(sequence="ACGT", quality_scores="").split("\t")
    assert f[10] == "*\n"
    # tags: NULL -> no field, integer letters as i, H upper-cased, empty B arrays, unknown letters as Z
    line = one_line(Xi=-5, XZ="", XH="1a2b", XA="~", Xa=33, XB=[], XF=[], Xs=[-1, 300], Xq="q q").rstrip("\n")
    assert line.split("\t")[11:] == ["Xi:i:-5", "XZ:Z:", "XH:H:1A2B", "XA:A:~", "Xa:A:!", "XB:B:C", "XF:B:f", "Xs:B:s,-1,300", "Xq:Z:q q"]


@pytest.mark.parametrize("bits,text", [(0x7fc00000, "NaN"), (0xffc00001, "NaN"), (0x7f800000, "inf"), (0xff800000, "-inf"), (0, "0"),
                                       (0x80000000, "-0"), (1, "0." + "0" * 44 + "1"), (0x3f800000, "1"), (0xbfc00000, "-1.5"),
                                       (0x3dcccccd, "0.1"), (0x7f7fffff, "340282350000000000000000000000000000000"), (0x33d6bf95, "0.0000001")])
def test_float_text_corners(bits, text):
    assert SW.f32_text(bits) == text
    f = one_line(Xf=float(np.array([bits], np.uint32).view(np.float32)[0]), XF=[float(np.array([bits], np.uint32).view(np.float32)[0])] * 2)
    assert f"Xf:f:{text}\t" in f and f"XF:B:f,{text},{text}" in f


def test_float_text_matches_the_c_oracle_rule(tmp_path):
    """The Python restatement against tests/native/f32_text_check.cpp's rule (oracle/bam_oracle.c::rust_f32_to_string) on the
    bit patterns that program checks: edges, every exponent's corners, random words, subnormals, "human" values."""
    src = (ROOT / "tests" / "native" / "f32_text_check.cpp").read_text().split("int main")[0]
    src = src.replace("../../datafusion-bio-formats_b200", str(ROOT / "datafusion-bio-formats_b200"))
    src += ('int main() { unsigned b; char out[128]; while (scanf("%x", &b) == 1) { float v; memcpy(&v, &b, 4); '
            'oracle_rule(v, out); printf("%s\\n", out); } return 0; }\n')
    (tmp_path / "rule.cpp").write_text(src)
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-o", str(tmp_path / "rule"), str(tmp_path / "rule.cpp")])
    rng = random.Random(12345)
    bits = [0x00000000, 0x80000000, 0x00000001, 0x007fffff, 0x00800000, 0x00800001, 0x7f7fffff, 0x7f800000, 0xff800000, 0x7fc00000,
            0x3f800000, 0x3fc00000, 0x3dcccccd, 0x33d6bf95, 0x60ad78ec, 0x4b800000, 0x4b7fffff, 0x3f7fffff, 0x34000000, 0x01000000, 0x7e800000]
    bits += [(e << 23) | m for e in range(255) for m in (0, 1, 0x7fffff, 0x400000)]
    bits += [rng.getrandbits(32) for _ in range(12000)] + [rng.randrange(0x800000) for _ in range(3000)]
    bits += [int(np.array([np.float32(rng.randint(-1000000, 1000000) / 1000.0)]).view(np.uint32)[0]) for _ in range(3000)]
    out = subprocess.run([str(tmp_path / "rule")], input="\n".join("%x" % b for b in bits), capture_output=True, text=True, check=True).stdout.split("\n")
    bad = [(hex(b), SW.f32_text(b), o) for b, o in zip(bits, out) if SW.f32_text(b) != o]
    assert not bad, bad[:10]


def test_header_and_zero_rows(tmp_path):
    s = rule_schema()
    p = tmp_path / "none.sam"
    assert SW.write_sam(p, [], s, RULE_TAG_NAMES) == 0
    assert p.read_bytes() == b"@HD\tVN:1.6\n@SQ\tSN:chr1\tLN:249250621\n@SQ\tSN:chr2\tLN:1000\n"
    SW.write_sam(p, [pa.RecordBatch.from_pylist([], schema=s)], s, RULE_TAG_NAMES, True, {"bio.bam.sort_order": "coordinate"})
    assert p.read_bytes().startswith(b"@HD\tVN:1.6\tSO:coordinate\n")


# ---- host checks ------------------------------------------------------------------------------------------------------------

def test_sam_writer_validates_the_schema_and_refuses_without_gpu(tmp_path):
    """Columns, tag types and tag names are checked on the host before the device is touched; no CPU path behind it."""
    import bamscan
    s = rule_schema()
    out = tmp_path / "o.sam"
    with pytest.raises(bamscan.BamScanError, match="Required column 'flags' not found") as e:
        bamscan.SamWriteExec(str(out), pa.schema([f for f in s if f.name != "flags"]), []).execute([])
    assert e.value.code == -7
    bad = pa.schema(list(s) + [tf("Xz", pa.int32(), "Z")])
    with pytest.raises(bamscan.BamScanError, match="type mismatch") as e:
        bamscan.SamWriteExec(str(out), bad, ["Xz"]).execute([])
    assert e.value.code == -7
    for tag in ("1X", "X_", "X-"):
        with pytest.raises(bamscan.BamScanError, match=r"\[A-Za-z\]\[A-Za-z0-9\]") as e:
            bamscan.SamWriteExec(str(out), pa.schema(list(s) + [tf(tag, pa.int32(), "i")]), [tag]).execute([])
        assert e.value.code == -7
    assert not out.exists()
    with pytest.raises(bamscan.BamScanError, match="plain SAM output is out of scope"):
        bamscan.BamWriteExec(str(tmp_path / "o.SAM"), s, [])
    assert bamscan.is_sam_path("a.sam") and bamscan.is_sam_path("A.SaM") and not bamscan.is_sam_path("a.sam.gz")
    if _gpu_present():
        return
    for tags in ([], RULE_TAG_NAMES, ["1X"]):                        # (a tag name not in the schema is not a column: skipped)
        with pytest.raises(bamscan.BamScanError, match="no CPU path") as e:
            bamscan.SamWriteExec(str(out), s, tags).execute([])
        assert e.value.code == -4 and not out.exists()
    for path in ("p.sam", "P.SAM"):
        with pytest.raises(bamscan.BamScanError, match="no CPU path"):
            bamscan.BamTableProvider.new_for_write(str(tmp_path / path), s, RULE_TAG_NAMES).insert_into([])
        assert not (tmp_path / path).exists()


CPP_CHECK = r"""
#include <cstdio>
#include "bamscan.hpp"

static ArrowSchema field(const char* name, const char* fmt) { ArrowSchema s{}; s.format = fmt; s.name = name; return s; }

int main(int argc, char** argv) {
  ArrowSchema c[11] = {field("name", "u"), field("chrom", "u"), field("start", "I"), field("flags", "I"), field("cigar", "u"),
                       field("mapping_quality", "I"), field("mate_chrom", "u"), field("mate_start", "I"), field("sequence", "u"),
                       field("quality_scores", "u"), field("template_length", "i")};
  ArrowSchema* kids[11];
  for (int i = 0; i < 11; i++) kids[i] = &c[i];
  ArrowSchema st = field("", "+s");
  st.n_children = 10; st.children = kids;
  try { bamscan_cpp::SamWriteExec w(argv[1], "@HD\tVN:1.6\n", {"chr1"}, {1000}, &st); return 1; }
  catch (const bamscan_cpp::Error& e) { std::printf("partial %d %s\n", e.code, e.what()); }
  st.n_children = 11;
  try {
    bamscan_cpp::SamWriteExec w(argv[1], "@HD\tVN:1.6\n", {"chr1"}, {1000}, &st);
    std::printf("opened %llu\n", (unsigned long long)w.finish());
  } catch (const bamscan_cpp::Error& e) { std::printf("full %d %s\n", e.code, e.what()); }
  return 0;
}
"""


def test_cpp_sam_writer_compiles_and_checks_the_schema(tmp_path):
    """include/bamscan.hpp's SamWriteExec compiles with -Wall -Werror against the library; the schema check runs on the host."""
    lib = ROOT / "datafusion-bio-formats_b200"
    src = tmp_path / "sam_write.cpp"
    src.write_text(CPP_CHECK)
    exe = tmp_path / "sam_write"
    r = subprocess.run(["g++", "-std=c++17", "-O1", "-Wall", "-Werror", f"-I{ROOT / 'include'}", "-o", str(exe), str(src),
                        str(lib / "libbamscan.so"), f"-Wl,-rpath,{lib}"], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    out = tmp_path / "o.sam"
    r = subprocess.run([str(exe), str(out)], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "partial -7 Required column 'template_length' not found" in r.stdout, r.stdout
    if _gpu_present():
        assert "opened 0" in r.stdout and out.read_bytes() == b"@HD\tVN:1.6\n"
    else:
        assert "full -4" in r.stdout and not out.exists()
