"""CPU: the plain-SAM scan's host side and its oracle.
- oracle/sam_oracle.py on every golden BAM rendered to SAM equals the BAM oracle on the BAM itself (schema and header metadata as
  parsed JSON, every column), except the documented cell: end of a placed read whose CIGAR spans nothing;
- csrc/f32_parse.h (the transcoder's `f` parser) compiled for the host against exact rational rounding;
- planning without a GPU: SAM open, schema, describe, partition counts and block-range cuts on line starts;
- the SAM header / tag-inference parser under ASan + UBSan on corrupted SAM text."""
import random
import struct
import subprocess
from fractions import Fraction
from pathlib import Path

import numpy as np
import pytest

import sam_render
from conftest import GOLDEN

ROOT = Path(__file__).resolve().parent.parent
CSRC = ROOT / "datafusion-bio-formats_b200" / "csrc"
FIXTURES = ["multi_chrom.bam", "bam_with_tags.bam", "10x_pbmc_tags.bam", "nanopore_custom_tags.bam", "no_coor_only.bam"]


def _render(tmp_path, name):
    p = tmp_path / (name[:-4] + ".sam")
    p.write_bytes(sam_render.bam_to_sam((GOLDEN / name).read_bytes()))
    return p


def _all_tags(path):
    from oracle.bam_oracle import OracleBam
    return sorted({t for aux in OracleBam(str(path))._iter_aux(1 << 30) for t in aux})


@pytest.mark.parametrize("fixture", FIXTURES)
def test_oracle_on_rendered_sam_equals_bam_oracle(tmp_path, fixture):
    from oracle.bam_oracle import OracleBam, schema_equal
    from oracle.sam_oracle import OracleSam
    sam = _render(tmp_path, fixture)
    for tags in (None, _all_tags(GOLDEN / fixture)):
        for zero_based in (True, False):
            for binary_cigar in (False, True):
                ob = OracleBam(str(GOLDEN / fixture), zero_based, tags, binary_cigar)
                os_ = OracleSam(str(sam), zero_based, tags, binary_cigar)
                assert schema_equal(ob.schema, os_.schema)
                a, b = ob.scan().to_pydict(), os_.scan().to_pydict()
                for name in a:
                    want = a[name]
                    if name == "end":
                        want = [e if e is not None or s is None or s - (0 if zero_based else 1) == 0 else s - (0 if zero_based else 1) for e, s in zip(want, a["start"])]
                    assert b[name] == want, (fixture, tags, name)


def test_oracle_edge_rules():
    from oracle.sam_oracle import SamError, parse_sam
    text = (b"@SQ\tSN:c\tLN:10\nr\t0\tc\t+2\t5\t*\t=\t0\t+3\tAC\t*\tXA:i:70000\tXB:i:-3\tXE:B:f\r\n"
            b"s\t4\t*\t0\t0\t*\t*\t0\t0\t*\t*")
    _h, names, _l, ok, recs, no_qual, _end_null = parse_sam(text)
    assert ok and names == ["c"] and len(recs) == 2 and no_qual == {0}
    r = recs[0]
    assert struct.unpack_from("<iii", r, 4)[:2] == (0, 1) and r.endswith(b"XAI" + struct.pack("<I", 70000) + b"XBc\xfd" + b"XEBf\0\0\0\0")
    for bad, what in ((b"r\t0\tc\t1\t0\t*\t*\t0\t0\t*\t*\tXA:i:1\tXA:i:2", "duplicate"), (b"", "fewer than 11"), (b"@x\t0\tc\t1\t0\t*\t*\t0\t0\t*\t*", "QNAME")):
        with pytest.raises(SamError, match=what):
            parse_sam(b"@SQ\tSN:c\tLN:10\nok\t0\tc\t1\t0\t*\t*\t0\t0\t*\t*\n" + bad + b"\nok\t0\tc\t1\t0\t*\t*\t0\t0\t*\t*\n")


@pytest.fixture(scope="module")
def f32_driver(tmp_path_factory):
    exe = tmp_path_factory.mktemp("f32p") / "f32_parse_driver"
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-o", str(exe), str(ROOT / "tests" / "native" / "f32_parse_driver.cpp")])
    return exe


def _parse_all(exe, strings):
    out = subprocess.run([str(exe)], input="\n".join(strings) + "\n", capture_output=True, text=True, check=True).stdout.split()
    assert len(out) == len(strings)
    return out


def test_f32_parse_round_trips_shortest_text(f32_driver):
    rng = np.random.default_rng(5)
    bits = np.concatenate([rng.integers(0, 0x7F800000, 200000, dtype=np.uint32), np.arange(0, 2000, dtype=np.uint32),
                           np.uint32(0x00800000) + np.arange(-500, 500, dtype=np.int64).astype(np.uint32),
                           np.array([0x7F7FFFFF, 0x7F7FFFFE, 0x3F800000, 0x4B800000, 0x33800000], dtype=np.uint32)])
    bits = np.concatenate([bits, bits[:20000] | np.uint32(0x80000000)])
    strings = [str(v) for v in bits.view(np.float32)]
    got = _parse_all(f32_driver, strings)
    bad = [(s, g, f"{b:08x}") for s, g, b in zip(strings, got, bits) if g != f"{b:08x}"]
    assert not bad, bad[:10]


def _value(b):
    e, m = b >> 23, b & 0x7FFFFF
    return Fraction(m if e == 0 else m | 0x800000) * Fraction(2) ** ((e if e else 1) - 150)


def _exact_decimal(fr: Fraction, extra=0) -> str:
    """Fraction with a power-of-two denominator as an exact decimal string (+ `extra` trailing digits)."""
    k = 0
    while fr.denominator != 1:
        fr *= 10; k += 1
    digits = str(fr.numerator).rjust(k + 1, "0")
    s = digits[:len(digits) - k] + ("." + digits[len(digits) - k:] if k else "")
    return s + ("" if k else ".") + "0" * extra if extra else s


def test_f32_parse_against_exact_rounding(f32_driver):
    from oracle.sam_oracle import f32_from_text
    rng = random.Random(11)
    strings = ["3.4028235e38", "3.4028236e38", "340282356779733661637539395458142568448", "340282356779733661637539395458142568447",
               "7.006492321624085e-46", "7.006492321624086e-46", "7.0064923216240862e-46", "1e-46", "1e39", "0.0", "-0", "1e-400",
               "1e400", "+1.5", ".5", "5.", "1E+2", "00012.5000", "inf", "-Infinity", "NaN", "1e", "e5", "", "+", "1.2.3", "0x10", "1_0"]
    for _ in range(3000):                       # random decimals: mantissa up to 30 digits, exponents across the range
        m = str(rng.randrange(1, 10 ** rng.randrange(1, 30)))
        strings.append(f"{m[:1]}.{m[1:]}e{rng.randrange(-50, 40)}" if len(m) > 1 else f"{m}e{rng.randrange(-50, 40)}")
    for _ in range(1500):                       # exact halfway points (ties to even) and their neighbours one digit away
        b = rng.choice([rng.randrange(1, 0x7F7FFFFF), rng.randrange(1, 0x00800000)])
        h = (_value(b) + _value(b + 1)) / 2
        s = _exact_decimal(h)
        strings.append(s)
        strings.append(s + "000000001" if "." in s else s + ".000000001")
        if s.endswith("5"):
            strings.append(s[:-1] + "4" + "9" * 30)
    got = _parse_all(f32_driver, strings)
    for s, g in zip(strings, got):
        try:
            want = f"{f32_from_text(s):08x}"
        except ValueError:
            want = "err"
        assert g == want, (s, g, want)


def test_planning_without_gpu(tmp_path):
    import bamscan
    sam = _render(tmp_path, "multi_chrom.bam")
    prov = bamscan.BamTableProvider(str(sam), tag_fields=["NM", "MD", "RG"])
    from oracle.sam_oracle import OracleSam
    from oracle.bam_oracle import schema_equal
    assert schema_equal(prov.schema(), OracleSam(str(sam), tag_fields=["NM", "MD", "RG"]).schema)
    assert prov.scan(None, [], None).output_partition_count() == 1
    assert prov.supports_filters_pushdown([("chrom", "=", ["chr1"])]) == ["Inexact"]     # as for a BAM without an index
    data = sam.read_bytes()
    body = 0
    while data[body:body + 1] == b"@":                                  # the header: the leading lines that start with '@'
        body = data.index(b"\n", body) + 1
    for n in (2, 3, 8):
        plan = prov.scan(None, [], None, target_partitions=n, partition_mode="block_range")
        assert plan.output_partition_count() == n
        starts = [r["first_uoff"] for p in range(n) for r in plan.partition_ranges(p)]
        assert starts[0] == body and starts == sorted(starts)
        assert all(data[s - 1:s] == b"\n" for s in starts) and all(r["exact_start"] for p in range(n) for r in plan.partition_ranges(p))
    for name in FIXTURES:                                              # describe(): the same rows as on the BAM
        sam = _render(tmp_path, name)
        assert bamscan.BamTableProvider(str(sam)).describe().equals(bamscan.BamTableProvider(str(GOLDEN / name), index_path="").describe()), name


def test_sam_inference_narrows_integers_by_value(tmp_path):
    import bamscan
    p = tmp_path / "t.sam"
    p.write_text("@SQ\tSN:c\tLN:10\nr\t0\tc\t1\t0\t*\t*\t0\t0\t*\t*\tXA:i:70000\tXB:i:-70000\tXC:i:65535\tXF:f:1e3\tXL:B:S,1\tXH:H:0A\tXQ:B:c,1,200\tXR:i:1\n")
    s = bamscan.BamTableProvider(str(p), tag_fields=["XA", "XB", "XC", "XF", "XL", "XH", "XQ", "XR"]).schema()
    types = {f.name: str(f.type) for f in s}
    assert types["XA"] == "uint32" and types["XB"] == "int32" and types["XC"] == "int32" and types["XF"] == "float"
    assert types["XL"] == "list<item: uint16>" and types["XH"] == "string"
    # a field the scan refuses (200 is outside B:c) infers nothing, and the walk stops there as the BAM walk does
    assert types["XQ"] == "string" and types["XR"] == "string"


def test_gzip_sam_refused_at_open(tmp_path):
    import gzip
    import bamscan
    p = tmp_path / "z.sam"
    p.write_bytes(gzip.compress(b"@SQ\tSN:c\tLN:10\n"))
    with pytest.raises(bamscan.BamScanError) as ei:
        bamscan.BamTableProvider(str(p))
    assert ei.value.code == -5


def test_sam_host_parsers_under_sanitizers(tmp_path):
    exe = tmp_path / "shd"
    cmd = ["g++", "-O1", "-g", "-std=c++17", "-fsanitize=address,undefined", "-fno-omit-frame-pointer", "-o", str(exe),
           str(ROOT / "tests" / "native" / "sam_host_driver.cpp")] + [str(CSRC / f) for f in ("host_file.cpp", "host_schema.cpp", "host_index.cpp", "host_plan.cpp")] + ["-lz"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0 and "sanitize" in r.stderr:
        pytest.skip("no sanitizer runtime for g++ here")
    assert r.returncode == 0, r.stderr[-2000:]

    def run(path):
        r = subprocess.run([str(exe), str(path)], capture_output=True, text=True)
        assert r.returncode == 0 and "Sanitizer" not in r.stderr and "runtime error" not in r.stderr, (r.stdout, r.stderr[:3000])
        return dict(kv.split("=") for kv in r.stdout.split(":", 1)[1].split())

    srcs = [sam_render.bam_to_sam((GOLDEN / n).read_bytes())[:200000] for n in FIXTURES]
    f = tmp_path / "f.sam"
    # the valid files reach every SAM parser: header + references, pseudo-blocks, tag inference, plans on line starts
    for n, src in zip(FIXTURES, srcs):
        f.write_bytes(src)
        got = run(f)
        assert got["format"] == "2" and got["rc"] == "0" and got["header_ok"] == "1" and int(got["n_ref"]) > 0, (n, got)
        assert int(got["blocks"]) > 0 and int(got["ranges"]) >= 6 and (int(got["tags"]) > 0 or n == "no_coor_only.bam"), (n, got)
    f.write_bytes(b"@SQ\tSN:c\tLN:" + b"9" * 40 + b"\nr\t0\tc\t1\t0\t*\t*\t0\t0\t*\t*\n")     # an LN of 40 digits: a header that does not parse
    assert run(f)["header_ok"] == "0"
    rng = random.Random(17)
    for it in range(80):
        b = bytearray(rng.choice(srcs))
        for _ in range(rng.randrange(1, 12)):
            k = rng.randrange(len(b))
            b[k] = rng.choice([9, 10, 13, 44, 58, 64, 0, rng.randrange(256)])
        if it % 4 == 0:
            b = b[:rng.randrange(1, len(b))]
        f.write_bytes(bytes(b))
        assert run(f)["format"] == "2"
