"""GPU: f32 text and f32 parsing on the device against exact references, through the public API only --
oracle/f32_exact.py::display for f32 -> text (csrc/f32_text.h), oracle/sam_oracle.py::f32_from_text for text -> f32
(csrc/f32_parse.h).  Bit set B is tests/test_f32_exact.py's (every power of two and its neighbours, every exponent's
corners, the subnormal corners, the pinned values, 200 k random words).
a. SAM writer: B, then 800 k more random words, each as a Float32 `f` tag and as `B:f` list elements (lists of 0, 1, 31, 32,
   33 and ~1000 elements, so element offsets cross group and warp edges); every value in the file equals display (numpy's
   Dragon4 for the 800 k extra words: test_f32_exact checks it against display); the whole file of B equals the Python
   oracle's text (its float text taken from display, which test_f32_exact shows equal to it on B).
b. BAM scan of float tags into Utf8 columns (unknown tags, inference off), one tag per record over B and three per record,
   under the default decode kernel and the warp decode kernel; both decode passes (length, bytes) run f32_to_text.
c. SAM scan: adversarial decimal strings as `f` tags and `B:f` elements, bit for bit (sign of -0 and NaN included).
d. The files of (a) read back by the SAM scan: every non-NaN pattern identical, every NaN a NaN."""
import random
from fractions import Fraction

import numpy as np
import pyarrow as pa
import pytest

from oracle import sam_write_oracle as SW
from test_f32_exact import PINS, bit_set_b, float_tag_bam, float_tag_texts, map_all
from test_sam_oracle import _exact_decimal, _value
from test_sam_write_oracle import rule_schema, tf

pytestmark = pytest.mark.gpu

LENGTHS = [0, 1, 31, 32, 33, 1000, 999, 1001]
OVERRIDES = {"bio.bam.sort_order": "unsorted"}
TAGS = ["Yf", "Yb"]


@pytest.fixture(scope="module")
def sets():
    """(B, display of B, 800 k extra random words not in B, numpy's text of them)."""
    from oracle.f32_exact import display
    b = bit_set_b()
    extra = np.setdiff1d(np.random.default_rng(31).integers(0, 2**32, 820_000, dtype=np.uint64).astype(np.uint32), b)[:800_000]
    extra = np.random.default_rng(32).permutation(extra)
    assert len(extra) == 800_000
    return b, map_all(display, b), extra, _numpy_texts(extra)


def _numpy_texts(bits):
    out = []
    for b, x in zip(bits, bits.view(np.float32)):
        mag = int(b) & 0x7FFFFFFF
        out.append("NaN" if mag > 0x7F800000 else ("-inf" if b >> 31 else "inf") if mag == 0x7F800000
                   else np.format_float_positional(x, unique=True, trim="-"))
    return out


def _schema():
    s = rule_schema()
    return pa.schema(list(s)[:12] + [tf("Yf", pa.float32(), "f"), tf("Yb", pa.list_(pa.float32()), "B:f")], metadata=s.metadata)


def _batch(scalars, elems):
    """One row per scalar (Yf); the first rows also carry Yb lists over `elems`, lengths cycling through LENGTHS."""
    n = len(scalars)
    offs, k = [0], 0
    while offs[-1] < len(elems):
        offs.append(min(offs[-1] + LENGTHS[k % len(LENGTHS)], len(elems)))
        k += 1
    assert k <= n
    offsets = pa.array(offs + [offs[-1]] * (n - k), pa.int32())
    lists = pa.ListArray.from_arrays(offsets, pa.array(elems.view(np.float32), pa.float32()),
                                     mask=pa.array(np.arange(n) >= k))
    core = dict(name=pa.array([f"r{i}" for i in range(n)]), chrom=pa.array(["chr1"] * n), start=pa.array(np.full(n, 99, np.uint32)),
                end=pa.nulls(n, pa.uint32()), flags=pa.array(np.zeros(n, np.uint32)), cigar=pa.array(["4M"] * n),
                mapping_quality=pa.array(np.full(n, 60, np.uint32)), mate_chrom=pa.nulls(n, pa.string()), mate_start=pa.nulls(n, pa.uint32()),
                sequence=pa.array(["ACGT"] * n), quality_scores=pa.array(["IIII"] * n), template_length=pa.array(np.zeros(n, np.int32)))
    s = _schema()
    cols = [core[f.name] for f in list(s)[:12]] + [pa.array(scalars.view(np.float32), pa.float32()), lists]
    return pa.RecordBatch.from_arrays(cols, schema=s), [offs[i + 1] - offs[i] for i in range(k)]


def _write(path, batch):
    import bamscan
    ex = bamscan.SamWriteExec(str(path), batch.schema, TAGS, True, OVERRIDES)
    assert ex.execute([batch.slice(0, batch.num_rows // 3), batch.slice(batch.num_rows // 3)]) == batch.num_rows


def _file_values(path):
    """(every Yf:f: value, every Yb:B:f element, the element count of every Yb field), in file order."""
    yf, yb, lens = [], [], []
    for line in path.read_bytes().decode().split("\n"):
        if not line or line[0] == "@":
            continue
        for f in line.split("\t")[11:]:
            if f.startswith("Yf:f:"):
                yf.append(f[5:])
            elif f.startswith("Yb:B:f"):
                e = f[7:].split(",") if len(f) > 6 else []
                yb += e
                lens.append(len(e))
    return yf, yb, lens


def _oracle_text(batch, texts):
    """SW.sam_text([batch], ...) with SW.f32_text answered from `texts` ({bits: display(bits)}): test_f32_exact shows the two
    equal on B, and the Python oracle's float text would take minutes here."""
    from oracle.f32_exact import display
    with pytest.MonkeyPatch.context() as mp:
        mp.setattr(SW, "f32_text", lambda b: texts.get(b) or display(b))
        return SW.sam_text([batch], batch.schema, TAGS, True, OVERRIDES)


def _mismatch(bits, got, want):
    bad = [(f"{int(b):08x}", g, w) for b, g, w in zip(bits, got, want) if g != w]
    return f"{len(bad)} differ: {bad[:10]}" if bad else ""


def _sam_scan(path, tags):
    import bamscan
    p = bamscan.BamTableProvider(str(path), None, True, tags)
    t = p.scan(None, [], None).collect()
    p.close()
    return t


def _bits_equal(got: np.ndarray, want: np.ndarray):
    """Float32 bits: identical, except that a NaN is any NaN."""
    nan_w = (want & 0x7FFFFFFF) > 0x7F800000
    nan_g = (got & 0x7FFFFFFF) > 0x7F800000
    bad = np.nonzero((got != want) & ~(nan_w & nan_g))[0]
    return [(f"{want[i]:08x}", f"{got[i]:08x}") for i in bad[:10]], len(bad)


@pytest.fixture(scope="module")
def written(sets, tmp_path_factory):
    """(a)'s two files: B as scalars and (reversed) as list elements; the extra words likewise."""
    b, _tb, extra, _te = sets
    d = tmp_path_factory.mktemp("f32w")
    out = {}
    for name, words in (("b", b), ("extra", extra)):
        batch, lens = _batch(words, words[::-1].copy())
        _write(d / f"{name}.sam", batch)
        out[name] = (d / f"{name}.sam", batch, lens)
    return out


def test_sam_writer_float_text(sets, written):
    b, tb, extra, te = sets
    for name, words, texts in (("b", b, tb), ("extra", extra, te)):
        path, _batch_, lens = written[name]
        yf, yb, got_lens = _file_values(path)
        assert got_lens == lens, name
        assert len(yf) == len(yb) == len(words), name
        assert not (m := _mismatch(words, yf, texts)), f"{name} f: {m}"
        assert not (m := _mismatch(words[::-1], yb, texts[::-1])), f"{name} B:f: {m}"
    for bits, text in PINS:
        i = int(np.searchsorted(b, bits))
        assert b[i] == bits and tb[i] == text


def test_sam_writer_file_equals_the_oracle(sets, written):
    path, batch, _lens = written["b"]
    want = _oracle_text(batch, dict(zip(sets[0].tolist(), sets[1])))
    got = path.read_bytes()
    if got != want:
        i = next((k for k in range(min(len(got), len(want))) if got[k] != want[k]), min(len(got), len(want)))
        raise AssertionError(f"{len(got)} bytes, oracle {len(want)}; first difference at {i}: {got[i:i + 60]!r} vs {want[i:i + 60]!r}")


@pytest.mark.parametrize("flags", [0, 2], ids=["default_decode", "warp_decode"])
def test_bam_scan_float_tags_into_utf8(sets, flags, tmp_path):
    import bamscan
    b, tb, _extra, _te = sets
    perm = np.random.default_rng(9).permutation(len(b))[:60_000]
    multi = b[perm]
    tags = float_tag_bam(tmp_path / "f.bam", b, multi)
    p = bamscan.BamTableProvider(str(tmp_path / "f.bam"), None, True, tags, False, False, 100, None, index_path="", debug_flags=flags)
    t = p.scan(None, [], None).collect()
    p.close()
    for tag in tags:
        assert t.schema.field(tag).type == pa.string()
    got = float_tag_texts({tag: t[tag].to_pylist() for tag in tags}, len(b))
    want = tb + [tb[i] for i in perm]
    assert not (m := _mismatch(np.concatenate([b, multi]), got, want)), m


def adversarial_strings():
    """Decimal strings where a parser goes wrong (see the module doc, c)."""
    rng = random.Random(2026)
    out = []
    def halfway(b):
        return (_value(b) + (_value(b + 1) if b + 1 < 0x7F800000 else Fraction(2) ** 128)) / 2
    words = [0, 1, 2, 0x7FFFFE, 0x7FFFFF, 0x800000, 0x3F7FFFFF, 0x3F800000, 0x4B7FFFFF, 0x7F7FFFFE, 0x7F7FFFFF]
    words += [rng.randrange(1, 0x7F7FFFFF) for _ in range(300)] + [rng.randrange(1, 0x800000) for _ in range(100)]
    for b in words:                                   # exact halfway points (ties to even) and +-1 in a far digit
        s = _exact_decimal(halfway(b))
        frac = s if "." in s else s + "."
        out += [s, "-" + s, frac + "0" * 40 + "1"]
        digits = s.replace(".", "").lstrip("0")
        if digits.endswith("5"):                      # the same number minus one unit 30 digits further down
            out.append(s[:-1] + "4" + "9" * 30)
    for _ in range(200):                              # 112..130 significant digits; a non-zero tail past the 120th
        b = rng.randrange(0x800000, 0x7F7FFFFF)
        s = _exact_decimal(halfway(b)).replace(".", "")
        d = s.lstrip("0")[:rng.randrange(112, 131)]
        d = d + "0" * (rng.randrange(112, 131) - len(d))
        tail = d[:120] + "".join(rng.choice("0000000001") for _ in range(len(d) - 120))
        e = rng.randrange(-60, 20)
        out += [f"{d[0]}.{d[1:]}e{e}", f"{tail[0]}.{tail[1:]}e{e}", f"{tail[:-1]}1e{e - len(tail)}"]
    out += ["0" * 300 + "1.5", "-" + "0" * 250 + "3.4028235e38", "0." + "0" * 300 + "1e301", "0." + "0" * 400 + "7e355",
            "0" * 500, "0." + "0" * 500, "-0." + "0" * 200 + "1e-10", "0" * 200 + "16777217", "0." + "0" * 40 + "1401298464324817e-5"]
    out += ["1e100000", "-1e100000", "1e-100000", "-1e-100000", "0e100000", "-0e-100000", "123456789e-100000", "0.000001e+100000",
            "1" + "0" * 100 + "e-100100", "1E+99999", "1e+0100000"]
    for nd in (7, 8):                                 # the fast path's edges
        for e in (-11, -10, 10, 11):
            for _ in range(25):
                m = str(rng.randrange(10 ** (nd - 1), 10 ** nd))
                out += [f"{m}e{e}", f"-{m}e{e}", f"{m[0]}.{m[1:]}e{e + nd - 1}"]
            out += [f"{'9' * nd}e{e}", f"1{'0' * (nd - 1)}e{e}"]
    for w in ("inf", "infinity", "nan"):
        for v in (w, w.upper(), w.capitalize(), "iNf" if w == "inf" else w.title().swapcase()):
            out += [v, "+" + v, "-" + v]
    return out


def test_sam_scan_parses_floats_exactly(tmp_path):
    from oracle.sam_oracle import f32_from_text
    strings = adversarial_strings()
    want = np.array([f32_from_text(s) for s in strings], np.uint32)
    n, k = len(strings), 3
    lines = [f"s{i}\t4\t*\t0\t0\t*\t*\t0\t0\t*\t*\tYx:f:{s}\tYl:B:f," + ",".join(strings[(k * i + j) % n] for j in range(k))
             for i, s in enumerate(strings)]
    path = tmp_path / "f.sam"
    path.write_text("@HD\tVN:1.6\n" + "\n".join(lines) + "\n")
    t = _sam_scan(path, ["Yx", "Yl"])
    assert t.num_rows == n and t.schema.field("Yx").type == pa.float32()
    got = t["Yx"].combine_chunks().to_numpy().view(np.uint32)
    bad = [(strings[i][:80], f"{got[i]:08x}", f"{want[i]:08x}") for i in np.nonzero(got != want)[0][:10]]
    assert not bad, bad
    got = t["Yl"].combine_chunks().flatten().to_numpy().view(np.uint32)
    idx = [(k * i + j) % n for i in range(n) for j in range(k)]
    bad = [(strings[i][:80], f"{g:08x}", f"{want[i]:08x}") for i, g in zip(idx, got) if g != want[i]][:10]
    assert len(got) == len(idx) and not bad, bad


def test_written_floats_read_back(written):
    for name in ("b", "extra"):
        path, batch, _lens = written[name]
        t = _sam_scan(path, TAGS)
        assert t.num_rows == batch.num_rows
        assert t.schema.field("Yf").type == pa.float32() and t.schema.field("Yb").type == pa.list_(pa.float32())
        for col in TAGS:
            w = batch.column(batch.schema.get_field_index(col))
            g = t[col].combine_chunks()
            if col == "Yb":
                assert g.null_count == w.null_count and g.value_lengths().equals(w.value_lengths())
                w, g = w.flatten(), g.flatten()
            bad, nbad = _bits_equal(g.to_numpy().view(np.uint32), w.to_numpy().view(np.uint32))
            assert not nbad, f"{name} {col}: {nbad} differ (want, got): {bad}"
