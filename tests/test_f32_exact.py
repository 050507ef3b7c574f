"""CPU: the text of an f32 (Rust's `f32` Display) against an exact reference.

oracle/f32_exact.py::display states the definition with fractions.Fraction -- the fewest significant digits of any
decimal inside the float's rounding interval, the closer of two, the even last digit on a tie -- and is itself checked
against numpy's Dragon4, an independent implementation of the same definition.  Then each of the three implementations
of the rule is checked against display on bit set B:
- csrc/f32_text.h compiled for the host (what the BAM scan and the SAM writer run on the device);
- the C oracle's rule (oracle/bam_oracle.c::rust_f32_to_string), through an OracleBam scan of float tags into Utf8 columns;
- the Python oracle (oracle/sam_write_oracle.py::f32_text).
Bit set B: every power of two and its two neighbours, every exponent with mantissas 0, 1, 0x400000 and 0x7fffff, the
subnormal corners, the pinned values, and 200 k seeded random words; each with both signs where the sign is free.

The values a rule "correctly round to N digits, take it when it reads back" gets wrong are powers of two, where the
interval below is half as wide as the one above: the rounded N-digit value can miss the narrow lower half while the one
above is inside the upper half (PINS)."""
import subprocess
from pathlib import Path

import numpy as np
import pytest

from conftest import _bgzf, _rec

ROOT = Path(__file__).resolve().parent.parent

# (bits, text): the powers of two whose shortest text is one digit shorter than the correctly rounded rule finds, and ties
PINS = [
    (0x0F800000, "0.000000000000000000000000000012621775"),      # 2^-96
    (0x8F800000, "-0.000000000000000000000000000012621775"),
    (0x6B000000, "154742510000000000000000000"),                  # 2^87
    (0xEB000000, "-154742510000000000000000000"),
    (0x6C800000, "1237940100000000000000000000"),                 # 2^90
    (0xEC800000, "-1237940100000000000000000000"),
    (0x4986F3A6, "1105524.8"),                                    # 1105524.75: halfway, the even digit is above
    (0x4986F3A2, "1105524.2"),                                    # 1105524.25: halfway, the even digit is below
]


def bit_set_b(n_random=200_000, seed=20261021):
    """Bit set B (module doc) as a sorted uint32 array without duplicates."""
    pow2 = [e << 23 for e in range(1, 255)]
    words = pow2 + [b - 1 for b in pow2] + [b + 1 for b in pow2]
    words += [(e << 23) | m for e in range(256) for m in (0, 1, 0x400000, 0x7FFFFF)]
    sub = [1 << k for k in range(23)]
    words += sub + [b + 1 for b in sub] + [b - 1 for b in sub] + [0x7FFFFE, 0x400001, 0x3FFFFF, 0x800001]
    words += [b for b, _t in PINS]
    words += [b | 0x80000000 for b in words]
    rnd = np.random.default_rng(seed).integers(0, 2**32, n_random, dtype=np.uint64).astype(np.uint32)
    return np.unique(np.concatenate([np.array(words, np.uint32), rnd]))


def map_all(fn, bits):
    """[fn(b) for b in bits] on all cores (fn: a module-level function of an int)."""
    import multiprocessing
    from concurrent.futures import ProcessPoolExecutor
    with ProcessPoolExecutor(mp_context=multiprocessing.get_context("spawn")) as ex:
        return list(ex.map(fn, (int(b) for b in bits), chunksize=2048))


def float_tag_bam(path, values, multi):
    """A BAM of unmapped records: record i carries values[i] as the float tag Yf; then records with the float tags Yg, Yh and
    Yi together, carrying multi[3 j], multi[3 j + 1], multi[3 j + 2].  -> the tag names (unknown to the tag registry)."""
    text = "@HD\tVN:1.6\tSO:unsorted\n@SQ\tSN:chrA\tLN:1000\n"
    hdr = b"BAM\1" + np.int32(len(text)).tobytes() + text.encode() + np.int32(1).tobytes() + np.int32(5).tobytes() + b"chrA\0" + np.int32(1000).tobytes()
    recs = [_rec(-1, -1, f"f{i}", 0, 4, [], "", [], -1, -1, 0, b"Yff" + int(b).to_bytes(4, "little")) for i, b in enumerate(values)]
    multi = np.asarray(multi, np.uint32).reshape(-1, 3)
    recs += [_rec(-1, -1, f"m{j}", 0, 4, [], "", [], -1, -1, 0, b"".join(t + b"f" + int(b).to_bytes(4, "little") for t, b in zip((b"Yg", b"Yh", b"Yi"), w)))
             for j, w in enumerate(multi)]
    Path(path).write_bytes(_bgzf(hdr + b"".join(recs)))
    return ["Yf", "Yg", "Yh", "Yi"]


def float_tag_texts(columns, n_single):
    """The texts a scan of float_tag_bam must give, in its records' order: Yf for the first n_single rows, Yg / Yh / Yi after."""
    yf = columns["Yf"][:n_single]
    rest = [t for row in zip(columns["Yg"][n_single:], columns["Yh"][n_single:], columns["Yi"][n_single:]) for t in row]
    return yf + rest


@pytest.fixture(scope="module")
def bits_b():
    from oracle.f32_exact import display
    b = bit_set_b()
    return b, map_all(display, b)


def _host_f32_text(tmp_path, bits):
    exe = tmp_path / "f32_text_driver"
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-o", str(exe), str(ROOT / "tests" / "native" / "f32_text_driver.cpp")])
    out = subprocess.run([str(exe)], input="\n".join("%x" % b for b in bits) + "\n", capture_output=True, text=True, check=True).stdout.split("\n")
    assert len(out) == len(bits) + 1 and out[-1] == ""
    return out[:-1]


def _mismatches(bits, got, want):
    return [(f"{b:08x}", g, w) for b, g, w in zip(bits, got, want) if g != w]


def test_reference_equals_numpy_dragon4(bits_b):
    bits, want = bits_b
    assert len(bits) > 200_000
    f = bits.view(np.float32)
    bad = []
    for b, x, w in zip(bits, f, want):
        mag = int(b) & 0x7FFFFFFF
        if mag > 0x7F800000:
            ok = w == "NaN"
        elif mag == 0x7F800000:
            ok = w == ("-inf" if b >> 31 else "inf")
        else:
            ok = w == np.format_float_positional(x, unique=True, trim="-")
        if not ok:
            bad.append((f"{b:08x}", w))
    assert not bad, bad[:10]


@pytest.mark.parametrize("bits,text", PINS, ids=[f"{b:08x}" for b, _t in PINS])
def test_pinned_texts(bits, text, tmp_path):
    from oracle.f32_exact import display
    from oracle import sam_write_oracle as SW
    assert display(bits) == text
    assert SW.f32_text(bits) == text
    assert _host_f32_text(tmp_path, [bits]) == [text]


def test_device_routine_equals_reference(bits_b, tmp_path):
    """csrc/f32_text.h, host build; the length-only call (the size passes) is checked by the driver too."""
    bits, want = bits_b
    bad = _mismatches(bits, _host_f32_text(tmp_path, bits), want)
    assert not bad, f"{len(bad)} differ: {bad[:10]}"


def test_c_oracle_rule_equals_reference(bits_b, tmp_path):
    """oracle/bam_oracle.c::rust_f32_to_string: float tags read into Utf8 columns (unknown tags, inference off), one tag per
    record over all of B and three tags per record over the first 30 k words in reverse."""
    from oracle.bam_oracle import OracleBam
    bits, want = bits_b
    multi = bits[:30_000][::-1]
    tags = float_tag_bam(tmp_path / "f.bam", bits, multi)
    cols = OracleBam(str(tmp_path / "f.bam"), tag_fields=tags, infer_tag_types=False).scan().to_pydict()
    got = float_tag_texts(cols, len(bits))
    bad = _mismatches(np.concatenate([bits, multi]), got, want + want[:30_000][::-1])
    assert not bad, f"{len(bad)} differ: {bad[:10]}"


def test_c_oracle_rule_copy_equals_reference(bits_b, tmp_path):
    """The restatement of the C rule in tests/native/f32_text_check.cpp (which checks f32_text.h on its own patterns)."""
    bits, want = bits_b
    src = (ROOT / "tests" / "native" / "f32_text_check.cpp").read_text().split("int main")[0]
    src = src.replace("../../datafusion-bio-formats_b200", str(ROOT / "datafusion-bio-formats_b200"))
    src += ('int main() { unsigned b; char out[128]; while (scanf("%x", &b) == 1) { float v; memcpy(&v, &b, 4); '
            'oracle_rule(v, out); printf("%s\\n", out); } return 0; }\n')
    (tmp_path / "rule.cpp").write_text(src)
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-o", str(tmp_path / "rule"), str(tmp_path / "rule.cpp")])
    out = subprocess.run([str(tmp_path / "rule")], input="\n".join("%x" % b for b in bits), capture_output=True, text=True, check=True).stdout.split("\n")
    bad = _mismatches(bits, out, want)
    assert not bad, f"{len(bad)} differ: {bad[:10]}"


def test_python_oracle_equals_reference(bits_b):
    from oracle import sam_write_oracle as SW
    bits, want = bits_b
    bad = _mismatches(bits, map_all(SW.f32_text, bits), want)
    assert not bad, f"{len(bad)} differ: {bad[:10]}"
