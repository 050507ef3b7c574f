"""Members with more LZ77 matches than the CTA inflate kernel's match list holds: the resolver takes them in output-ordered
batches.  CPU: the host model (tools/inflate_sim.cpp --list-cap) with a small cap equals zlib.  GPU: such files, scanned with the
CTA-per-member kernel forced (debug_flags bit 4), equal the oracle."""
import random
import re
import subprocess
from pathlib import Path

import pyarrow as pa
import pytest

from conftest import gen_bam, write_bgzf

ROOT = Path(__file__).resolve().parent.parent


def _word_fastq(path: Path, reads=20000, seed=7) -> Path:
    """FASTQ whose sequence and quality lines are random strings of a few short words, deflated at level 1: ~10 000 short
    matches per 64 KB member."""
    rng = random.Random(seed)
    words, qwords = ["ACGT", "TTGA", "CAGG", "GATC"], ["II?", "+@5", "FFF:", "#,"]
    text = "".join(f"@r{i}\n" + "".join(rng.choice(words) for _ in range(25))[:100] + "\n+\n"
                   + "".join(rng.choice(qwords) for _ in range(40))[:100] + "\n" for i in range(reads))
    write_bgzf(path, text.encode(), level=1)
    return path


@pytest.fixture(scope="module")
def files(tmp_path_factory):
    d = tmp_path_factory.mktemp("batched")
    return {"bam": gen_bam(d, "short", 30000, seed=3, level=1), "fastq": _word_fastq(d / "words.fastq.bgz")}


@pytest.fixture(scope="module")
def inflate_sim(tmp_path_factory):
    exe = tmp_path_factory.mktemp("isim") / "inflate_sim"
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-o", str(exe), str(ROOT / "tools" / "inflate_sim.cpp"), "-lz"])
    return exe


@pytest.mark.parametrize("kind", ["bam", "fastq"])
@pytest.mark.parametrize("cap", [256, 4096])
def test_host_model_batched_resolve_equals_zlib(inflate_sim, files, kind, cap):
    r = subprocess.run([str(inflate_sim), str(files[kind]), "--resolve", "6", "--list-cap", str(cap), "--max-members", "40"],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    m = re.search(r"members=(\d+) bad=(\d+) .* matches/member\(max\)=(\d+) list-batches=(\d+)", r.stdout)
    assert m, r.stdout
    members, bad, most, batches = (int(x) for x in m.groups())
    assert members == 40 and bad == 0
    assert most > 8192 and batches > members        # members of more than one batch (the kernel's list holds 3136)


@pytest.mark.gpu
def test_gpu_batched_resolve_bam(files):
    import bamscan
    from oracle.bam_oracle import OracleBam
    tags = ["NM", "MD", "AS", "RG"]
    want = pa.Table.from_batches([OracleBam(str(files["bam"]), tag_fields=tags).scan()])
    p = bamscan.BamTableProvider(str(files["bam"]), None, True, tags, False, True, 100, None, index_path="", debug_flags=16)
    got = p.scan(None, [], None).collect()
    assert got.num_rows == want.num_rows
    for name in want.schema.names:
        assert got[name].combine_chunks().equals(want[name].combine_chunks()), name
    p.close()


@pytest.mark.gpu
def test_gpu_batched_resolve_fastq(files):
    import bamscan
    from oracle.fastq_oracle import OracleFastq
    want = pa.Table.from_batches([OracleFastq(files["fastq"]).scan()])
    p = bamscan.FastqTableProvider(str(files["fastq"]), debug_flags=16)
    got = p.scan().collect()
    assert got.num_rows == want.num_rows == 20000
    for name in want.schema.names:
        assert got[name].combine_chunks().equals(want[name].combine_chunks()), name
    p.close()
