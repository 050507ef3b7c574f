"""GPU: the SAM write path (bamscan_sam_writer_open + bamscan_writer_*) against oracle/sam_write_oracle.py.  The written file
equals the oracle's text byte for byte, and the GPU SAM scan reads it back to what the GPU BAM scan reads from the BAM writer's
file of the same batches (up to the differences DESIGN 3.9 lists)."""
import random

import numpy as np
import pyarrow as pa
import pytest

from conftest import GOLDEN, gen_bam, make_edge_bam
from oracle import bam_write_oracle as W
from oracle import sam_write_oracle as SW
from oracle.bam_oracle import OracleBam
from test_gpu_write import FIXTURE_TAGS
from test_sam_write_oracle import (REFUSAL_IDS, REFUSALS, RULE_TAG_NAMES, _no_qual_rows, assert_round_trip, fixture_batch, refusal_batch,
                                   row, rule_schema, tf)

pytestmark = pytest.mark.gpu


def gpu_write(path, batches, schema, tags, zero_based=True, overrides=None):
    import bamscan
    ex = bamscan.SamWriteExec(str(path), schema, tags, zero_based, overrides)
    n = ex.execute(batches)
    return n, ex.stats


def check_text(path, want: bytes):
    got = open(path, "rb").read()
    if got != want:
        i = next((k for k in range(min(len(got), len(want))) if got[k] != want[k]), min(len(got), len(want)))
        raise AssertionError(f"{path}: {len(got)} bytes, oracle {len(want)}; first difference at {i}: {got[i:i + 40]!r} vs {want[i:i + 40]!r}")


def one_batch(table: pa.Table, schema):
    t = table.combine_chunks()
    return t.to_batches()[0] if t.num_rows else pa.RecordBatch.from_pylist([], schema=schema)


def gpu_scan(path, zero_based, tags, **kw):
    import bamscan
    p = bamscan.BamTableProvider(str(path), None, zero_based, tags, index_path="", **kw) if str(path).endswith(".bam") else \
        bamscan.BamTableProvider(str(path), None, zero_based, tags, **kw)
    t = pa.Table.from_batches(list(p.scan(None, [], None).execute(0)), schema=p.schema())
    p.close()
    return one_batch(t, t.schema)


def write_and_compare(tmp_path, batches, schema, tags, zero_based=True, what=""):
    """GPU SAM file == oracle text; GPU SAM scan of it == GPU BAM scan of the BAM writer's file of the same batches."""
    import bamscan
    sam, bam = tmp_path / "o.sam", tmp_path / "o.bam"
    n, st = gpu_write(sam, batches, schema, tags, zero_based, {"bio.bam.sort_order": "unsorted"})
    want = SW.sam_text(batches, schema, tags, zero_based, {"bio.bam.sort_order": "unsorted"})
    check_text(sam, want)
    assert n == sum(b.num_rows for b in batches) == st["rows"] and st["bam_bytes"] == st["compressed_bytes"] == len(want)
    assert st["members"] == 0 and st["ms_deflate"] == 0
    bamscan.BamWriteExec(str(bam), schema, tags, zero_based, {"bio.bam.sort_order": "unsorted"}).execute(batches)
    if n:
        whole = one_batch(pa.Table.from_batches(batches, schema=schema), schema)
        assert_round_trip(gpu_scan(sam, zero_based, tags), gpu_scan(bam, zero_based, tags), _no_qual_rows(whole), what)
    return want


@pytest.mark.parametrize("name", sorted(FIXTURE_TAGS))
@pytest.mark.parametrize("zero_based", [True, False])
@pytest.mark.parametrize("tagset", ["listed", "all"])
def test_fixtures_are_byte_exact_and_read_back(name, zero_based, tagset, tmp_path):
    if tagset == "all":
        b, schema, tags, _recs = fixture_batch(name, zero_based)
    else:
        tags = FIXTURE_TAGS[name]
        o = OracleBam(str(GOLDEN / name), zero_based=zero_based, tag_fields=tags)
        b, schema = o.scan(None), o.schema
    write_and_compare(tmp_path, [b], schema, tags, zero_based, f"{name} {tagset}")


def test_edge_bam(tmp_path):
    src = tmp_path / "edge.bam"
    make_edge_bam(src, missing_qual=True)
    tags = ["NM", "MD", "XS", "XF", "XB", "XA", "XI", "XU"]
    o = OracleBam(str(src), tag_fields=tags)
    write_and_compare(tmp_path, [o.scan(None)], o.schema, tags, True, "edge")


@pytest.mark.parametrize("mode,reads", [("short", 60000), ("long", 400)])
def test_synthetic_sliced_batches_and_partitions(mode, reads, syn_dir, tmp_path):
    """60 k short reads (group of 8 lanes per row) and 400 long reads with MM / ML (a warp per row), in empty and sliced batches;
    read back over 1 / 2 / 4 / 8 block-range partitions with the seam check."""
    import bamscan
    path = gen_bam(syn_dir, mode, reads, seed=7)
    tags = ["NM", "MD", "AS", "RG"] if mode == "short" else ["NM", "MD", "MM", "ML"]
    o = OracleBam(str(path), tag_fields=tags)
    b = o.scan(None)
    n = b.num_rows
    cuts = [0, 1, 17, n // 3, n // 3, (2 * n) // 3 + 5, n]
    if mode == "short":
        cuts = [0, 1, 17, 17 + 8192, n // 3, n // 3, (2 * n) // 3 + 5, n]
    parts = [b.slice(x, y - x) for x, y in zip(cuts, cuts[1:])]
    write_and_compare(tmp_path, parts, o.schema, tags, True, mode)
    want = gpu_scan(tmp_path / "o.sam", True, tags)
    p = bamscan.BamTableProvider(str(tmp_path / "o.sam"), None, True, tags, chunk_inflated_bytes=4 << 20)
    for tp in (1, 2, 4, 8):
        plan = p.scan(None, [], None, target_partitions=tp, partition_mode="block_range")
        got, stats = [], []
        for i in range(plan.output_partition_count()):
            got += list(plan.execute(i))
            stats.append(plan.last_stats)
        assert pa.Table.from_batches(got, schema=plan.schema()).equals(pa.Table.from_batches([want])), f"{tp} partitions"
        if len(stats) > 1:
            bamscan.check_partition_seams(stats)
    p.close()


def test_binary_cigar_column(syn_dir, tmp_path):
    path = gen_bam(syn_dir, "short", 5000, seed=3)
    o = OracleBam(str(path), tag_fields=["NM"], binary_cigar=True)
    b = o.scan(None)
    assert b.schema.field("cigar").type == pa.binary()
    _n, _st = gpu_write(tmp_path / "b.sam", [b], o.schema, ["NM"])
    text = SW.sam_text([b], o.schema, ["NM"])
    check_text(tmp_path / "b.sam", text)
    o2 = OracleBam(str(path), tag_fields=["NM"])
    assert text == SW.sam_text([o2.scan(None)], o2.schema, ["NM"])       # the same lines as from the text CIGAR column


def random_rows(rng, n, refs):
    """Seeded rows over every accepted corner of the rules (the refused ones are test_each_refusal_rule's)."""
    def maybe(p, v):
        return None if rng.random() < p else v
    rows = []
    for i in range(n):
        r = rng.random()
        if r < 0.1:
            cig, L = rng.choice(["*", ""]), rng.randint(0, 40)
        else:
            cig = "".join(f"{rng.choice([0, 1, 2, 9, 10, 99, 100, 12345, 268435455])}{rng.choice('MIDNSHP=X')}" for _ in range(rng.randint(1, 12)))
            if rng.random() < 0.1:
                cig = "0" + cig
            L = rng.randint(0, 60)
        seq = rng.choice(["*", "", None]) if rng.random() < 0.08 else "".join(rng.choice("ACGTNacgtn=.MRSVWYHKDBxz") for _ in range(L))
        has_seq = seq not in ("*", "", None)
        qual = rng.choice(["*", "", None]) if (not has_seq or rng.random() < 0.15) else "".join(chr(rng.choice([9, 32, 33, 34, 73, 126])) for _ in range(len(seq)))
        rows.append(dict(
            name=rng.choice([None, "*", "r" * rng.randint(1, 254), f"read{i}", "a/1?~!"]), chrom=maybe(0.15, rng.choice(refs + ["chrNope"])),
            start=maybe(0.15, rng.choice([0, 1, 16383, 5_000_000, 2**29])), end=None, flags=rng.choice([0, 4, 99, 65535]), cigar=cig,
            mapping_quality=rng.choice([0, 60, 255, 256, 300]), mate_chrom=maybe(0.3, rng.choice(refs + ["=", "chrNope"])),
            mate_start=maybe(0.3, rng.choice([0, 7, 2**31 - 2])), sequence=seq, quality_scores=qual, template_length=rng.choice([0, -1, 2**31 - 1, -2**31]),
            Xi=maybe(0.3, rng.choice([0, -2**31, 2**31 - 1])), Xf=maybe(0.3, rng.choice([0.0, -0.0, -1.5, 3.4028234663852886e38, 1e-45, float("inf"), float("-inf"), float("nan")])),
            Xd=maybe(0.3, rng.choice([0.1, -2.5e-40, 1e30])), XZ=maybe(0.3, rng.choice(["", "10A5", "x y" * 100, "~!"])),
            XH=maybe(0.3, rng.choice(["", "1a2B", "ff" * 40])), XA=maybe(0.3, rng.choice("AZ~!")), Xa=maybe(0.3, rng.randint(33, 126)),
            XB=maybe(0.3, [rng.randint(0, 255) for _ in range(rng.randint(0, 70))]), XF=maybe(0.3, [rng.choice([0.5, -2.0, 1e-7, float("nan")]) for _ in range(rng.randint(0, 5))]),
            Xs=maybe(0.3, [rng.randint(-32768, 32767) for _ in range(rng.randint(0, 33))]), Xq=maybe(0.3, rng.choice(["", "q q"]))))
    return rows


def test_seeded_random_rows_against_the_oracle(tmp_path):
    s = rule_schema()
    rows = random_rows(random.Random(20261020), 4000, ["chr1", "chr2"])
    b = pa.RecordBatch.from_pylist(rows, schema=s)
    for zb in (True, False):
        n, _st = gpu_write(tmp_path / f"r{int(zb)}.sam", [b.slice(0, 1111), b.slice(1111)], s, RULE_TAG_NAMES, zb)
        assert n == 4000
        check_text(tmp_path / f"r{int(zb)}.sam", SW.sam_text([b], s, RULE_TAG_NAMES, zb))


@pytest.mark.parametrize("change,code,msg,shared", REFUSALS, ids=REFUSAL_IDS)
def test_each_refusal_rule(change, code, msg, shared, tmp_path):
    import bamscan
    b = refusal_batch(change, bad_row=37, n=100)
    with pytest.raises(SW.WriteError, match=f"row 37: .*({msg})"):
        SW.render_batch(b, ["chr1", "chr2"], RULE_TAG_NAMES)
    with pytest.raises(bamscan.BamScanError, match=f"row 37: .*({msg})") as e:
        gpu_write(tmp_path / "bad.sam", [b], rule_schema(), RULE_TAG_NAMES)
    assert e.value.code == code
    with pytest.raises(bamscan.BamScanError, match=f"row 30: .*({msg})"):
        gpu_write(tmp_path / "bad2.sam", [b.slice(7)], rule_schema(), RULE_TAG_NAMES)
    if shared:                                                   # the BAM writer refuses it with the same class
        with pytest.raises(bamscan.BamScanError, match="row 37") as e2:
            bamscan.BamWriteExec(str(tmp_path / "bad.bam"), rule_schema(), RULE_TAG_NAMES).execute([b])
        assert e2.value.code == code


def test_device_batches_are_written_in_place(syn_dir, tmp_path):
    import bamscan
    tags = ["NM", "MD", "AS", "RG"]
    path = gen_bam(syn_dir, "short", 30000, seed=11)
    p = bamscan.BamTableProvider(str(path), None, True, tags, index_path="", chunk_inflated_bytes=4 << 20)    # several device batches
    host = list(p.scan(None, [], None).execute(0))
    gpu_write(tmp_path / "h.sam", host, p.schema(), tags)
    ex = bamscan.SamWriteExec(str(tmp_path / "d.sam"), p.schema(), tags)
    assert ex.execute(p.scan(None, [], None).execute_device(0)) == 30000 and ex.stats["arrow_bytes"] == 0 and ex.stats["batches"] > 1
    p.close()
    assert (tmp_path / "d.sam").read_bytes() == (tmp_path / "h.sam").read_bytes() == SW.sam_text(host, host[0].schema, tags)


def test_insert_into_sam_targets(tmp_path):
    """`INSERT OVERWRITE` into a provider made for a .sam file, and into a provider opened on a .sam file (its own file)."""
    import bamscan
    o = OracleBam(str(GOLDEN / "multi_chrom.bam"), tag_fields=["NM", "MD"])
    b = o.scan(None)
    pw = bamscan.BamTableProvider.new_for_write(str(tmp_path / "x.SAM"), o.schema, ["NM", "MD"], True, sort_on_write=True)
    assert pw.insert_into([b]) == b.num_rows
    check_text(tmp_path / "x.SAM", SW.sam_text([b], o.schema, ["NM", "MD"], True, {"bio.bam.sort_order": "coordinate"}))
    with pytest.raises(NotImplementedError):
        pw.insert_into([b], "append")
    own = tmp_path / "own.sam"
    own.write_bytes((tmp_path / "x.SAM").read_bytes())
    po = bamscan.BamTableProvider(str(own), None, True, ["NM", "MD"])
    keep = [x.slice(0, x.num_rows // 2) for x in po.scan(None, [], None).execute(0)]
    schema = po.schema()
    assert po.insert_into(keep) == sum(x.num_rows for x in keep)
    po.close()
    check_text(own, SW.sam_text(keep, schema, ["NM", "MD"], True, {"bio.bam.sort_order": "unsorted"}))
    back = gpu_scan(own, True, ["NM", "MD"])
    assert back.num_rows == sum(x.num_rows for x in keep)


def test_small_files(tmp_path):
    s = rule_schema()
    header = W.build_bam_header(s)[0].encode()
    n, st = gpu_write(tmp_path / "none.sam", [], s, RULE_TAG_NAMES)
    assert n == 0 and (tmp_path / "none.sam").read_bytes() == header and st["bam_bytes"] == len(header)
    gpu_write(tmp_path / "empty.sam", [pa.RecordBatch.from_pylist([], schema=s)], s, RULE_TAG_NAMES)
    assert (tmp_path / "empty.sam").read_bytes() == header
    one = pa.RecordBatch.from_pylist([row(Xi=-5, XZ="z", XB=[1, 2])], schema=s)
    gpu_write(tmp_path / "one.sam", [one], s, RULE_TAG_NAMES)
    assert (tmp_path / "one.sam").read_bytes() == header + b"r\t0\tchr1\t100\t60\t4M\t*\t0\t0\tACGT\tIIII\tXi:i:-5\tXZ:Z:z\tXB:B:C,1,2\n"


def test_random_float_bit_patterns(tmp_path):
    """>= 100 k random f32 bit patterns (NaN payloads, infinities, subnormals included) as a Float32 tag and as B:f elements."""
    rng = np.random.default_rng(77)
    bits = rng.integers(0, 2**32, size=100_000, dtype=np.uint64).astype(np.uint32)
    bits[:8] = [0, 0x80000000, 1, 0x7f7fffff, 0x7f800000, 0xff800000, 0x7fc00001, 0x00800000]
    vals = bits.view(np.float32)
    n = len(vals)
    s = rule_schema()
    cols = []
    for f in s:
        if f.name == "Xf":
            cols.append(pa.array(vals, pa.float32()))
        elif f.name == "XF":                                     # one element per row, in the other order
            cols.append(pa.ListArray.from_arrays(pa.array(np.arange(n + 1, dtype=np.int32)), pa.array(vals[::-1].copy(), pa.float32())))
        else:
            cols.append(pa.array([row(name=f"r{i}")[f.name] if f.name in row() else None for i in range(n)], f.type))
    b = pa.RecordBatch.from_arrays(cols, schema=s)
    b, b2 = b.slice(0, n // 2), b.slice(n // 2)
    gpu_write(tmp_path / "f.sam", [b, b2], s, RULE_TAG_NAMES)
    check_text(tmp_path / "f.sam", SW.sam_text([b, b2], s, RULE_TAG_NAMES))
