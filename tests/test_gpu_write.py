"""GPU: the write path (SURVEY 8 f4) through the C ABI (bamscan_writer_*), checked against oracle/bam_write_oracle.py:
the INFLATED BAM stream of the written file is bit-exact (header + every record byte), every BGZF member is well formed
(BSIZE chain, CRC-32, ISIZE, 0xff00-byte members, EOF marker), and reading the file back gives the batches that went in."""
import struct
import zlib

import pyarrow as pa
import pytest

from conftest import GOLDEN, gen_bam, make_edge_bam
from oracle import bam_write_oracle as W
from oracle.bam_oracle import OracleBam

pytestmark = pytest.mark.gpu

FIXTURE_TAGS = {"multi_chrom.bam": ["NM", "MD"], "bam_with_tags.bam": ["NM", "MD", "AS", "XS"], "10x_pbmc_tags.bam": ["CB", "UB", "NH", "xf"],
                "nanopore_custom_tags.bam": ["pt", "NM", "de", "MM", "ML"], "multi_chrom_large.bam": ["NM", "MD", "RG"], "no_coor_only.bam": []}


def gpu_write(path, batches, schema, tags, zero_based=True, overrides=None, compression=0):
    import bamscan
    ex = bamscan.BamWriteExec(str(path), schema, tags, zero_based, overrides, compression=compression)
    n = ex.execute(batches)
    return n, ex.stats


def check_file(path, batches, schema, tags, zero_based=True, overrides=None):
    data = open(path, "rb").read()
    stream, sizes = W.inflate_bgzf(data)                       # strict: member headers, BSIZE chain, CRC-32, ISIZE
    assert data.endswith(W.BGZF_EOF) and sizes[-1] == 0
    assert all(s == W.BGZF_BLOCK for s in sizes[:-2]) and 0 < sizes[-2] <= W.BGZF_BLOCK
    want = W.bam_stream(batches, schema, tags, zero_based, overrides)
    assert len(stream) == len(want)
    if stream != want:
        i = next(k for k in range(len(want)) if stream[k] != want[k])
        raise AssertionError(f"inflated stream differs from the oracle at byte {i}: {stream[i:i+16].hex()} vs {want[i:i+16].hex()}")
    return len(data)


@pytest.mark.parametrize("name", sorted(FIXTURE_TAGS))
@pytest.mark.parametrize("zero_based", [True, False])
def test_fixture_write_is_bit_exact_and_reads_back(name, zero_based, tmp_path):
    import bamscan
    tags = FIXTURE_TAGS[name]
    o = OracleBam(str(GOLDEN / name), zero_based=zero_based, tag_fields=tags)
    batch = o.scan(None)
    out = tmp_path / "out.bam"
    n, st = gpu_write(out, [batch], o.schema, tags, zero_based, {"bio.bam.sort_order": "unsorted"})
    assert n == batch.num_rows == st["rows"]
    check_file(out, [batch], o.schema, tags, zero_based, {"bio.bam.sort_order": "unsorted"})
    # read -> write -> read (write_test.rs::test_read_add_write_read_round_trip), the reading done by the GPU scan
    p = bamscan.BamTableProvider(str(out), None, zero_based, tags, index_path="")
    back = pa.Table.from_batches(list(p.scan(None, [], None).execute(0)), schema=p.schema()) if batch.num_rows else None
    if back is not None:
        for i, f in enumerate(batch.schema):
            assert back.column(i).combine_chunks().equals(batch.column(i)), f.name
        assert p.schema().metadata[b"bio.bam.sort_order"] == b"unsorted"


def test_edge_bam_and_every_tag_type(tmp_path):
    src = tmp_path / "edge.bam"
    make_edge_bam(src, missing_qual=False)
    tags = ["NM", "MD", "XS", "XF", "XB", "XA", "XI", "XU"]
    o = OracleBam(str(src), tag_fields=tags)
    batch = o.scan(None)
    out = tmp_path / "o.bam"
    gpu_write(out, [batch], o.schema, tags)
    check_file(out, [batch], o.schema, tags)

    def tf(name, typ, spec):
        return pa.field(name, typ, True, {"bio.bam.tag.tag": name, "bio.bam.tag.type": spec})
    fields = [tf("Xc", pa.int32(), "c"), tf("XC", pa.int32(), "C"), tf("Xs", pa.int32(), "s"), tf("XS", pa.int32(), "S"), tf("Xi", pa.int32(), "i"),
              tf("XI", pa.uint32(), "I"), tf("Xf", pa.float32(), "f"), tf("XZ", pa.string(), "Z"), tf("XH", pa.string(), "H"), tf("XA", pa.string(), "A"),
              tf("XB", pa.list_(pa.uint8()), "B:C"), tf("Xb", pa.list_(pa.int16()), "B:s"), tf("XF", pa.list_(pa.float32()), "B:f"),
              tf("Xa", pa.uint32(), "A"), tf("Xl", pa.list_(pa.int32()), "B"), tf("XL", pa.list_(pa.uint32()), "B:I"),
              # column types only a query can produce (CAST, arithmetic): every integer width and Float64 (sam_tag_io.rs:390-438, 292-303)
              tf("Y1", pa.int8(), "c"), tf("Y2", pa.uint8(), "C"), tf("Y3", pa.int16(), "s"), tf("Y4", pa.uint16(), "S"), tf("Y5", pa.int64(), "i"),
              tf("Y6", pa.uint64(), "I"), tf("Y7", pa.float64(), "f"), tf("Y8", pa.int64(), "A"), tf("Y9", pa.int64(), "C")]
    schema = pa.schema(list(o.schema)[:12] + fields, metadata=o.schema.metadata)
    base = batch.select(range(12)).to_pylist()
    rows = []
    for i, r in enumerate(base):
        r = dict(r)
        if i % 2 == 0:
            r.update(Xc=-5 - i, XC=200, Xs=-3000, XS=60000, Xi=-70000, XI=4000000000, Xf=1.5, XZ="hello", XH="1a2b", XA="q", XB=[1, 2, 255], Xb=[-1, 300],
                     XF=[0.5, -2.0], Xa=65, Xl=[-5, 70000], XL=[0, 4294967295],
                     Y1=-128, Y2=255, Y3=-32768, Y4=65535, Y5=-2**31, Y6=2**32 - 1, Y7=-1.5e-3, Y8=126, Y9=7)
        else:
            r.update(XZ="", XB=[], XF=[1e-7])
        rows.append(r)
    b2 = pa.RecordBatch.from_pylist(rows, schema=schema)
    names = [f.name for f in fields]
    out2 = tmp_path / "o2.bam"
    gpu_write(out2, [b2], schema, names + ["NM"])
    check_file(out2, [b2], schema, names + ["NM"])


@pytest.mark.parametrize("mode,reads", [("short", 60000), ("long", 400)])
def test_synthetic_multi_batch_and_slices(mode, reads, syn_dir, tmp_path):
    path = gen_bam(syn_dir, mode, reads, seed=7)
    tags = ["NM", "MD", "AS", "RG"] if mode == "short" else ["NM", "MD", "MM", "ML"]
    o = OracleBam(str(path), tag_fields=tags)
    batch = o.scan(None)
    n = batch.num_rows
    cuts = [0, 1, 17, n // 3, n // 3, (2 * n) // 3 + 5, n]                    # an empty batch and sliced batches (array offset != 0)
    if mode == "short":
        cuts = [0, 1, 17, 17 + 8192, n // 3, n // 3, (2 * n) // 3 + 5, n]      # a batch of exactly two scan tiles (4096 rows each)
    parts = [batch.slice(a, b - a) for a, b in zip(cuts, cuts[1:])]
    out = tmp_path / "o.bam"
    rows, st = gpu_write(out, parts, o.schema, tags)
    assert rows == n
    size = check_file(out, parts, o.schema, tags)
    # the device DEFLATE is a real compressor: within 1.45 x of zlib level 6 on the same stream, far below stored
    stream = W.bam_stream([batch], o.schema, tags, True)
    z6 = sum(len(W.bgzf_member(stream[i:i + W.BGZF_BLOCK])) for i in range(0, len(stream), W.BGZF_BLOCK))
    assert size < 1.45 * z6 and size < 0.75 * len(stream), (size, z6, len(stream))
    # stored members (compression = 1) carry the same stream
    out1 = tmp_path / "o1.bam"
    gpu_write(out1, [batch], o.schema, tags, compression=1)
    assert check_file(out1, [batch], o.schema, tags) > len(stream)


def test_binary_cigar_column(syn_dir, tmp_path):
    path = gen_bam(syn_dir, "short", 5000, seed=3)
    o = OracleBam(str(path), tag_fields=["NM"], binary_cigar=True)
    batch = o.scan(None)
    assert batch.schema.field("cigar").type == pa.binary()
    out = tmp_path / "o.bam"
    gpu_write(out, [batch], o.schema, ["NM"])
    check_file(out, [batch], o.schema, ["NM"])


def test_insert_into_overwrites_the_providers_file(tmp_path):
    """== `INSERT OVERWRITE`: TableProvider::insert_into (table_provider.rs:1117-1177)."""
    import shutil, bamscan
    dst = tmp_path / "t.bam"
    shutil.copyfile(GOLDEN / "multi_chrom.bam", dst)      # contents only: a read-only checkout's mode would make dst read-only
    p = bamscan.BamTableProvider(str(dst), None, True, ["NM"], index_path="")
    batches = list(p.scan(None, [], None).execute(0))
    keep = [b.slice(0, b.num_rows // 2) for b in batches]
    with pytest.raises(NotImplementedError):
        p.insert_into(keep, "append")
    n = p.insert_into(keep)
    assert n == sum(b.num_rows for b in keep)
    p2 = bamscan.BamTableProvider(str(dst), None, True, ["NM"], index_path="")
    back = list(p2.scan(None, [], None).execute(0))
    assert pa.Table.from_batches(back).equals(pa.Table.from_batches(keep))
    # new_for_write (table_provider.rs:639-664): a provider for a file that does not exist yet; sort_on_write only labels the header
    fresh = tmp_path / "fresh.bam"
    pw = bamscan.BamTableProvider.new_for_write(str(fresh), p.schema(), ["NM"], True, sort_on_write=True)
    assert pw.insert_into(keep) == n
    p3 = bamscan.BamTableProvider(str(fresh), None, True, ["NM"], index_path="")
    assert pa.Table.from_batches(list(p3.scan(None, [], None).execute(0))).equals(pa.Table.from_batches(keep))
    assert p3.schema().metadata[b"bio.bam.sort_order"] == b"coordinate"
    assert p2.schema().metadata[b"bio.bam.sort_order"] == b"unsorted"        # write_test.rs::test_sort_on_write_false_sets_unsorted


def test_data_errors_surface(tmp_path):
    import bamscan
    o = OracleBam(str(GOLDEN / "multi_chrom.bam"), tag_fields=[])
    batch = o.scan(None).slice(0, 50)
    cols = {f.name: batch.column(i) for i, f in enumerate(batch.schema)}

    def with_col(name, values):
        arrs = [pa.array(values, type=batch.schema.field(name).type) if f.name == name else cols[f.name] for f in batch.schema]
        return pa.RecordBatch.from_arrays(arrs, schema=batch.schema)
    flags = cols["flags"].to_pylist(); flags[7] = 65536
    with pytest.raises(bamscan.BamScanError, match="row 7.*16-bit SAM flags"):       # serializer.rs::test_batch_to_bam_records_rejects_flag_overflow
        gpu_write(tmp_path / "e1.bam", [with_col("flags", flags)], o.schema, [])
    cig = cols["cigar"].to_pylist(); cig[3] = "10M5"
    with pytest.raises(bamscan.BamScanError, match="row 3.*CIGAR"):
        gpu_write(tmp_path / "e2.bam", [with_col("cigar", cig)], o.schema, [])
    q = cols["quality_scores"].to_pylist(); q[9] = q[9][:-1]
    with pytest.raises(bamscan.BamScanError, match="row 9.*length mismatch"):
        gpu_write(tmp_path / "e3.bam", [with_col("quality_scores", q)], o.schema, [])
    tf = pa.field("Xc", pa.int32(), True, {"bio.bam.tag.tag": "Xc", "bio.bam.tag.type": "c"})
    s2 = pa.schema(list(batch.schema) + [tf], metadata=o.schema.metadata)
    b2 = pa.RecordBatch.from_arrays(list(batch.columns) + [pa.array([1] * 49 + [128], type=pa.int32())], schema=s2)
    with pytest.raises(bamscan.BamScanError, match="row 49") as e:
        gpu_write(tmp_path / "e4.bam", [b2], s2, ["Xc"])
    assert e.value.code == -7
    for typ, val, spec in ((pa.int64(), 2**31, "i"), (pa.uint64(), 2**63 + 5, "I"), (pa.float64(), 1e39, "f"), (pa.float64(), float("nan"), "f")):
        tfw = pa.field("Yw", typ, True, {"bio.bam.tag.tag": "Yw", "bio.bam.tag.type": spec})
        sw = pa.schema(list(batch.schema) + [tfw], metadata=o.schema.metadata)
        bw = pa.RecordBatch.from_arrays(list(batch.columns) + [pa.array([None] * 20 + [val] + [None] * 29, type=typ)], schema=sw)
        with pytest.raises(bamscan.BamScanError, match="row 20") as e:
            gpu_write(tmp_path / "e8.bam", [bw], sw, ["Yw"])
        assert e.value.code == -7
        with pytest.raises(W.WriteError):
            W.encode_batch(bw, ["chr1"], ["Yw"], True)
    bad = pa.schema(list(batch.schema) + [pa.field("Xz", pa.int32(), True, {"bio.bam.tag.tag": "Xz", "bio.bam.tag.type": "Z"})])
    with pytest.raises(bamscan.BamScanError, match="type mismatch"):
        gpu_write(tmp_path / "e5.bam", [], bad, ["Xz"])
    with pytest.raises(bamscan.BamScanError, match="Required column 'flags'"):
        gpu_write(tmp_path / "e6.bam", [], pa.schema([f for f in batch.schema if f.name != "flags"]), [])
    ms = cols["mate_start"].to_pylist(); ms[11] = 2**31
    with pytest.raises(bamscan.BamScanError, match="row 11.*position does not fit"):
        gpu_write(tmp_path / "e7.bam", [with_col("mate_start", ms)], o.schema, [])


def test_incompressible_and_tiny_members(tmp_path):
    """Random names / qualities do not shrink: such members fall back to stored blocks; a file of one record is one tiny member."""
    import random
    rng = random.Random(5)
    o = OracleBam(str(GOLDEN / "multi_chrom.bam"), tag_fields=[])
    schema = o.schema
    rows = []
    for i in range(3000):
        L = 250
        rows.append(dict(name="".join(chr(rng.randint(33, 126)) for _ in range(40)), chrom=None, start=None, end=None, flags=4, cigar="*", mapping_quality=0,
                         mate_chrom=None, mate_start=None, sequence="".join(rng.choice("=ACMGRSVTWYHKDBN") for _ in range(L)),
                         quality_scores="".join(chr(33 + rng.randint(0, 93)) for _ in range(L)), template_length=rng.randint(-2**31, 2**31 - 1)))
    b = pa.RecordBatch.from_pylist(rows, schema=schema)
    out = tmp_path / "r.bam"
    gpu_write(out, [b], schema, [])
    check_file(out, [b], schema, [])
    out1 = tmp_path / "one.bam"
    gpu_write(out1, [b.slice(0, 1)], schema, [])
    check_file(out1, [b.slice(0, 1)], schema, [])
    out0 = tmp_path / "none.bam"
    gpu_write(out0, [], schema, [])
    check_file(out0, [], schema, [])


def test_degenerate_alphabets_and_long_runs(tmp_path):
    """Constant columns: matches of the maximum length 258, a distance code with one used symbol, literal alphabets of a few
    symbols (the forced second symbol keeps both Huffman codes complete); zlib must accept every member."""
    o = OracleBam(str(GOLDEN / "multi_chrom.bam"), tag_fields=[])
    schema = o.schema
    rows = [dict(name="r", chrom="chr1", start=7, end=None, flags=0, cigar="1000M", mapping_quality=60, mate_chrom="=", mate_start=7, sequence="A" * 1000,
                 quality_scores="I" * 1000, template_length=0) for _ in range(2000)]
    b = pa.RecordBatch.from_pylist(rows, schema=schema)
    out = tmp_path / "runs.bam"
    _n, st = gpu_write(out, [b], schema, [])
    size = check_file(out, [b], schema, [])
    assert size < st["bam_bytes"] / 30                                      # (one 258-byte match costs ~2.5 bytes; zlib reaches more with its longer look-ahead)
    # two symbols only: alternating qualities, one base
    rows2 = [dict(r, quality_scores="!~" * 500, name="q") for r in rows[:300]]
    b2 = pa.RecordBatch.from_pylist(rows2, schema=schema)
    out2 = tmp_path / "alt.bam"
    gpu_write(out2, [b2], schema, [])
    check_file(out2, [b2], schema, [])


def test_random_rows_against_the_oracle(tmp_path):
    """Seeded random rows over the corners of the column rules: NULL / "*" / empty names, chromosomes outside the header, "=" mates of
    unplaced reads, NULL positions, position 0 in both coordinate systems, "*" / empty CIGAR + sequence + qualities, odd lengths,
    lower-case and unknown bases, qualities below '!', every tag kind with NULLs and empty values."""
    import random
    rng = random.Random(20261019)
    o = OracleBam(str(GOLDEN / "multi_chrom.bam"), tag_fields=[])
    refs = [d["name"] for d in __import__("json").loads(o.schema.metadata[b"bio.bam.reference_sequences"])]

    def tf(name, typ, spec):
        return pa.field(name, typ, True, {"bio.bam.tag.tag": name, "bio.bam.tag.type": spec})
    tag_fields = [tf("NM", pa.int32(), "i"), tf("XC", pa.uint32(), "C"), tf("Xs", pa.int32(), "s"), tf("Xf", pa.float32(), "f"), tf("MD", pa.string(), "Z"),
                  tf("XH", pa.string(), "H"), tf("XA", pa.string(), "A"), tf("ML", pa.list_(pa.uint8()), "B:C"), tf("Xi", pa.list_(pa.int32()), "B:i"),
                  tf("XF", pa.list_(pa.float32()), "B:f"), tf("XS", pa.list_(pa.uint16()), "B")]
    schema = pa.schema(list(o.schema)[:12] + tag_fields, metadata=o.schema.metadata)
    names = [f.name for f in tag_fields]

    def maybe(p, v):
        return None if rng.random() < p else v

    def cigar_and_len():
        r = rng.random()
        if r < 0.1:
            return rng.choice(["*", ""]), rng.randint(0, 40)
        ops, qlen = [], 0
        for _ in range(rng.randint(1, 12)):
            n, op = rng.choice([1, 2, 9, 10, 99, 100, 12345, 268435455]), rng.choice("MIDNSHP=X")
            ops.append(f"{n}{op}")
        return "".join(ops), rng.randint(0, 60)

    rows = []
    for i in range(3000):
        cig, L = cigar_and_len()
        seq = rng.choice(["*", "", None]) if rng.random() < 0.08 else "".join(rng.choice("ACGTNacgtn=MRSVWYHKDBxz.") for _ in range(L))
        has_seq = seq not in ("*", "", None)
        qual = rng.choice(["*", ""]) if (not has_seq or rng.random() < 0.15) else "".join(chr(rng.choice([32, 33, 34, 73, 126])) for _ in range(len(seq)))
        chrom = maybe(0.15, rng.choice(refs + ["chrNope"]))
        rows.append(dict(
            name=rng.choice([None, "*", "", "r" * rng.randint(1, 254), f"read{i}"]), chrom=chrom, start=maybe(0.15, rng.choice([0, 1, 16383, 16384, 5_000_000, 2**29])),
            end=None, flags=rng.choice([0, 4, 99, 65535]), cigar=cig, mapping_quality=rng.choice([0, 60, 255, 256, 300]),
            mate_chrom=maybe(0.3, rng.choice(refs + ["=", "chrNope"])), mate_start=maybe(0.3, rng.choice([0, 7, 2**31 - 2])), sequence=seq, quality_scores=qual,
            template_length=rng.choice([0, -1, 2**31 - 1, -2**31]),
            NM=maybe(0.3, rng.choice([0, -2**31, 2**31 - 1])), XC=maybe(0.3, rng.randint(0, 255)), Xs=maybe(0.3, rng.randint(-32768, 32767)),
            Xf=maybe(0.3, rng.choice([0.0, -1.5, 3.4028234663852886e38, 1e-45])), MD=maybe(0.3, rng.choice(["", "10A5", "x" * 300])),
            XH=maybe(0.3, rng.choice(["", "1a2B", "FF" * 40])), XA=maybe(0.3, rng.choice("AZ~!")), ML=maybe(0.3, [rng.randint(0, 255) for _ in range(rng.randint(0, 70))]),
            Xi=maybe(0.3, [rng.choice([0, -2**31, 2**31 - 1]) for _ in range(rng.randint(0, 9))]), XF=maybe(0.3, [rng.choice([0.5, -2.0]) for _ in range(rng.randint(0, 5))]),
            XS=maybe(0.3, [rng.randint(0, 65535) for _ in range(rng.randint(0, 33))])))
    batch = pa.RecordBatch.from_pylist(rows, schema=schema)
    for zero_based in (True, False):
        out = tmp_path / f"rnd{int(zero_based)}.bam"
        gpu_write(out, [batch.slice(0, 1111), batch.slice(1111)], schema, names, zero_based)
        check_file(out, [batch], schema, names, zero_based)


@pytest.mark.parametrize("mode,reads,tags", [("short", 30000, ["NM", "MD", "AS", "RG"]), ("long", 300, ["NM", "MD", "MM", "ML"])])
def test_device_batches_are_written_in_place(mode, reads, tags, syn_dir, tmp_path):
    """SURVEY 8 f2 + f4: batches that stay in HBM (bamscan_execute_device / bamscan_next_device) go straight into
    bamscan_writer_write_device -- no D2H, no H2D -- and the file equals the oracle's."""
    import bamscan
    path = gen_bam(syn_dir, mode, reads, seed=11)
    o = OracleBam(str(path), tag_fields=tags)
    want = o.scan(None)
    p = bamscan.BamTableProvider(str(path), None, True, tags, index_path="", chunk_inflated_bytes=4 << 20)    # several device batches
    plan = p.scan(None, [], None)
    out = tmp_path / "dev.bam"
    ex = bamscan.BamWriteExec(str(out), p.schema(), tags, True)
    n = ex.execute(plan.execute_device(0))
    assert n == want.num_rows and ex.stats["arrow_bytes"] == 0 and ex.stats["batches"] > 1
    check_file(out, [want], o.schema, tags)
