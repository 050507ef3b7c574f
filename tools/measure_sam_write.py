#!/usr/bin/env python3
"""SAM write path on one GPU: device ms per stage (validation = enc_cigar_kernel + enc_size_kernel, size = sam_size_kernel, scan =
the 64-bit length scan, render = sam_records_kernel) from a torch.profiler run of its own, the render kernel's bytes/s (Arrow bytes
read + text written) as a share of the HBM data-sheet peak, end-to-end rows/s to a file on tmpfs alternated with the BAM writer on
the same batches, the CPU oracle on a slice, and the output checked against the oracle on seeded sample rows at the timed size.

Workloads: config-2 short reads of tools/bamgen (tags NM MD AS RG), config-5 long reads (NM MD MM ML, ML a B:C array), and the
config-2 rows with a Float32 tag of random bit patterns on every row (f32_to_text on every row).
usage  python tools/measure_sam_write.py [short=20000000] [long=200000] [float_rows=4000000]  -> markdown on stdout.  Files go
under BAMSCAN_BENCH_DIR (default /dev/shm/bamscan_bench); the written outputs are deleted at the end."""
import os
import subprocess
import sys
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
for p in (str(ROOT), str(ROOT / "datafusion-bio-formats_b200")):
    sys.path.insert(0, p)

import numpy as np  # noqa: E402
import pyarrow as pa  # noqa: E402

import bench  # noqa: E402

HBM_PEAK = 7.7e12              # B200 data sheet, HBM3e, one GPU
STAGES = {"validation": ("enc_cigar_kernel", "enc_size_kernel"), "size": ("sam_size_kernel",), "scan": ("len_tile_sums_kernel", "len_offsets_kernel"),
          "render": ("sam_records_kernel",)}


def gpu_info():
    return subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], text=True).strip().splitlines()[0]


def stage_ms(write):
    """Device ms per stage of one call of write(), from CUDA kernel events of torch.profiler."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.init()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        write()
        torch.cuda.synchronize()
    out = {k: 0.0 for k in STAGES}
    for ev in prof.events():
        if ev.device_type.name != "CUDA":
            continue
        us = getattr(ev, "device_time_total", None)
        us = ev.cuda_time_total if us is None else us
        for k, names in STAGES.items():
            if any(n in ev.name for n in names):
                out[k] += us / 1e3
    return out


def sample_check(path, batches, schema, tags, n_sample=20000, seed=5):
    """The written file against the oracle: header, line count, and n_sample seeded rows rendered by the oracle."""
    from oracle import bam_write_oracle as W
    from oracle import sam_write_oracle as SW
    data = np.fromfile(path, dtype=np.uint8)
    text, names, _l = W.build_bam_header(schema, {"bio.bam.sort_order": "unsorted"})
    h = len(text.encode())
    assert data[:h].tobytes() == text.encode(), "header differs"
    ends = np.flatnonzero(data[h:] == 10) + h
    rows = sum(b.num_rows for b in batches)
    assert len(ends) == rows, (len(ends), rows)
    idx = np.sort(np.random.default_rng(seed).choice(rows, size=min(n_sample, rows), replace=False))
    offs = np.cumsum([0] + [b.num_rows for b in batches])
    parts = [b.take(pa.array(idx[(idx >= offs[k]) & (idx < offs[k + 1])] - offs[k])) for k, b in enumerate(batches)]   # (per batch: a whole-table
    sub = pa.Table.from_batches(parts, schema=schema).combine_chunks().to_batches()[0]                                 # take overflows Utf8 offsets)
    want = SW.render_batch(sub, names, tags, True).split(b"\n")[:-1]
    starts = np.concatenate([[h], ends[:-1] + 1])
    for k, i in enumerate(idx):
        got = data[starts[i]:ends[i]].tobytes()
        assert got == want[k], f"row {i}: {got[:80]!r} vs {want[k][:80]!r}"
    return len(idx)


def cpu_rate(batches, schema, tags, n=20000):
    from oracle import bam_write_oracle as W
    from oracle import sam_write_oracle as SW
    _t, names, _l = W.build_bam_header(schema)
    sl = pa.Table.from_batches(batches, schema=schema).slice(0, n).combine_chunks().to_batches()[0]
    t0 = time.perf_counter()
    SW.render_batch(sl, names, tags, True)
    return sl.num_rows / (time.perf_counter() - t0)


def run(label, batches, schema, tags, out_dir):
    import bamscan
    sam, bam = out_dir / "m.sam", out_dir / "m.bam"
    rows = sum(b.num_rows for b in batches)
    res = {"label": label, "rows": rows, "sam": [], "bam": []}
    for rep in range(3):                                       # alternated, rep 0 warms both paths
        for kind, cls, path in (("sam", bamscan.SamWriteExec, sam), ("bam", bamscan.BamWriteExec, bam)):
            ex = cls(str(path), schema, tags, True, {"bio.bam.sort_order": "unsorted"})
            t0 = time.perf_counter()
            n = ex.execute(batches)
            dt = time.perf_counter() - t0
            assert n == rows
            if rep:
                res[kind].append(dict(wall_s=dt, **ex.stats))
            print(f"[{label}] rep {rep} {kind}: {dt:.3f} s", file=sys.stderr, flush=True)
    res["file_bytes"] = sam.stat().st_size
    per_row = max(1, res["file_bytes"] // rows)                # (the CPU oracle's cost grows with the row: ~20 MB of text per check)
    res["checked_rows"] = sample_check(sam, batches, schema, tags, n_sample=max(500, min(20000, 20_000_000 // per_row)))
    try:
        res["stages"] = stage_ms(lambda: bamscan.SamWriteExec(str(sam), schema, tags, True, {"bio.bam.sort_order": "unsorted"}).execute(batches))
    except Exception as e:                                     # (reported as not measured)
        res["stages"] = None
        print(f"[{label}] profiler run failed: {e!r}", file=sys.stderr, flush=True)
    res["cpu_rows"] = max(200, min(20000, 20_000_000 // per_row))
    res["cpu_rows_per_s"] = cpu_rate(batches, schema, tags, res["cpu_rows"])
    sam.unlink(); bam.unlink()
    return res


def report(r):
    sam, bam = r["sam"][-1], r["bam"][-1]
    st = r["stages"]
    render_bytes = sam["arrow_bytes"] + sam["bam_bytes"]
    print(f"### {r['label']}: {r['rows']:,} rows, {r['file_bytes'] / 1e9:.3f} GB of SAM text\n")
    if st is None:
        print("- device ms per stage: not measured (the profiler run failed)")
    else:
        print("| stage | device ms (torch.profiler, one write) |\n|---|---:|")
        for k in STAGES:
            print(f"| {k} | {st[k]:.2f} |")
        print(f"| sum | {sum(st.values()):.2f} |\n")
    if st is not None and st["render"] > 0:
        print(f"- render: {render_bytes / 1e9:.2f} GB (Arrow bytes read {sam['arrow_bytes'] / 1e9:.2f} + text written {sam['bam_bytes'] / 1e9:.2f}) in "
          f"{st['render']:.2f} ms = {render_bytes / (st['render'] / 1e3) / 1e12:.2f} TB/s, {100 * render_bytes / (st['render'] / 1e3) / HBM_PEAK:.1f} % of the "
          f"7.7 TB/s HBM data-sheet peak (counted from the writer's stats: Arrow bytes staged for the batch, SAM text bytes)")
    for kind, x in (("SAM", sam), ("BAM", bam)):
        walls = [y["wall_s"] for y in r[kind.lower()]]
        print(f"- {kind} writer, host batches -> file on tmpfs: wall {', '.join(f'{w:.3f}' for w in walls)} s -> "
              f"{r['rows'] / min(walls) / 1e6:.2f} M rows/s end to end; device encode {x['ms_encode']:.1f} ms, deflate {x['ms_deflate']:.1f} ms; "
              f"file {x['compressed_bytes'] / 1e9:.3f} GB")
    print(f"- CPU oracle (oracle/sam_write_oracle.py, one thread, first {r['cpu_rows']:,} rows): {r['cpu_rows_per_s'] / 1e3:.2f} k rows/s")
    print(f"- output check: header, {r['rows']:,} lines, and {r['checked_rows']:,} seeded sample rows equal to the oracle's lines\n")


def main():
    short = int(sys.argv[1]) if len(sys.argv) > 1 else 20_000_000
    long_ = int(sys.argv[2]) if len(sys.argv) > 2 else 200_000
    frows = int(sys.argv[3]) if len(sys.argv) > 3 else 4_000_000
    import bamscan
    info = gpu_info()
    out_dir = Path(os.environ.get("BAMSCAN_BENCH_DIR", "/dev/shm/bamscan_bench"))
    out_dir.mkdir(parents=True, exist_ok=True)
    results = []
    for label, reads, seed, mode, tags in (("config-2 short reads", short, 2, "short", ["NM", "MD", "AS", "RG"]),
                                           ("config-5 long reads", long_, 5, "long", ["NM", "MD", "MM", "ML"])):
        path, _ = bench.ensure_bam(reads, seed, False, mode=mode)
        p = bamscan.BamTableProvider(str(path), None, True, tags, index_path="")
        batches = list(p.scan(None, [], None).execute(0))
        schema = p.schema()
        p.close()
        results.append(run(label, batches, schema, tags, out_dir))
        if mode == "short":
            t = pa.Table.from_batches(batches, schema=schema).slice(0, frows)
            bits = np.random.default_rng(3).integers(0, 2**32, size=t.num_rows, dtype=np.uint64).astype(np.uint32)
            fs = pa.schema(list(schema) + [pa.field("Xf", pa.float32(), True, {"bio.bam.tag.tag": "Xf", "bio.bam.tag.type": "f"})], metadata=schema.metadata)
            ft = t.append_column(fs.field("Xf"), pa.array(bits.view(np.float32), pa.float32())).cast(fs)
            fb = ft.to_batches(max_chunksize=1 << 20)
            del batches, t
            results.append(run("config-2 rows + a Float32 tag of random bits", fb, fs, tags + ["Xf"], out_dir))
            del fb, ft
    print(f"# SAM write path, measured\n\n`python tools/measure_sam_write.py {short} {long_} {frows}` on **{info}** (name, power limit, max SM clock, "
          f"read by nvidia-smi in the same run).\n")
    for r in results:
        report(r)


if __name__ == "__main__":
    main()
