#!/usr/bin/env python3
"""BGZF-FASTA scan on one GPU, two seeded shapes from `bamgen --fasta`:
  genome  the 25 records of a human-sized assembly (about 3.1 Gb, 60-column lines, runs of lower case and N);
  short   20 M records of 300 residues, one-line and wrapped at 60 columns.
Per shape: device-resident CUDA-event time per stage (run_device_resident), inflated GB/s, the sequence copy kernel's algorithmic
bytes (text read once + sequence written once) over its time (torch.profiler, in a run of its own), end to end through the ABI
(host batches), and the CPU restatement (oracle/fasta_oracle.py, one thread) on a 64 MB sample.  The card's name and power limit are
read in the same run.  usage: python tools/measure_fasta.py [out.md] [short_records=20000000]"""
import os
import subprocess
import sys
import tempfile
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT)); sys.path.insert(0, str(ROOT / "datafusion-bio-formats_b200"))
OUT = Path(sys.argv[1]) if len(sys.argv) > 1 else ROOT / "profiles" / "r4_fasta.md"
SHORT = int(sys.argv[2]) if len(sys.argv) > 2 else 20_000_000


def card():
    return subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], text=True).strip().splitlines()[0]


def bamgen():
    exe = ROOT / "tools" / "_build" / "bamgen"
    if not exe.exists():
        exe.parent.mkdir(exist_ok=True)
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-pthread", "-o", str(exe), str(ROOT / "tools" / "bamgen.cpp"), "-lz"])
    return exe


def rows_and_seq_bytes(batches):
    rows = n = 0
    for b in batches:
        c = b.column("sequence")
        o = np.frombuffer(c.buffers()[1], np.int32)[c.offset:c.offset + b.num_rows + 1]
        rows += b.num_rows
        n += int(o[-1] - o[0])
    return rows, n


def kernel_ms(fn):
    """Sums of CUDA kernel time by kernel name over one call of fn (torch.profiler; CUPTI sees the library's kernels too)."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.init()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    out = {}
    for e in prof.events():
        if e.device_type.name == "CUDA":
            key = e.name.split("(")[0].replace("void ", "").replace("bamscan::", "")
            out[key] = out.get(key, 0.0) + e.device_time / 1e3
    return out


def measure(shape, path, info):
    import bamscan
    from oracle.bam_write_oracle import inflate_bgzf
    from oracle.fasta_oracle import parse_records
    rows = {}
    p = bamscan.FastaTableProvider(str(path))
    plan = p.scan()
    plan.run_device_resident(0, 1)                                   # warm-up (module load, allocations)
    st = plan.run_device_resident(0, 3)
    rows["records"] = st["rows"]
    rows["inflated GB"] = st["inflated_bytes"] / 1e9
    rows["device-resident ms (mean of 3)"] = st["ms_total"]
    rows["  inflate ms (last run)"] = st["ms_inflate"]
    rows["  framing ms (last run)"] = st["ms_boundary"]
    rows["  lines + columns ms (last run)"] = st["ms_decode"]
    rows["device-resident inflated GB/s"] = st["inflated_bytes"] / st["ms_total"] / 1e6
    # end to end through the ABI: open, plan and host batches of all three columns (nothing kept)
    t0 = time.perf_counter()
    p2 = bamscan.FastaTableProvider(str(path))
    full, n_seq = rows_and_seq_bytes(p2.scan().execute(0))
    t1 = time.perf_counter()
    assert full == st["rows"]
    rows["sequence GB"] = n_seq / 1e9
    rows["end to end s"] = t1 - t0
    rows["end to end inflated GB/s"] = st["inflated_bytes"] / (t1 - t0) / 1e9
    rows["end to end M records/s"] = full / (t1 - t0) / 1e6
    # kernel times, one device-resident run under the profiler
    ks = kernel_ms(lambda: plan.run_device_resident(0, 1))
    seq_ms = ks.get("fa_seq_kernel", 0.0)
    rows["fa_seq_kernel ms"] = seq_ms
    rows["fa_seq_kernel (text read + sequence written) GB/s"] = (st["inflated_bytes"] + n_seq) / seq_ms / 1e6 if seq_ms else float("nan")
    for k in ("fq_count_kernel", "fq_lines_kernel", "fa_count_kernel", "fa_starts_kernel", "fa_lines_kernel", "fa_lengths_kernel", "fa_copy_kernel<8>"):
        rows[f"{k} ms"] = ks.get(k, 0.0)
    infl = sum(v for k, v in ks.items() if "inflate" in k)
    rows["inflate kernels ms (profiled run)"] = infl
    p.close(); p2.close()
    # CPU restatement on a 64 MB sample
    data = path.read_bytes()
    off, take = 0, 0
    while take < (64 << 20) and off < len(data):
        bsize = int.from_bytes(data[off + 16:off + 18], "little") + 1
        off += bsize; take += 0xff00
    text, _ = inflate_bgzf(data[:off])
    cut = text.rfind(b"\n>") + 1 if shape == "short" else len(text)
    t0 = time.perf_counter()
    recs = parse_records(text[:cut])
    dt = time.perf_counter() - t0
    rows["CPU oracle MB/s (one thread, 64 MB sample)"] = cut / dt / 1e6
    rows["CPU oracle records/s (one thread)"] = len(recs) / dt
    return rows


def main():
    info = card()
    base = Path(os.environ.get("BAMSCAN_BENCH_DIR", tempfile.mkdtemp(prefix="bamscan_fasta_")))
    base.mkdir(parents=True, exist_ok=True)
    results = {}
    for shape, n in (("genome", 25), ("short", SHORT)):
        path = base / f"{shape}.fa.bgz"
        t0 = time.time()
        subprocess.check_call([str(bamgen()), "--fasta", shape, "--reads", str(n), "--seed", "20", "--out", str(path)])
        print(f"[{shape}] generated {path.stat().st_size / 1e9:.2f} GB in {time.time() - t0:.1f} s", file=sys.stderr)
        results[shape] = measure(shape, path, info)
        path.unlink()
        print(f"[{shape}] {results[shape]}", file=sys.stderr)
    lines = ["# BGZF-FASTA scan on one GPU (`tools/measure_fasta.py`)", "",
             f"Card (nvidia-smi name, power limit, max SM clock): **{info}**.", "",
             "Inputs from `bamgen --fasta <shape> --seed 20` (zlib level 6 BGZF members of 0xff00 bytes): *genome* is 25 records "
             "(about 3.1 Gb, 60-column lines, runs of lower case and N); *short* is "
             f"{SHORT:,} records of 300 residues, alternately on one line and wrapped at 60 columns.", "",
             "Device-resident times are CUDA events around the whole partition with the compressed file staged in HBM (mean of 3 "
             "runs after a warm-up). Kernel times come from a separate run under torch.profiler. The copy kernel's bytes are the "
             "text read once plus the sequence written once. End to end is `FastaTableProvider.scan().execute(0)` to host Arrow "
             "batches. The CPU oracle is the pure-Python restatement on one thread.", "",
             "| | genome | short |", "|---|---:|---:|"]
    for k in results["genome"]:
        a, b = results["genome"][k], results["short"][k]
        fmt = (lambda v: f"{v:,}") if isinstance(a, int) else (lambda v: f"{v:,.3f}")
        lines.append(f"| {k} | {fmt(a)} | {fmt(b)} |")
    OUT.parent.mkdir(parents=True, exist_ok=True)
    OUT.write_text("\n".join(lines) + "\n")
    print("\n".join(lines))


if __name__ == "__main__":
    main()
