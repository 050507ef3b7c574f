#!/usr/bin/env python3
"""FASTQ write path on one GPU: device encode + deflate time, end to end from host batches and scan -> device batches -> write,
file size against zlib level 6 on the same 0xff00-byte members, and the CPU restatement (oracle/fastq_write_oracle.py + zlib,
one thread) on a sample.  Data: the 101 bp generator of tools/measure_fastq.py (its BGZF file is the input of the scans).
usage  python tools/measure_fastq_write.py [reads=20000000]  -> markdown on stdout.  Files go under BAMSCAN_BENCH_DIR
(default /dev/shm/bamscan_bench); the written outputs are deleted at the end."""
import os, subprocess, sys, time, zlib
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT)); sys.path.insert(0, str(ROOT / "datafusion-bio-formats_b200")); sys.path.insert(0, str(ROOT / "tools"))
import measure_fastq as MF  # noqa: E402  (reads sys.argv[1] for the read count)

reads = MF.reads


def gpu_name():
    try:
        return subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], text=True).strip().splitlines()[0]
    except Exception as e:       # (the device itself is checked by the writer: there is no CPU path)
        return f"unknown ({e})"


def first_members_text(path, n_members):
    """Inflated text of the first n BGZF members of a file."""
    out, off = [], 0
    with open(path, "rb") as f:
        raw = f.read(n_members * 65536)
    for _ in range(n_members):
        size = int.from_bytes(raw[off + 16:off + 18], "little") + 1
        out.append(zlib.decompress(raw[off + 18:off + size - 8], -15))
        off += size
    return b"".join(out)


PER_JOB = 250_000          # reads per generator job of tools/measure_fastq.py (seed 1000 + job)


def _job_text(k):
    n = min(PER_JOB, reads - k * PER_JOB)
    return MF.make_text(k * PER_JOB, n, 1000 + k) if n > 0 else b""


def _z6_members_of_job(k):
    """zlib level 6 bytes (BGZF member framing included) of the exact 0xff00-byte members of the whole text whose first byte
    lies in generator job k; a member that crosses into job k + 1 takes its tail from there."""
    from oracle.bam_write_oracle import bgzf_member
    text = _job_text(k)
    g0 = k * PER_JOB * len(MF.make_text(0, 1, 0))      # fixed-width records: the job's offset in the whole text
    nxt = _job_text(k + 1)[:0xff00]
    both = text + nxt
    m0 = (g0 + 0xff00 - 1) // 0xff00
    total = 0
    for m in range(m0, (g0 + len(text) + 0xff00 - 1) // 0xff00):
        a = m * 0xff00 - g0
        total += len(bgzf_member(both[a:a + 0xff00]))
    return total


def zlib6_exact_members():
    """The whole text recompressed with zlib level 6 in exact 0xff00-byte members (the writer's member size), in parallel."""
    from concurrent.futures import ProcessPoolExecutor
    with ProcessPoolExecutor(max_workers=min(32, os.cpu_count() or 8)) as ex:
        return sum(ex.map(_z6_members_of_job, range((reads + PER_JOB - 1) // PER_JOB)))


def main():
    import pyarrow as pa
    import bamscan
    from oracle import fastq_write_oracle as FW
    from oracle.bam_write_oracle import bgzf_member
    src, info = MF.ensure_file()
    print(f"[fastq-write] {src}: {info}", file=sys.stderr, flush=True)
    text_bytes = info["inflated_bytes"]
    t0 = time.perf_counter()
    z6_bytes = zlib6_exact_members()                   # (the generator's own file ends a member early at every job boundary)
    print(f"[fastq-write] zlib-6 on exact 0xff00 members: {z6_bytes} bytes in {time.perf_counter() - t0:.1f} s", file=sys.stderr, flush=True)
    base = src.parent
    prov = bamscan.FastqTableProvider(str(src))
    schema = prov.schema()
    host = list(prov.scan().execute(0))
    assert sum(b.num_rows for b in host) == reads
    results = {}
    for label, comp, source in (("host batches -> BGZF", 0, "host"), ("host batches -> plain text", 2, "host"),
                                ("scan -> device batches -> BGZF", 0, "device")):
        out = base / ("w.fastq" if comp == 2 else "w.fastq.bgz")
        for rep in range(2):                           # the second repetition is reported (pooled buffers and staging warm)
            ex = bamscan.FastqWriteExec(str(out), schema, comp)
            t0 = time.perf_counter()
            n = ex.execute(prov.scan().execute_device(0) if source == "device" else host)
            wall = time.perf_counter() - t0
        st = ex.stats
        assert n == reads and st["bam_bytes"] == text_bytes, (n, st)
        size = out.stat().st_size
        head = out.read_bytes()[:1 << 21] if comp == 2 else first_members_text(out, 32)
        want = _job_text(0)[:len(head)]
        assert head == want, "written text differs from the generator's"
        results[label] = (wall, st, size)
        print(f"[fastq-write] {label}: {wall:.3f} s, stats {st}, file {size}", file=sys.stderr, flush=True)
        out.unlink()
    # CPU restatement on a sample: render + zlib level 6 members, one thread
    sample = min(reads, 200_000)
    tb = pa.Table.from_batches(host).slice(0, sample).combine_chunks().to_batches()[0]
    t0 = time.perf_counter()
    txt = FW.render_batch(tb)
    blob = b"".join(bgzf_member(txt[i:i + 0xff00]) for i in range(0, len(txt), 0xff00))
    cpu_s = time.perf_counter() - t0
    assert txt == _job_text(0)[:len(txt)] and len(blob) > 0     # (the generator's random draws depend on the job size)
    print(f"GPU: {gpu_name()}\n")
    print(f"{reads} reads x {MF.READ_LEN} bp, {text_bytes / 1e9:.2f} GB of FASTQ text.\n")
    print("| path | device encode ms | device deflate ms | reads/s (device: encode + deflate) | wall s | reads/s (end to end) | file GB | file / text | file / zlib-6 |")
    print("|---|---:|---:|---:|---:|---:|---:|---:|---:|")
    for label, (wall, st, size) in results.items():
        dev = st["ms_encode"] + st["ms_deflate"]
        plain = "plain" in label
        print(f"| {label} | {st['ms_encode']:.1f} | {st['ms_deflate']:.1f} | {reads / dev * 1e3 / 1e6:.1f} M | {wall:.3f} | {reads / wall / 1e6:.1f} M | "
              f"{size / 1e9:.3f} | {size / text_bytes:.3f} | {'-' if plain else f'{size / z6_bytes:.3f}'} |")
    print(f"\nzlib level 6 on the same text in exact 0xff00-byte BGZF members (EOF marker excluded): {z6_bytes / 1e9:.3f} GB ({z6_bytes / text_bytes:.3f} of the text); "
          f"the GPU files include the 28-byte EOF marker.")
    print(f"Device encode rate: {text_bytes / (results['host batches -> BGZF'][1]['ms_encode'] / 1e3) / 1e9:.1f} GB/s of FASTQ text written; "
          f"deflate: {text_bytes / (results['host batches -> BGZF'][1]['ms_deflate'] / 1e3) / 1e9:.1f} GB/s of text in.")
    print(f"CPU restatement (oracle/fastq_write_oracle.py render + zlib level 6 members, 1 thread) on {sample} reads: {sample / cpu_s / 1e6:.3f} M reads/s.")
    prov.close()


if __name__ == "__main__":
    main()
