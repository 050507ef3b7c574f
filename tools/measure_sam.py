#!/usr/bin/env python3
"""Plain-SAM scan against the BAM scan of the SAME reads, on one GPU.

usage  python tools/measure_sam.py [reads=20000000] [--out DIR]   -> markdown on stdout (and DIR/r3_sam.md when --out is given)

Input: the config-2 shape of bench.py (tools/bamgen.cpp short mode, 150 bp paired-end, seed 2, the bench's tag set), written
once as BGZF BAM and once as SAM text (`bamgen --sam`: the same header and records).  Files go to a temporary directory.

For each format, in the same call:
- device-resident reads/s (bamscan_run_device_resident: input staged in HBM, untimed) and the per-stage split of BamScanStats:
  ms_inflate (BAM: inflate; SAM: the ingest copy), ms_boundary (BAM: record boundaries; SAM: line framing + transcode to BAM),
  ms_decode;
- end-to-end reads/s (execute(): H2D from the page cache, D2H of every Arrow batch);
- the bytes-based fraction of HBM peak over the device-resident time.  SAM: text read + BAM records written + BAM records read
  + Arrow written.  BAM: BGZF read + inflated written + inflated read + Arrow written.  The BAM records a SAM chunk is
  transcoded into have the BAM file's record bytes (same records), so the BAM file's inflated size stands for them;
- the CPU arm: oracle/sam_oracle.py (Python parser + transcode + bam_oracle.c) on one thread, on a sample of the SAM.
The card's name, power limit and maximum SM clock are read in the same call and printed with the numbers.
"""
import argparse
import subprocess
import sys
import tempfile
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT)); sys.path.insert(0, str(ROOT / "datafusion-bio-formats_b200"))
TAGS = ["NM", "MD", "AS", "RG"]          # bench.py's config-2 tag set
HBM_PEAK = 7.7e12                        # B200 data sheet, bytes/s (one GPU, 1000 W)


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True)
    except FileNotFoundError:
        out = None
    if out is None or out.returncode != 0:
        raise SystemExit("nvidia-smi failed: this measurement needs a GPU")
    return out.stdout.strip().splitlines()[0]


def bamgen():
    exe = ROOT / "tools" / "_build" / "bamgen"
    src = ROOT / "tools" / "bamgen.cpp"
    if not exe.exists() or exe.stat().st_mtime < src.stat().st_mtime:
        exe = Path(tempfile.gettempdir()) / "bamgen_measure_sam"
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-pthread", "-o", str(exe), str(src), "-lz"])
    return exe


def measure(path, reads, repeats=3):
    import bamscan
    prov = bamscan.BamTableProvider(str(path), tag_fields=TAGS, index_path="")
    plan = prov.scan(None, [], None)
    plan.run_device_resident(0, 1)                                   # warm-up: module load, buffers
    st = plan.run_device_resident(0, repeats)                        # ms_total: mean over the repeats
    assert st["rows"] == reads, (st["rows"], reads)
    e2e = []
    for _ in range(2):
        t0 = time.perf_counter(); n = 0
        for b in plan.execute(0):
            n += b.num_rows
            del b
        e2e.append(time.perf_counter() - t0)
        assert n == reads, (n, reads)
    prov.close()
    return st, min(e2e)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("reads", nargs="?", type=int, default=20_000_000)
    ap.add_argument("--out", default=None, help="directory for r3_sam.md")
    a = ap.parse_args()
    reads = a.reads + (a.reads & 1)
    gpu = card()
    exe = bamgen()
    with tempfile.TemporaryDirectory(dir="/dev/shm" if Path("/dev/shm").is_dir() else None) as td:
        bam, sam = Path(td) / "r.bam", Path(td) / "r.sam"
        for out, extra in ((bam, []), (sam, ["--sam"])):
            subprocess.check_call([str(exe), "--mode", "short", "--reads", str(reads), "--seed", "2", "--out", str(out), "--level", "6"] + extra,
                                  stdout=subprocess.DEVNULL)
        res = {}
        for name, path in (("BAM", bam), ("SAM", sam)):
            res[name] = measure(path, reads)
            print(f"[sam] {name}: {res[name]}", file=sys.stderr, flush=True)
        bam_records = res["BAM"][0]["inflated_bytes"]               # (header included: a few KB)
        # CPU arm: the oracle on the first lines of the SAM, one thread
        sample = min(reads, 200_000)
        with open(sam, "rb") as f:
            head = b"".join(f.readline() for _ in range(sample + 40))
        lines = head.split(b"\n")
        n_hdr = sum(1 for ln in lines if ln.startswith(b"@"))
        part = Path(td) / "sample.sam"
        part.write_bytes(b"\n".join(lines[:n_hdr + sample]) + b"\n")
        from oracle.sam_oracle import OracleSam
        t0 = time.perf_counter()
        o = OracleSam(str(part), tag_fields=TAGS)
        nrows = o.scan().num_rows
        cpu_s = time.perf_counter() - t0
        o.close()
    rows = []
    for name in ("BAM", "SAM"):
        st, e2e_s = res[name]
        ms = st["ms_total"]
        if name == "SAM":
            traffic = st["inflated_bytes"] + 2 * bam_records + st["arrow_bytes"]
        else:
            traffic = st["compressed_bytes"] + 2 * st["inflated_bytes"] + st["arrow_bytes"]
        rows.append(f"| {name} | {st['compressed_bytes'] / 1e9:.2f} | {ms:.1f} | {reads / ms * 1e3 / 1e6:.1f} M | {st['ms_inflate']:.1f} | "
                    f"{st['ms_boundary']:.1f} | {st['ms_decode']:.1f} | {traffic / 1e9:.2f} | {traffic / (ms / 1e3) / HBM_PEAK:.3f} | "
                    f"{e2e_s * 1e3:.0f} | {reads / e2e_s / 1e6:.1f} M |")
    md = [f"# Plain SAM against BAM, same {reads} reads (config-2 shape: bamgen short, seed 2, tags {', '.join(TAGS)})", "",
          f"Card: {gpu} (name, power limit, max SM clock, read in the same call).", "",
          "| format | input GB | device ms | reads/s (device) | ingest / inflate ms | framing + transcode / boundaries ms | decode ms | "
          "bytes moved GB | fraction of HBM peak (7.7 TB/s) | e2e ms | reads/s (e2e) |",
          "|---|---:|---:|---:|---:|---:|---:|---:|---:|---:|---:|"] + rows + [
          "",
          f"CPU arm: oracle/sam_oracle.py on the first {nrows} reads, one thread: {nrows / cpu_s / 1e6:.3f} M reads/s.",
          "Stage times are CUDA-event sums over the scan's chunks; a stage that overlaps the next chunk's work is counted whole."]
    text = "\n".join(md) + "\n"
    print(text)
    if a.out:
        Path(a.out).mkdir(parents=True, exist_ok=True)
        (Path(a.out) / "r3_sam.md").write_text(text)


if __name__ == "__main__":
    main()
