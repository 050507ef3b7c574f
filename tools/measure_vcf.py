#!/usr/bin/env python3
"""BGZF-VCF scan on one GPU, two seeded inputs from tests/vcf_inputs.py:
  sites      sites-only lines (gnomAD-like): 12 declared INFO keys plus 24 integer keys per line and a VEP-like CSQ list of
             0.5-2 kB, about 5 M records;
  genotypes  200 k records x 2 504 samples of FORMAT GT (about 10 kB lines; FORMAT and samples are skipped by the scan).
Per input: device-resident CUDA-event time per stage (run_device_resident: ms_inflate, ms_boundary = the newline scan and line
framing, ms_decode = the VCF kernels), rows/s and inflated GB/s, kernel launches, kernel times by name (torch.profiler, in a run of
its own), and end to end through the ABI (host batches).  The card's name and power limit are read in the same run.
With a fourth argument, instead: one genotype input of that many records x 2 504 samples carrying FORMAT GT:DP:AD:GQ:PL
(tests/vcf_format_inputs.py), scanned (a) without FORMAT columns, (b) with format_fields=["GT"] and (c) with all five.
usage: python tools/measure_vcf.py [out.md] [sites_records=5000000] [genotype_records=200000] [format_records]"""
import os
import subprocess
import sys
import tempfile
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
for p in (str(ROOT), str(ROOT / "datafusion-bio-formats_b200"), str(ROOT / "tests")):
    sys.path.insert(0, p)
OUT = Path(sys.argv[1]) if len(sys.argv) > 1 else ROOT / "profiles" / "r4_vcf.md"
SITES = int(sys.argv[2]) if len(sys.argv) > 2 else 5_000_000
GENOTYPES = int(sys.argv[3]) if len(sys.argv) > 3 else 200_000
FORMAT_RECORDS = int(sys.argv[4]) if len(sys.argv) > 4 else 0


def card():
    return subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], text=True).strip().splitlines()[0]


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


def measure(path, format_fields=None):
    import bamscan
    rows = {}
    p = bamscan.VcfTableProvider(str(path), format_fields=format_fields)
    plan = p.scan()
    plan.run_device_resident(0, 1)                                   # warm-up (module load, allocations)
    st = plan.run_device_resident(0, 3)
    rows["records"] = st["rows"]
    rows["inflated GB"] = st["inflated_bytes"] / 1e9
    rows["device-resident ms (mean of 3)"] = st["ms_total"]
    rows["  inflate ms (last run)"] = st["ms_inflate"]
    rows["  framing ms (last run)"] = st["ms_boundary"]
    rows["  VCF kernels ms (last run)"] = st["ms_decode"]
    rows["kernel launches (last run)"] = st["kernel_launches"]
    rows["device-resident M rows/s"] = st["rows"] / st["ms_total"] / 1e3
    rows["device-resident inflated GB/s"] = st["inflated_bytes"] / st["ms_total"] / 1e6
    t0 = time.perf_counter()
    p2 = bamscan.VcfTableProvider(str(path), format_fields=format_fields)
    n = sum(b.num_rows for b in p2.scan().execute(0))
    t1 = time.perf_counter()
    assert n == st["rows"]
    rows["end to end s"] = t1 - t0
    rows["end to end M rows/s"] = n / (t1 - t0) / 1e6
    rows["end to end inflated GB/s"] = st["inflated_bytes"] / (t1 - t0) / 1e9
    ks = kernel_ms(lambda: plan.run_device_resident(0, 1))
    for k in sorted(ks):
        if "vcf" in k or "fq_" in k or "sam_frame" in k:
            rows[f"{k} ms"] = ks[k]
    rows["inflate kernels ms (profiled run)"] = sum(v for k, v in ks.items() if "inflate" in k)
    p.close(); p2.close()
    return rows


def main_format():
    from vcf_format_inputs import FIVE, format_text
    from vcf_inputs import bgzf_parallel
    info = card()
    base = Path(os.environ.get("BAMSCAN_BENCH_DIR", tempfile.mkdtemp(prefix="bamscan_vcf_")))
    base.mkdir(parents=True, exist_ok=True)
    path = base / "format.vcf.gz"
    t0 = time.time()
    text = format_text(FORMAT_RECORDS)
    path.write_bytes(bgzf_parallel(text))
    print(f"[format] generated {len(text) / 1e9:.2f} GB text, {path.stat().st_size / 1e9:.2f} GB file in {time.time() - t0:.1f} s", file=sys.stderr)
    del text
    cases = {"(a) no FORMAT": None, "(b) GT": ["GT"], "(c) GT DP AD GQ PL": FIVE}
    results = {}
    for name, sel in cases.items():
        results[name] = measure(path, sel)
        print(f"[{name}] {results[name]}", file=sys.stderr)
    path.unlink()
    keys = list(dict.fromkeys(k for r in results.values() for k in r))
    lines = ["# VCF FORMAT columns on one GPU (`tools/measure_vcf.py`, FORMAT input)", "",
             f"Card (nvidia-smi name, power limit, max SM clock): **{info}**.", "",
             f"Input from `tests/vcf_format_inputs.py::format_text`: {FORMAT_RECORDS:,} records x 2 504 samples of FORMAT "
             "GT:DP:AD:GQ:PL (every seventh line GT:PL:DP), zlib level 1 BGZF members of 0xff00 bytes.", "",
             "Device-resident times are CUDA events around the whole partition with the compressed file staged in HBM (mean of 3 "
             "runs after a warm-up); the stage split is of the last run. Kernel times come from a separate run under "
             "torch.profiler. End to end is `VcfTableProvider.scan().execute(0)` to host Arrow batches of every column.", "",
             "| | " + " | ".join(cases) + " |", "|---|" + "---:|" * len(cases)]
    for k in keys:
        vals = [r.get(k, 0.0) for r in results.values()]
        fmt = (lambda v: f"{v:,}") if all(isinstance(v, int) for v in vals) else (lambda v: f"{v:,.3f}")
        lines.append(f"| {k} | " + " | ".join(fmt(v) for v in vals) + " |")
    OUT.parent.mkdir(parents=True, exist_ok=True)
    OUT.write_text("\n".join(lines) + "\n")
    print("\n".join(lines))


def main():
    if FORMAT_RECORDS:
        return main_format()
    from vcf_inputs import bgzf_parallel, genotypes_text, sites_text
    info = card()
    base = Path(os.environ.get("BAMSCAN_BENCH_DIR", tempfile.mkdtemp(prefix="bamscan_vcf_")))
    base.mkdir(parents=True, exist_ok=True)
    results = {}
    for name, make in (("sites", lambda: sites_text(SITES)), ("genotypes", lambda: genotypes_text(GENOTYPES))):
        path = base / f"{name}.vcf.gz"
        t0 = time.time()
        path.write_bytes(bgzf_parallel(make()))
        print(f"[{name}] generated {path.stat().st_size / 1e9:.2f} GB in {time.time() - t0:.1f} s", file=sys.stderr)
        results[name] = measure(path)
        path.unlink()
        print(f"[{name}] {results[name]}", file=sys.stderr)
    keys = list(dict.fromkeys(list(results["sites"]) + list(results["genotypes"])))
    lines = ["# BGZF-VCF scan on one GPU (`tools/measure_vcf.py`)", "",
             f"Card (nvidia-smi name, power limit, max SM clock): **{info}**.", "",
             f"Inputs from `tests/vcf_inputs.py` (zlib level 1 BGZF members of 0xff00 bytes): *sites* is {SITES:,} sites-only records "
             "with 36 INFO keys and a CSQ list of 0.5-2 kB per line; *genotypes* is "
             f"{GENOTYPES:,} records with FORMAT GT and 2 504 samples.", "",
             "Device-resident times are CUDA events around the whole partition with the compressed file staged in HBM (mean of 3 "
             "runs after a warm-up); the stage split is of the last run. Kernel times come from a separate run under "
             "torch.profiler. End to end is `VcfTableProvider.scan().execute(0)` to host Arrow batches of every column.", "",
             "| | sites | genotypes |", "|---|---:|---:|"]
    for k in keys:
        a, b = results["sites"].get(k, 0.0), results["genotypes"].get(k, 0.0)
        fmt = (lambda v: f"{v:,}") if isinstance(a, int) and isinstance(b, int) else (lambda v: f"{v:,.3f}")
        lines.append(f"| {k} | {fmt(a)} | {fmt(b)} |")
    OUT.parent.mkdir(parents=True, exist_ok=True)
    OUT.write_text("\n".join(lines) + "\n")
    print("\n".join(lines))


if __name__ == "__main__":
    main()
