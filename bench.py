#!/usr/bin/env python3
"""bench.py -- BAM->Arrow scan throughput (BASELINE.json metric) on N B200s of one node.

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K --warmup W   # CPU restatement of the reference path, all host threads

A step = one full-projection scan (12 core columns + NM, MD, AS, RG) of the synthetic 150 bp WGS-like BAM of
BASELINE.json configs[1] (100 M reads by default; --reads / BAMSCAN_BENCH_READS overrides), written once per box by the
repo's own writer (tools/bamgen.cpp, seed 2, zlib level 6) under /dev/shm.

value   : reads/s, device resident (compressed bytes already in HBM, Arrow buffers stay in HBM), CUDA-event time, max over ranks
e2e     : same scan through the public provider API: H2D of the compressed bytes from pinned host memory and D2H of every
          Arrow buffer inside the timed region
roofline: the inflate stage (dominant), algorithmic bytes = compressed bytes read + inflated bytes written, per launch
N > 1   : STRONG scaling of the ONE file (BASELINE config 2, "by BGZF block range"): the plan has N block-range partitions,
          rank r scans partition r on its own GPU (ranks > 0 find their first record by speculation); no collective on the
          data path.  `replicas` keeps the round-1 number (every rank scans a whole copy) beside it.
verify  : at N = 1, config 2 (or with --verify; --no-verify skips it), outside every timed region, the default product path
          over a <= 10 M-read file of the same generator is compared with the oracle, every row of every column
          (oracle/verify.py); the result goes into the line's "verify" key.
--config: 2 (default) full projection | 3 fixed-width projection | 4 BAI region query chr1:50M-150M | 5 long reads
--dump-outputs DIR: after the timed steps, <= 64 MB of what the last end-to-end step handed its caller, as float .npy files
          (column_arrays): 16 windows of 1024 rows at seeded offsets, so two builds can be compared output for output
"""
import argparse
import json
import os
import statistics
import struct
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np
import pyarrow as pa
import pyarrow.compute as pc

ROOT = Path(__file__).resolve().parent
PKG = ROOT / "datafusion-bio-formats_b200"
for p in (str(ROOT), str(PKG)):
    if p not in sys.path:
        sys.path.insert(0, p)

TAGS = ["NM", "MD", "AS", "RG"]


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def ensure_bam(reads: int, seed: int, want_bai: bool, mode: str = "short") -> tuple[Path, dict]:
    base = Path(os.environ.get("BAMSCAN_BENCH_DIR", "/dev/shm/bamscan_bench"))
    base.mkdir(parents=True, exist_ok=True)
    path = base / f"wgs_{mode}_{reads}_s{seed}.bam"
    meta = path.with_suffix(".json")
    if path.exists() and meta.exists() and (not want_bai or Path(str(path) + ".bai").exists()):
        return path, json.loads(meta.read_text())
    exe = ROOT / "tools" / "_build" / "bamgen"          # built by __graft_entry__.build()
    src = ROOT / "tools" / "bamgen.cpp"
    if not exe.exists() or exe.stat().st_mtime < src.stat().st_mtime:
        exe = base / "bamgen"                            # the source tree may be read-only: build beside the data
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-pthread", "-o", str(exe), str(src), "-lz"])
    t0 = time.time()
    out = subprocess.check_output([str(exe), "--mode", mode, "--reads", str(reads), "--seed", str(seed), "--out", str(path),
                                   "--level", "6", "--bai"])
    info = json.loads(out.decode().strip().splitlines()[-1])
    info["generate_s"] = round(time.time() - t0, 1)
    meta.write_text(json.dumps(info))
    log(f"[bench] generated {path} in {info['generate_s']} s: {info}")
    return path, info


DUMP_BYTES = 64 << 20
DUMP_WINDOWS, DUMP_WINDOW_ROWS = 16, 1024


def dump_windows(rows: int, seed: int = 0):
    """Row windows [lo, hi) of one step's output to dump, in row order: DUMP_WINDOW_ROWS rows at a seeded offset inside
    each of DUMP_WINDOWS equal strata, or the whole output when it is smaller."""
    if rows <= DUMP_WINDOWS * DUMP_WINDOW_ROWS:
        return [(0, rows)]
    rng = np.random.default_rng(seed)
    stratum = rows // DUMP_WINDOWS
    starts = [k * stratum + int(rng.integers(0, stratum - DUMP_WINDOW_ROWS + 1)) for k in range(DUMP_WINDOWS)]
    return [(lo, lo + DUMP_WINDOW_ROWS) for lo in starts]


def keep_window_rows(batch, first_row: int, windows, kept: list):
    """Appends (row index, copy of the rows) to `kept` for the rows of `batch` that fall in `windows`; `first_row` is the
    index of the batch's first row in the step's output.  Only the copies outlive the batch."""
    for lo, hi in windows:
        lo, hi = max(lo, first_row), min(hi, first_row + batch.num_rows)
        if lo < hi:
            kept.append((lo, batch.take(pa.array(np.arange(lo - first_row, hi - first_row)))))


def _is_bytes(t):
    return pa.types.is_string(t) or pa.types.is_binary(t)


def column_arrays(name, col):
    """One Arrow column as float arrays: numbers as float64 with NaN for null; strings and binaries as their UTF-8 / raw
    bytes (float32) plus per-row byte lengths (float64, NaN for null); lists as their flattened values plus lengths."""
    f64 = lambda a: np.asarray(a.to_numpy(zero_copy_only=False), dtype=np.float64)
    t = col.type
    if _is_bytes(t):
        data = b"".join(v.encode() if isinstance(v, str) else v for v in col.to_pylist() if v is not None)
        return {f"{name}.bytes": np.frombuffer(data, np.uint8).astype(np.float32), f"{name}.lengths": f64(pc.binary_length(col))}
    if pa.types.is_list(t) and not _is_bytes(t.value_type):
        return {f"{name}.values": f64(pc.cast(pc.list_flatten(col), pa.float64())), f"{name}.lengths": f64(pc.list_value_length(col))}
    if pa.types.is_integer(t) or pa.types.is_floating(t):
        return {name: f64(pc.cast(col, pa.float64()))}
    raise TypeError(f"column {name}: no float form for {t}")


def dump_outputs(out_dir: Path, kept, windows, prefix: str, budget: int) -> dict:
    """Writes the rows in `kept` (keep_window_rows, row order) as out_dir/<prefix><name>.npy: row_index.npy plus one file
    per column_arrays entry.  When they would exceed `budget` bytes, every window keeps the same number of leading rows."""
    out_dir.mkdir(parents=True, exist_ok=True)
    if not kept:
        np.save(out_dir / f"{prefix}row_index.npy", np.zeros(0, np.float64))
        return {"dir": str(out_dir), "rows": 0, "bytes": 0}
    t = pa.Table.from_batches([b for _, b in kept]).combine_chunks()
    index = np.concatenate([np.arange(lo, lo + b.num_rows) for lo, b in kept])
    lengths = lambda a: np.nan_to_num(np.asarray(a.to_numpy(zero_copy_only=False), dtype=np.float64))
    cost, files = np.full(t.num_rows, 8.0), 1       # bytes each row adds to the files: row_index, then per column
    for col in t.columns:
        cost += 8.0                                  # the value, or the length
        if _is_bytes(col.type):
            cost += 4.0 * lengths(pc.binary_length(col)); files += 2
        elif pa.types.is_list(col.type):
            cost += 8.0 * lengths(pc.list_value_length(col)); files += 2
        else:
            files += 1
    starts = np.array([lo for lo, _ in windows])
    offset = index - starts[np.searchsorted(starts, index, side="right") - 1]          # a row's place in its window
    cost_upto = np.cumsum(np.bincount(offset, weights=cost))
    per_window = int(np.searchsorted(cost_upto, budget - 128 * files, side="right"))   # 128: an .npy header
    sel = np.flatnonzero(offset < per_window)
    t = t.take(pa.array(sel))
    arrays = {"row_index": index[sel].astype(np.float64)}
    for name, col in zip(t.column_names, t.columns):
        arrays.update(column_arrays(name, col))
    total = 0
    for name, arr in arrays.items():
        path = out_dir / f"{prefix}{name}.npy"
        np.save(path, arr)
        total += path.stat().st_size
    return {"dir": str(out_dir), "rows": len(sel), "bytes": total}


def bai_linear_offsets(bai_path: Path):
    """Record-start virtual offsets from a BAI linear index (every ioffset is the start of a record)."""
    d = bai_path.read_bytes()
    assert d[:4] == b"BAI\1"
    n_ref = struct.unpack_from("<i", d, 4)[0]
    p = 8
    offs = set()
    for _ in range(n_ref):
        n_bin = struct.unpack_from("<i", d, p)[0]; p += 4
        for _ in range(n_bin):
            _bin, n_chunk = struct.unpack_from("<Ii", d, p); p += 8 + 16 * n_chunk
        n_intv = struct.unpack_from("<i", d, p)[0]; p += 4
        offs.update(struct.unpack_from(f"<{n_intv}Q", d, p)); p += 8 * n_intv
    offs.discard(0)
    return sorted(offs)


class ClockSampler:
    """Samples SM clock / throttle reasons DURING the timed region through in-process NVML (nvidia_ml_py): a polling
    nvidia-smi child perturbs short timed regions (its start-up alone costs hundreds of ms of driver time)."""

    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.sm, self.reasons, self.power = [], set(), []
        self.max_sm = None
        self._stop = threading.Event()
        self._thread = None
        self.h = None
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            idx = int(vis.split(",")[gpu_index]) if vis and vis.split(",")[gpu_index].isdigit() else gpu_index
            self.h = pynvml.nvmlDeviceGetHandleByIndex(idx)
            self.nv = pynvml
            self.max_sm = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception as e:   # pragma: no cover
            log(f"[bench] NVML unavailable ({e}); clocks not sampled")

    def _loop(self):
        nv = self.nv
        while not self._stop.is_set():
            try:
                self.sm.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h) if hasattr(nv, "nvmlDeviceGetCurrentClocksEventReasons") \
                    else nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in self.REASONS.items():
                    if r & bit:
                        self.reasons.add(name)
                self.power.append(nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0)
            except Exception:
                pass
            self._stop.wait(0.1)

    def start(self):
        if self.h is not None:
            self._thread = threading.Thread(target=self._loop, daemon=True)
            self._thread.start()

    def stop(self) -> dict:
        self._stop.set()
        if self._thread:
            self._thread.join(timeout=2)
        sm_load = sorted(self.sm)[len(self.sm) // 2:] if self.sm else []    # samples under load = upper half
        return {"sm_mhz": statistics.median(sm_load) if sm_load else None, "sm_max_mhz": self.max_sm,
                "reasons": sorted(self.reasons), "samples": len(self.sm), "power_w_max": max(self.power) if self.power else None}


def peaks():
    f = ROOT / "MEASURED_PEAKS.json"
    if f.exists():
        return float(json.loads(f.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


CONFIG_KEYS = ("workload", "reads", "projection", "tags", "partitioning", "sample_reads_per_step")


def make_config(reads, projection, partitioning, sample):
    return {"workload": f"synthetic {reads}-read 150bp WGS-like BAM (BGZF lvl 6, tools/bamgen.cpp seed 2)", "reads": reads,
            "projection": "all 12 core columns + tags" if projection is None else "chrom,start,end,mapping_quality,flags",
            "tags": TAGS if projection is None else [], "partitioning": partitioning, "sample_reads_per_step": sample}


def inflate_only_cpu(path, members=3000):
    """zlib raw inflate + crc32 of the first `members` BGZF members on one thread (BASELINE.md 4: the reference links libdeflate,
    which is ~2x faster than zlib and absent from this image)."""
    import zlib
    data = open(path, "rb").read(members * 30000)
    off, n, out_bytes = 0, 0, 0
    t0 = time.perf_counter()
    while off + 28 <= len(data) and n < members:
        bsize = struct.unpack_from("<H", data, off + 16)[0]
        xlen = struct.unpack_from("<H", data, off + 10)[0]
        if off + bsize + 1 > len(data):
            break
        payload = data[off + 12 + xlen: off + bsize + 1 - 8]
        raw = zlib.decompress(payload, -15)
        zlib.crc32(raw)
        out_bytes += len(raw); off += bsize + 1; n += 1
    dt = time.perf_counter() - t0
    return {"inflated_gbps": out_bytes / dt / 1e9, "members": n, "threads": 1, "library": "zlib (python binding)"}


def oracle_threads_scan(o, offs, total_reads, sample_reads, threads, steps=1, warmup=0):
    """`threads` block-range partitions of a bounded prefix, one sequential decode loop each (the reference's one-thread-per-
    partition model), batches of 8192 rows built and dropped."""
    frac = min(1.0, sample_reads / total_reads)
    hi = max(threads + 1, min(int(len(offs) * frac), len(offs) - 1))
    cuts = [o.first_record_voffset] + [offs[(hi * k) // threads] for k in range(1, threads)] + [offs[hi] if frac < 1.0 else 0]
    results = [None] * threads

    def work(i):
        _b, st = o.scan(None, start_voffset=cuts[i], stop_voffset=cuts[i + 1], batch_rows=8192, want_stats=True)
        results[i] = st

    def step():
        ths = [threading.Thread(target=work, args=(i,)) for i in range(threads)]
        t0 = time.perf_counter()
        for t in ths: t.start()
        for t in ths: t.join()
        return time.perf_counter() - t0, sum(r["rows"] for r in results), sum(r["inflated_bytes"] for r in results)

    for _ in range(warmup):
        step()
    tt, rows, infl = 0.0, 0, 0
    for _ in range(steps):
        dt, r, ib = step()
        tt += dt; rows += r; infl += ib
    return tt, rows, infl


def run_reference(args, path, info, rank, world):
    """The reference's CPU path, restated (oracle/): one sequential decode loop per partition, all host threads."""
    if rank != 0:
        return
    from oracle.bam_oracle import OracleBam
    cores = os.cpu_count() or 1
    offs = bai_linear_offsets(Path(str(path) + ".bai"))
    o = OracleBam(str(path), tag_fields=TAGS)
    total_reads = info["reads"]
    target = min(total_reads, int(os.environ.get("BAMSCAN_REF_SAMPLE_READS", 1_000_000 * cores)))
    tt, rows, infl = oracle_threads_scan(o, offs, total_reads, target, cores, args.steps, args.warmup)
    value = rows / tt
    per_step = rows // args.steps
    sample = f"first {per_step} reads of the {total_reads}-read file per step, {cores} block-range partitions seeded from BAI linear-index record starts, batches of 8192 rows built and dropped"
    line = {
        "impl": "reference", "metric": "bam_scan_reads_per_s", "value": value, "unit": "reads/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1000 * tt / args.steps, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "inflated_gbps": infl / tt / 1e9,
        "config": make_config(total_reads, None, f"{cores} block-range partitions on {cores} host threads", per_step),
        "note": "CPU restatement of the reference path (noodles + libdeflate are not buildable here; zlib inflate, ~2x slower than libdeflate); a bounded prefix per step",
        "cpu_baseline": {"value": value, "unit": "reads/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "reads/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def bind_to_gpu_numa(local):
    """Pins this rank's threads (and therefore its pinned-memory allocations) to the CPUs next to its GPU."""
    try:
        import pynvml
        pynvml.nvmlInit()
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        idx = int(vis.split(",")[local]) if vis and vis.split(",")[local].isdigit() else local
        bus = pynvml.nvmlDeviceGetPciInfo(pynvml.nvmlDeviceGetHandleByIndex(idx)).busId
        bus = (bus.decode() if isinstance(bus, bytes) else bus).lower()
        if len(bus.split(":")[0]) == 8:
            bus = bus[4:]
        cpus = Path(f"/sys/bus/pci/devices/{bus}/local_cpulist").read_text().strip()
        ids = set()
        for part in cpus.split(","):
            a, _, b = part.partition("-")
            ids.update(range(int(a), int(b or a) + 1))
        if ids:
            os.sched_setaffinity(0, ids)
            return cpus
    except Exception as e:   # pragma: no cover
        log(f"[bench] NUMA binding skipped ({e})")
    return None


def traffic_from_profile(kernel_sources):
    """DRAM bytes per launch of the dominant kernel from the committed ncu pass (tools/ncu_traffic.py), valid only for the
    kernel source it was taken on: a stale capture reads as null, never as a number."""
    import hashlib
    f = ROOT / "profiles" / "r2_inflate_traffic.json"
    if not f.exists():
        return None, "no ncu traffic capture committed (profiles/r2_inflate_traffic.json)"
    d = json.loads(f.read_text())
    h = hashlib.sha256(b"".join((PKG / "csrc" / k).read_bytes() for k in kernel_sources)).hexdigest()[:16]
    if d.get("source_sha") != h:
        return None, f"ncu capture is for kernel source {d.get('source_sha')}, tree has {h}: stale, not reported"
    return d, "ncu --set full, dram__bytes_read.sum + dram__bytes_write.sum per launch (tools/ncu_traffic.py)"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--reads", type=int, default=int(os.environ.get("BAMSCAN_BENCH_READS", 100_000_000)))
    ap.add_argument("--seed", type=int, default=2)
    ap.add_argument("--projection", default="full", choices=["full", "fixed"])
    ap.add_argument("--config", type=int, default=2, choices=[2, 3, 4, 5])
    ap.add_argument("--verify", action="store_true", help="(default at N = 1, config 2) compare the product path with the oracle outside the timed regions")
    ap.add_argument("--no-verify", action="store_true")
    ap.add_argument("--no-replicas", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", type=Path,
                    help="write a fixed, seeded row sample of the last timed end-to-end step's RecordBatches to DIR/<name>.npy")
    args = ap.parse_args()
    if args.config == 3:
        args.projection = "fixed"

    rank = int(os.environ.get("RANK", 0)); world = int(os.environ.get("WORLD_SIZE", 1)); local = int(os.environ.get("LOCAL_RANK", 0))

    if args.impl == "reference":
        if rank == 0:
            path, info = ensure_bam(args.reads, args.seed, True)
            run_reference(args, path, info, rank, world)
        return

    numa = bind_to_gpu_numa(local) if world > 1 else None
    import torch
    dist = None
    if world > 1:
        import torch.distributed as dist
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    else:
        torch.cuda.set_device(local)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def all_max(x):
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        if dist is not None:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def all_sum(x):
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        if dist is not None:
            dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    def gather(obj):
        if dist is None:
            return [obj]
        out = [None] * world
        dist.all_gather_object(out, obj)
        return out

    long_reads = args.config == 5
    if long_reads:
        args.reads = min(args.reads, int(os.environ.get("BAMSCAN_BENCH_LONG_READS", 1_000_000)))
    if rank == 0:
        path, info = ensure_bam(args.reads, args.seed if not long_reads else 5, True, mode="long" if long_reads else "short")
    barrier()
    if rank != 0:
        path, info = ensure_bam(args.reads, args.seed if not long_reads else 5, True, mode="long" if long_reads else "short")

    import bamscan
    tags = TAGS if not long_reads else ["NM", "MD", "MM", "ML"]
    t_open = time.time()
    provider = bamscan.BamTableProvider(str(path), None, True, tags, False, True, 100, None, device_id=local,
                                        index_path=None if args.config == 4 else "",
                                        debug_flags=int(os.environ.get("BAMSCAN_DEBUG_FLAGS", "0")))   # (A/B runs of the profiles; default 0 = product path)
    projection = None if args.projection == "full" else [1, 2, 3, 6, 4]
    filters = [("chrom", "=", ["chr1"]), ("start", "between", [50_000_000, 150_000_000])] if args.config == 4 else []
    if args.config == 4:
        plan = provider.scan(projection, filters, None, target_partitions=world)          # balance_partitions regions, one per GPU
        partitioning = f"BAI region query chr1:50000000-150000000, {plan.output_partition_count()} balance_partitions regions over {world} GPU(s)"
    else:
        # block_range with N partitions: rank r owns the records that start in its block range (N = 1: the reference's sequential scan)
        plan = provider.scan(projection, [], None, target_partitions=world, partition_mode="block_range")
        partitioning = f"{world} BGZF block-range partition(s) of one file, one per GPU"
    n_parts = plan.output_partition_count()
    my_parts = [p for p in range(n_parts) if p % world == rank]
    log(f"[bench r{rank}] open+plan {time.time() - t_open:.1f}s, partitions {my_parts} of {n_parts}, numa cpus {numa}")

    def dev_pass(repeats):
        tot = None
        for p in my_parts:
            st = plan.run_device_resident(p, repeats)
            if tot is None:
                tot = dict(st)
            else:
                for k, v in st.items():
                    tot[k] = tot[k] + v
        return tot or {"rows": 0, "ms_total": 0.0, "ms_inflate": 0.0, "ms_boundary": 0.0, "ms_decode": 0.0, "chunks": 0, "compressed_bytes": 0,
                       "inflated_bytes": 0, "arrow_bytes": 0, "kernel_launches": 0, "boundary_repairs": 0, "boundary_seam_mismatches": 0, "blocks": 0}

    # ---------------- device-resident value ----------------
    if args.warmup > 0:
        dev_pass(args.warmup)
    sampler = ClockSampler(local)
    sampler.start()
    barrier()
    t0 = time.perf_counter()
    st = dev_pass(args.steps)
    barrier()
    wall_dev = time.perf_counter() - t0
    clocks = sampler.stop()
    dev_s_max = all_max(st["ms_total"] / 1000.0 * args.steps)
    rows_all = int(all_sum(st["rows"]))
    value = rows_all * args.steps / dev_s_max
    per_rank = gather({"rank": rank, "rows": st["rows"], "ms_per_step": st["ms_total"], "ms_inflate": st["ms_inflate"], "ms_boundary": st["ms_boundary"],
                       "ms_decode": st["ms_decode"], "chunks": st["chunks"], "members": st["blocks"], "boundary_repairs": st["boundary_repairs"],
                       "seam_mismatches": st["boundary_seam_mismatches"], "first_record": "exact (header end)" if rank == 0 else "speculated",
                       "last_chunk_members": st["blocks"] % 22496 if st["chunks"] else 0, "kernel_launches": st["kernel_launches"],
                       "first_record_uoff": st.get("first_record_uoff", 0), "end_chain_uoff": st.get("end_chain_uoff", 0)})

    # ---------------- end to end through the provider API ----------------
    def e2e_step(windows=None, kept=None):
        n = 0
        for p in my_parts:
            for b in plan.execute(p):
                if windows:
                    keep_window_rows(b, n, windows, kept)    # a batch is a whole inflate wave (GBs): copy the rows, not it
                n += b.num_rows
                del b
        return n

    for _ in range(max(1, args.warmup)):   # warm-up: the pinned arena pool settles after a few scans
        step_rows = e2e_step()
    windows = dump_windows(step_rows) if args.dump_outputs else None
    kept = []
    barrier()
    t0 = time.perf_counter()
    e2e_rows = 0
    for i in range(args.steps):
        e2e_rows += e2e_step(windows if i == args.steps - 1 else None, kept)
    barrier()
    e2e_s = all_max(time.perf_counter() - t0)
    dumped = None
    if args.dump_outputs:
        prefix = f"rank{rank}." if world > 1 else ""
        dumped = dump_outputs(args.dump_outputs, kept, windows, prefix, DUMP_BYTES // world)
        log(f"[bench r{rank}] wrote {dumped['rows']} sampled rows of {step_rows} ({dumped['bytes']} bytes) to {args.dump_outputs}")
    est = plan.last_stats if my_parts else {"h2d_bytes": 0, "d2h_bytes": 0}
    e2e_value = all_sum(e2e_rows) / e2e_s
    h2d_all, d2h_all = all_sum(est["h2d_bytes"]), all_sum(est["d2h_bytes"])

    # ---------------- round-1 number beside it: every rank scans a whole copy ----------------
    replicas = None
    if world > 1 and not args.no_replicas and args.config in (2, 3):
        rplan = provider.scan(projection, [], None, target_partitions=1, partition_mode="block_range")
        rplan.run_device_resident(0, 1)
        barrier()
        rst = rplan.run_device_resident(0, 2)
        barrier()
        r_s = all_max(rst["ms_total"] / 1000.0 * 2)
        replicas = {"value": world * rst["rows"] * 2 / r_s, "unit": "reads/s", "note": "every rank scans one whole copy of the file (weak scaling, what round 1 reported)"}

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return

    if args.config != 4 and world > 1:
        # every partition must start where its predecessor's record chain landed: the speculated starts are proven, or the run fails
        bamscan.check_partition_seams([dict(rows=r["rows"], first_record_uoff=r["first_record_uoff"], end_chain_uoff=r["end_chain_uoff"]) for r in per_rank])
    peak, peak_src = peaks()
    launches_inflate = max(1, st["chunks"])
    infl_alg = st["compressed_bytes"] + st["inflated_bytes"]
    infl_gbs = infl_alg / (st["ms_inflate"] / 1000.0) / 1e9 if st["ms_inflate"] > 0 else 0.0
    scan_alg = st["inflated_bytes"] + st["arrow_bytes"]
    tr, tr_note = traffic_from_profile(["kernels_inflate.cuh", "kernels_inflate_cta.cuh", "inflate_cta_core.h"])
    # the same kernel timed ALONE on the first chunk of rank 0's partition (in the scan the next chunk's inflate overlaps this
    # chunk's decode kernels, so its in-pipeline duration includes what it loses to them)
    alone = None
    if my_parts and not long_reads:
        try:
            bi = plan.bench_inflate(my_parts[0], 3)
            ab = bi["inflated_bytes"] + bi["compressed_bytes"]
            alone = {"ms_per_launch": bi["ms_per_launch"], "alg_bytes_per_launch": ab, "achieved": ab / (bi["ms_per_launch"] / 1e3) / 1e9,
                     "frac": ab / (bi["ms_per_launch"] / 1e3) / 1e9 / peak, "inflated_gbps": bi["inflated_bytes"] / (bi["ms_per_launch"] / 1e3) / 1e9,
                     "note": "first chunk of rank 0's partition, 3 launches after one warm-up, nothing else on the GPU"}
        except Exception as e:      # the scan numbers stand without it
            alone = {"error": str(e)}
    line = {
        "metric": "bam_scan_reads_per_s", "value": value, "unit": "reads/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1000 * dev_s_max / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "u8", "data": "synthetic",
        "config": make_config(info["reads"], projection, partitioning, rows_all) if not long_reads else
        {"workload": f"synthetic {info['reads']}-read long-read BAM (10 kb, long CIGARs, MM/ML), tools/bamgen.cpp seed 5", "reads": info["reads"],
         "projection": "all 12 core columns + tags", "tags": tags, "partitioning": partitioning, "sample_reads_per_step": rows_all},
        "bytes_rank0": {"compressed": st["compressed_bytes"], "inflated": st["inflated_bytes"], "arrow": st["arrow_bytes"],
                        "l2": "inputs (>= 10x L2) stream from HBM; no reuse between steps"},
        "inflated_gbps": info["inflated_bytes"] * (rows_all / max(1, info["reads"])) * args.steps / dev_s_max / 1e9,
        "scan_roofline_frac_rank0": (scan_alg / (st["ms_total"] / 1000.0) / 1e9) / peak if st["ms_total"] else None,
        "stage_ms_rank0": {"inflate": st["ms_inflate"], "boundary": st["ms_boundary"], "decode": st["ms_decode"], "total": st["ms_total"]},
        "roofline": {"kernel": "inflate stage of rank 0: inflate_cta_kernel (CTA per BGZF member, CRC-32 fused) on every chunk; event bracket around the launch",
                     "bound": "hbm", "achieved": infl_gbs, "peak": peak, "unit": "GB/s", "frac": infl_gbs / peak,
                     "traffic": (tr["dram_bytes_per_launch"] if tr else None), "traffic_note": tr_note,
                     "peak_source": peak_src, "launches": launches_inflate,
                     "alg_bytes_per_launch": infl_alg / launches_inflate, "ms_per_launch": st["ms_inflate"] / launches_inflate,
                     "kernel_alone": alone},
        "e2e": {"value": e2e_value, "unit": "reads/s", "h2d_bytes_per_step": int(h2d_all), "d2h_bytes_per_step": int(d2h_all),
                "ms_per_step": 1000 * e2e_s / args.steps, "d2h_gbps_aggregate": d2h_all / (e2e_s / args.steps) / 1e9},
        "gpu_launches": int(sum(r["kernel_launches"] for r in per_rank) * args.steps),
        "per_rank": per_rank,
        "clocks": clocks, "wall_s_device_region": wall_dev,
    }
    if replicas:
        line["replicas"] = replicas
    if dumped:
        line["dump_outputs"] = dumped
    if world == 1 and args.config == 2:
        # CPU baseline beside it (bounded samples): the oracle port on all host threads, on one thread, and inflate alone
        from oracle.bam_oracle import OracleBam
        o = OracleBam(str(path), tag_fields=TAGS)
        cores = os.cpu_count() or 1
        offs = bai_linear_offsets(Path(str(path) + ".bai"))
        n_all = min(info["reads"], int(os.environ.get("BAMSCAN_CPU_SAMPLE_READS", 500_000 * cores)))
        tt, r_all, ib = oracle_threads_scan(o, offs, info["reads"], n_all, cores)
        n_one = min(info["reads"], 2_000_000)
        t0 = time.perf_counter()
        cst = o.time_scan(None, max_records=n_one, batch_rows=8192)
        dt = time.perf_counter() - t0
        line["cpu_baseline"] = {"value": r_all / tt, "unit": "reads/s", "cores": cores, "kind": "port",
                                "sample": f"first {r_all} reads as {cores} block-range partitions on {cores} threads; zlib inflate + crc32, batches of 8192 built and dropped",
                                "inflated_gbps": ib / tt / 1e9,
                                "one_thread": {"value": cst["rows"] / dt, "unit": "reads/s", "cores": 1, "sample": f"first {cst['rows']} reads, one sequential loop",
                                               "inflated_gbps": cst["inflated_bytes"] / dt / 1e9},
                                "inflate_only": inflate_only_cpu(path)}
    if (args.verify or (world == 1 and args.config == 2)) and not args.no_verify:
        # parity at the benchmarked shape, outside every timed region: the DEFAULT product path (no chunk cap, no forced kernels,
        # >= 2 full inflate launches) over a <= 10 M-read file of the same generator against the oracle on all host threads
        t_v = time.time()
        try:
            from oracle.bam_oracle import OracleBam
            from oracle.verify import verify_full_scan
            vreads = min(args.reads, int(os.environ.get("BAMSCAN_VERIFY_READS", 10_000_000)))
            vpath, _vinfo = ensure_bam(vreads, args.seed, True)
            vp = bamscan.BamTableProvider(str(vpath), None, True, TAGS, False, True, 100, None, device_id=local, index_path="")
            vo = OracleBam(str(vpath), tag_fields=TAGS)
            rep = verify_full_scan(vo, str(vpath) + ".bai", vp.scan(None, [], None).execute(0), n_parts=max(8, vreads // 1_000_000), threads=os.cpu_count())
            rep.pop("checksums", None)
            rep["result"] = "bit-exact: per-column checksums over every row + RecordBatch equality on 3 windows"
        except Exception as e:      # a parity failure must show up IN the line, not instead of it
            rep = {"result": f"FAILED: {type(e).__name__}: {e}"[:500]}
        rep["seconds"] = round(time.time() - t_v, 1)
        line["verify"] = rep
    if world == 1 and args.config == 2 and not args.no_verify:
        # SURVEY 8 f4 beside it (outside every timed region of the scan): the first ~4 M rows of the verify file go back out through
        # bamscan_writer_* (Arrow -> BAM records -> BGZF members compressed on the GPU), and the GPU scan reads the file back
        try:
            import pyarrow as pa
            wreads = min(args.reads, int(os.environ.get("BAMSCAN_VERIFY_READS", 10_000_000)))
            wpath, winfo = ensure_bam(wreads, args.seed, True)
            wp = bamscan.BamTableProvider(str(wpath), None, True, TAGS, False, True, 100, None, device_id=local, index_path="")
            batches, nrows = [], 0
            for b in wp.scan(None, [], None).execute(0):
                batches.append(b); nrows += b.num_rows
                if nrows >= 4_000_000:
                    break
            out = wpath.parent / "bench_written.bam"
            best = None
            for _ in range(2):
                ex = bamscan.BamWriteExec(str(out), wp.schema(), TAGS, True, {"bio.bam.sort_order": "unsorted"}, device_id=local)
                t0 = time.perf_counter()
                n = ex.execute(batches)
                dt = time.perf_counter() - t0
                if best is None or dt < best[0]:
                    best = (dt, ex.stats)
            dt, wst = best
            rp = bamscan.BamTableProvider(str(out), None, True, TAGS, False, True, 100, None, device_id=local, index_path="")
            back = pa.Table.from_batches(list(rp.scan(None, [], None).execute(0)))
            want = pa.Table.from_batches(batches)
            same = back.num_rows == want.num_rows and all(back.column(i).combine_chunks().equals(want.column(i).combine_chunks()) for i in range(want.num_columns))
            line["write_path"] = {"rows": n, "e2e_reads_per_s": n / dt, "device_reads_per_s": n / (wst["ms_total"] / 1e3), "encode_ms": wst["ms_encode"], "deflate_ms": wst["ms_deflate"],
                                  "arrow_bytes_h2d": wst["arrow_bytes"], "bam_stream_bytes": wst["bam_bytes"], "file_bytes": wst["compressed_bytes"], "members": wst["members"],
                                  "compression_ratio": wst["bam_bytes"] / max(1, wst["compressed_bytes"]), "kernel_launches": wst["kernel_launches"],
                                  "read_back": "equal to the batches written (GPU scan of the written file, every column)" if same else "DIFFERS",
                                  "note": "bamscan_writer_* (INSERT OVERWRITE): enc_size / enc_records / bgzf_deflate kernels; best of 2; file on tmpfs"}
            out.unlink(missing_ok=True)
        except Exception as e:
            line["write_path"] = {"error": f"{type(e).__name__}: {e}"[:300]}
    print(json.dumps(line), flush=True)
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
