"""bamscan -- python host mirror of the reference's BAM table provider over the C ABI (include/bamscan.h).

Mirrors, name for name, the interface DataFusion drives in the reference
(datafusion/bio-format-bam/src/table_provider.rs:314-335, 381-390, 928-1115; physical_exec.rs:84-173):

    provider = BamTableProvider(file_path, None, coordinate_system_zero_based, tag_fields, binary_cigar,
                                infer_tag_types, infer_tag_sample_size, tag_type_hints)
    provider.schema()                                  -> pyarrow.Schema
    provider.supports_filters_pushdown(filters)        -> ["Inexact" | "Unsupported", ...]
    plan = provider.scan(projection, filters, limit, target_partitions=...)   -> BamExec
    plan.output_partition_count()
    for batch in plan.execute(partition): ...          -> pyarrow.RecordBatch

Everything below the method signatures is libbamscan.so (CUDA, sm_100a).  There is no CPU path: importing works
anywhere (so CPU-only CI can check symbols), but opening a file without a GPU raises BamScanError.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

import pyarrow as pa

_HERE = Path(__file__).resolve().parent
LIB_PATH = _HERE.parent / "libbamscan.so"

EXPORTED_SYMBOLS = [
    "bamscan_open", "bamscan_open_fastq", "bamscan_open_fasta", "bamscan_close", "bamscan_schema", "bamscan_describe_tags", "bamscan_classify_filters", "bamscan_plan",
    "bamscan_plan_num_partitions", "bamscan_plan_schema", "bamscan_plan_free", "bamscan_plan_num_ranges",
    "bamscan_plan_range_info", "bamscan_plan_partition_regions", "bamscan_extract_regions", "bamscan_balance_partitions",
    "bamscan_execute", "bamscan_next", "bamscan_execute_device", "bamscan_next_device",
    "bamscan_stream_free", "bamscan_run_device_resident", "bamscan_stream_stats", "bamscan_bench_inflate",
    "bamscan_probe_pcie", "bamscan_check_partition_seams", "bamscan_last_error", "bamscan_version",
    "bamscan_writer_open", "bamscan_writer_write", "bamscan_writer_write_device", "bamscan_writer_finish", "bamscan_writer_stats", "bamscan_writer_free",
    "bamscan_fastq_writer_open", "bamscan_sam_writer_open",
]


class BamScanError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"[{code}] {msg}")
        self.code = code


class _Options(C.Structure):
    _fields_ = [("struct_size", C.c_uint32), ("coordinate_system_zero_based", C.c_int32), ("binary_cigar", C.c_int32),
                ("has_tag_fields", C.c_int32), ("n_tag_fields", C.c_int32), ("tag_fields", C.POINTER(C.c_char_p)),
                ("infer_tag_types", C.c_int32), ("infer_tag_sample_size", C.c_int32),
                ("n_tag_type_hints", C.c_int32), ("tag_type_hints", C.POINTER(C.c_char_p)),
                ("device_id", C.c_int32), ("batch_rows", C.c_int32), ("chunk_inflated_bytes", C.c_uint64),
                ("segment_bytes", C.c_uint32), ("skip_crc", C.c_int32), ("debug_flags", C.c_int32), ("decode_all_tag_fields", C.c_int32)]


class _Filter(C.Structure):
    _fields_ = [("column", C.c_int32), ("op", C.c_int32), ("n_values", C.c_int32),
                ("num_values", C.POINTER(C.c_double)), ("str_values", C.POINTER(C.c_char_p))]


class RegionAnalysis(C.Structure):
    _fields_ = [("unsatisfiable", C.c_int32), ("has_start", C.c_int32), ("has_end", C.c_int32), ("n_chroms", C.c_int32),
                ("start", C.c_uint64), ("end", C.c_uint64), ("residual_mask", C.c_uint64), ("chroms", C.c_ubyte * 4096)]


class RegionEstimate(C.Structure):
    _fields_ = [("chrom", C.c_char_p), ("has_start", C.c_int32), ("has_end", C.c_int32), ("start", C.c_uint64), ("end", C.c_uint64),
                ("estimated_bytes", C.c_uint64), ("contig_length", C.c_uint64), ("unmapped_count", C.c_uint64),
                ("nonempty_bin_positions", C.POINTER(C.c_uint64)), ("n_bin_positions", C.c_int32), ("leaf_bin_span", C.c_uint64)]


class AssignedRegion(C.Structure):
    _fields_ = [("partition", C.c_int32), ("estimate_index", C.c_int32), ("has_start", C.c_int32), ("has_end", C.c_int32),
                ("start", C.c_uint64), ("end", C.c_uint64), ("unmapped_tail", C.c_int32), ("partition_total_estimated_bytes", C.c_uint64)]


class Stats(C.Structure):
    _fields_ = [("rows", C.c_uint64), ("batches", C.c_uint64), ("chunks", C.c_uint64),
                ("compressed_bytes", C.c_uint64), ("inflated_bytes", C.c_uint64), ("arrow_bytes", C.c_uint64),
                ("h2d_bytes", C.c_uint64), ("d2h_bytes", C.c_uint64),
                ("blocks", C.c_uint64), ("kernel_launches", C.c_uint64), ("boundary_repairs", C.c_uint64),
                ("ms_total", C.c_double), ("ms_inflate", C.c_double), ("ms_boundary", C.c_double), ("ms_decode", C.c_double),
                ("boundary_seam_mismatches", C.c_uint64), ("first_record_uoff", C.c_uint64), ("end_chain_uoff", C.c_uint64),
                ("inflate_retries", C.c_uint64)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


class _WriteOptions(C.Structure):
    _fields_ = [("struct_size", C.c_uint32), ("coordinate_system_zero_based", C.c_int32), ("n_tag_fields", C.c_int32),
                ("tag_fields", C.POINTER(C.c_char_p)), ("device_id", C.c_int32), ("compression", C.c_int32)]


class WriteStats(C.Structure):
    _fields_ = [("rows", C.c_uint64), ("batches", C.c_uint64), ("members", C.c_uint64), ("arrow_bytes", C.c_uint64),
                ("bam_bytes", C.c_uint64), ("compressed_bytes", C.c_uint64), ("ms_encode", C.c_double), ("ms_deflate", C.c_double),
                ("ms_total", C.c_double), ("kernel_launches", C.c_uint64)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


_OPS = {"=": 0, "==": 0, "!=": 1, "<": 2, "<=": 3, ">": 4, ">=": 5, "between": 6, "not_between": 7, "in": 8, "not_in": 9,
        "other": 100}
CORE_COLUMNS = ["name", "chrom", "start", "end", "flags", "cigar", "mapping_quality", "mate_chrom", "mate_start",
                "sequence", "quality_scores", "template_length"]

_lib = None


def load_library():
    """Loads libbamscan.so; fails loudly when the CUDA extension has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise BamScanError(-4, f"{LIB_PATH} is missing: build it with `make -C {LIB_PATH.parent / 'csrc'}` "
                               "(there is no CPU fallback)")
    L = C.CDLL(str(LIB_PATH))
    L.bamscan_last_error.restype = C.c_char_p
    L.bamscan_version.restype = C.c_char_p
    L.bamscan_open.argtypes = [C.c_char_p, C.c_char_p, C.POINTER(_Options), C.POINTER(C.c_void_p)]
    L.bamscan_open_fastq.argtypes = [C.c_char_p, C.POINTER(_Options), C.POINTER(C.c_void_p)]
    L.bamscan_open_fasta.argtypes = [C.c_char_p, C.POINTER(_Options), C.POINTER(C.c_void_p)]
    L.bamscan_close.argtypes = [C.c_void_p]
    L.bamscan_schema.argtypes = [C.c_void_p, C.c_void_p]
    L.bamscan_describe_tags.argtypes = [C.c_void_p, C.c_int32, C.c_char_p, C.c_uint64, C.POINTER(C.c_uint64)]
    L.bamscan_classify_filters.argtypes = [C.c_void_p, C.POINTER(_Filter), C.c_int32, C.POINTER(C.c_uint8)]
    L.bamscan_plan.argtypes = [C.c_void_p, C.POINTER(C.c_int32), C.c_int32, C.POINTER(_Filter), C.c_int32, C.c_int64,
                               C.c_int32, C.c_int32, C.POINTER(C.c_void_p)]
    L.bamscan_plan_num_partitions.argtypes = [C.c_void_p]
    L.bamscan_plan_schema.argtypes = [C.c_void_p, C.c_void_p]
    L.bamscan_plan_free.argtypes = [C.c_void_p]
    L.bamscan_plan_num_ranges.argtypes = [C.c_void_p, C.c_int32]
    L.bamscan_plan_range_info.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.POINTER(C.c_uint64)]
    L.bamscan_plan_partition_regions.argtypes = [C.c_void_p, C.c_int32, C.POINTER(AssignedRegion), C.c_int32]
    L.bamscan_extract_regions.argtypes = [C.POINTER(_Filter), C.c_int32, C.c_int32, C.POINTER(RegionAnalysis)]
    L.bamscan_balance_partitions.argtypes = [C.POINTER(RegionEstimate), C.c_int32, C.c_int32, C.POINTER(AssignedRegion), C.c_int32,
                                             C.POINTER(C.c_int32), C.POINTER(C.c_int32)]
    L.bamscan_execute.argtypes = [C.c_void_p, C.c_int32, C.POINTER(C.c_void_p)]
    L.bamscan_next.argtypes = [C.c_void_p, C.c_void_p]
    L.bamscan_stream_free.argtypes = [C.c_void_p]
    L.bamscan_run_device_resident.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.POINTER(Stats)]
    L.bamscan_stream_stats.argtypes = [C.c_void_p, C.POINTER(Stats)]
    L.bamscan_bench_inflate.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.POINTER(C.c_double), C.POINTER(C.c_uint64),
                                        C.POINTER(C.c_uint64)]
    L.bamscan_probe_pcie.argtypes = [C.c_int32, C.c_uint64, C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_double)]
    L.bamscan_writer_open.argtypes = [C.c_char_p, C.c_char_p, C.c_int32, C.POINTER(C.c_char_p), C.POINTER(C.c_int32), C.c_void_p,
                                      C.POINTER(_WriteOptions), C.POINTER(C.c_void_p)]
    L.bamscan_writer_write.argtypes = [C.c_void_p, C.c_void_p]
    L.bamscan_writer_write_device.argtypes = [C.c_void_p, C.c_void_p]
    L.bamscan_writer_finish.argtypes = [C.c_void_p, C.POINTER(C.c_uint64)]
    L.bamscan_writer_stats.argtypes = [C.c_void_p, C.POINTER(WriteStats)]
    L.bamscan_writer_free.argtypes = [C.c_void_p]
    L.bamscan_fastq_writer_open.argtypes = [C.c_char_p, C.c_void_p, C.POINTER(_WriteOptions), C.POINTER(C.c_void_p)]
    L.bamscan_sam_writer_open.argtypes = L.bamscan_writer_open.argtypes
    _lib = L
    return L


def _check(rc):
    if rc < 0:
        raise BamScanError(rc, load_library().bamscan_last_error().decode("utf-8", "replace"))
    return rc


def _strs(values):
    if not values:
        return None, []
    enc = [v.encode() for v in values]
    return (C.c_char_p * len(enc))(*enc), enc


class _FilterPack:
    """Converts [(column, op, values)] into BamScanFilter[]; column is a name or a schema index."""

    def __init__(self, filters, schema_names):
        self.keep = []
        filters = filters or []
        self.n = len(filters)
        self.arr = (_Filter * max(1, self.n))()
        for i, (col, op, vals) in enumerate(filters):
            idx = schema_names.index(col) if isinstance(col, str) and col in schema_names else (col if isinstance(col, int) else -1)
            self.arr[i].column = idx
            self.arr[i].op = _OPS[op]
            vals = list(vals) if isinstance(vals, (list, tuple)) else [vals]
            self.arr[i].n_values = len(vals)
            if vals and all(isinstance(v, str) for v in vals):
                a, enc = _strs(vals)
                self.keep += [a, enc]
                self.arr[i].str_values = a
            elif vals:
                a = (C.c_double * len(vals))(*[float(v) for v in vals])
                self.keep.append(a)
                self.arr[i].num_values = a


class BamExec:
    """== BamExec : ExecutionPlan (physical_exec.rs:39-173)."""

    def __init__(self, provider, handle):
        self._provider = provider
        self._h = handle

    def __del__(self):
        try:
            if self._h:
                load_library().bamscan_plan_free(self._h)
                self._h = None
        except Exception:
            pass

    def output_partition_count(self) -> int:
        return load_library().bamscan_plan_num_partitions(self._h)

    def partition_ranges(self, partition: int):
        """Block ranges (+ row rule) a partition scans: list of dicts (bamscan_plan_range_info)."""
        L = load_library()
        keys = ["block_begin", "block_end", "coff_begin", "coff_end", "exact_start", "first_uoff", "stop_uoff",
                "region_mode", "region_ref", "region_start", "region_end", "estimated_bytes", "start_voffset", "stop_voffset"]
        out = []
        for r in range(L.bamscan_plan_num_ranges(self._h, partition)):
            buf = (C.c_uint64 * 14)()
            _check(L.bamscan_plan_range_info(self._h, partition, r, buf))
            d = dict(zip(keys, list(buf)))
            d["region_ref"] = C.c_int64(d["region_ref"]).value
            out.append(d)
        return out

    def partition_regions(self, partition: int):
        """GenomicRegions assigned to a partition (PartitionAssignment::regions): list of dicts."""
        L = load_library()
        n = L.bamscan_plan_partition_regions(self._h, partition, None, 0)
        arr = (AssignedRegion * max(1, n))()
        L.bamscan_plan_partition_regions(self._h, partition, arr, n)
        return [dict(ref=a.estimate_index, start=a.start if a.has_start else None, end=a.end if a.has_end else None,
                     unmapped_tail=bool(a.unmapped_tail), estimated_bytes=a.partition_total_estimated_bytes) for a in arr[:n]]

    def schema(self) -> pa.Schema:
        cs = _ArrowSchemaStruct()
        _check(load_library().bamscan_plan_schema(self._h, C.byref(cs)))
        return pa.Schema._import_from_c(C.addressof(cs))

    def execute(self, partition: int):
        """Generator of pyarrow.RecordBatch for one partition (== execute(partition) + poll_next)."""
        L = load_library()
        schema = self.schema()
        st = C.c_void_p()
        _check(L.bamscan_execute(self._h, partition, C.byref(st)))
        try:
            while True:
                arr = _ArrowArrayStruct()
                rc = _check(L.bamscan_next(st, C.byref(arr)))
                if rc == 0:
                    break
                if len(schema) == 0:
                    sa = pa.Array._import_from_c(C.addressof(arr), pa.struct([]))
                    yield pa.RecordBatch.from_struct_array(sa)   # zero columns, row count kept (alignment_utils.rs:360-363)
                else:
                    yield pa.RecordBatch._import_from_c(C.addressof(arr), schema)
            s = Stats()
            L.bamscan_stream_stats(st, C.byref(s))
            self.last_stats = s.as_dict()
        finally:
            L.bamscan_stream_free(st)

    def execute_device(self, partition: int):
        """Generator of DeviceBatch for one partition: the batch stays in HBM (Arrow C Device Data Interface, SURVEY 8 f2)."""
        L = load_library()
        schema = self.schema()
        st = C.c_void_p()
        _check(L.bamscan_execute_device(self._h, partition, C.byref(st)))
        try:
            while True:
                dev = ArrowDeviceArrayStruct()
                rc = _check(L.bamscan_next_device(st, C.byref(dev)))
                if rc == 0:
                    break
                yield DeviceBatch(dev, schema)
            s = Stats()
            L.bamscan_stream_stats(st, C.byref(s))
            self.last_stats = s.as_dict()
        finally:
            L.bamscan_stream_free(st)

    def collect(self) -> pa.Table:
        """All partitions in partition order (CoalescePartitionsExec over the leaf).  Block-range partitions > 0 speculate
        their first record: the seams are checked (each partition must start where its predecessor's chain landed)."""
        schema = self.schema()
        batches = []
        stats = []
        for p in range(self.output_partition_count()):
            batches += list(self.execute(p))
            stats.append(self.last_stats)
        if len(stats) > 1 and all(len(self.partition_ranges(p)) == 1 and self.partition_ranges(p)[0]["region_mode"] == 0 for p in range(len(stats))):
            check_partition_seams(stats)
        if len(schema) == 0:
            return batches
        return pa.Table.from_batches(batches, schema=schema)

    def run_device_resident(self, partition=0, repeats=1) -> dict:
        s = Stats()
        _check(load_library().bamscan_run_device_resident(self._h, partition, repeats, C.byref(s)))
        return s.as_dict()

    def bench_inflate(self, partition=0, repeats=10) -> dict:
        ms = C.c_double(); ib = C.c_uint64(); cb = C.c_uint64()
        _check(load_library().bamscan_bench_inflate(self._h, partition, repeats, C.byref(ms), C.byref(ib), C.byref(cb)))
        return {"ms_per_launch": ms.value, "inflated_bytes": ib.value, "compressed_bytes": cb.value}


class _ArrowSchemaStruct(C.Structure):
    _fields_ = [("format", C.c_char_p), ("name", C.c_char_p), ("metadata", C.c_void_p), ("flags", C.c_int64),
                ("n_children", C.c_int64), ("children", C.c_void_p), ("dictionary", C.c_void_p), ("release", C.c_void_p),
                ("private_data", C.c_void_p)]


class _ArrowArrayStruct(C.Structure):
    _fields_ = [("length", C.c_int64), ("null_count", C.c_int64), ("offset", C.c_int64), ("n_buffers", C.c_int64),
                ("n_children", C.c_int64), ("buffers", C.c_void_p), ("children", C.c_void_p), ("dictionary", C.c_void_p),
                ("release", C.c_void_p), ("private_data", C.c_void_p)]


class ArrowDeviceArrayStruct(C.Structure):
    _fields_ = [("array", _ArrowArrayStruct), ("device_id", C.c_int64), ("device_type", C.c_int32), ("sync_event", C.c_void_p),
                ("reserved", C.c_int64 * 3)]


ARROW_DEVICE_CUDA = 2
_cudart = None


def _cuda_memcpy_d2h(dst_addr: int, src_addr: int, n: int):
    """cudaMemcpy(dst, src, n, DeviceToHost) through libcudart (tests / debugging of the device hand-off only)."""
    global _cudart
    if _cudart is None:
        import glob
        cands = glob.glob("/usr/local/cuda/lib64/libcudart.so*")
        try:
            import torch
            cands += glob.glob(os.path.join(os.path.dirname(torch.__file__), "lib", "libcudart*.so*"))
            cands += glob.glob(os.path.join(os.path.dirname(os.path.dirname(torch.__file__)), "nvidia", "cuda_runtime", "lib", "libcudart.so*"))
        except Exception:
            pass
        if not cands:
            raise RuntimeError("libcudart not found")
        _cudart = C.CDLL(sorted(cands)[-1])
        _cudart.cudaMemcpy.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_int]
        _cudart.cudaDeviceSynchronize.argtypes = []
    if n:
        rc = _cudart.cudaMemcpy(dst_addr, src_addr, n, 2)
        if rc != 0:
            raise RuntimeError(f"cudaMemcpy D2H failed ({rc})")


class DeviceBatch:
    """One batch in HBM: an ArrowDeviceArray (device_type CUDA) plus the projected schema.  `release()` (or garbage collection)
    returns the device allocation to the engine; `to_host()` copies it back as a pyarrow.RecordBatch (tests, debugging)."""

    def __init__(self, dev: ArrowDeviceArrayStruct, schema: pa.Schema):
        self._dev = dev
        self.schema = schema
        self.num_rows = dev.array.length
        self.device_id = dev.device_id
        self.device_type = dev.device_type

    def release(self):
        a = self._dev.array
        if a.release:
            C.CFUNCTYPE(None, C.POINTER(_ArrowArrayStruct))(a.release)(C.byref(a))

    def __del__(self):
        try:
            self.release()
        except Exception:
            pass

    @staticmethod
    def _host(addr, nbytes):
        import numpy as np
        buf = np.empty(max(1, nbytes), dtype=np.uint8)
        _cuda_memcpy_d2h(buf.ctypes.data, addr, nbytes)
        return pa.py_buffer(buf[:nbytes].tobytes())

    def _child(self, node: _ArrowArrayStruct, typ: pa.DataType) -> pa.Array:
        import numpy as np
        n, off = node.length, node.offset
        bufs = C.cast(node.buffers, C.POINTER(C.c_void_p))
        validity = self._host(bufs[0], (off + n + 7) // 8) if bufs[0] else None
        if pa.types.is_string(typ) or pa.types.is_binary(typ) or pa.types.is_list(typ):
            offs = self._host(bufs[1], 4 * (off + n + 1))
            o = np.frombuffer(offs, dtype=np.int32)
            if pa.types.is_list(typ):
                kids = C.cast(node.children, C.POINTER(C.POINTER(_ArrowArrayStruct)))
                child = self._child(kids[0].contents, typ.value_type)
                return pa.Array.from_buffers(typ, n, [validity, offs], null_count=-1, offset=off, children=[child])
            data = self._host(bufs[2], int(o[-1]) if len(o) else 0)
            return pa.Array.from_buffers(typ, n, [validity, offs, data], null_count=-1, offset=off)
        return pa.Array.from_buffers(typ, n, [validity, self._host(bufs[1], (off + n) * (typ.bit_width // 8))], null_count=-1, offset=off)

    def to_host(self) -> pa.RecordBatch:
        if self._dev.sync_event:
            _cuda_memcpy_d2h(0, 0, 0)
            _cudart.cudaDeviceSynchronize()           # (a consumer kernel would cudaStreamWaitEvent on *sync_event instead)
        a = self._dev.array
        if len(self.schema) == 0:
            return pa.RecordBatch.from_struct_array(pa.array([{}] * a.length, type=pa.struct([])))
        kids = C.cast(a.children, C.POINTER(C.POINTER(_ArrowArrayStruct)))
        cols = [self._child(kids[i].contents, self.schema.field(i).type) for i in range(a.n_children)]
        return pa.RecordBatch.from_arrays(cols, schema=self.schema)


class BamTableProvider:
    """== BamTableProvider (table_provider.rs:314-335); constructor arguments follow `new` (:381-390)."""

    def __init__(self, file_path, object_storage_options=None, coordinate_system_zero_based=True, tag_fields=None,
                 binary_cigar=False, infer_tag_types=True, infer_tag_sample_size=100, tag_type_hints=None, *,
                 index_path=None, device_id=0, batch_rows=0, chunk_inflated_bytes=0, segment_bytes=0, skip_crc=False,
                 debug_flags=0, decode_all_tag_fields=False):
        if object_storage_options is not None:
            raise BamScanError(-5, "remote object storage is out of scope for this build (local files only)")
        L = load_library()
        o = _Options()
        o.struct_size = C.sizeof(_Options)
        o.coordinate_system_zero_based = int(coordinate_system_zero_based)
        o.binary_cigar = int(binary_cigar)
        o.has_tag_fields = int(tag_fields is not None)
        self._tag_arr, self._tag_enc = _strs(list(tag_fields or []))
        o.n_tag_fields = len(tag_fields or [])
        if self._tag_arr is not None:
            o.tag_fields = self._tag_arr
        o.infer_tag_types = int(infer_tag_types)
        o.infer_tag_sample_size = int(infer_tag_sample_size)
        self._hint_arr, self._hint_enc = _strs(list(tag_type_hints or []))
        o.n_tag_type_hints = len(tag_type_hints or [])
        if self._hint_arr is not None:
            o.tag_type_hints = self._hint_arr
        o.device_id = device_id
        o.batch_rows = batch_rows
        o.chunk_inflated_bytes = chunk_inflated_bytes
        o.segment_bytes = segment_bytes
        o.skip_crc = int(skip_crc)
        o.debug_flags = debug_flags
        o.decode_all_tag_fields = int(decode_all_tag_fields)
        self._h = C.c_void_p()
        _check(L.bamscan_open(str(file_path).encode(), index_path.encode() if index_path is not None else None, C.byref(o), C.byref(self._h)))
        self.file_path = str(file_path)
        self.device_id = device_id
        self._schema = None

    def close(self):
        if self._h:
            load_library().bamscan_close(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def schema(self) -> pa.Schema:
        if self._schema is None:
            cs = _ArrowSchemaStruct()
            _check(load_library().bamscan_schema(self._h, C.byref(cs)))
            self._schema = pa.Schema._import_from_c(C.addressof(cs))
        return self._schema

    def table_type(self) -> str:
        return "Base"

    @classmethod
    def try_new_with_inferred_schema(cls, file_path, object_storage_options=None, coordinate_system_zero_based=True,
                                     tag_fields=None, sample_size=None, binary_cigar=False, **kw):
        """== BamTableProvider::try_new_with_inferred_schema (table_provider.rs:568-621): `new` with tag types always inferred
        from the first `sample_size` (default 100) records and no hints."""
        return cls(file_path, object_storage_options, coordinate_system_zero_based, tag_fields, binary_cigar, True,
                   100 if sample_size is None else sample_size, None, **kw)

    def describe(self, ctx=None, sample_size=None) -> pa.Table:
        """== BamTableProvider::describe (table_provider.rs:703-927): one row per core column and per aux tag found in the first
        `sample_size` (default 100) records: column_name, data_type, nullable, category ("core" / "tag"), sam_type, description.
        `ctx` (the reference's SessionContext, which only wraps the batch in a DataFrame) is accepted and ignored."""
        L = load_library()
        need = C.c_uint64(0)
        buf = C.create_string_buffer(1 << 16)
        rc = L.bamscan_describe_tags(self._h, int(sample_size or 0), buf, len(buf), C.byref(need))
        if rc != 0 and need.value > len(buf):
            buf = C.create_string_buffer(need.value)
            rc = L.bamscan_describe_tags(self._h, int(sample_size or 0), buf, len(buf), C.byref(need))
        _check(rc)
        binary = pa.types.is_binary(self.schema().field("cigar").type)
        zero_based = (self.schema().metadata or {}).get(b"bio.coordinate_system_zero_based", b"true") == b"true"
        rows = [("name", "Utf8", True, "Read name/query template name"), ("chrom", "Utf8", True, "Reference sequence name"),
                ("start", "UInt32", True, "Leftmost mapping position (%s)" % ("0-based" if zero_based else "1-based")),
                ("end", "UInt32", True, "Rightmost mapping position"), ("flags", "UInt32", False, "Bitwise flags"),
                ("cigar", "Binary" if binary else "Utf8", False, "CIGAR (binary LE u32 ops)" if binary else "CIGAR string"),
                ("mapping_quality", "UInt32", False, "Mapping quality (0-255)"), ("mate_chrom", "Utf8", True, "Mate reference sequence name"),
                ("mate_start", "UInt32", True, "Mate position"), ("sequence", "Utf8", False, "Segment sequence"),
                ("quality_scores", "Utf8", False, "Base quality scores"), ("template_length", "Int32", False, "Template length (TLEN)")]
        cols = [[r[0] for r in rows], [r[1] for r in rows], [r[2] for r in rows], ["core"] * 12, [None] * 12, [r[3] for r in rows]]
        for line in buf.value.decode().splitlines():
            tag, sam, typ, desc = line.split("\t", 3)
            for c, v in zip(cols, (tag, typ, True, "tag", sam, desc)):
                c.append(v)
        schema = pa.schema([pa.field("column_name", pa.utf8(), False), pa.field("data_type", pa.utf8(), False),
                            pa.field("nullable", pa.bool_(), False), pa.field("category", pa.utf8(), False),
                            pa.field("sam_type", pa.utf8(), True), pa.field("description", pa.utf8(), False)])
        return pa.Table.from_arrays([pa.array(c, f.type) for c, f in zip(cols, schema)], schema=schema)

    def supports_filters_pushdown(self, filters):
        pack = _FilterPack(filters, self.schema().names)
        out = (C.c_uint8 * max(1, pack.n))()
        _check(load_library().bamscan_classify_filters(self._h, pack.arr, pack.n, out))
        return ["Inexact" if out[i] else "Unsupported" for i in range(pack.n)]

    def scan(self, projection=None, filters=None, limit=None, *, target_partitions=1, partition_mode="reference") -> BamExec:
        L = load_library()
        pack = _FilterPack(filters, self.schema().names)
        if projection is None:
            proj, n_proj = None, -1
        else:
            proj = (C.c_int32 * max(1, len(projection)))(*projection)
            n_proj = len(projection)
        ph = C.c_void_p()
        mode = {"reference": 0, "block_range": 1}[partition_mode]
        _check(L.bamscan_plan(self._h, proj, n_proj, pack.arr, pack.n, -1 if limit is None else int(limit),
                              int(target_partitions), mode, C.byref(ph)))
        return BamExec(self, ph)


    @classmethod
    def new_for_write(cls, output_path, schema: pa.Schema, tag_fields=None, coordinate_system_zero_based=True, sort_on_write=False, *, device_id=0):
        """== BamTableProvider::new_for_write (table_provider.rs:639-664): a provider for a file that does not exist yet; only
        schema() and insert_into() are meaningful on it."""
        self = cls.__new__(cls)
        self._h = None
        self.file_path = str(output_path)
        self.device_id = device_id
        self._schema = schema
        self._write_tag_fields = list(tag_fields) if tag_fields is not None else None
        self._write_zero_based = bool(coordinate_system_zero_based)
        self._sort_on_write = bool(sort_on_write)
        return self

    def insert_into(self, batches, insert_op="overwrite", *, sort_on_write=None, compression=0):
        """== TableProvider::insert_into (table_provider.rs:1117-1177) + BamWriteExec::execute: `INSERT OVERWRITE` of `batches`
        (an iterable of pyarrow.RecordBatch with this provider's schema) into this provider's file.  Returns the row count (the
        reference's one-row `count` batch).  sort_on_write is DataFusion's SortExec in front of the writer, not part of it: the
        rows are written in arrival order and only the header's SO field follows the flag, as in the reference.  A `.sam` path
        (is_sam_path) is written as plain SAM text through SamWriteExec; `compression` applies to BAM only."""
        if insert_op != "overwrite":
            raise NotImplementedError("BAM insert_into only supports OVERWRITE mode")
        schema = self.schema()
        md = {k.decode(): v.decode() for k, v in (schema.metadata or {}).items()}
        zero_based = md.get("bio.coordinate_system_zero_based", "true").lower() != "false"      # table_provider.rs:1133-1136 (the schema decides)
        tags = [f.name for f in schema if f.metadata and b"bio.bam.tag.tag" in f.metadata]
        for t in getattr(self, "_write_tag_fields", None) or []:                                 # explicitly requested tags are honoured too (:1146-1154)
            if t not in tags:
                tags.append(t)
        if sort_on_write is None:
            sort_on_write = getattr(self, "_sort_on_write", False)
        overrides = {"bio.bam.sort_order": "coordinate" if sort_on_write else "unsorted"}
        if is_sam_path(self.file_path):                                                          # plain SAM text (compression is not read)
            ex = SamWriteExec(self.file_path, schema, tags, zero_based, overrides, device_id=getattr(self, "device_id", 0))
        else:
            ex = BamWriteExec(self.file_path, schema, tags, zero_based, overrides, device_id=getattr(self, "device_id", 0), compression=compression)
        n = ex.execute(batches)
        self.last_write_stats = ex.stats
        return n


# ---- SURVEY 8 f4: the write path -------------------------------------------------------------------------------------
_SQ_TAGS = {"AH", "AN", "AS", "DS", "M5", "SP", "TP", "UR"}
_RG_TAGS = {"BC", "CN", "DT", "FO", "KS", "PG", "PI", "PM", "PU"}
_PG_TAGS = {"PP", "DS"}


def build_bam_header(schema: pa.Schema, tag_fields=None, overrides=None):
    """== build_bam_header (bio-format-bam/src/header_builder.rs:43-186) followed by noodles' SAM header writer: the header
    text and the reference dictionary reconstructed from the bio.bam.* schema metadata (defaults: VN 1.6, no @SQ).  In the
    Rust host this function stays the reference's own; it is restated here because the tests drive the ABI from python.
    Extra per-line fields sit in a HashMap in the reference (arbitrary order); here they are written in sorted key order."""
    import json
    md = {(k.decode() if isinstance(k, bytes) else k): (v.decode() if isinstance(v, bytes) else v) for k, v in (schema.metadata or {}).items()}
    md.update(overrides or {})

    def arr(key):
        try:
            return json.loads(md[key]) if key in md else []
        except Exception:
            return []

    ver = md.get("bio.bam.file_format_version", "1.6").split(".")
    ver = f"{int(ver[0])}.{int(ver[1])}" if len(ver) == 2 and all(p.isdigit() for p in ver) else "1.6"
    hd = ["VN:" + ver] + [f"{t}:{md[k]}" for k, t in (("bio.bam.sort_order", "SO"), ("bio.bam.group_order", "GO"), ("bio.bam.subsort_order", "SS")) if k in md]
    lines, names, lens = ["@HD\t" + "\t".join(hd)], [], []

    def extra(d, allowed):
        return [f"{k}:{v}" for k, v in sorted((d.get("other_fields") or {}).items()) if k in allowed]

    for sq in arr("bio.bam.reference_sequences"):
        if int(sq["length"]) == 0:
            raise BamScanError(-6, "Reference sequence length cannot be zero")
        lines.append("\t".join(["@SQ", f"SN:{sq['name']}", f"LN:{int(sq['length'])}"] + extra(sq, _SQ_TAGS)))
        names.append(sq["name"]); lens.append(int(sq["length"]))
    for rg in arr("bio.bam.read_groups"):
        f = [f"{t}:{rg[k]}" for k, t in (("sample", "SM"), ("platform", "PL"), ("library", "LB"), ("description", "DS")) if rg.get(k) is not None]
        lines.append("\t".join(["@RG", f"ID:{rg['id']}"] + f + extra(rg, _RG_TAGS)))
    for pg in arr("bio.bam.program_info"):
        f = [f"{t}:{pg[k]}" for k, t in (("name", "PN"), ("version", "VN"), ("command_line", "CL")) if pg.get(k) is not None]
        lines.append("\t".join(["@PG", f"ID:{pg['id']}"] + f + extra(pg, _PG_TAGS)))
    lines += [f"@CO\t{c}" for c in arr("bio.bam.comments")]
    return "\n".join(lines) + "\n", names, lens


class BamWriteExec:
    """== BamWriteExec (bio-format-bam/src/write_exec.rs:43-110): new(input, output_path, compression, tag_fields,
    coordinate_system_zero_based, schema_metadata_overrides, sort_on_write); `execute` consumes the batches and returns the
    count.  Only BGZF BAM output: a `.sam` path is refused here, SamWriteExec writes plain SAM."""

    def __init__(self, output_path, input_schema: pa.Schema, tag_fields=None, coordinate_system_zero_based=True,
                 schema_metadata_overrides=None, *, device_id=0, compression=0):
        if is_sam_path(output_path):
            raise BamScanError(-5, "plain SAM output is out of scope for BamWriteExec (BGZF BAM only): use SamWriteExec")
        self.output_path = str(output_path)
        self.schema = input_schema
        self.tag_fields = list(tag_fields or [])
        self.zero_based = bool(coordinate_system_zero_based)
        self.overrides = dict(schema_metadata_overrides or {})
        self.device_id = device_id
        self.compression = compression
        self.stats = None

    def execute(self, batches) -> int:
        n, self.stats = _open_and_drive(load_library().bamscan_writer_open, self, batches)
        return n


def is_sam_path(path) -> bool:
    """The reference's `is_sam`: a path ending in `.sam`, in any case, is plain SAM text (scan and write)."""
    return str(path).lower().endswith(".sam")


class SamWriteExec:
    """The SAM write path (bamscan_sam_writer_open): the rows BamWriteExec accepts, written as plain SAM text -- the header of
    build_bam_header(input_schema, tag_fields, overrides), then one line per row in arrival order (no BGZF).  Rows the BAM writer
    refuses are refused with the same error; so are rows whose line would not read back as the same row (DESIGN 3.9).
    `execute` takes pyarrow.RecordBatch or DeviceBatch and returns the row count; `.stats` after it."""

    def __init__(self, output_path, input_schema: pa.Schema, tag_fields=None, coordinate_system_zero_based=True,
                 schema_metadata_overrides=None, *, device_id=0):
        self.output_path = str(output_path)
        self.schema = input_schema
        self.tag_fields = list(tag_fields or [])
        self.zero_based = bool(coordinate_system_zero_based)
        self.overrides = dict(schema_metadata_overrides or {})
        self.device_id = device_id
        self.compression = 0
        self.stats = None

    def execute(self, batches) -> int:
        n, self.stats = _open_and_drive(load_library().bamscan_sam_writer_open, self, batches)
        return n


def _open_and_drive(open_fn, ex, batches):
    """bamscan_writer_open / bamscan_sam_writer_open with ex's header, references, tags and options, then _drive_writer."""
    text, names, lens = build_bam_header(ex.schema, ex.tag_fields, ex.overrides)
    o = _WriteOptions()
    o.struct_size = C.sizeof(_WriteOptions)
    o.coordinate_system_zero_based = int(ex.zero_based)
    tag_arr, _keep = _strs(ex.tag_fields)
    o.n_tag_fields = len(ex.tag_fields)
    if tag_arr is not None:
        o.tag_fields = tag_arr
    o.device_id = ex.device_id
    o.compression = ex.compression
    name_arr, _keep2 = _strs(names)
    len_arr = (C.c_int32 * max(1, len(lens)))(*lens)
    cs = _ArrowSchemaStruct()
    pa.struct(list(ex.schema))._export_to_c(C.addressof(cs))
    h = C.c_void_p()
    try:
        _check(open_fn(ex.output_path.encode(), text.encode(), len(names), name_arr, len_arr, C.addressof(cs), C.byref(o), C.byref(h)))
    finally:
        if cs.release:
            C.CFUNCTYPE(None, C.c_void_p)(cs.release)(C.addressof(cs))
    return _drive_writer(h, batches, ex.schema)


def _drive_writer(h, batches, schema: pa.Schema):
    """Feeds `batches` (pyarrow.RecordBatch or DeviceBatch with `schema`'s columns) to an open writer handle, finishes it and
    frees it.  -> (rows written, stats dict)."""
    L = load_library()
    try:
        for b in batches:
            if b.schema.names != schema.names:
                raise BamScanError(-7, "batch columns differ from the writer's input schema")
            if isinstance(b, DeviceBatch):                   # stays in HBM: bamscan_writer_write_device
                _check(L.bamscan_writer_write_device(h, C.byref(b._dev)))
                continue
            ca = _ArrowArrayStruct()
            sa = b.to_struct_array()
            sa._export_to_c(C.addressof(ca))
            try:
                _check(L.bamscan_writer_write(h, C.addressof(ca)))
            finally:
                if ca.release:
                    C.CFUNCTYPE(None, C.c_void_p)(ca.release)(C.addressof(ca))
        n = C.c_uint64()
        _check(L.bamscan_writer_finish(h, C.byref(n)))
        st = WriteStats()
        _check(L.bamscan_writer_stats(h, C.byref(st)))
        return int(n.value), st.as_dict()
    finally:
        L.bamscan_writer_free(h)


FASTQ_SCHEMA = pa.schema([pa.field("name", pa.string(), False), pa.field("description", pa.string(), True),
                          pa.field("sequence", pa.string(), False), pa.field("quality_scores", pa.string(), False)])


def fastq_compression_for(output_path) -> int:
    """Compression a FASTQ path asks for by its extension: `.bgz`, `.bgzf` and `.gz` -> BGZF (0), anything else -> plain text
    (2).  BGZF is valid multi-member gzip, so a `.gz` file is written as BGZF too."""
    return 0 if str(output_path).lower().endswith((".bgz", ".bgzf", ".gz")) else 2


class FastqWriteExec:
    """The FASTQ write path (bamscan_fastq_writer_open): rows of `input_schema`'s name / description / sequence / quality_scores
    columns (looked up by name; description optional; other columns ignored) encoded as FASTQ text on the device, into BGZF
    members (compression 0, or 1 = stored blocks) or plain text (2).  compression None: by the path's extension
    (fastq_compression_for).  `execute` takes pyarrow.RecordBatch or DeviceBatch and returns the row count; `.stats` after it.
    Bases and qualities are written as stored: reads of a BAM scan are not reverse-complemented."""

    def __init__(self, output_path, input_schema: pa.Schema, compression=None, *, device_id=0):
        self.output_path = str(output_path)
        self.schema = input_schema
        self.compression = fastq_compression_for(output_path) if compression is None else int(compression)
        self.device_id = device_id
        self.stats = None

    def execute(self, batches) -> int:
        L = load_library()
        o = _WriteOptions()
        o.struct_size = C.sizeof(_WriteOptions)
        o.device_id = self.device_id
        o.compression = self.compression
        cs = _ArrowSchemaStruct()
        pa.struct(list(self.schema))._export_to_c(C.addressof(cs))
        h = C.c_void_p()
        try:
            _check(L.bamscan_fastq_writer_open(self.output_path.encode(), C.addressof(cs), C.byref(o), C.byref(h)))
        finally:
            if cs.release:
                C.CFUNCTYPE(None, C.c_void_p)(cs.release)(C.addressof(cs))
        n, self.stats = _drive_writer(h, batches, self.schema)
        return n


class FastqTableProvider(BamTableProvider):
    """== FastqTableProvider (bio-format-fastq/src/table_provider.rs:46-75) for BGZF-compressed FASTQ: `new(file_path,
    object_storage_options)`; schema name / description / sequence / quality_scores (Utf8, description nullable).  `scan` with
    target_partitions > 1 uses BGZF block ranges balanced by compressed bytes; partition_mode="reference" cuts by block count from
    the companion .gzi exactly as get_bgzf_partition_bounds does (physical_exec.rs:140-175; no .gzi: one partition); everything
    else is BamTableProvider's."""

    def __init__(self, file_path, object_storage_options=None, *, device_id=0, batch_rows=0, chunk_inflated_bytes=0,
                 skip_crc=False, debug_flags=0):
        if object_storage_options is not None:
            raise BamScanError(-5, "remote object storage is out of scope for this build (local files only)")
        L = load_library()
        o = _Options()
        o.struct_size = C.sizeof(_Options)
        o.device_id = device_id
        o.batch_rows = batch_rows
        o.chunk_inflated_bytes = chunk_inflated_bytes
        o.skip_crc = int(skip_crc)
        o.debug_flags = debug_flags
        self._h = C.c_void_p()
        _check(L.bamscan_open_fastq(str(file_path).encode(), C.byref(o), C.byref(self._h)))
        self.file_path = str(file_path)
        self.device_id = device_id
        self._schema = None

    def scan(self, projection=None, filters=None, limit=None, *, target_partitions=1, partition_mode=None) -> BamExec:
        if partition_mode is None:
            partition_mode = "block_range" if target_partitions > 1 else "reference"
        return super().scan(projection, None, limit, target_partitions=target_partitions, partition_mode=partition_mode)

    @classmethod
    def new_for_write(cls, output_path, schema: pa.Schema = None, *, device_id=0):
        """A provider for a FASTQ file that does not exist yet (default schema: the FASTQ scan's); only schema() and
        insert_into() are meaningful on it."""
        self = cls.__new__(cls)
        self._h = None
        self.file_path = str(output_path)
        self.device_id = device_id
        self._schema = FASTQ_SCHEMA if schema is None else schema
        return self

    def insert_into(self, batches, insert_op="overwrite", *, compression=None):
        """`INSERT OVERWRITE` of `batches` (pyarrow.RecordBatch or DeviceBatch with this provider's schema) into this provider's
        file through FastqWriteExec; compression None picks BGZF or plain text by the file's extension.  Returns the row count."""
        if insert_op != "overwrite":
            raise NotImplementedError("FASTQ insert_into only supports OVERWRITE mode")
        ex = FastqWriteExec(self.file_path, self.schema(), compression, device_id=getattr(self, "device_id", 0))
        n = ex.execute(batches)
        self.last_write_stats = ex.stats
        return n


class FastaTableProvider(BamTableProvider):
    """A provider for BGZF-compressed FASTA (bamscan_open_fasta): `FastaTableProvider(file_path, object_storage_options)`;
    schema name / description / sequence (Utf8, description nullable).  `scan` with target_partitions > 1 uses BGZF block ranges
    balanced by compressed bytes (a record belongs to the range that holds its '>'); no filter is pushed down and `limit` is not
    applied, as for FastqTableProvider; everything else is BamTableProvider's."""

    def __init__(self, file_path, object_storage_options=None, *, device_id=0, batch_rows=0, chunk_inflated_bytes=0,
                 skip_crc=False, debug_flags=0):
        if object_storage_options is not None:
            raise BamScanError(-5, "remote object storage is out of scope for this build (local files only)")
        L = load_library()
        o = _Options()
        o.struct_size = C.sizeof(_Options)
        o.device_id = device_id
        o.batch_rows = batch_rows
        o.chunk_inflated_bytes = chunk_inflated_bytes
        o.skip_crc = int(skip_crc)
        o.debug_flags = debug_flags
        self._h = C.c_void_p()
        _check(L.bamscan_open_fasta(str(file_path).encode(), C.byref(o), C.byref(self._h)))
        self.file_path = str(file_path)
        self.device_id = device_id
        self._schema = None

    def scan(self, projection=None, filters=None, limit=None, *, target_partitions=1) -> BamExec:
        mode = "block_range" if target_partitions > 1 else "reference"
        return super().scan(projection, None, limit, target_partitions=target_partitions, partition_mode=mode)


def check_partition_seams(stats_list):
    """Raises BamScanError unless every block-range partition starts where the chain of the one before it landed
    (bamscan_check_partition_seams).  stats_list: last_stats dicts (or run_device_resident results) in partition order."""
    arr = (Stats * len(stats_list))()
    for i, d in enumerate(stats_list):
        for k, _t in Stats._fields_:
            setattr(arr[i], k, d.get(k, 0))
    _check(load_library().bamscan_check_partition_seams(arr, len(stats_list)))


def extract_genomic_regions(filters, coordinate_system_zero_based: bool) -> dict:
    """== extract_genomic_regions (genomic_filter.rs:51-100) over [(column, op, values)]."""
    pack = _FilterPack(filters, CORE_COLUMNS)
    out = RegionAnalysis()
    _check(load_library().bamscan_extract_regions(pack.arr, pack.n, int(coordinate_system_zero_based), C.byref(out)))
    raw = bytes(out.chroms)
    chroms = [c.decode() for c in raw.split(b"\0")[:out.n_chroms]]
    start = out.start if out.has_start else None
    end = out.end if out.has_end else None
    regions = [] if out.unsatisfiable else [dict(chrom=c, start=start, end=end, unmapped_tail=False) for c in chroms]
    return dict(regions=regions, unsatisfiable=bool(out.unsatisfiable), start=start, end=end,
                residual=[i for i in range(pack.n) if (out.residual_mask >> i) & 1])


def balance_partitions(estimates, target_partitions: int):
    """== balance_partitions (partition_balancer.rs:61-295).  estimates: list of dicts with keys chrom, bytes and optionally
    start, end, contig_length, unmapped_count, bins, leaf_bin_span.  Returns a list of partitions:
    dict(regions=[dict(chrom, start, end, unmapped_tail)], total_estimated_bytes)."""
    n = len(estimates)
    arr = (RegionEstimate * max(1, n))()
    keep = []
    for i, e in enumerate(estimates):
        name = e["chrom"].encode(); keep.append(name)
        arr[i].chrom = name
        arr[i].has_start = int(e.get("start") is not None); arr[i].start = e.get("start") or 0
        arr[i].has_end = int(e.get("end") is not None); arr[i].end = e.get("end") or 0
        arr[i].estimated_bytes = e["bytes"]; arr[i].contig_length = e.get("contig_length") or 0
        arr[i].unmapped_count = e.get("unmapped_count", 0)
        bins = e.get("bins") or []
        if bins:
            b = (C.c_uint64 * len(bins))(*bins); keep.append(b)
            arr[i].nonempty_bin_positions = b
        arr[i].n_bin_positions = len(bins); arr[i].leaf_bin_span = e.get("leaf_bin_span", 0)
    cap = 64 * max(1, n) + 4 * max(1, target_partitions) + 64
    out = (AssignedRegion * cap)()
    n_out, n_parts = C.c_int32(), C.c_int32()
    _check(load_library().bamscan_balance_partitions(arr, n, target_partitions, out, cap, C.byref(n_out), C.byref(n_parts)))
    parts = [dict(regions=[], total_estimated_bytes=0) for _ in range(n_parts.value)]
    for a in out[:n_out.value]:
        p = parts[a.partition]
        p["total_estimated_bytes"] = a.partition_total_estimated_bytes
        p["regions"].append(dict(chrom=estimates[a.estimate_index]["chrom"], start=a.start if a.has_start else None,
                                 end=a.end if a.has_end else None, unmapped_tail=bool(a.unmapped_tail)))
    return parts


def probe_pcie(device_id=0, nbytes=1 << 30) -> dict:
    a, b, c = C.c_double(), C.c_double(), C.c_double()
    _check(load_library().bamscan_probe_pcie(device_id, nbytes, C.byref(a), C.byref(b), C.byref(c)))
    return {"h2d_gbps": a.value, "d2h_gbps": b.value, "bidir_gbps": c.value, "bytes": nbytes}
