//! `GpuBamTableProvider` / `GpuBamExec`: the DataFusion-facing pair of the reference
//! (`datafusion/bio-format-bam/src/table_provider.rs:926-1115`, `physical_exec.rs:84-173`) with everything below the two
//! traits replaced by `libbamscan.so`.  Planning (schema, filter classification, region extraction, partition balancing)
//! and execution (BGZF ingest, inflate, record framing, columnar decode) all happen behind the C ABI; Arrow data comes
//! back through the Arrow C Data Interface and is imported zero-copy.
//!
//! SOURCE-ONLY: no Rust toolchain exists where this repository is built; the Python mirror
//! (`datafusion-bio-formats_b200/bamscan/__init__.py`) is the binding that the tests exercise.  The constructor keeps the
//! reference's argument list so that call sites (`BamTableProvider::new(...)`) only change the type name.

pub mod ffi;
pub mod write;

use arrow::array::{Array, StructArray};
use arrow::datatypes::{DataType, Schema, SchemaRef};
use arrow::ffi::{from_ffi, FFI_ArrowArray, FFI_ArrowSchema};
use arrow::record_batch::{RecordBatch, RecordBatchOptions};
use async_trait::async_trait;
use datafusion::catalog::{Session, TableProvider};
use datafusion::common::{DataFusionError, Result, ScalarValue};
use datafusion::datasource::TableType;
use datafusion::execution::{SendableRecordBatchStream, TaskContext};
use datafusion::logical_expr::{BinaryExpr, Expr, Operator, TableProviderFilterPushDown};
use datafusion::physical_expr::EquivalenceProperties;
use datafusion::physical_plan::empty::EmptyExec;
use datafusion::physical_plan::execution_plan::{Boundedness, EmissionType};
use datafusion::physical_plan::stream::RecordBatchStreamAdapter;
use datafusion::physical_plan::{DisplayAs, DisplayFormatType, ExecutionPlan, Partitioning, PlanProperties};
use std::any::Any;
use std::ffi::{c_char, CStr, CString};
use std::fmt::{Debug, Formatter};
use std::sync::Arc;

fn last_error() -> DataFusionError {
    let msg = unsafe { CStr::from_ptr(ffi::bamscan_last_error()) }.to_string_lossy().into_owned();
    DataFusionError::Execution(msg)
}

/// Owns a `BamScanHandle*` (one per file and device).
struct Handle(*mut ffi::BamScanHandle);
unsafe impl Send for Handle {}
unsafe impl Sync for Handle {} // the library serialises access to a handle's shared state (`BamScanHandle::mu`)
impl Drop for Handle {
    fn drop(&mut self) {
        unsafe { ffi::bamscan_close(self.0) }
    }
}

/// Owns a `BamScanPlan*`; must not outlive its handle (it holds an `Arc<Handle>`).
struct Plan {
    raw: *mut ffi::BamScanPlan,
    _handle: Arc<Handle>,
}
unsafe impl Send for Plan {}
unsafe impl Sync for Plan {}
impl Drop for Plan {
    fn drop(&mut self) {
        unsafe { ffi::bamscan_plan_free(self.raw) }
    }
}

pub struct GpuBamTableProvider {
    handle: Arc<Handle>,
    schema: SchemaRef,
    device_id: i32,
}

impl GpuBamTableProvider {
    /// Same arguments, same meaning as `BamTableProvider::new` (`table_provider.rs:381-529`); `object_storage_options`
    /// must be `None` (local files only).  `device_id` selects the GPU.
    #[allow(clippy::too_many_arguments)]
    pub fn new(
        file_path: String,
        coordinate_system_zero_based: bool,
        tag_fields: Option<Vec<String>>,
        binary_cigar: bool,
        infer_tag_types: bool,
        infer_tag_sample_size: usize,
        tag_type_hints: Option<Vec<String>>,
        device_id: i32,
    ) -> Result<Self> {
        let c_path = CString::new(file_path).map_err(|e| DataFusionError::Execution(e.to_string()))?;
        let to_c = |v: &Option<Vec<String>>| -> Vec<CString> { v.iter().flatten().map(|s| CString::new(s.as_str()).unwrap()).collect() };
        let tags_c = to_c(&tag_fields);
        let hints_c = to_c(&tag_type_hints);
        let tags_p: Vec<*const c_char> = tags_c.iter().map(|s| s.as_ptr()).collect();
        let hints_p: Vec<*const c_char> = hints_c.iter().map(|s| s.as_ptr()).collect();
        let opts = ffi::BamScanOptions {
            struct_size: std::mem::size_of::<ffi::BamScanOptions>() as u32,
            coordinate_system_zero_based: coordinate_system_zero_based as i32,
            binary_cigar: binary_cigar as i32,
            has_tag_fields: tag_fields.is_some() as i32,
            n_tag_fields: tags_p.len() as i32,
            tag_fields: tags_p.as_ptr(),
            infer_tag_types: infer_tag_types as i32,
            infer_tag_sample_size: infer_tag_sample_size as i32,
            n_tag_type_hints: hints_p.len() as i32,
            tag_type_hints: hints_p.as_ptr(),
            device_id,
            batch_rows: 0, // 0 = one batch per decode slice; pass SessionConfig::batch_size here for the reference's batch shape
            chunk_inflated_bytes: 0,
            segment_bytes: 0,
            skip_crc: 0,
            debug_flags: 0,
            decode_all_tag_fields: 0,
            has_format_fields: 0,
            n_format_fields: 0,
            format_fields: std::ptr::null(),
        };
        let mut raw = std::ptr::null_mut();
        // index_path = NULL: discover `<file>.bai` / `.csi` next to the file like `discover_bam_index` does
        if unsafe { ffi::bamscan_open(c_path.as_ptr(), std::ptr::null(), &opts, &mut raw) } != 0 {
            return Err(last_error());
        }
        let handle = Arc::new(Handle(raw));
        let mut c_schema = FFI_ArrowSchema::empty();
        if unsafe { ffi::bamscan_schema(handle.0, &mut c_schema) } != 0 {
            return Err(last_error());
        }
        let schema = Arc::new(Schema::try_from(&c_schema)?); // fields + the bio.bam.* metadata of determine_schema
        Ok(Self { handle, schema, device_id })
    }

    pub fn device_id(&self) -> i32 {
        self.device_id
    }
}

impl Debug for GpuBamTableProvider {
    fn fmt(&self, f: &mut Formatter<'_>) -> std::fmt::Result {
        f.debug_struct("GpuBamTableProvider").field("device_id", &self.device_id).finish()
    }
}

/// One conjunct of the WHERE clause in the ABI's form.  Owns the C strings and numbers the raw struct points at.
struct OwnedFilter {
    column: i32,
    op: i32,
    nums: Vec<f64>,
    strs: Vec<CString>,
    str_ptrs: Vec<*const c_char>,
}

impl OwnedFilter {
    fn other() -> Self {
        Self { column: -1, op: ffi::OP_OTHER, nums: vec![], strs: vec![], str_ptrs: vec![] }
    }
    fn raw(&self) -> ffi::BamScanFilter {
        ffi::BamScanFilter {
            column: self.column,
            op: self.op,
            n_values: self.nums.len().max(self.strs.len()) as i32,
            num_values: if self.nums.is_empty() { std::ptr::null() } else { self.nums.as_ptr() },
            str_values: if self.str_ptrs.is_empty() { std::ptr::null() } else { self.str_ptrs.as_ptr() },
        }
    }
    fn push(&mut self, v: &ScalarValue) -> bool {
        match v {
            ScalarValue::Utf8(Some(s)) | ScalarValue::LargeUtf8(Some(s)) | ScalarValue::Utf8View(Some(s)) => {
                self.strs.push(CString::new(s.as_str()).unwrap());
                true
            }
            ScalarValue::Int8(Some(x)) => { self.nums.push(*x as f64); true }
            ScalarValue::Int16(Some(x)) => { self.nums.push(*x as f64); true }
            ScalarValue::Int32(Some(x)) => { self.nums.push(*x as f64); true }
            ScalarValue::Int64(Some(x)) => { self.nums.push(*x as f64); true }
            ScalarValue::UInt8(Some(x)) => { self.nums.push(*x as f64); true }
            ScalarValue::UInt16(Some(x)) => { self.nums.push(*x as f64); true }
            ScalarValue::UInt32(Some(x)) => { self.nums.push(*x as f64); true }
            ScalarValue::UInt64(Some(x)) => { self.nums.push(*x as f64); true }
            _ => false,
        }
    }
    fn seal(mut self) -> Self {
        self.str_ptrs = self.strs.iter().map(|s| s.as_ptr()).collect();
        self
    }
}

fn literal(e: &Expr) -> Option<&ScalarValue> {
    match e {
        Expr::Literal(v, _) => Some(v),
        _ => None,
    }
}

/// `Column op Literal`, `Column [NOT] BETWEEN a AND b`, `Column [NOT] IN (..)`; anything else is OP_OTHER (classified
/// Unsupported and ignored by planning), so that filter indices stay aligned with `supports_filters_pushdown`.
fn convert(expr: &Expr, schema: &Schema) -> OwnedFilter {
    let col_index = |e: &Expr| match e {
        Expr::Column(c) => schema.index_of(&c.name).ok().map(|i| i as i32),
        _ => None,
    };
    match expr {
        Expr::BinaryExpr(BinaryExpr { left, op, right }) => {
            let (col, lit, flipped) = match (col_index(left), literal(right), literal(left), col_index(right)) {
                (Some(c), Some(l), _, _) => (c, l, false),
                (_, _, Some(l), Some(c)) => (c, l, true),
                _ => return OwnedFilter::other(),
            };
            let op = match (op, flipped) {
                (Operator::Eq, _) => ffi::OP_EQ,
                (Operator::NotEq, _) => ffi::OP_NE,
                (Operator::Lt, false) | (Operator::Gt, true) => ffi::OP_LT,
                (Operator::LtEq, false) | (Operator::GtEq, true) => ffi::OP_LE,
                (Operator::Gt, false) | (Operator::Lt, true) => ffi::OP_GT,
                (Operator::GtEq, false) | (Operator::LtEq, true) => ffi::OP_GE,
                _ => return OwnedFilter::other(),
            };
            let mut f = OwnedFilter { column: col, op, nums: vec![], strs: vec![], str_ptrs: vec![] };
            if f.push(lit) { f.seal() } else { OwnedFilter::other() }
        }
        Expr::Between(b) => match (col_index(&b.expr), literal(&b.low), literal(&b.high)) {
            (Some(c), Some(lo), Some(hi)) => {
                let op = if b.negated { ffi::OP_NOT_BETWEEN } else { ffi::OP_BETWEEN };
                let mut f = OwnedFilter { column: c, op, nums: vec![], strs: vec![], str_ptrs: vec![] };
                if f.push(lo) && f.push(hi) { f.seal() } else { OwnedFilter::other() }
            }
            _ => OwnedFilter::other(),
        },
        Expr::InList(l) => match col_index(&l.expr) {
            Some(c) => {
                let op = if l.negated { ffi::OP_NOT_IN } else { ffi::OP_IN };
                let mut f = OwnedFilter { column: c, op, nums: vec![], strs: vec![], str_ptrs: vec![] };
                for item in &l.list {
                    match literal(item) {
                        Some(v) if f.push(v) => {}
                        _ => return OwnedFilter::other(),
                    }
                }
                f.seal()
            }
            None => OwnedFilter::other(),
        },
        _ => OwnedFilter::other(),
    }
}

/// DataFusion hands `scan` the conjuncts it was told are pushable; nested ANDs are flattened first.
fn flatten<'a>(e: &'a Expr, out: &mut Vec<&'a Expr>) {
    if let Expr::BinaryExpr(BinaryExpr { left, op: Operator::And, right }) = e {
        flatten(left, out);
        flatten(right, out);
    } else {
        out.push(e);
    }
}

#[async_trait]
impl TableProvider for GpuBamTableProvider {
    fn as_any(&self) -> &dyn Any {
        self
    }
    fn schema(&self) -> SchemaRef {
        self.schema.clone()
    }
    fn table_type(&self) -> TableType {
        TableType::Base
    }

    fn supports_filters_pushdown(&self, filters: &[&Expr]) -> Result<Vec<TableProviderFilterPushDown>> {
        let owned: Vec<OwnedFilter> = filters.iter().map(|e| convert(e, &self.schema)).collect();
        let raw: Vec<ffi::BamScanFilter> = owned.iter().map(|f| f.raw()).collect();
        let mut out = vec![0u8; raw.len()];
        if unsafe { ffi::bamscan_classify_filters(self.handle.0, raw.as_ptr(), raw.len() as i32, out.as_mut_ptr()) } != 0 {
            return Err(last_error());
        }
        Ok(out
            .into_iter()
            .map(|c| if c == ffi::PUSHDOWN_INEXACT { TableProviderFilterPushDown::Inexact } else { TableProviderFilterPushDown::Unsupported })
            .collect())
    }

    async fn scan(&self, state: &dyn Session, projection: Option<&Vec<usize>>, filters: &[Expr], limit: Option<usize>) -> Result<Arc<dyn ExecutionPlan>> {
        let mut conjuncts = Vec::new();
        for f in filters {
            flatten(f, &mut conjuncts);
        }
        let owned: Vec<OwnedFilter> = conjuncts.iter().map(|e| convert(e, &self.schema)).collect();
        let raw: Vec<ffi::BamScanFilter> = owned.iter().map(|f| f.raw()).collect();
        let proj: Option<Vec<i32>> = projection.map(|p| p.iter().map(|&i| i as i32).collect());
        let (proj_ptr, n_proj) = match &proj {
            Some(p) => (p.as_ptr(), p.len() as i32),
            None => (std::ptr::null(), -1), // -1 = no projection (all columns); 0 = empty projection (COUNT(*))
        };
        let mut raw_plan = std::ptr::null_mut();
        let rc = unsafe {
            ffi::bamscan_plan(
                self.handle.0,
                proj_ptr,
                n_proj,
                raw.as_ptr(),
                raw.len() as i32,
                limit.map(|l| l as i64).unwrap_or(-1),
                state.config().target_partitions() as i32,
                ffi::PARTITION_REFERENCE,
                &mut raw_plan,
            )
        };
        if rc != 0 {
            return Err(last_error());
        }
        let plan = Arc::new(Plan { raw: raw_plan, _handle: self.handle.clone() });
        let mut c_schema = FFI_ArrowSchema::empty();
        if unsafe { ffi::bamscan_plan_schema(plan.raw, &mut c_schema) } != 0 {
            return Err(last_error());
        }
        let schema: SchemaRef = Arc::new(Schema::try_from(&c_schema)?);
        let n = unsafe { ffi::bamscan_plan_num_partitions(plan.raw) };
        if n == 0 {
            // unsatisfiable genomic filters (table_provider.rs:1005-1010)
            return Ok(Arc::new(EmptyExec::new(schema)));
        }
        let cache = PlanProperties::new(
            EquivalenceProperties::new(schema.clone()),
            Partitioning::UnknownPartitioning(n as usize),
            EmissionType::Final,
            Boundedness::Bounded,
        );
        Ok(Arc::new(GpuBamExec { plan, schema, cache: Arc::new(cache) }))
    }
}

pub struct GpuBamExec {
    plan: Arc<Plan>,
    schema: SchemaRef,
    cache: Arc<PlanProperties>,
}

impl Debug for GpuBamExec {
    fn fmt(&self, f: &mut Formatter<'_>) -> std::fmt::Result {
        f.debug_struct("GpuBamExec").field("schema", &self.schema).finish()
    }
}

impl DisplayAs for GpuBamExec {
    fn fmt_as(&self, _t: DisplayFormatType, f: &mut Formatter) -> std::fmt::Result {
        let cols: Vec<&str> = self.schema.fields().iter().map(|f| f.name().as_str()).collect();
        write!(f, "GpuBamExec: projection=[{}]", cols.join(", "))
    }
}

/// One partition's batches: what `get_local_bam_sync` / `get_indexed_stream` produce in the reference.
struct GpuBamStream {
    raw: *mut ffi::BamScanStream,
    schema: SchemaRef,
    _plan: Arc<Plan>,
}
unsafe impl Send for GpuBamStream {} // driven by one thread at a time, like the reference's per-partition loops

impl Iterator for GpuBamStream {
    type Item = Result<RecordBatch>;
    fn next(&mut self) -> Option<Self::Item> {
        let mut arr = FFI_ArrowArray::empty();
        match unsafe { ffi::bamscan_next(self.raw, &mut arr) } {
            0 => None,
            1 => Some((|| {
                let c_schema = FFI_ArrowSchema::try_from(&DataType::Struct(self.schema.fields().clone()))?;
                let data = unsafe { from_ffi(arr, &c_schema) }?;
                let sa = StructArray::from(data);
                // a zero-column batch keeps its row count (alignment_utils.rs:360-363)
                let opts = RecordBatchOptions::new().with_row_count(Some(sa.len()));
                Ok(RecordBatch::try_new_with_options(self.schema.clone(), sa.columns().to_vec(), &opts)?)
            })()),
            _ => Some(Err(last_error())),
        }
    }
}

impl Drop for GpuBamStream {
    fn drop(&mut self) {
        unsafe { ffi::bamscan_stream_free(self.raw) }
    }
}

impl ExecutionPlan for GpuBamExec {
    fn name(&self) -> &str {
        "GpuBamExec"
    }
    fn as_any(&self) -> &dyn Any {
        self
    }
    fn properties(&self) -> &Arc<PlanProperties> {
        &self.cache
    }
    fn children(&self) -> Vec<&Arc<dyn ExecutionPlan>> {
        vec![]
    }
    fn with_new_children(self: Arc<Self>, _children: Vec<Arc<dyn ExecutionPlan>>) -> Result<Arc<dyn ExecutionPlan>> {
        Ok(self)
    }

    fn execute(&self, partition: usize, _context: Arc<TaskContext>) -> Result<SendableRecordBatchStream> {
        let mut raw = std::ptr::null_mut();
        if unsafe { ffi::bamscan_execute(self.plan.raw, partition as i32, &mut raw) } != 0 {
            return Err(last_error());
        }
        let it = GpuBamStream { raw, schema: self.schema.clone(), _plan: self.plan.clone() };
        // The library hands out one batch per decode slice (a few million rows) unless `batch_rows` was set at open();
        // DataFusion's CoalesceBatches / downstream operators accept either.  The blocking calls run on the executing
        // task's thread, as the reference's synchronous per-partition readers do (sync_stream.rs:34-43).
        Ok(Box::pin(RecordBatchStreamAdapter::new(self.schema.clone(), futures::stream::iter(it))))
    }
}

/// A provider for BGZF-compressed FASTA (`bamscan_open_fasta`), shaped like the BAM one: name, description (nullable) and
/// sequence; no filter is pushed down (DataFusion applies them), `limit` is passed on and not applied, and with
/// `target_partitions` > 1 the file is cut into BGZF block ranges balanced by compressed bytes (a record belongs to the range
/// that holds its '>').  Scans return `GpuBamExec`, which streams the batches exactly as for BAM.
pub struct GpuFastaTableProvider {
    handle: Arc<Handle>,
    schema: SchemaRef,
    device_id: i32,
}

impl GpuFastaTableProvider {
    /// `object_storage_options` must be `None` (local files only).  `device_id` selects the GPU.
    pub fn new(file_path: String, object_storage_options: Option<String>, device_id: i32) -> Result<Self> {
        if object_storage_options.is_some() {
            return Err(DataFusionError::NotImplemented("remote object storage is out of scope for this build (local files only)".into()));
        }
        let c_path = CString::new(file_path).map_err(|e| DataFusionError::Execution(e.to_string()))?;
        let opts = ffi::BamScanOptions {
            struct_size: std::mem::size_of::<ffi::BamScanOptions>() as u32,
            coordinate_system_zero_based: 1,
            binary_cigar: 0,
            has_tag_fields: 0,
            n_tag_fields: 0,
            tag_fields: std::ptr::null(),
            infer_tag_types: 0,
            infer_tag_sample_size: 0,
            n_tag_type_hints: 0,
            tag_type_hints: std::ptr::null(),
            device_id,
            batch_rows: 0,
            chunk_inflated_bytes: 0,
            segment_bytes: 0,
            skip_crc: 0,
            debug_flags: 0,
            decode_all_tag_fields: 0,
            has_format_fields: 0,
            n_format_fields: 0,
            format_fields: std::ptr::null(),
        };
        let mut raw = std::ptr::null_mut();
        if unsafe { ffi::bamscan_open_fasta(c_path.as_ptr(), &opts, &mut raw) } != 0 {
            return Err(last_error());
        }
        let handle = Arc::new(Handle(raw));
        let mut c_schema = FFI_ArrowSchema::empty();
        if unsafe { ffi::bamscan_schema(handle.0, &mut c_schema) } != 0 {
            return Err(last_error());
        }
        let schema = Arc::new(Schema::try_from(&c_schema)?);
        Ok(Self { handle, schema, device_id })
    }

    pub fn device_id(&self) -> i32 {
        self.device_id
    }
}

impl Debug for GpuFastaTableProvider {
    fn fmt(&self, f: &mut Formatter<'_>) -> std::fmt::Result {
        f.debug_struct("GpuFastaTableProvider").field("device_id", &self.device_id).finish()
    }
}

#[async_trait]
impl TableProvider for GpuFastaTableProvider {
    fn as_any(&self) -> &dyn Any {
        self
    }
    fn schema(&self) -> SchemaRef {
        self.schema.clone()
    }
    fn table_type(&self) -> TableType {
        TableType::Base
    }

    fn supports_filters_pushdown(&self, filters: &[&Expr]) -> Result<Vec<TableProviderFilterPushDown>> {
        Ok(vec![TableProviderFilterPushDown::Unsupported; filters.len()])
    }

    async fn scan(&self, state: &dyn Session, projection: Option<&Vec<usize>>, _filters: &[Expr], limit: Option<usize>) -> Result<Arc<dyn ExecutionPlan>> {
        let proj: Option<Vec<i32>> = projection.map(|p| p.iter().map(|&i| i as i32).collect());
        let (proj_ptr, n_proj) = match &proj {
            Some(p) => (p.as_ptr(), p.len() as i32),
            None => (std::ptr::null(), -1),
        };
        let target = state.config().target_partitions() as i32;
        let mode = if target > 1 { ffi::PARTITION_BLOCK_RANGE } else { ffi::PARTITION_REFERENCE };
        let mut raw_plan = std::ptr::null_mut();
        let rc = unsafe {
            ffi::bamscan_plan(self.handle.0, proj_ptr, n_proj, std::ptr::null(), 0, limit.map(|l| l as i64).unwrap_or(-1), target, mode, &mut raw_plan)
        };
        if rc != 0 {
            return Err(last_error());
        }
        let plan = Arc::new(Plan { raw: raw_plan, _handle: self.handle.clone() });
        let mut c_schema = FFI_ArrowSchema::empty();
        if unsafe { ffi::bamscan_plan_schema(plan.raw, &mut c_schema) } != 0 {
            return Err(last_error());
        }
        let schema: SchemaRef = Arc::new(Schema::try_from(&c_schema)?);
        let n = unsafe { ffi::bamscan_plan_num_partitions(plan.raw) };
        let cache = PlanProperties::new(
            EquivalenceProperties::new(schema.clone()),
            Partitioning::UnknownPartitioning(n as usize),
            EmissionType::Final,
            Boundedness::Bounded,
        );
        Ok(Arc::new(GpuBamExec { plan, schema, cache: Arc::new(cache) }))
    }
}

/// A provider for BGZF-compressed VCF (`bamscan_open_vcf`), shaped like the BAM one: chrom, start, end, id, ref, alt, qual and
/// filter, then one column per selected `##INFO` field (Flag -> Boolean, Number=1 -> Int32 / Float32 / Utf8, any other Number ->
/// a list of those), then one column `format_<ID>` per selected FORMAT field holding one element per sample (`format_fields`
/// `None` or empty selects none, unlike `info_fields`; rules in bamscan.h).  `info_fields` `None` selects every `##INFO` field in header order;
/// at most 112 INFO columns can be projected in one scan (more fail with BAMSCAN_ERR_UNSUPPORTED).  No filter is pushed down
/// (DataFusion applies them), `limit` is passed on and not applied, and with `target_partitions` > 1 the file is cut into BGZF
/// block ranges balanced by compressed bytes (a line belongs to the range that holds its first byte).  Scans return
/// `GpuBamExec`, which streams the batches exactly as for BAM.
pub struct GpuVcfTableProvider {
    handle: Arc<Handle>,
    schema: SchemaRef,
    device_id: i32,
}

impl GpuVcfTableProvider {
    /// `object_storage_options` must be `None` (local files only).  `device_id` selects the GPU.
    pub fn new(file_path: String, info_fields: Option<Vec<String>>, object_storage_options: Option<String>, coordinate_system_zero_based: bool,
               device_id: i32, format_fields: Option<Vec<String>>) -> Result<Self> {
        if object_storage_options.is_some() {
            return Err(DataFusionError::NotImplemented("remote object storage is out of scope for this build (local files only)".into()));
        }
        let c_path = CString::new(file_path).map_err(|e| DataFusionError::Execution(e.to_string()))?;
        let c_ids: Vec<CString> = info_fields.iter().flatten().map(|s| CString::new(s.as_str())).collect::<std::result::Result<_, _>>()
            .map_err(|e| DataFusionError::Execution(e.to_string()))?;
        let id_ptrs: Vec<*const c_char> = c_ids.iter().map(|c| c.as_ptr()).collect();
        let c_fmt: Vec<CString> = format_fields.iter().flatten().map(|s| CString::new(s.as_str())).collect::<std::result::Result<_, _>>()
            .map_err(|e| DataFusionError::Execution(e.to_string()))?;
        let fmt_ptrs: Vec<*const c_char> = c_fmt.iter().map(|c| c.as_ptr()).collect();
        let opts = ffi::BamScanOptions {
            struct_size: std::mem::size_of::<ffi::BamScanOptions>() as u32,
            coordinate_system_zero_based: coordinate_system_zero_based as i32,
            binary_cigar: 0,
            has_tag_fields: info_fields.is_some() as i32,
            n_tag_fields: id_ptrs.len() as i32,
            tag_fields: if id_ptrs.is_empty() { std::ptr::null() } else { id_ptrs.as_ptr() },
            infer_tag_types: 0,
            infer_tag_sample_size: 0,
            n_tag_type_hints: 0,
            tag_type_hints: std::ptr::null(),
            device_id,
            batch_rows: 0,
            chunk_inflated_bytes: 0,
            segment_bytes: 0,
            skip_crc: 0,
            debug_flags: 0,
            decode_all_tag_fields: 0,
            has_format_fields: format_fields.is_some() as i32,
            n_format_fields: fmt_ptrs.len() as i32,
            format_fields: if fmt_ptrs.is_empty() { std::ptr::null() } else { fmt_ptrs.as_ptr() },
        };
        let mut raw = std::ptr::null_mut();
        if unsafe { ffi::bamscan_open_vcf(c_path.as_ptr(), &opts, &mut raw) } != 0 {
            return Err(last_error());
        }
        let handle = Arc::new(Handle(raw));
        let mut c_schema = FFI_ArrowSchema::empty();
        if unsafe { ffi::bamscan_schema(handle.0, &mut c_schema) } != 0 {
            return Err(last_error());
        }
        let schema = Arc::new(Schema::try_from(&c_schema)?);
        Ok(Self { handle, schema, device_id })
    }

    pub fn device_id(&self) -> i32 {
        self.device_id
    }
}

impl Debug for GpuVcfTableProvider {
    fn fmt(&self, f: &mut Formatter<'_>) -> std::fmt::Result {
        f.debug_struct("GpuVcfTableProvider").field("device_id", &self.device_id).finish()
    }
}

#[async_trait]
impl TableProvider for GpuVcfTableProvider {
    fn as_any(&self) -> &dyn Any {
        self
    }
    fn schema(&self) -> SchemaRef {
        self.schema.clone()
    }
    fn table_type(&self) -> TableType {
        TableType::Base
    }

    fn supports_filters_pushdown(&self, filters: &[&Expr]) -> Result<Vec<TableProviderFilterPushDown>> {
        Ok(vec![TableProviderFilterPushDown::Unsupported; filters.len()])
    }

    async fn scan(&self, state: &dyn Session, projection: Option<&Vec<usize>>, _filters: &[Expr], limit: Option<usize>) -> Result<Arc<dyn ExecutionPlan>> {
        let proj: Option<Vec<i32>> = projection.map(|p| p.iter().map(|&i| i as i32).collect());
        let (proj_ptr, n_proj) = match &proj {
            Some(p) => (p.as_ptr(), p.len() as i32),
            None => (std::ptr::null(), -1),
        };
        let target = state.config().target_partitions() as i32;
        let mode = if target > 1 { ffi::PARTITION_BLOCK_RANGE } else { ffi::PARTITION_REFERENCE };
        let mut raw_plan = std::ptr::null_mut();
        let rc = unsafe {
            ffi::bamscan_plan(self.handle.0, proj_ptr, n_proj, std::ptr::null(), 0, limit.map(|l| l as i64).unwrap_or(-1), target, mode, &mut raw_plan)
        };
        if rc != 0 {
            return Err(last_error());
        }
        let plan = Arc::new(Plan { raw: raw_plan, _handle: self.handle.clone() });
        let mut c_schema = FFI_ArrowSchema::empty();
        if unsafe { ffi::bamscan_plan_schema(plan.raw, &mut c_schema) } != 0 {
            return Err(last_error());
        }
        let schema: SchemaRef = Arc::new(Schema::try_from(&c_schema)?);
        let n = unsafe { ffi::bamscan_plan_num_partitions(plan.raw) };
        let cache = PlanProperties::new(
            EquivalenceProperties::new(schema.clone()),
            Partitioning::UnknownPartitioning(n as usize),
            EmissionType::Final,
            Boundedness::Bounded,
        );
        Ok(Arc::new(GpuBamExec { plan, schema, cache: Arc::new(cache) }))
    }
}
