//! The write path behind `BamWriteExec::execute` (`datafusion/bio-format-bam/src/write_exec.rs:195-350`): `write_bam_stream` with
//! the noodles writer and `batch_to_bam_records` replaced by `bamscan_writer_*` (Arrow batches -> BAM records -> BGZF members on
//! the GPU).  `build_bam_header` (`header_builder.rs:43-186`) stays the reference's own function; its result crosses the ABI as SAM
//! text plus the reference dictionary.  SOURCE-ONLY like the rest of this crate.

use crate::ffi;
use arrow::array::{Array, RecordBatch, StructArray};
use arrow::datatypes::{DataType, SchemaRef};
use arrow::ffi::{to_ffi, FFI_ArrowSchema};
use datafusion::common::{DataFusionError, Result};
use std::ffi::{c_char, CStr, CString};

fn last_error() -> DataFusionError {
    let msg = unsafe { CStr::from_ptr(ffi::bamscan_last_error()) }.to_string_lossy().into_owned();
    DataFusionError::Execution(msg)
}

/// Owns a `BamWriter*`; dropping it without `finish` discards the tail like dropping the reference's writer would.
pub struct GpuBamWriter(*mut ffi::BamWriter);
unsafe impl Send for GpuBamWriter {}

impl GpuBamWriter {
    /// `sam_header_text`: the header `build_bam_header(&effective_schema, &tag_fields)` gives, serialised with
    /// `noodles_sam::io::Writer::write_header`; `references`: `header.reference_sequences()` as (name, length).
    pub fn open(
        output_path: &str,
        sam_header_text: &str,
        references: &[(String, i32)],
        input_schema: &SchemaRef,
        tag_fields: &[String],
        coordinate_system_zero_based: bool,
        device_id: i32,
    ) -> Result<Self> {
        let c_path = CString::new(output_path).map_err(|e| DataFusionError::Execution(e.to_string()))?;
        let c_text = CString::new(sam_header_text).map_err(|e| DataFusionError::Execution(e.to_string()))?;
        let names: Vec<CString> = references.iter().map(|(n, _)| CString::new(n.as_str()).unwrap()).collect();
        let name_ptrs: Vec<*const c_char> = names.iter().map(|n| n.as_ptr()).collect();
        let lens: Vec<i32> = references.iter().map(|(_, l)| *l).collect();
        let tags: Vec<CString> = tag_fields.iter().map(|t| CString::new(t.as_str()).unwrap()).collect();
        let tag_ptrs: Vec<*const c_char> = tags.iter().map(|t| t.as_ptr()).collect();
        let c_schema = FFI_ArrowSchema::try_from(&DataType::Struct(input_schema.fields().clone()))?;
        let opts = ffi::BamWriteOptions {
            struct_size: std::mem::size_of::<ffi::BamWriteOptions>() as u32,
            coordinate_system_zero_based: coordinate_system_zero_based as i32,
            n_tag_fields: tag_ptrs.len() as i32,
            tag_fields: tag_ptrs.as_ptr(),
            device_id,
            compression: 0,
        };
        let mut raw: *mut ffi::BamWriter = std::ptr::null_mut();
        let rc = unsafe {
            ffi::bamscan_writer_open(c_path.as_ptr(), c_text.as_ptr(), names.len() as i32, name_ptrs.as_ptr(), lens.as_ptr(), &c_schema, &opts, &mut raw)
        };
        if rc != 0 {
            return Err(last_error());
        }
        Ok(Self(raw))
    }

    /// == `batch_to_bam_records` + `writer.write_records` for one batch (write_exec.rs:322-337).
    pub fn write(&mut self, batch: &RecordBatch) -> Result<()> {
        let (array, _schema) = to_ffi(&StructArray::from(batch.clone()).into_data())?;
        if unsafe { ffi::bamscan_writer_write(self.0, &array) } != 0 {
            return Err(last_error());
        }
        Ok(())
    }

    /// == `writer.finish(&header)`; returns the row count of the reference's one-row `count` batch (write_exec.rs:339-349).
    pub fn finish(self) -> Result<u64> {
        let mut rows = 0u64;
        if unsafe { ffi::bamscan_writer_finish(self.0, &mut rows) } != 0 {
            return Err(last_error());
        }
        Ok(rows)
    }
}

impl Drop for GpuBamWriter {
    fn drop(&mut self) {
        unsafe { ffi::bamscan_writer_free(self.0) }
    }
}

/// FASTQ output for `FastqTableProvider::insert_into`: `bamscan_fastq_writer_open` + the same `bamscan_writer_*` calls.  The
/// name / description / sequence / quality_scores columns are looked up by name (description optional, other columns ignored);
/// `compression`: 0 BGZF, 1 BGZF with stored blocks, 2 plain text.  Bases are written as stored (no reverse-complementing).
pub struct GpuFastqWriter(*mut ffi::BamWriter);
unsafe impl Send for GpuFastqWriter {}

impl GpuFastqWriter {
    /// `compression` None: BGZF for `.bgz` / `.bgzf` / `.gz` paths, plain text otherwise.
    pub fn open(output_path: &str, input_schema: &SchemaRef, compression: Option<i32>, device_id: i32) -> Result<Self> {
        let c_path = CString::new(output_path).map_err(|e| DataFusionError::Execution(e.to_string()))?;
        let lower = output_path.to_ascii_lowercase();
        let bgzf = [".bgz", ".bgzf", ".gz"].iter().any(|s| lower.ends_with(s));
        let c_schema = FFI_ArrowSchema::try_from(&DataType::Struct(input_schema.fields().clone()))?;
        let opts = ffi::BamWriteOptions {
            struct_size: std::mem::size_of::<ffi::BamWriteOptions>() as u32,
            coordinate_system_zero_based: 1,
            n_tag_fields: 0,
            tag_fields: std::ptr::null(),
            device_id,
            compression: compression.unwrap_or(if bgzf { 0 } else { 2 }),
        };
        let mut raw: *mut ffi::BamWriter = std::ptr::null_mut();
        if unsafe { ffi::bamscan_fastq_writer_open(c_path.as_ptr(), &c_schema, &opts, &mut raw) } != 0 {
            return Err(last_error());
        }
        Ok(Self(raw))
    }

    /// One batch (host memory), not consumed.
    pub fn write(&mut self, batch: &RecordBatch) -> Result<()> {
        let (array, _schema) = to_ffi(&StructArray::from(batch.clone()).into_data())?;
        if unsafe { ffi::bamscan_writer_write(self.0, &array) } != 0 {
            return Err(last_error());
        }
        Ok(())
    }

    /// Flushes the last member and the EOF marker (BGZF) and closes the file; returns the row count.
    pub fn finish(self) -> Result<u64> {
        let mut rows = 0u64;
        if unsafe { ffi::bamscan_writer_finish(self.0, &mut rows) } != 0 {
            return Err(last_error());
        }
        Ok(rows)
    }
}

impl Drop for GpuFastqWriter {
    fn drop(&mut self) {
        unsafe { ffi::bamscan_writer_free(self.0) }
    }
}

/// SAM output for `.sam` targets (the reference's `is_sam` rule): `bamscan_sam_writer_open` with `GpuBamWriter::open`'s
/// arguments, then the same `bamscan_writer_*` calls.  The file is the header text as given and one SAM line per row (no BGZF).
/// Rows are accepted and refused as by the BAM writer, plus the SAM-only refusals of DESIGN 3.9.  SOURCE-ONLY: never compiled here.
pub struct GpuSamWriter(*mut ffi::BamWriter);
unsafe impl Send for GpuSamWriter {}

impl GpuSamWriter {
    pub fn open(
        output_path: &str,
        sam_header_text: &str,
        references: &[(String, i32)],
        input_schema: &SchemaRef,
        tag_fields: &[String],
        coordinate_system_zero_based: bool,
        device_id: i32,
    ) -> Result<Self> {
        let c_path = CString::new(output_path).map_err(|e| DataFusionError::Execution(e.to_string()))?;
        let c_text = CString::new(sam_header_text).map_err(|e| DataFusionError::Execution(e.to_string()))?;
        let names: Vec<CString> = references.iter().map(|(n, _)| CString::new(n.as_str()).unwrap()).collect();
        let name_ptrs: Vec<*const c_char> = names.iter().map(|n| n.as_ptr()).collect();
        let lens: Vec<i32> = references.iter().map(|(_, l)| *l).collect();
        let tags: Vec<CString> = tag_fields.iter().map(|t| CString::new(t.as_str()).unwrap()).collect();
        let tag_ptrs: Vec<*const c_char> = tags.iter().map(|t| t.as_ptr()).collect();
        let c_schema = FFI_ArrowSchema::try_from(&DataType::Struct(input_schema.fields().clone()))?;
        let opts = ffi::BamWriteOptions {
            struct_size: std::mem::size_of::<ffi::BamWriteOptions>() as u32,
            coordinate_system_zero_based: coordinate_system_zero_based as i32,
            n_tag_fields: tag_ptrs.len() as i32,
            tag_fields: tag_ptrs.as_ptr(),
            device_id,
            compression: 0,
        };
        let mut raw: *mut ffi::BamWriter = std::ptr::null_mut();
        let rc = unsafe {
            ffi::bamscan_sam_writer_open(c_path.as_ptr(), c_text.as_ptr(), names.len() as i32, name_ptrs.as_ptr(), lens.as_ptr(), &c_schema, &opts, &mut raw)
        };
        if rc != 0 {
            return Err(last_error());
        }
        Ok(Self(raw))
    }

    /// One batch (host memory), not consumed.
    pub fn write(&mut self, batch: &RecordBatch) -> Result<()> {
        let (array, _schema) = to_ffi(&StructArray::from(batch.clone()).into_data())?;
        if unsafe { ffi::bamscan_writer_write(self.0, &array) } != 0 {
            return Err(last_error());
        }
        Ok(())
    }

    /// Writes the remaining lines and closes the file; returns the row count.
    pub fn finish(self) -> Result<u64> {
        let mut rows = 0u64;
        if unsafe { ffi::bamscan_writer_finish(self.0, &mut rows) } != 0 {
            return Err(last_error());
        }
        Ok(rows)
    }
}

impl Drop for GpuSamWriter {
    fn drop(&mut self) {
        unsafe { ffi::bamscan_writer_free(self.0) }
    }
}
