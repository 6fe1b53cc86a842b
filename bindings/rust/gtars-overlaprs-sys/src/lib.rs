//! Raw FFI declarations for include/gtars_gpu.h (one `extern "C"` item per header entry point).
//! WRITTEN, NOT BUILT in this repository's environment (no Rust toolchain); kept in lock-step with the header by
//! tests/test_abi.py, which checks the header against the symbols libgtars_gpu.so exports.
#![allow(non_camel_case_types)]
use std::os::raw::{c_char, c_void};

#[repr(C)] pub struct gtgpu_ctx { _p: [u8; 0] }
#[repr(C)] pub struct gtgpu_index { _p: [u8; 0] }
#[repr(C)] pub struct gtgpu_igd { _p: [u8; 0] }
#[repr(C)] pub struct gtgpu_buf { _p: [u8; 0] }

pub const GTGPU_OK: i32 = 0;
pub const GTGPU_KIND_BITS: i32 = 0;
pub const GTGPU_KIND_AILIST: i32 = 1;
pub const GTGPU_UNKNOWN_CHROM: u32 = 0xFFFF_FFFF;

extern "C" {
    pub fn gtgpu_last_error() -> *const c_char;
    pub fn gtgpu_version() -> *const c_char;
    pub fn gtgpu_device_count(out_n: *mut i32) -> i32;
    pub fn gtgpu_init(device: i32, stream_or_null: *mut c_void, out_ctx: *mut *mut gtgpu_ctx) -> i32;
    pub fn gtgpu_init_multi(n_devices: i32, device_ids: *const i32, out_ctx: *mut *mut gtgpu_ctx) -> i32;
    pub fn gtgpu_ctx_devices(ctx: *const gtgpu_ctx, out_n: *mut i32, out_ids: *mut i32, cap: i32) -> i32;
    pub fn gtgpu_shutdown(ctx: *mut gtgpu_ctx) -> i32;
    pub fn gtgpu_synchronize(ctx: *mut gtgpu_ctx) -> i32;
    pub fn gtgpu_launch_count(ctx: *mut gtgpu_ctx, out_n: *mut u64) -> i32;
    pub fn gtgpu_timing_enable(ctx: *mut gtgpu_ctx, on: i32) -> i32;
    pub fn gtgpu_timing_read(ctx: *mut gtgpu_ctx, out_ms: *mut f32, cap: u32, out_n: *mut u32) -> i32;
    pub fn gtgpu_host_alloc(bytes: u64, out_ptr: *mut *mut c_void) -> i32;
    pub fn gtgpu_host_free(ptr: *mut c_void) -> i32;
    pub fn gtgpu_buf_data(buf: *const gtgpu_buf) -> *const c_void;
    pub fn gtgpu_buf_len(buf: *const gtgpu_buf) -> u64;
    pub fn gtgpu_buf_free(buf: *mut gtgpu_buf) -> i32;
    pub fn gtgpu_index_build(ctx: *mut gtgpu_ctx, kind: i32, n_chroms: u32, chrom_offsets: *const u64, starts: *const u32,
                             ends: *const u32, vals: *const u32, out_index: *mut *mut gtgpu_index) -> i32;
    pub fn gtgpu_index_free(index: *mut gtgpu_index) -> i32;
    pub fn gtgpu_index_info(index: *const gtgpu_index, info: *mut u64) -> i32;
    pub fn gtgpu_count(index: *mut gtgpu_index, n: u64, chr: *const u32, start: *const u32, end: *const u32,
                       min_overlap: i32, out_counts: *mut u32) -> i32;
    pub fn gtgpu_bits_count(index: *mut gtgpu_index, n: u64, chr: *const u32, start: *const u32, end: *const u32,
                            out_counts: *mut u64) -> i32;
    pub fn gtgpu_any(index: *mut gtgpu_index, n: u64, chr: *const u32, start: *const u32, end: *const u32,
                     min_overlap: i32, out_any: *mut u8) -> i32;
    pub fn gtgpu_find(index: *mut gtgpu_index, n: u64, chr: *const u32, start: *const u32, end: *const u32,
                      min_overlap: i32, out_offsets: *mut u64, out_vals: *mut *mut gtgpu_buf) -> i32;
    pub fn gtgpu_tokenize_files(index: *mut gtgpu_index, n_files: u64, file_offsets: *const u64, chr: *const u32,
                                start: *const u32, end: *const u32, unk_id: u32, out_file_token_offsets: *mut u64,
                                out_ids: *mut *mut gtgpu_buf) -> i32;
    pub fn gtgpu_tokenize_files_runs(index: *mut gtgpu_index, n_files: u64, file_offsets: *const u64, n_runs: u64,
                                     run_offsets: *const u64, run_chr: *const u32, start: *const u32, end: *const u32,
                                     unk_id: u32, out_file_token_offsets: *mut u64, out_ids: *mut *mut gtgpu_buf) -> i32;
    pub fn gtgpu_tokenize_files_compact(index: *mut gtgpu_index, n_files: u64, file_offsets: *const u64, n_runs: u64,
                                        run_offsets: *const u64, run_chr: *const u32, start: *const u32, width16: *const u16,
                                        n_wide: u64, wide_index: *const u64, wide_end: *const u32, unk_id: u32,
                                        out_file_token_offsets: *mut u64, out_ids: *mut *mut gtgpu_buf) -> i32;
    pub fn gtgpu_parse_bed(ctx: *mut gtgpu_ctx, text: *const u8, n_bytes: u64, n_names: u32, names: *const u8,
                           name_offsets: *const u32, out_n: *mut u64, out_chr: *mut *mut gtgpu_buf,
                           out_start: *mut *mut gtgpu_buf, out_end: *mut *mut gtgpu_buf) -> i32;
    pub fn gtgpu_tokenize_bed(index: *mut gtgpu_index, text: *const u8, n_bytes: u64, n_names: u32, names: *const u8,
                              name_offsets: *const u32, unk_id: u32, out_ids: *mut *mut gtgpu_buf) -> i32;
    /// Tokenizer::encode(RegionSet::try_from(file f)) for every file of a batch (file f = text[file_offsets[f], file_offsets[f + 1]),
    /// any total size) in one device pass; out_file_token_offsets (n_files + 1) index *out_ids as in gtgpu_tokenize_files.
    pub fn gtgpu_tokenize_bed_files(index: *mut gtgpu_index, n_files: u64, text: *const c_char, file_offsets: *const u64, n_names: u32,
                                    names: *const u8, name_offsets: *const u32, unk_id: u32, out_file_token_offsets: *mut u64,
                                    out_ids: *mut *mut gtgpu_buf) -> i32;
    /// The same from gzip members: file f = members [file_members[f], file_members[f + 1]) of gz / member_offsets.
    pub fn gtgpu_tokenize_bed_files_gz(index: *mut gtgpu_index, n_files: u64, file_members: *const u64, n_members: u64, gz: *const u8,
                                       member_offsets: *const u64, n_names: u32, names: *const u8, name_offsets: *const u32,
                                       unk_id: u32, out_file_token_offsets: *mut u64, out_ids: *mut *mut gtgpu_buf) -> i32;
    pub fn gtgpu_tokenize_fragments_text(index: *mut gtgpu_index, text: *const u8, n_bytes: u64, n_names: u32, names: *const u8,
                                         name_offsets: *const u32, unk_id: u32, out_n_barcodes: *mut u32,
                                         out_barcode_spans: *mut *mut gtgpu_buf, out_barcode_offsets: *mut *mut gtgpu_buf,
                                         out_ids: *mut *mut gtgpu_buf) -> i32;
    pub fn gtgpu_tokenize_fragments(index: *mut gtgpu_index, n: u64, chr: *const u32, start: *const u32, end: *const u32,
                                    barcode_id: *const u32, n_barcodes: u32, unk_id: u32, out_barcode_offsets: *mut u64,
                                    out_ids: *mut *mut gtgpu_buf) -> i32;
    pub fn gtgpu_tokenize_fragments_dev(index: *mut gtgpu_index, n: u64, d_chr: *const u32, d_start: *const u32, d_end: *const u32,
                                        d_barcode_id: *const u32, n_barcodes: u32, unk_id: u32, d_out_barcode_offsets: *mut u64,
                                        d_out_ids: *mut u32, ids_capacity: u64, d_out_total: *mut u64) -> i32;
    pub fn gtgpu_marshal_compact(n: u64, chr: *const u32, start: *const u32, end: *const u32, n_files: u64, file_offsets: *const u64,
                                 threads: i32, out_width16: *mut u16, run_capacity: u64, out_run_offsets: *mut u64,
                                 out_run_chr: *mut u32, out_n_runs: *mut u64, wide_capacity: u64, out_wide_index: *mut u64,
                                 out_wide_end: *mut u32, out_n_wide: *mut u64) -> i32;
    pub fn gtgpu_tokenize_files_packed(index: *mut gtgpu_index, n_files: u64, file_offsets: *const u64, n_runs: u64,
                                       run_offsets: *const u64, run_chr: *const u32, width_bits: u32, packed: *const u32,
                                       anchors: *const u32, n_exc: u64, exc_index: *const u64, exc_start: *const u32,
                                       exc_end: *const u32, unk_id: u32, out_file_token_offsets: *mut u64,
                                       out_ids: *mut *mut gtgpu_buf) -> i32;
    pub fn gtgpu_marshal_packed(n: u64, chr: *const u32, start: *const u32, end: *const u32, n_files: u64, file_offsets: *const u64,
                                threads: i32, width_bits: u32, out_packed: *mut u32, out_anchors: *mut u32, run_capacity: u64,
                                out_run_offsets: *mut u64, out_run_chr: *mut u32, out_n_runs: *mut u64, exc_capacity: u64,
                                out_exc_index: *mut u64, out_exc_start: *mut u32, out_exc_end: *mut u32, out_n_exc: *mut u64,
                                out_width_bits: *mut u32) -> i32;
    pub fn gtgpu_gzip_members(gz: *const u8, n_bytes: u64, capacity: u64, out_member_offsets: *mut u64, out_n_members: *mut u64) -> i32;
    pub fn gtgpu_gunzip(ctx: *mut gtgpu_ctx, n_members: u64, gz: *const u8, member_offsets: *const u64,
                        out_text: *mut *mut gtgpu_buf, out_member_offsets: *mut u64) -> i32;
    pub fn gtgpu_tokenize_bed_gz(index: *mut gtgpu_index, n_members: u64, gz: *const u8, member_offsets: *const u64, n_names: u32,
                                 names: *const u8, name_offsets: *const u32, unk_id: u32, out_ids: *mut *mut gtgpu_buf) -> i32;
    pub fn gtgpu_tokenize_fragments_gz(index: *mut gtgpu_index, n_members: u64, gz: *const u8, member_offsets: *const u64,
                                       n_names: u32, names: *const u8, name_offsets: *const u32, unk_id: u32,
                                       out_n_barcodes: *mut u32, out_barcode_spans: *mut *mut gtgpu_buf,
                                       out_barcode_offsets: *mut *mut gtgpu_buf, out_ids: *mut *mut gtgpu_buf,
                                       out_text: *mut *mut gtgpu_buf) -> i32;
    pub fn gtgpu_tokenize_fragments_file(index: *mut gtgpu_index, text: *const u8, n_bytes: u64, n_names: u32, names: *const u8,
                                         name_offsets: *const u32, unk_id: u32, out_n_barcodes: *mut u32,
                                         out_barcode_names: *mut *mut gtgpu_buf, out_barcode_name_offsets: *mut *mut gtgpu_buf,
                                         out_barcode_offsets: *mut *mut gtgpu_buf, out_ids: *mut *mut gtgpu_buf) -> i32;
    pub fn gtgpu_tokenize_fragments_file_gz(index: *mut gtgpu_index, n_members: u64, gz: *const u8, member_offsets: *const u64,
                                            n_names: u32, names: *const u8, name_offsets: *const u32, unk_id: u32,
                                            out_n_barcodes: *mut u32, out_barcode_names: *mut *mut gtgpu_buf,
                                            out_barcode_name_offsets: *mut *mut gtgpu_buf, out_barcode_offsets: *mut *mut gtgpu_buf,
                                            out_ids: *mut *mut gtgpu_buf) -> i32;
    pub fn gtgpu_score_matrix(index: *mut gtgpu_index, n_files: u64, file_offsets: *const u64, n: u64, chr: *const u32,
                              start: *const u32, end: *const u32, mode: i32, n_cols: u64, out_counts: *mut u32) -> i32;
    pub fn gtgpu_score_matrix_dev(index: *mut gtgpu_index, n_files: u64, d_file_offsets: *const u64, n: u64,
                                  d_chr: *const u32, d_start: *const u32, d_end: *const u32, mode: i32, n_cols: u64,
                                  d_out_counts: *mut u32) -> i32;
    pub fn gtgpu_score_barcodes(index: *mut gtgpu_index, n: u64, chr: *const u32, start: *const u32, end: *const u32,
                                barcode_id: *const u32, n_barcodes: u32, out_barcode_offsets: *mut u64,
                                out_peaks: *mut *mut gtgpu_buf, out_counts: *mut *mut gtgpu_buf) -> i32;
    pub fn gtgpu_score_matrix_text(index: *mut gtgpu_index, text: *const u8, n_bytes: u64, n_names: u32, names: *const u8,
                                   name_offsets: *const u32, mode: i32, n_cols: u64, out_row: *mut u32) -> i32;
    pub fn gtgpu_score_matrix_gz(index: *mut gtgpu_index, n_members: u64, gz: *const u8, member_offsets: *const u64, n_names: u32,
                                 names: *const u8, name_offsets: *const u32, mode: i32, n_cols: u64, out_row: *mut u32) -> i32;
    pub fn gtgpu_score_barcodes_text(index: *mut gtgpu_index, text: *const u8, n_bytes: u64, n_names: u32, names: *const u8,
                                     name_offsets: *const u32, out_n_barcodes: *mut u32, out_barcode_names: *mut *mut gtgpu_buf,
                                     out_barcode_name_offsets: *mut *mut gtgpu_buf, out_barcode_offsets: *mut *mut gtgpu_buf,
                                     out_peaks: *mut *mut gtgpu_buf, out_counts: *mut *mut gtgpu_buf) -> i32;
    pub fn gtgpu_score_barcodes_gz(index: *mut gtgpu_index, n_members: u64, gz: *const u8, member_offsets: *const u64, n_names: u32,
                                   names: *const u8, name_offsets: *const u32, out_n_barcodes: *mut u32,
                                   out_barcode_names: *mut *mut gtgpu_buf, out_barcode_name_offsets: *mut *mut gtgpu_buf,
                                   out_barcode_offsets: *mut *mut gtgpu_buf, out_peaks: *mut *mut gtgpu_buf,
                                   out_counts: *mut *mut gtgpu_buf) -> i32;
    pub fn gtgpu_igd_build(ctx: *mut gtgpu_ctx, n_files: u64, file_offsets: *const u64, n_chroms: u32, chr: *const u32,
                           start: *const u32, end: *const u32, out_igd: *mut *mut gtgpu_igd) -> i32;
    /// An IGD from its BED files' text (file f = text[file_offsets[f], file_offsets[f + 1]), any size), parsed on the device;
    /// the chromosome names come back in id order (bytes + n_chroms + 1 u64 offsets).
    pub fn gtgpu_igd_build_bed(ctx: *mut gtgpu_ctx, n_files: u64, text: *const c_char, file_offsets: *const u64, out_n_chroms: *mut u32,
                               out_chrom_names: *mut *mut gtgpu_buf, out_chrom_name_offsets: *mut *mut gtgpu_buf,
                               out_igd: *mut *mut gtgpu_igd) -> i32;
    /// The same from gzip members: file f = members [file_members[f], file_members[f + 1]) of gz / member_offsets.
    pub fn gtgpu_igd_build_bed_gz(ctx: *mut gtgpu_ctx, n_files: u64, file_members: *const u64, n_members: u64, gz: *const u8,
                                  member_offsets: *const u64, out_n_chroms: *mut u32, out_chrom_names: *mut *mut gtgpu_buf,
                                  out_chrom_name_offsets: *mut *mut gtgpu_buf, out_igd: *mut *mut gtgpu_igd) -> i32;
    pub fn gtgpu_igd_free(igd: *mut gtgpu_igd) -> i32;
    /// Igd::save of a database built any way: the .igd file's bytes (u8 buffer), and per file the .tsv region count and width
    /// sum (n_files each).  names: the chromosome names by id (n_names + 1 u32 offsets), n_names == the igd's chromosome count.
    pub fn gtgpu_igd_serialize(igd: *mut gtgpu_igd, n_names: u32, names: *const u8, name_offsets: *const u32,
                               out_igd_bytes: *mut *mut gtgpu_buf, out_file_regions: *mut u64, out_file_width_sums: *mut u64) -> i32;
    pub fn gtgpu_igd_info(igd: *const gtgpu_igd, info: *mut u64) -> i32;
    pub fn gtgpu_igd_count_set_overlaps(igd: *mut gtgpu_igd, n_sets: u64, set_offsets: *const u64, chr: *const u32,
                                        start: *const u32, end: *const u32, min_overlap: i32, out: *mut u64) -> i32;
    pub fn gtgpu_igd_count_region_hits(igd: *mut gtgpu_igd, n_sets: u64, set_offsets: *const u64, chr: *const u32,
                                       start: *const u32, end: *const u32, min_overlap: i32, out: *mut u64) -> i32;
    pub fn gtgpu_igd_count_dev(igd: *mut gtgpu_igd, binary: i32, n: u64, d_set_of: *const u32, d_chr: *const u32,
                               d_start: *const u32, d_end: *const u32, min_overlap: i32, d_out: *mut u64) -> i32;
    /// count_region_hits (binary = 1) / count_set_overlaps (binary = 0) of query sets given as BED files (set s = text[file_offsets[s],
    /// file_offsets[s + 1])), parsed on the device; names map through the caller's table.  out: [n_sets x n_files];
    /// out_set_regions: every set's region lines.
    pub fn gtgpu_igd_count_bed(igd: *mut gtgpu_igd, binary: i32, n_sets: u64, text: *const c_char, file_offsets: *const u64, n_names: u32,
                               names: *const u8, name_offsets: *const u32, min_overlap: i32, out: *mut u64,
                               out_set_regions: *mut u64) -> i32;
    /// The same from gzip members: set s = members [file_members[s], file_members[s + 1]) of gz / member_offsets.
    pub fn gtgpu_igd_count_bed_gz(igd: *mut gtgpu_igd, binary: i32, n_sets: u64, file_members: *const u64, n_members: u64, gz: *const u8,
                                  member_offsets: *const u64, n_names: u32, names: *const u8, name_offsets: *const u32,
                                  min_overlap: i32, out: *mut u64, out_set_regions: *mut u64) -> i32;
    pub fn gtgpu_comm_unique_id(out_id: *mut u8) -> i32;
    pub fn gtgpu_comm_init(ctx: *mut gtgpu_ctx, world: i32, rank: i32, id: *const u8) -> i32;
    pub fn gtgpu_comm_free(ctx: *mut gtgpu_ctx) -> i32;
    pub fn gtgpu_igd_count_sharded(ctx: *mut gtgpu_ctx, igd: *mut gtgpu_igd, binary: i32, n_files_global: u64, n_sets: u64,
                                   set_offsets: *const u64, chr: *const u32, start: *const u32, end: *const u32,
                                   min_overlap: i32, out: *mut u64) -> i32;
    pub fn gtgpu_count_dev(index: *mut gtgpu_index, n: u64, d_chr: *const u32, d_start: *const u32, d_end: *const u32,
                           min_overlap: i32, d_out_counts: *mut u32) -> i32;
    pub fn gtgpu_find_dev(index: *mut gtgpu_index, n: u64, d_chr: *const u32, d_start: *const u32, d_end: *const u32,
                          min_overlap: i32, n_files: u64, d_file_offsets: *const u64, d_out_ids: *mut u32, ids_capacity: u64,
                          d_out_offsets: *mut u64, d_out_file_token_offsets: *mut u64, d_out_total: *mut u64) -> i32;
    pub fn gtgpu_unk_rule_dev(ctx: *mut gtgpu_ctx, n_files: u64, d_raw_file_token_offsets: *const u64, d_raw_ids: *const u32,
                              unk_id: u32, d_out_file_token_offsets: *mut u64, d_out_ids: *mut u32, d_out_n_empty: *mut u64) -> i32;
}
