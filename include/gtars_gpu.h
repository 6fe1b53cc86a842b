/* gtars_gpu.h — C ABI of the B200-native interval-overlap engine (libgtars_gpu.so).
 *
 * This is the drop-in boundary for gtars' data-parallel hot path: the bodies of the batch-shaped Rust APIs
 * cited on each entry point below would, under a `cuda` cargo feature, marshal their inputs into flat SoA
 * arrays and call these functions (binding sketch: INTEGRATION.md, bindings/rust/).  The reference has no FFI
 * seam today (SURVEY.md §8b), so every entry point names the reference function whose body it replaces.
 *
 * Conventions
 *  - every function returns an int32 status (GTGPU_OK = 0); nothing throws or unwinds across the boundary;
 *    gtgpu_last_error() returns a thread-local message for the last failing call on this thread.
 *  - gtgpu_init gives a context on ONE CUDA device; gtgpu_init_multi gives one context that owns SEVERAL devices of the
 *    same process (SURVEY.md 8b): indexes built on it are replicated, IGD databases sharded by region set, and the host
 *    entry points shard their work over the devices internally — query blocks / files / fragments for count, find,
 *    tokenize and scoring (no collective), database columns + one ncclAllGather between the devices for the IGD / LOLA
 *    count matrices — and return exactly what a single device returns.  That is what makes all GPUs of a box reachable
 *    behind the unchanged Tokenizer::encode / run_lola signatures of a single Python / R / Rust process.  The
 *    process-per-GPU form (one ctx per rank + gtgpu_comm_*) stays available for MPI / torchrun style launches.
 *  - chromosome names are mapped to dense uint32 ids by the caller; GTGPU_UNKNOWN_CHROM (or any id >= n_chroms)
 *    means "chromosome not in the index" and contributes no hits, exactly like the reference's map lookups
 *    (gtars-tokenizers/src/tokenizer.rs:144, gtars-overlaprs/src/multi_chrom_overlapper.rs:231-234,
 *    gtars-igd/src/igd.rs:519-522).
 *  - coordinates are half-open [start,end), uint32 for overlaprs/tokenizers (Interval<u32,u32>), int32 semantics
 *    for IGD (the reference casts u32→i32, igd.rs:295-296,549-550; values must be < 2^31).
 *  - "host" entry points take caller-owned host arrays (pinned memory — see gtgpu_host_alloc — makes the copies
 *    true DMA) and include H2D/D2H; "_dev" entry points take device pointers, are asynchronous on the ctx stream
 *    and move no data.  Outputs of unknown size are returned as library-owned pinned buffers (gtgpu_buf).
 *  - there is NO CPU fallback: without a usable CUDA device gtgpu_init fails.
 */
#ifndef GTARS_GPU_H
#define GTARS_GPU_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GTGPU_OK 0
#define GTGPU_ERR_INVALID 1   /* bad argument */
#define GTGPU_ERR_CUDA 2      /* CUDA runtime error (message has the cudaError string) */
#define GTGPU_ERR_NOMEM 3     /* host or device allocation failed */
#define GTGPU_ERR_CAPACITY 4  /* caller-provided device output buffer too small; *out_total has the need */
#define GTGPU_ERR_NCCL 5      /* NCCL not loadable / collective failed */
#define GTGPU_ERR_UNSUPPORTED 6

#define GTGPU_KIND_BITS 0   /* gtars_overlaprs::Bits   — hits in ascending (start,end,insertion) order */
#define GTGPU_KIND_AILIST 1 /* gtars_overlaprs::AIList — component-major, descending position         */

#define GTGPU_UNKNOWN_CHROM 0xFFFFFFFFu

typedef struct gtgpu_ctx gtgpu_ctx;
typedef struct gtgpu_index gtgpu_index; /* immutable after build; usable from several host threads */
typedef struct gtgpu_igd gtgpu_igd;
typedef struct gtgpu_buf gtgpu_buf;     /* library-owned pinned host result buffer */

/* ---- library / context ------------------------------------------------------------------------------- */
const char* gtgpu_last_error(void);
const char* gtgpu_version(void);
int32_t gtgpu_device_count(int32_t* out_n);
/* stream_or_null: a cudaStream_t to run on (e.g. the caller's / torch's current stream) or NULL for an
 * internal non-blocking stream. */
int32_t gtgpu_init(int32_t device, void* stream_or_null, gtgpu_ctx** out_ctx);
/* One context over n_devices CUDA devices of this process (device_ids NULL = devices 0 .. n_devices-1), each with its own
 * internal streams, scratch and pinned staging; n_devices == 1 equals gtgpu_init(device_ids[0], NULL).  "_dev" entry points
 * (device pointers) and the text-ingest entry points run on the first device.  gtgpu_ctx_devices reports the devices. */
int32_t gtgpu_init_multi(int32_t n_devices, const int32_t* device_ids, gtgpu_ctx** out_ctx);
int32_t gtgpu_ctx_devices(const gtgpu_ctx* ctx, int32_t* out_n, int32_t* out_ids, int32_t cap);
int32_t gtgpu_shutdown(gtgpu_ctx* ctx);
int32_t gtgpu_synchronize(gtgpu_ctx* ctx);
/* Number of kernels this ctx (all its devices) has launched so far (bench.py's gpu_launches). */
int32_t gtgpu_launch_count(gtgpu_ctx* ctx, uint64_t* out_n);

/* Kernel timing: when enabled, every launch of a dominant kernel (fused find / count / IGD count) is bracketed by
 * CUDA events on the ctx stream (up to 256 launches are kept, then recording stops).  gtgpu_timing_read
 * synchronises the stream, writes the elapsed milliseconds of the first min(cap, recorded) launches, returns how
 * many were recorded in *out_n and clears the log. */
int32_t gtgpu_timing_enable(gtgpu_ctx* ctx, int32_t on);
int32_t gtgpu_timing_read(gtgpu_ctx* ctx, float* out_ms, uint32_t cap, uint32_t* out_n);

/* pinned host memory for caller-side SoA arrays */
int32_t gtgpu_host_alloc(uint64_t bytes, void** out_ptr);
int32_t gtgpu_host_free(void* ptr);

/* result buffers */
const void* gtgpu_buf_data(const gtgpu_buf* buf);
uint64_t gtgpu_buf_len(const gtgpu_buf* buf); /* elements (4-byte ids unless the entry point says otherwise), not bytes */
int32_t gtgpu_buf_free(gtgpu_buf* buf);       /* returns the pinned block to the ctx cache */

/* ---- index: Overlapper::build per chromosome -------------------------------------------------------------
 * Replaces Bits::build (gtars-overlaprs/src/bits.rs:101-128) / AIList::build (ailist.rs:105-151) for every
 * chromosome of a MultiChromOverlapper (multi_chrom_overlapper.rs:130-200) or of a tokenizer core
 * (gtars-tokenizers/src/utils/mod.rs:49-99).  Chromosome c owns intervals [chrom_offsets[c], chrom_offsets[c+1])
 * given in the caller's INSERTION order; the library performs the reference's stable sort / decomposition so
 * hit order semantics live in one place.  vals may be NULL (val = global insertion index).
 * A chromosome with no intervals behaves as "absent". */
int32_t gtgpu_index_build(gtgpu_ctx* ctx, int32_t kind, uint32_t n_chroms, const uint64_t* chrom_offsets,
                          const uint32_t* starts, const uint32_t* ends, const uint32_t* vals,
                          gtgpu_index** out_index);
int32_t gtgpu_index_free(gtgpu_index* index);
/* info[0]=n_intervals, [1]=n_segments (chromosome×AIList component), [2]=device bytes, [3]=lut shift,
 * [4]=max components on one chromosome, [5]=1 if every interval has start<=end, [6]=bin-table bins,
 * [7]=bin-table windows served by the generic walk (too many candidates), [8]=bin-table shift,
 * [9]=bin-table windows with a pooled candidate list (nested intervals / several AIList components),
 * [10]=1 if every window is a plain record (the lean find kernel serves the index, the full kernel is queued behind it
 * as an on-device fallback), [11]=1 once a launch on this index had to take that fallback (the lean kernel is then no
 * longer tried; the flag is read lazily, so it shows at the latest after the launch following the fallback) */
int32_t gtgpu_index_info(const gtgpu_index* index, uint64_t info[12]);

/* ---- batch queries, host buffers ------------------------------------------------------------------------ */
/* MultiChromOverlapper::count_overlaps (multi_chrom_overlapper.rs:483-498): out_counts[i] = number of indexed
 * intervals overlapping query i; min_overlap is applied only when > 1 (bp of overlap), as in the reference.
 * Databases whose search tables exceed the L2 (tens of millions of intervals) are served by bucketing the batch by
 * table slice on the device first (DESIGN.md 4.2); the output is the same array in the caller's query order. */
int32_t gtgpu_count(gtgpu_index* index, uint64_t n, const uint32_t* chr, const uint32_t* start,
                    const uint32_t* end, int32_t min_overlap, uint32_t* out_counts);
/* Bits::count (bits.rs:337-344), the two-binary-search identity, with the reference's wrapping usize
 * arithmetic (`start+1` wraps in u32; the difference wraps in u64).  Index must be GTGPU_KIND_BITS. */
int32_t gtgpu_bits_count(gtgpu_index* index, uint64_t n, const uint32_t* chr, const uint32_t* start,
                         const uint32_t* end, uint64_t* out_counts);
/* MultiChromOverlapper::any_overlaps (multi_chrom_overlapper.rs:501-516). */
int32_t gtgpu_any(gtgpu_index* index, uint64_t n, const uint32_t* chr, const uint32_t* start,
                  const uint32_t* end, int32_t min_overlap, uint8_t* out_any);
/* Overlapper::find for a batch (bits.rs:141-156, ailist.rs:153-178; callers: find_overlaps_regions
 * multi_chrom_overlapper.rs:524-550, IndexedRegionSet::find_overlaps indexed_region_set.rs:145-263):
 * out_offsets[n+1] (caller-allocated), *out_vals = the hits' vals, query-major, in the reference's per-backend
 * iteration order. */
int32_t gtgpu_find(gtgpu_index* index, uint64_t n, const uint32_t* chr, const uint32_t* start,
                   const uint32_t* end, int32_t min_overlap, uint64_t* out_offsets, gtgpu_buf** out_vals);
/* Tokenizer::encode for a batch of calls (gtars-tokenizers/src/tokenizer.rs:140-171): "file" f is one encode()
 * call over queries [file_offsets[f], file_offsets[f+1]); its ids are the concatenated vals of every query's
 * hits, or the single id unk_id when the whole call produced none.  out_file_token_offsets has n_files+1
 * entries.  (Duplicate-universe remapping, SURVEY.md §8a A9, is folded into vals by the caller at build time.) */
int32_t gtgpu_tokenize_files(gtgpu_index* index, uint64_t n_files, const uint64_t* file_offsets,
                             const uint32_t* chr, const uint32_t* start, const uint32_t* end, uint32_t unk_id,
                             uint64_t* out_file_token_offsets, gtgpu_buf** out_ids);

/* gtgpu_tokenize_files for queries whose chromosome ids come as RUNS: run r covers queries
 * [run_offsets[r], run_offsets[r+1]) and all of them lie on chromosome run_chr[r].  A BED file read by
 * RegionSet::try_from is sorted by chromosome (gtars-core/src/models/region_set.rs:502-505), so a file contributes a
 * handful of runs; the per-query chromosome array is then rebuilt on the device and never crosses PCIe (a third of
 * the input bytes).  run_offsets has n_runs + 1 entries, starts at 0 and ends at file_offsets[n_files]. */
int32_t gtgpu_tokenize_files_runs(gtgpu_index* index, uint64_t n_files, const uint64_t* file_offsets, uint64_t n_runs,
                                  const uint64_t* run_offsets, const uint32_t* run_chr, const uint32_t* start,
                                  const uint32_t* end, uint32_t unk_id, uint64_t* out_file_token_offsets,
                                  gtgpu_buf** out_ids);

/* gtgpu_tokenize_files_runs with the ends as 16-bit widths: end[i] = start[i] + width16[i], except for the queries
 * listed in wide_index (strictly increasing), whose end is wide_end[k] — regions wider than 65 535 bp, or with
 * end < start.  Peak-sized regions then cost 6 bytes of PCIe traffic each instead of 8 (the host entry point is
 * H2D-bound); results are identical to gtgpu_tokenize_files on the expanded arrays. */
int32_t gtgpu_tokenize_files_compact(gtgpu_index* index, uint64_t n_files, const uint64_t* file_offsets, uint64_t n_runs,
                                     const uint64_t* run_offsets, const uint32_t* run_chr, const uint32_t* start,
                                     const uint16_t* width16, uint64_t n_wide, const uint64_t* wide_index,
                                     const uint32_t* wide_end, uint32_t unk_id, uint64_t* out_file_token_offsets,
                                     gtgpu_buf** out_ids);

/* Host-side marshalling for gtgpu_tokenize_files_compact (no device work; `threads` host threads, 0 = all cores): from the
 * flat per-query arrays a caller holds after mapping chromosome names to ids it derives the chromosome runs (cut at every
 * file boundary as well), the 16-bit widths (out_width16[n], caller-allocated — pinned memory makes the later copy DMA)
 * and the exception list of queries wider than 65 534 bp or with end < start.  out_run_offsets needs run_capacity + 1
 * entries.  *out_n_runs / *out_n_wide always receive the counts; GTGPU_ERR_CAPACITY when a capacity was too small. */
int32_t gtgpu_marshal_compact(uint64_t n, const uint32_t* chr, const uint32_t* start, const uint32_t* end, uint64_t n_files,
                              const uint64_t* file_offsets, int32_t threads, uint16_t* out_width16, uint64_t run_capacity,
                              uint64_t* out_run_offsets, uint32_t* out_run_chr, uint64_t* out_n_runs, uint64_t wide_capacity,
                              uint64_t* out_wide_index, uint32_t* out_wide_end, uint64_t* out_n_wide);

/* gtgpu_tokenize_files_runs with start AND width in ONE 32-bit word per query ("packed" wire format, 4.125 bytes of PCIe
 * traffic per region instead of 6): queries are taken in blocks of 32 (block b = queries [32 b, 32 b + 32)), every block
 * has an anchor, and
 *     start[i] = anchors[i / 32] + (packed[i] & ((1 << (32 - width_bits)) - 1)),   end[i] = start[i] + (packed[i] >> (32 - width_bits))
 * except for the queries listed in exc_index (strictly increasing), which are (exc_start[k], exc_end[k]).  A file read by
 * RegionSet::try_from is sorted by (chromosome, start) (gtars-core/src/models/region_set.rs:502-505), so inside a block the
 * offsets are small; what does not fit (the far side of a chromosome / file boundary inside a block, wide or reversed
 * regions) is an exception.  anchors has ceil(n / 32) entries; width_bits is 1..24.  Results are identical to
 * gtgpu_tokenize_files on the expanded arrays. */
int32_t gtgpu_tokenize_files_packed(gtgpu_index* index, uint64_t n_files, const uint64_t* file_offsets, uint64_t n_runs,
                                    const uint64_t* run_offsets, const uint32_t* run_chr, uint32_t width_bits,
                                    const uint32_t* packed, const uint32_t* anchors, uint64_t n_exc, const uint64_t* exc_index,
                                    const uint32_t* exc_start, const uint32_t* exc_end, uint32_t unk_id,
                                    uint64_t* out_file_token_offsets, gtgpu_buf** out_ids);

/* Host-side marshalling for gtgpu_tokenize_files_packed (no device work; `threads` host threads, 0 = all cores): chromosome
 * runs as in gtgpu_marshal_compact, packed words (out_packed[n]), block anchors (out_anchors[ceil(n / 32)]; the start of the
 * block's first query, or of the first query after a descent when that leaves fewer exceptions) and the exception list.
 * width_bits = 0 lets the packer choose the split (6..16 bits of width, fewest exceptions on a sample of blocks);
 * *out_width_bits receives the split used.  Unsorted inputs still round-trip exactly — as exceptions, 16 bytes each — so a
 * caller compares *out_n_exc with n before preferring this format.  GTGPU_ERR_CAPACITY when a capacity was too small (the
 * needed counts are returned). */
int32_t gtgpu_marshal_packed(uint64_t n, const uint32_t* chr, const uint32_t* start, const uint32_t* end, uint64_t n_files,
                             const uint64_t* file_offsets, int32_t threads, uint32_t width_bits, uint32_t* out_packed,
                             uint32_t* out_anchors, uint64_t run_capacity, uint64_t* out_run_offsets, uint32_t* out_run_chr,
                             uint64_t* out_n_runs, uint64_t exc_capacity, uint64_t* out_exc_index, uint32_t* out_exc_start,
                             uint32_t* out_exc_end, uint64_t* out_n_exc, uint32_t* out_width_bits);

/* tokenize_fragment_file (gtars-tokenizers/src/utils/fragments.rs:12-82) over pre-parsed fragments: every fragment
 * is one Tokenizer::tokenize call (a fragment with no hit, or on an unknown chromosome, yields unk_id), ids are
 * appended to the fragment's barcode list in input order.  barcode_id[i] < n_barcodes (dense ids, mapped by the
 * caller); output is barcode-major: out_barcode_offsets[n_barcodes + 1] + ids. */
int32_t gtgpu_tokenize_fragments(gtgpu_index* index, uint64_t n, const uint32_t* chr, const uint32_t* start,
                                 const uint32_t* end, const uint32_t* barcode_id, uint32_t n_barcodes, uint32_t unk_id,
                                 uint64_t* out_barcode_offsets, gtgpu_buf** out_ids);

/* gtgpu_tokenize_fragments with everything device-resident and asynchronous on the ctx stream: d_out_barcode_offsets has
 * n_barcodes + 1 entries, d_out_ids room for ids_capacity >= n ids, *d_out_total (device u64) receives the number of ids
 * — one per hit, one unk_id per fragment without a hit — or UINT64_MAX when they did not fit ids_capacity (the output is
 * then incomplete; the host entry point re-runs with an exact buffer by itself). */
int32_t gtgpu_tokenize_fragments_dev(gtgpu_index* index, uint64_t n, const uint32_t* d_chr, const uint32_t* d_start,
                                     const uint32_t* d_end, const uint32_t* d_barcode_id, uint32_t n_barcodes,
                                     uint32_t unk_id, uint64_t* d_out_barcode_offsets, uint32_t* d_out_ids,
                                     uint64_t ids_capacity, uint64_t* d_out_total);

/* ---- BED text ingest ----------------------------------------------------------------------------------------------------
 * gtgpu_parse_bed replaces the parse + sort of RegionSet::try_from (gtars-core/src/models/region_set.rs:60-185,
 * :502-505) for query files: `text` is the (decompressed) file, n_bytes < 4 GiB.  Lines are split on '\n' (a trailing
 * '\r' is dropped); lines starting with "browser", "track" or "#" are skipped, and so is a first line whose second
 * field is not a number; every other line needs three tab-separated fields with start and end accepted by Rust's
 * str::parse::<u32>() — otherwise GTGPU_ERR_INVALID with the 1-based line number; no region at all is an error too
 * (EmptyRegionSet).  Chromosome names are mapped through the caller's table (names back to back, name_offsets has
 * n_names + 1 entries); a name that is not in it becomes GTGPU_UNKNOWN_CHROM.  Output: the regions in the reference's
 * sorted order — stable, by chromosome STRING then start — with unknown names after all known ones (they cannot
 * produce output).  gtgpu_tokenize_bed = parse + sort + Tokenizer::encode of that one file, text in, token ids out. */
int32_t gtgpu_parse_bed(gtgpu_ctx* ctx, const char* text, uint64_t n_bytes, uint32_t n_names, const char* names,
                        const uint32_t* name_offsets, uint64_t* out_n, gtgpu_buf** out_chr, gtgpu_buf** out_start,
                        gtgpu_buf** out_end);
int32_t gtgpu_tokenize_bed(gtgpu_index* index, const char* text, uint64_t n_bytes, uint32_t n_names, const char* names,
                           const uint32_t* name_offsets, uint32_t unk_id, gtgpu_buf** out_ids);
/* Tokenizer::encode(RegionSet::try_from(file f)) for a batch of n_files BED files in one device pass.  Inputs as in
 * gtgpu_igd_count_bed / _gz: file f = text[file_offsets[f], file_offsets[f+1]) of any total size, or the gzip members
 * [file_members[f], file_members[f+1]) of gz / member_offsets (as in gtgpu_gunzip; inflated whole into device memory,
 * GTGPU_ERR_NOMEM when that text does not fit).  Line rules, windows of about GTGPU_INGEST_WINDOW bytes, the header rule per
 * file and the errors are those of gtgpu_igd_build_bed (GTGPU_ERR_INVALID: a malformed line, "file k, line j", j 1-based in file
 * k; a file without a region line, "file k: ... 0 regions found"; GTGPU_ERR_UNSUPPORTED: more than 262 144 distinct names or
 * 2^32 - 1 region lines or more).  Chromosome names map through the caller's table as in gtgpu_tokenize_bed; a name not in it
 * produces no hits.  Every file's regions are stable-sorted by (chromosome string, start) on the device unless every file is
 * already in that order.  Outputs as gtgpu_tokenize_files: out_file_token_offsets (n_files + 1, caller-allocated) into *out_ids;
 * file f's ids equal gtgpu_tokenize_bed on file f alone (hits in the backend's order, [unk_id] for a file without a token).
 * n_files == 0 gives the offsets [0] and an empty buffer.  On a multi-device ctx the call runs on the first device. */
int32_t gtgpu_tokenize_bed_files(gtgpu_index* index, uint64_t n_files, const char* text, const uint64_t* file_offsets,
                                 uint32_t n_names, const char* names, const uint32_t* name_offsets, uint32_t unk_id,
                                 uint64_t* out_file_token_offsets, gtgpu_buf** out_ids);
int32_t gtgpu_tokenize_bed_files_gz(gtgpu_index* index, uint64_t n_files, const uint64_t* file_members, uint64_t n_members,
                                    const uint8_t* gz, const uint64_t* member_offsets, uint32_t n_names, const char* names,
                                    const uint32_t* name_offsets, uint32_t unk_id, uint64_t* out_file_token_offsets,
                                    gtgpu_buf** out_ids);

/* tokenize_fragment_file (gtars-tokenizers/src/utils/fragments.rs:12-82) from the file's (decompressed) text: lines
 * starting with '#' are skipped, every other line needs at least five whitespace-separated fields (chr start end
 * barcode ...) with start and end accepted by str::parse::<u32>() — otherwise GTGPU_ERR_INVALID with the 0-based line
 * number the reference reports.  Barcodes become dense ids in first-appearance order through a device hash table
 * (64-bit FNV-1a + byte comparison against the first appearance; a true hash collision is reported as
 * GTGPU_ERR_UNSUPPORTED).  Outputs: *out_n_barcodes; *out_barcode_spans = (byte offset, length) of each barcode's first
 * occurrence in `text` (u32 pairs, so the caller recovers the strings); *out_barcode_offsets = n_barcodes + 1 u64
 * offsets into *out_ids (gtgpu_buf_len counts 8-byte elements); ids as gtgpu_tokenize_fragments returns them.  n_bytes < 4 GiB
 * (GTGPU_ERR_UNSUPPORTED beyond); gtgpu_tokenize_fragments_file takes any size and returns the names themselves. */
int32_t gtgpu_tokenize_fragments_text(gtgpu_index* index, const char* text, uint64_t n_bytes, uint32_t n_names,
                                      const char* names, const uint32_t* name_offsets, uint32_t unk_id,
                                      uint32_t* out_n_barcodes, gtgpu_buf** out_barcode_spans,
                                      gtgpu_buf** out_barcode_offsets, gtgpu_buf** out_ids);

/* ---- gzip on the device ------------------------------------------------------------------------------------------------
 * The reference reads `.gz` inputs through flate2's MultiGzDecoder (gtars-core/src/utils.rs:115-126): the text is the
 * concatenation of the file's gzip members.  A DEFLATE stream is sequential, so the device inflates MEMBERS in parallel, one
 * warp each: a bgzip'ed fragment file is thousands of independent <= 64 KiB BGZF members, a tokenization batch thousands of
 * one-member `.bed.gz` files back to back.  (One multi-gigabyte single-member stream is a job for the host's zlib.)
 *
 * gtgpu_gzip_members (host only): member boundaries of a gzip buffer — BGZF blocks are split by their BSIZE field, anything
 * else is one member to the end of the buffer.  out_member_offsets needs n_members + 1 entries (`capacity` of them are
 * available; *out_n_members always receives the count, GTGPU_ERR_CAPACITY when it did not fit).
 * gtgpu_gunzip: member k = gz[member_offsets[k], member_offsets[k+1]) (whole members; several files may simply be laid
 * back to back).  *out_text (byte elements) = the members' texts concatenated, out_member_offsets[n_members + 1] where each
 * starts.  Every member's ISIZE and CRC-32 are verified; corrupt data, a unit that holds more than one member, or a member
 * with >= 4 GiB of text give GTGPU_ERR_INVALID naming the member.
 * gtgpu_tokenize_bed_gz / gtgpu_tokenize_fragments_gz = inflate + gtgpu_tokenize_bed / gtgpu_tokenize_fragments_text with
 * the text never leaving the device on its way to the parser (the fragment form also returns the text: the barcode spans
 * index into it). */
int32_t gtgpu_gzip_members(const uint8_t* gz, uint64_t n_bytes, uint64_t capacity, uint64_t* out_member_offsets,
                           uint64_t* out_n_members);
int32_t gtgpu_gunzip(gtgpu_ctx* ctx, uint64_t n_members, const uint8_t* gz, const uint64_t* member_offsets,
                     gtgpu_buf** out_text, uint64_t* out_member_offsets);
int32_t gtgpu_tokenize_bed_gz(gtgpu_index* index, uint64_t n_members, const uint8_t* gz, const uint64_t* member_offsets,
                              uint32_t n_names, const char* names, const uint32_t* name_offsets, uint32_t unk_id,
                              gtgpu_buf** out_ids);
int32_t gtgpu_tokenize_fragments_gz(gtgpu_index* index, uint64_t n_members, const uint8_t* gz, const uint64_t* member_offsets,
                                    uint32_t n_names, const char* names, const uint32_t* name_offsets, uint32_t unk_id,
                                    uint32_t* out_n_barcodes, gtgpu_buf** out_barcode_spans, gtgpu_buf** out_barcode_offsets,
                                    gtgpu_buf** out_ids, gtgpu_buf** out_text);

/* tokenize_fragment_file from ONE fragment file's bytes of any size, parsed on the device: the (decompressed) text, or its gzip
 * members (n_members, gz, member_offsets as in gtgpu_gunzip; inflated whole into device memory, GTGPU_ERR_NOMEM when that text
 * does not fit).  Line rules, chromosome names, malformed-line errors ("Invalid fragment file detected at line: i", 0-based,
 * '#' lines count, no output) and results are those of gtgpu_tokenize_fragments_text: every barcode is kept, including one
 * whose fragments all lie on unknown chromosomes.  The text is parsed in windows of about GTGPU_INGEST_WINDOW bytes (default
 * 2 GiB), as the scoring entry points do; at most 2^32 - 1 fragments per file and no more ids than gtgpu_tokenize_fragments
 * takes (GTGPU_ERR_UNSUPPORTED beyond).  Outputs: *out_n_barcodes; *out_barcode_names = the barcodes' bytes back to back in
 * first-appearance order (u8 elements); *out_barcode_name_offsets = n_barcodes + 1 u64 offsets into those bytes;
 * *out_barcode_offsets = n_barcodes + 1 u64 offsets into *out_ids (u32), as gtgpu_tokenize_fragments returns them.  On a
 * multi-device ctx these run on the first device.  gtgpu_tokenize_fragments_text / _gz run on the same windowed parse. */
int32_t gtgpu_tokenize_fragments_file(gtgpu_index* index, const char* text, uint64_t n_bytes, uint32_t n_names, const char* names,
                                      const uint32_t* name_offsets, uint32_t unk_id, uint32_t* out_n_barcodes,
                                      gtgpu_buf** out_barcode_names, gtgpu_buf** out_barcode_name_offsets,
                                      gtgpu_buf** out_barcode_offsets, gtgpu_buf** out_ids);
int32_t gtgpu_tokenize_fragments_file_gz(gtgpu_index* index, uint64_t n_members, const uint8_t* gz, const uint64_t* member_offsets,
                                         uint32_t n_names, const char* names, const uint32_t* name_offsets, uint32_t unk_id,
                                         uint32_t* out_n_barcodes, gtgpu_buf** out_barcode_names, gtgpu_buf** out_barcode_name_offsets,
                                         gtgpu_buf** out_barcode_offsets, gtgpu_buf** out_ids);

/* ---- gtars-scoring: fragments x consensus peaks ------------------------------------------------------------------------
 * gtgpu_score_matrix replaces region_scoring_from_fragments (gtars-scoring/src/fragment_scoring.rs:19-121) over
 * pre-parsed fragments: file f owns fragments [file_offsets[f], file_offsets[f+1]); the index is the ConsensusSet
 * (gtars-scoring/src/files.rs:60-99: one Bits per chromosome, val = id of the peak); out_counts is the row-major
 * n_files x n_cols CountMatrix<u32> (counts.rs:9-56; a val >= n_cols is ignored like CountMatrix::increment does).
 * GTGPU_SCORE_ATAC: every fragment is two lookups, the shifted start [start+4, start+5) and the end interval the
 * reference builds as Region{start: end-5, end: end-6} (fragment_scoring.rs:59-84, consts.rs START_SHIFT/END_SHIFT);
 * GTGPU_SCORE_CHIP: the fragment itself (:99-107).  u32 arithmetic wraps.  The _dev form takes device pointers. */
#define GTGPU_SCORE_ATAC 0
#define GTGPU_SCORE_CHIP 1
int32_t gtgpu_score_matrix(gtgpu_index* index, uint64_t n_files, const uint64_t* file_offsets, uint64_t n,
                           const uint32_t* chr, const uint32_t* start, const uint32_t* end, int32_t mode,
                           uint64_t n_cols, uint32_t* out_counts);
int32_t gtgpu_score_matrix_dev(gtgpu_index* index, uint64_t n_files, const uint64_t* d_file_offsets, uint64_t n,
                               const uint32_t* d_chr, const uint32_t* d_start, const uint32_t* d_end, int32_t mode,
                               uint64_t n_cols, uint32_t* d_out_counts);

/* region_scoring_from_fragments / barcode_scoring_from_fragments from ONE fragment file's bytes, parsed on the device: the
 * (decompressed) text, or its gzip members (n_members, gz, member_offsets as in gtgpu_gunzip; inflated whole into device memory,
 * GTGPU_ERR_NOMEM when that text does not fit).  Lines follow Fragment::from_str (gtars-core/src/models/fragments.rs:16-44):
 * '#' lines are skipped, every other line needs at least five whitespace-separated fields with start, end and the fifth
 * (support) field accepted by str::parse::<u32>() — otherwise GTGPU_ERR_INVALID, "Failed to parse fragment at line i" with the
 * 0-based line index the host parser reports ('#' lines count), and no output.  Chromosome names map through the caller's table
 * as in gtgpu_tokenize_fragments_text.  Any file size: the text is parsed in windows of about GTGPU_INGEST_WINDOW bytes (default
 * 2 GiB); at most 2^32 - 1 fragments per file (GTGPU_ERR_UNSUPPORTED beyond).
 * gtgpu_score_matrix_text / _gz: out_row (n_cols u32, overwritten) = the file's row of gtgpu_score_matrix, same mode and n_cols
 * rules.  gtgpu_score_barcodes_text / _gz: the content of gtgpu_score_barcodes for the file, barcodes numbered in
 * first-appearance order; only barcodes with at least one fragment on a chromosome of the name table are kept (the reference's
 * key set, files.rs:106-129 + fragment_scoring.rs:146-153: such a barcode has an entry even without a hit).  Outputs:
 * *out_n_barcodes (kept barcodes); *out_barcode_names = their bytes back to back in id order (u8 elements);
 * *out_barcode_name_offsets = n_barcodes + 1 u64 offsets into those bytes; *out_barcode_offsets = n_barcodes + 1 u64 offsets into
 * *out_peaks / *out_counts (u32 each), sorted by (barcode, peak).  On a multi-device ctx these run on the first device. */
int32_t gtgpu_score_matrix_text(gtgpu_index* index, const char* text, uint64_t n_bytes, uint32_t n_names, const char* names,
                                const uint32_t* name_offsets, int32_t mode, uint64_t n_cols, uint32_t* out_row);
int32_t gtgpu_score_matrix_gz(gtgpu_index* index, uint64_t n_members, const uint8_t* gz, const uint64_t* member_offsets,
                              uint32_t n_names, const char* names, const uint32_t* name_offsets, int32_t mode, uint64_t n_cols,
                              uint32_t* out_row);
int32_t gtgpu_score_barcodes_text(gtgpu_index* index, const char* text, uint64_t n_bytes, uint32_t n_names, const char* names,
                                  const uint32_t* name_offsets, uint32_t* out_n_barcodes, gtgpu_buf** out_barcode_names,
                                  gtgpu_buf** out_barcode_name_offsets, gtgpu_buf** out_barcode_offsets, gtgpu_buf** out_peaks,
                                  gtgpu_buf** out_counts);
int32_t gtgpu_score_barcodes_gz(gtgpu_index* index, uint64_t n_members, const uint8_t* gz, const uint64_t* member_offsets,
                                uint32_t n_names, const char* names, const uint32_t* name_offsets, uint32_t* out_n_barcodes,
                                gtgpu_buf** out_barcode_names, gtgpu_buf** out_barcode_name_offsets, gtgpu_buf** out_barcode_offsets,
                                gtgpu_buf** out_peaks, gtgpu_buf** out_counts);

/* barcode_scoring_from_fragments (fragment_scoring.rs:126-155): whole fragments, sparse barcode x peak counts.  The
 * reference returns HashMap<barcode, HashMap<peak, count>>; here the same content as CSR sorted by (barcode, peak):
 * out_barcode_offsets[n_barcodes + 1] index the (peak, count) pairs in *out_peaks / *out_counts. */
int32_t gtgpu_score_barcodes(gtgpu_index* index, uint64_t n, const uint32_t* chr, const uint32_t* start,
                             const uint32_t* end, const uint32_t* barcode_id, uint32_t n_barcodes,
                             uint64_t* out_barcode_offsets, gtgpu_buf** out_peaks, gtgpu_buf** out_counts);

/* ---- IGD / LOLA overlap-count matrices ------------------------------------------------------------------------------
 * gtgpu_igd_build replaces Igd::from_named_region_sets / from_region_sets (gtars-igd/src/igd.rs:249-317): file f owns
 * records [file_offsets[f], file_offsets[f+1]); records with start >= end, or negative as int32, are dropped as
 * Igd::add does (igd.rs:109-116).  chr ids must be < n_chroms. */
int32_t gtgpu_igd_build(gtgpu_ctx* ctx, uint64_t n_files, const uint64_t* file_offsets, uint32_t n_chroms,
                        const uint32_t* chr, const uint32_t* start, const uint32_t* end, gtgpu_igd** out_igd);
/* gtgpu_igd_build from the database's BED files, parsed on the device (Igd::from_named_region_sets over RegionSet::try_from of
 * every file, gtars-core/src/models/region_set.rs:60-185): file f = text[file_offsets[f], file_offsets[f+1]) of any total
 * size, or the gzip members [file_members[f], file_members[f+1]) of gz / member_offsets (as in gtgpu_gunzip; inflated whole into
 * device memory, GTGPU_ERR_NOMEM when that text does not fit).  Every file follows the line rules of gtgpu_parse_bed: browser /
 * track / '#' lines are skipped, a first line of the file whose second field is not a u32 is a header, every other line needs
 * three tab-separated fields with u32 start and end.  A file's end ends its last line (a line never spans two files).  A region
 * line that gtgpu_igd_build would drop (start >= end, or negative as int32) still counts as a region of its file.  Chromosome
 * ids are the names' first-appearance order over the region lines (files in order, lines in file order); *out_n_chroms names
 * come back as their bytes back to back (*out_chrom_names, u8) and n_chroms + 1 u64 offsets (*out_chrom_name_offsets): a
 * caller maps query chromosomes through them.  Errors (GTGPU_ERR_INVALID, no IGD): a malformed line ("file k, line j", j
 * 1-based within file k; reported before an empty file); a file without a region line ("file k: ... 0 regions found").
 * Distinct names are found with 64-bit FNV-1a + a byte comparison: a true hash collision, more than 262 144 distinct names or
 * 2^32 - 1 region lines give GTGPU_ERR_UNSUPPORTED.  The text is parsed in windows of about GTGPU_INGEST_WINDOW bytes (default
 * 2 GiB) on the first device of a multi-device ctx; the shards of a group are then copied from there to their devices. */
int32_t gtgpu_igd_build_bed(gtgpu_ctx* ctx, uint64_t n_files, const char* text, const uint64_t* file_offsets, uint32_t* out_n_chroms,
                            gtgpu_buf** out_chrom_names, gtgpu_buf** out_chrom_name_offsets, gtgpu_igd** out_igd);
int32_t gtgpu_igd_build_bed_gz(gtgpu_ctx* ctx, uint64_t n_files, const uint64_t* file_members, uint64_t n_members, const uint8_t* gz,
                               const uint64_t* member_offsets, uint32_t* out_n_chroms, gtgpu_buf** out_chrom_names,
                               gtgpu_buf** out_chrom_name_offsets, gtgpu_igd** out_igd);
int32_t gtgpu_igd_free(gtgpu_igd* igd);
/* Igd::save (gtars-igd/src/igd.rs:418-486) of a database built any way (gtgpu_igd_build, gtgpu_igd_build_bed / _gz, one device
 * or a group), written on the device: *out_igd_bytes (u8, gtgpu_buf_len = bytes) is the .igd file byte for byte as the
 * reference writes it after Igd::from_named_region_sets over the same sets: nbp 16384, gType 1, the contigs in the order
 * Igd::add created them (for gtgpu_igd_build: by the first kept record in the input arrays; for BED files, whose RegionSets the
 * reference sorts by (name, start): by the first file with a kept record on the name, then by name bytes), a kept record in
 * every tile it reaches, a tile stable-sorted by start, value 0.  Chromosomes without a kept record are not contigs.  The names
 * are indexed by chromosome id, in the table format of gtgpu_igd_count_bed (n_names + 1 u32 byte offsets; a name is cut to 40
 * bytes); n_names must equal the igd's chromosome count (else GTGPU_ERR_INVALID).  out_file_regions / out_file_width_sums
 * (n_files each, caller-allocated) receive the .tsv numbers of every input file: its region lines with start < end as u32
 * (records dropped as negative int32 included) and the wrapping u64 sum of their widths (int32 end - int32 start, widened);
 * Avg size = sum / regions.  More than 2^32 - 2 tile entries give GTGPU_ERR_UNSUPPORTED. */
int32_t gtgpu_igd_serialize(gtgpu_igd* igd, uint32_t n_names, const char* names, const uint32_t* name_offsets,
                            gtgpu_buf** out_igd_bytes, uint64_t* out_file_regions, uint64_t* out_file_width_sums);
/* info[0]=n_files, [1]=records kept, [2]=device bytes, [3]=lut shift */
int32_t gtgpu_igd_info(const gtgpu_igd* igd, uint64_t info[4]);
/* Igd::count_set_overlaps (igd.rs:544-556) / Igd::count_region_hits (igd.rs:563-590) for n_sets query sets at once:
 * set s owns queries [set_offsets[s], set_offsets[s+1]); out is [n_sets x n_files] row-major (caller-allocated).
 * Queries follow Igd::count_overlaps (igd.rs:504-540): int32 semantics, start >= end or end <= 0 -> nothing, negative
 * start clamps to 0.  min_overlap must be >= 1 (values <= 0 depend on the reference's tile layout). */
int32_t gtgpu_igd_count_set_overlaps(gtgpu_igd* igd, uint64_t n_sets, const uint64_t* set_offsets, const uint32_t* chr,
                                     const uint32_t* start, const uint32_t* end, int32_t min_overlap, uint64_t* out);
int32_t gtgpu_igd_count_region_hits(gtgpu_igd* igd, uint64_t n_sets, const uint64_t* set_offsets, const uint32_t* chr,
                                    const uint32_t* start, const uint32_t* end, int32_t min_overlap, uint64_t* out);
/* device-resident core: d_set_of[i] = set index of query i; d_out ([n_sets x n_files] u64) is accumulated into */
int32_t gtgpu_igd_count_dev(gtgpu_igd* igd, int32_t binary, uint64_t n, const uint32_t* d_set_of, const uint32_t* d_chr,
                            const uint32_t* d_start, const uint32_t* d_end, int32_t min_overlap, uint64_t* d_out);
/* Igd::count_region_hits (binary = 1) / Igd::count_set_overlaps (binary = 0) for n_sets query sets given as BED files, parsed on
 * the device: set s = text[file_offsets[s], file_offsets[s+1]) (any total size), or the gzip members [file_members[s],
 * file_members[s+1]) of gz / member_offsets (as in gtgpu_igd_build_bed_gz).  Line rules, windows, the header rule per file and
 * the errors ("file k, line j"; "file k: ... 0 regions found"; at most 262 144 distinct names and fewer than 2^32 - 1 region
 * lines, else GTGPU_ERR_UNSUPPORTED) are those of gtgpu_igd_build_bed.  Chromosome names map through the caller's table (the
 * database's names, as gtgpu_igd_build_bed returns them or as the caller of gtgpu_igd_build numbered them), looked up as
 * gtgpu_parse_bed does; a name not in it contributes no hits.  out = [n_sets x n_files] u64 row-major (caller-allocated,
 * overwritten); out_set_regions[s] = the region lines of set s (RegionSet::len: every region line, unknown names and start >= end
 * included: the |user set| / |universe| of run_lola's tables).  min_overlap >= 1.  On a multi-device ctx the parse runs on the
 * first device and every device reads the parsed queries from there. */
int32_t gtgpu_igd_count_bed(gtgpu_igd* igd, int32_t binary, uint64_t n_sets, const char* text, const uint64_t* file_offsets,
                            uint32_t n_names, const char* names, const uint32_t* name_offsets, int32_t min_overlap,
                            uint64_t* out, uint64_t* out_set_regions);
int32_t gtgpu_igd_count_bed_gz(gtgpu_igd* igd, int32_t binary, uint64_t n_sets, const uint64_t* file_members, uint64_t n_members,
                               const uint8_t* gz, const uint64_t* member_offsets, uint32_t n_names, const char* names,
                               const uint32_t* name_offsets, int32_t min_overlap, uint64_t* out, uint64_t* out_set_regions);

/* ---- multi-GPU: the LOLA database sharded by region set, one ncclAllGather (run_lola's count matrices,
 * gtars-lola/src/enrichment.rs:198-211) ------------------------------------------------------------------------------
 * This is the process-per-GPU form (a multi-device context does the same internally, see gtgpu_init_multi).
 * One process per GPU.  Rank 0 calls gtgpu_comm_unique_id and ships the 128 bytes to the other ranks by any means
 * (MPI, torch.distributed, a file); every rank then calls gtgpu_comm_init on its ctx.  NCCL is dlopen'ed on first
 * use.  With world W and n_files_global sets, rank r must have built its gtgpu_igd over global sets
 * [r*C, min((r+1)*C, n_files_global)), C = ceil(n_files_global / W); every rank passes the SAME query sets and
 * receives the full [n_sets x n_files_global] matrix.  Without a communicator (W = 1) it equals the local call. */
int32_t gtgpu_comm_unique_id(uint8_t out_id[128]);
int32_t gtgpu_comm_init(gtgpu_ctx* ctx, int32_t world, int32_t rank, const uint8_t id[128]);
int32_t gtgpu_comm_free(gtgpu_ctx* ctx);
int32_t gtgpu_igd_count_sharded(gtgpu_ctx* ctx, gtgpu_igd* igd, int32_t binary, uint64_t n_files_global,
                                uint64_t n_sets, const uint64_t* set_offsets, const uint32_t* chr, const uint32_t* start,
                                const uint32_t* end, int32_t min_overlap, uint64_t* out);

/* ---- batch queries, device-resident (asynchronous on the ctx stream) --------------------------------------- */
int32_t gtgpu_count_dev(gtgpu_index* index, uint64_t n, const uint32_t* d_chr, const uint32_t* d_start,
                        const uint32_t* d_end, int32_t min_overlap, uint32_t* d_out_counts);
/* Fused count → device-wide exclusive scan → emit in ONE pass over the queries (the device-resident core of
 * gtgpu_find / gtgpu_tokenize_files).  d_out_ids has room for ids_capacity ids; d_out_offsets (n+1 u64, per query)
 * and d_out_file_token_offsets (n_files+1 u64, RAW: before the [unk] rule; needs d_file_offsets) may each be NULL.
 * *d_out_total (device u64) receives the number of ids the call produces; when it exceeds ids_capacity the first
 * ids_capacity ids are written exactly and the surplus is not written, while the total and both offset arrays are still
 * complete (the host entry points then re-run with an exact buffer).  d_out_ids may be NULL when ids_capacity is 0.
 * The kernel's overflow flag (a tile whose ids do not fit its 32-bit sums, or a running total of 2^55 or more) is not
 * reported here; the host entry points fail with GTGPU_ERR_UNSUPPORTED on it. */
int32_t gtgpu_find_dev(gtgpu_index* index, uint64_t n, const uint32_t* d_chr, const uint32_t* d_start,
                       const uint32_t* d_end, int32_t min_overlap, uint64_t n_files, const uint64_t* d_file_offsets,
                       uint32_t* d_out_ids, uint64_t ids_capacity, uint64_t* d_out_offsets,
                       uint64_t* d_out_file_token_offsets, uint64_t* d_out_total);
/* The per-call [unk] rule of Tokenizer::tokenize (tokenizer.rs:158-160) applied to raw per-file id runs:
 * d_out_file_token_offsets[f] = raw[f] + #empty files before f; d_out_ids gets every file's ids, or unk_id for a
 * file with none (capacity >= raw total + n_files); *d_out_n_empty (device u64) = number of such files. */
int32_t gtgpu_unk_rule_dev(gtgpu_ctx* ctx, uint64_t n_files, const uint64_t* d_raw_file_token_offsets,
                           const uint32_t* d_raw_ids, uint32_t unk_id, uint64_t* d_out_file_token_offsets,
                           uint32_t* d_out_ids, uint64_t* d_out_n_empty);

#ifdef __cplusplus
}
#endif
#endif /* GTARS_GPU_H */
