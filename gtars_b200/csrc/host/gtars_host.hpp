// gtars_host.hpp — host-side mirror of the reference's public API for the interval-overlap path, in C++ (the reference's
// host language, Rust, is not available in this image).  Same names, argument meaning and error behaviour as the
// reference; every batch method marshals into flat SoA arrays and calls the C ABI of include/gtars_gpu.h — exactly what
// the feature-gated Rust bodies would do (INTEGRATION.md).  Nothing here computes an overlap on the CPU.
//
//   gtars_core::models::{Region, RegionSet}                      gtars-core/src/models/region.rs:11-17, region_set.rs:40-45
//   gtars_overlaprs::{OverlapperType, MultiChromOverlapper}       gtars-overlaprs/src/lib.rs:139-144, multi_chrom_overlapper.rs:86-88
//   gtars_overlaprs::IndexedRegionSet                             gtars-overlaprs/src/indexed_region_set.rs:81-87
//   gtars_tokenizers::{Universe, Tokenizer, tokenize_fragment_file}  universe/mod.rs:35-42, tokenizer.rs:36-280, utils/fragments.rs
//   gtars_igd::Igd, gtars_lola::run_lola (contingency counts)     gtars-igd/src/igd.rs:61-72, gtars-lola/src/enrichment.rs:182-297
#pragma once

#include <cstdint>
#include <map>
#include <memory>
#include <stdexcept>
#include <string>
#include <unordered_map>
#include <utility>
#include <array>
#include <vector>

#include "../../../include/gtars_gpu.h"

namespace gtars {

struct Error : std::runtime_error {
    using std::runtime_error::runtime_error;
};

// ---- gtars_core::models ------------------------------------------------------------------------------------------
struct Region {
    std::string chr;
    uint32_t start = 0, end = 0;
    std::string rest;  // remaining BED columns joined by tabs ("" = None)
};

struct RegionSet {
    std::vector<Region> regions;
    std::string header;
    // RegionSet::try_from(&Path) (region_set.rs:60-185): parses a (gzipped) BED file, then sorts by (chr, start).
    static RegionSet from_file(const std::string& path);
    static RegionSet from_regions(std::vector<Region> regions) {  // RegionSet::from(Vec<Region>): order kept
        RegionSet rs;
        rs.regions = std::move(regions);
        return rs;
    }
    void sort();  // region_set.rs:502-505, stable
    size_t len() const { return regions.size(); }
};

enum class OverlapperType { Bits = GTGPU_KIND_BITS, AIList = GTGPU_KIND_AILIST };

// Owns one gtgpu_ctx (one device).  Shared by every object built on it.
class Device {
   public:
    explicit Device(int device = 0);
    ~Device();
    gtgpu_ctx* ctx() const { return ctx_; }

   private:
    gtgpu_ctx* ctx_ = nullptr;
};

// Dense chromosome ids in first-appearance order; unknown names map to GTGPU_UNKNOWN_CHROM.
class ChromMap {
   public:
    uint32_t add(const std::string& name);
    uint32_t get(const std::string& name) const;
    size_t size() const { return names_.size(); }
    const std::string& name(uint32_t id) const { return names_[id]; }

   private:
    std::unordered_map<std::string, uint32_t> ids_;
    std::vector<std::string> names_;
};

struct FlatQueries {
    std::vector<uint32_t> chr, start, end;
};
FlatQueries flatten(const std::vector<Region>& regions, const ChromMap& cmap);

// get_dynamic_reader (gtars-core/src/utils.rs:115-126): the whole file, gunzipped iff the extension is "gz".
std::string read_file_bytes(const std::string& path);
// RegionSet::try_from's parse + sort of BED text ON THE DEVICE (gtgpu_parse_bed): dense chromosome ids through `cmap`
// (names it does not hold become GTGPU_UNKNOWN_CHROM and sort last), regions in the reference's sorted order.
FlatQueries parse_bed_text_device(const Device& dev, const std::string& text, const ChromMap& cmap);

// ---- gtars_io::gtok (gtok.rs:126-300): "GTOK", one flag byte (1 = u16 tokens, 2 = u32), little-endian tokens -----------------
void write_tokens_to_gtok(const std::string& filename, const std::vector<uint32_t>& tokens);   // u16 iff every token fits
std::vector<uint32_t> read_tokens_from_gtok(const std::string& filename);
void init_gtok_file(const std::string& filename);                                              // header + u32 flag
void append_tokens_to_gtok_file(const std::string& filename, const std::vector<uint32_t>& tokens);

// ---- gtars_overlaprs::MultiChromOverlapper / IndexedRegionSet ------------------------------------------------------
class MultiChromOverlapper {
   public:
    // RegionSet::into_multi_chrom_overlapper (multi_chrom_overlapper.rs:240-300): val = index of the region in `source`.
    MultiChromOverlapper(std::shared_ptr<Device> dev, const RegionSet& source, OverlapperType kind);
    ~MultiChromOverlapper();
    MultiChromOverlapper(const MultiChromOverlapper&) = delete;
    MultiChromOverlapper& operator=(const MultiChromOverlapper&) = delete;

    // multi_chrom_overlapper.rs:483-498 / :501-516 / :524-550.  min_overlap < 0 means None.
    std::vector<uint64_t> count_overlaps(const RegionSet& query, int32_t min_overlap = -1) const;
    std::vector<bool> any_overlaps(const RegionSet& query, int32_t min_overlap = -1) const;
    std::vector<std::vector<Region>> find_overlaps_regions(const RegionSet& query, int32_t min_overlap = -1) const;
    // IndexedRegionSet::find_overlaps (indexed_region_set.rs:145-263): indices into the source, per query.
    std::vector<std::vector<uint32_t>> find_overlaps_indices(const RegionSet& query, int32_t min_overlap = -1) const;
    // multi_chrom_overlapper.rs:449-480: deduplicated, sorted by (chr, start, end).
    RegionSet subset_by(const RegionSet& query, int32_t min_overlap = -1) const;

   private:
    std::shared_ptr<Device> dev_;
    gtgpu_index* index_ = nullptr;
    ChromMap cmap_;
    std::vector<Region> source_;  // coordinates only, to rebuild regions from vals
};

// gtars_overlaprs::IndexedRegionSet (indexed_region_set.rs:100-263): a RegionSet plus its overlap index; the
// index-returning queries report positions in the source set, sorted and de-duplicated per query.
class IndexedRegionSet {
   public:
    IndexedRegionSet(std::shared_ptr<Device> dev, RegionSet regions, OverlapperType kind = OverlapperType::AIList);  // :111-143
    const RegionSet& regions() const { return source_; }                                                    // :168
    RegionSet intersect_all(const RegionSet& query) const;                                                  // :201-216
    RegionSet subset_by_overlaps(const RegionSet& query, int32_t min_overlap = -1) const;                   // :218-232
    std::vector<uint64_t> count_overlaps(const RegionSet& query, int32_t min_overlap = -1) const;           // :234-238
    std::vector<bool> any_overlaps(const RegionSet& query, int32_t min_overlap = -1) const;                 // :240-244
    std::vector<std::vector<uint32_t>> find_overlaps(const RegionSet& query, int32_t min_overlap = -1) const;  // :246-263

   private:
    RegionSet source_;
    std::unique_ptr<MultiChromOverlapper> index_;
};

// ---- gtars_scoring ---------------------------------------------------------------------------------------------------------
enum class ScoringMode { Atac = GTGPU_SCORE_ATAC, Chip = GTGPU_SCORE_CHIP };  // scoring_modes.rs

struct CountMatrix {  // counts.rs:9-56, row-major u32
    std::vector<uint32_t> data;
    size_t rows = 0, cols = 0;
    const uint32_t* get(size_t row, size_t col) const { return row < rows && col < cols ? &data[row * cols + col] : nullptr; }
};

// ConsensusSet::new (files.rs:60-99): RegionSet::try_from(path); ids = rank of first appearance among distinct
// regions (chr, start, end, rest); one Bits per chromosome.
class ConsensusSet {
   public:
    ConsensusSet(std::shared_ptr<Device> dev, const std::string& path);
    ConsensusSet(std::shared_ptr<Device> dev, const RegionSet& regions);
    ~ConsensusSet();
    ConsensusSet(const ConsensusSet&) = delete;
    ConsensusSet& operator=(const ConsensusSet&) = delete;
    size_t len() const { return len_; }
    bool is_empty() const { return len_ == 0; }
    gtgpu_index* index() const { return index_; }
    const ChromMap& chroms() const { return cmap_; }

   private:
    void build(const RegionSet& rs);
    std::shared_ptr<Device> dev_;
    gtgpu_index* index_ = nullptr;
    ChromMap cmap_;
    size_t len_ = 0;
};

// region_scoring_from_fragments (fragment_scoring.rs:19-121): one row per fragment file (in the given order — the
// reference's glob yields sorted paths), one column per consensus region.
CountMatrix region_scoring_from_fragments(const std::vector<std::string>& fragment_files, const ConsensusSet& consensus,
                                          ScoringMode mode);
// barcode_scoring_from_fragments (fragment_scoring.rs:126-155): barcode -> (peak index -> count); barcodes in
// first-appearance order (the reference's map is unordered), only barcodes with at least one overlap appear.
std::vector<std::pair<std::string, std::map<uint32_t, uint32_t>>> barcode_scoring_from_fragments(const std::string& fragment_file,
                                                                                                 const ConsensusSet& consensus);

// The same two with every file's bytes parsed on the device (gtgpu_score_matrix_text / gtgpu_score_barcodes_text, or their
// _gz forms for bgzip'ed files), one call per file; results and errors as above (an error names the file).
CountMatrix region_scoring_from_fragments_device(const std::vector<std::string>& fragment_files, const ConsensusSet& consensus,
                                                 ScoringMode mode);
std::vector<std::pair<std::string, std::map<uint32_t, uint32_t>>> barcode_scoring_from_fragments_device(const std::string& fragment_file,
                                                                                                        const ConsensusSet& consensus);

// ---- gtars_tokenizers ----------------------------------------------------------------------------------------------------
struct SpecialTokens {
    std::string unk = "<unk>", pad = "<pad>", mask = "<mask>", cls = "<cls>", eos = "<eos>", bos = "<bos>", sep = "<sep>";
    std::vector<std::string> as_vec() const { return {unk, pad, mask, cls, eos, bos, sep}; }  // special_tokens.rs:59-71
};

struct Universe {
    std::vector<std::string> regions;                        // positional (file order, then special tokens)
    std::unordered_map<std::string, uint32_t> region_to_id;  // first-appearance rank (gtars-core utils.rs:240-252)
    std::unordered_map<uint32_t, std::string> id_to_region;  // positional (utils.rs:258-271)
    std::vector<std::string> special_tokens;
    static Universe from_file(const std::string& path);      // universe/mod.rs:123-197
    void add_token_to_universe(const std::string& tok);      // universe/mod.rs:51-56
    size_t len() const { return region_to_id.size(); }
};

class Tokenizer {
   public:
    static std::unique_ptr<Tokenizer> from_bed(std::shared_ptr<Device> dev, const std::string& path);     // tokenizer.rs:88-100
    static std::unique_ptr<Tokenizer> from_config(std::shared_ptr<Device> dev, const std::string& path);  // tokenizer.rs:60-83
    static std::unique_ptr<Tokenizer> from_auto(std::shared_ptr<Device> dev, const std::string& path);    // tokenizer.rs:129-138
    ~Tokenizer();

    std::vector<std::string> tokenize(const std::vector<Region>& regions) const;  // tokenizer.rs:140-163
    std::vector<uint32_t> encode(const std::vector<Region>& regions) const;       // tokenizer.rs:165-171
    // encode(RegionSet::try_from(path)) with the file's text parsed, sorted and tokenized on the device (gtgpu_tokenize_bed).
    std::vector<uint32_t> encode_bed_file(const std::string& path) const;
    // encode_bed_file(paths[f]) for every f in ONE device pass over all the files' text, of any total size
    // (gtgpu_tokenize_bed_files; gtgpu_tokenize_bed_files_gz when every path ends in ".gz").
    std::vector<std::vector<uint32_t>> encode_bed_files(const std::vector<std::string>& paths) const;
    // One encode() per region set, resolved in ONE device pass (the batch shape the GPU serves).
    std::vector<std::vector<uint32_t>> encode_batch(const std::vector<const std::vector<Region>*>& calls) const;
    std::vector<std::string> decode(const std::vector<uint32_t>& ids) const;      // tokenizer.rs:173-181
    // utils/fragments.rs:61-82: barcode -> token ids, every fragment one tokenize() call (per-fragment [unk]).
    std::vector<std::pair<std::string, std::vector<uint32_t>>> tokenize_fragment_file(const std::string& path) const;
    // The same with the file's text (any size; a bgzip'ed file is inflated on the device) parsed, barcodes numbered and
    // fragments tokenized on the device (gtgpu_tokenize_fragments_file / _gz); barcodes come back in first-appearance order.
    std::vector<std::pair<std::string, std::vector<uint32_t>>> tokenize_fragment_file_device(const std::string& path) const;
    // utils/fragments.rs:87-112: barcode -> (token id -> count).
    std::vector<std::pair<std::string, std::map<uint32_t, uint32_t>>> count_fragments_by_barcode(const std::string& path) const;

    size_t get_vocab_size() const { return universe_.len(); }
    int64_t convert_token_to_id(const std::string& tok) const;
    const std::string* convert_id_to_token(uint32_t id) const;
    const SpecialTokens& special_tokens() const { return special_; }
    uint32_t unk_id() const { return unk_id_; }
    const Universe& universe() const { return universe_; }
    OverlapperType kind() const { return kind_; }

   private:
    Tokenizer() = default;
    void build(std::shared_ptr<Device> dev, Universe universe, SpecialTokens special, OverlapperType kind);
    std::shared_ptr<Device> dev_;
    Universe universe_;
    SpecialTokens special_;
    OverlapperType kind_ = OverlapperType::Bits;
    gtgpu_index* index_ = nullptr;
    ChromMap cmap_;
    std::vector<std::string> id_to_first_token_;  // inverse of region_to_id (what encode(tokenize(x)) round-trips through)
    uint32_t unk_id_ = 0;
};

// ---- gtars_igd::Igd + the LOLA contingency block --------------------------------------------------------------------------
struct ContingencyCounts {  // gtars-lola/src/enrichment.rs:213-220 (i64: negatives pass through)
    int64_t a, b, c, d;
};

class Igd {
   public:
    // Igd::from_named_region_sets (igd.rs:285-317): file_idx = position in `sets`; regions with start >= end are skipped.
    Igd(std::shared_ptr<Device> dev, const std::vector<const RegionSet*>& sets);
    ~Igd();
    size_t num_files() const { return n_files_; }
    std::vector<uint64_t> count_set_overlaps(const RegionSet& regions, int32_t min_overlap = 1) const;  // igd.rs:544-556
    std::vector<uint64_t> count_region_hits(const RegionSet& regions, int32_t min_overlap = 1) const;   // igd.rs:563-590
    // Many query sets in one device pass: row-major [n_sets x n_files].
    std::vector<uint64_t> count_region_hits_batch(const std::vector<const RegionSet*>& sets, int32_t min_overlap, bool pairwise) const;

    // .igd on-disk format (igd.rs:320-486; header nbp, gType, nCtg; tiles per contig; records per tile; 40-byte
    // names; 16-byte LE records).  save_named_region_sets = from_named_region_sets + save: byte-for-byte the file
    // (and companion .tsv) the reference writes.  from_igd_file loads such a file straight into the device layout
    // (the tile copies of an interval collapse to one record: the closed-form count does not need tiles); the
    // number of files is taken from the companion .tsv when it exists, else from the largest file index.
    static void save_named_region_sets(const std::vector<std::pair<std::string, const RegionSet*>>& sets, const std::string& path,
                                       int32_t nbp = 16384);
    static std::unique_ptr<Igd> from_igd_file(std::shared_ptr<Device> dev, const std::string& path);
    // Igd::save of this database (names[f] = file f's name in the .tsv): `path` (.igd) and the companion .tsv, the same bytes
    // save_named_region_sets writes for the same sets, with the file built on the device (gtgpu_igd_serialize).  A database
    // loaded with from_igd_file writes its kept records under the given names.  A database Igd only.
    void save(const std::string& path, const std::vector<std::string>& names) const;
    // Igd(RegionSet::from_file(p) for p in paths) with every file's text parsed on the device (gtgpu_igd_build_bed): when every
    // path ends in ".gz" the gzip bytes go to the device inflater (gtgpu_igd_build_bed_gz), otherwise each file is read (".gz"
    // inflated by zlib) and the texts go back to back.  Chromosome ids follow the names' first appearance in the files.  Errors
    // name the file's path.
    static std::unique_ptr<Igd> from_bed_files(std::shared_ptr<Device> dev, const std::vector<std::string>& paths);
    // count_region_hits_batch (pairwise: count_set_overlaps) of query sets given as BED files, each parsed on the device
    // (gtgpu_igd_count_bed; the gzip form when every path ends in ".gz", as from_bed_files).  matrix: [paths x n_files];
    // set_regions: every file's region lines (RegionSet::len).  Errors name the file's path.  A database Igd only.
    struct BedCounts {
        std::vector<uint64_t> matrix, set_regions;
    };
    BedCounts count_bed_files(const std::vector<std::string>& paths, int32_t min_overlap, bool pairwise) const;
    // gtgpu_igd_info: n_files, records kept, device bytes, LUT shift (a database Igd only)
    std::array<uint64_t, 4> info() const;

    // Igd::from_single_region_set (igd.rs:609-634): two-set overlap queries; the subject index is kept per record.
    static std::unique_ptr<Igd> from_single_region_set(std::shared_ptr<Device> dev, const RegionSet& subject);
    // igd.rs:645-678: (query idx, subject idx) pairs, one per overlapping pair, sorted.
    std::vector<std::pair<uint32_t, uint32_t>> find_overlaps_regionset(const RegionSet& query, int32_t min_overlap = 1) const;
    // igd.rs:690-722: number of distinct subject regions overlapping each query region.
    std::vector<uint32_t> count_overlaps_per_query(const RegionSet& query, int32_t min_overlap = 1) const;

   private:
    Igd() = default;
    std::shared_ptr<Device> dev_;
    gtgpu_igd* igd_ = nullptr;
    ChromMap cmap_;
    size_t n_files_ = 0;
    // single-set mode: the kept subjects (0 <= start < end as i32, like Igd::add) in an overlap index, val = subject idx
    std::unique_ptr<MultiChromOverlapper> single_;
    std::vector<uint32_t> single_src_;
};

// run_lola up to the contingency tables (enrichment.rs:198-220): [user set][db set].  Fisher / ranking stay with the caller.
std::vector<std::vector<ContingencyCounts>> lola_contingency(const Igd& igd, const std::vector<const RegionSet*>& user_sets,
                                                             const RegionSet& universe, int32_t min_overlap = 1);
// lola_contingency([RegionSet(p) for p in user_paths], RegionSet(universe_path)) with every file parsed on the device, the
// universe counted as the last set of the same pass (Igd::count_bed_files).
std::vector<std::vector<ContingencyCounts>> lola_contingency_bed_files(const Igd& igd, const std::vector<std::string>& user_paths,
                                                                       const std::string& universe_path, int32_t min_overlap = 1);

}  // namespace gtars
