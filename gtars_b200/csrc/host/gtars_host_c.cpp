// gtars_host_c.cpp — a small handle-based C surface over gtars_host.hpp so that the Python package (ctypes) and the
// tests can drive the C++ host layer.  Every function returns NULL / non-zero on failure; gth_last_error() has the text.
#include <cstring>

#include "gtars_host.hpp"

using namespace gtars;

namespace {
thread_local std::string g_err;

struct Lists {  // a list of (optionally named) u32 lists
    std::vector<std::string> names;
    std::vector<std::vector<uint32_t>> lists;
};

template <class F>
auto guard(F&& f, decltype(f()) on_error) -> decltype(f()) {
    try {
        return f();
    } catch (const std::exception& e) {
        g_err = e.what();
        return on_error;
    }
}

std::vector<const RegionSet*> as_sets(uint64_t n, void** handles) {
    std::vector<const RegionSet*> v(n);
    for (uint64_t i = 0; i < n; ++i) v[i] = (const RegionSet*)handles[i];
    return v;
}

Lists* count_lists(const std::vector<std::pair<std::string, std::map<uint32_t, uint32_t>>>& counts) {
    Lists* l = new Lists();
    for (auto& kv : counts) {
        l->names.push_back(kv.first);
        std::vector<uint32_t> flat;
        for (auto& tc : kv.second) { flat.push_back(tc.first); flat.push_back(tc.second); }
        l->lists.push_back(std::move(flat));
    }
    return l;
}
}  // namespace

extern "C" {

const char* gth_last_error() { return g_err.c_str(); }

void* gth_device_new(int device) {
    return guard([&]() -> void* { return new std::shared_ptr<Device>(std::make_shared<Device>(device)); }, nullptr);
}
void gth_device_free(void* d) { delete (std::shared_ptr<Device>*)d; }

// ---- RegionSet -------------------------------------------------------------------------------------------------------------
void* gth_regionset_from_file(const char* path) {
    return guard([&]() -> void* { return new RegionSet(RegionSet::from_file(path)); }, nullptr);
}
void* gth_regionset_new(uint64_t n, const char** chr, const uint32_t* start, const uint32_t* end) {
    return guard([&]() -> void* {
        RegionSet* rs = new RegionSet();
        rs->regions.resize(n);
        for (uint64_t i = 0; i < n; ++i) rs->regions[i] = Region{chr[i], start[i], end[i], ""};
        return rs;
    }, nullptr);
}
void gth_regionset_free(void* rs) { delete (RegionSet*)rs; }
uint64_t gth_regionset_len(void* rs) { return ((RegionSet*)rs)->regions.size(); }
const char* gth_regionset_chr(void* rs, uint64_t i) { return ((RegionSet*)rs)->regions[i].chr.c_str(); }
uint32_t gth_regionset_start(void* rs, uint64_t i) { return ((RegionSet*)rs)->regions[i].start; }
uint32_t gth_regionset_end(void* rs, uint64_t i) { return ((RegionSet*)rs)->regions[i].end; }

// ---- lists ------------------------------------------------------------------------------------------------------------------
void gth_lists_free(void* l) { delete (Lists*)l; }
uint64_t gth_lists_n(void* l) { return ((Lists*)l)->lists.size(); }
uint64_t gth_lists_len(void* l, uint64_t i) { return ((Lists*)l)->lists[i].size(); }
const uint32_t* gth_lists_data(void* l, uint64_t i) { return ((Lists*)l)->lists[i].data(); }
const char* gth_lists_name(void* l, uint64_t i) { return ((Lists*)l)->names[i].c_str(); }

// ---- MultiChromOverlapper ------------------------------------------------------------------------------------------------------
void* gth_mco_new(void* dev, void* source, int kind) {
    return guard([&]() -> void* {
        return new MultiChromOverlapper(*(std::shared_ptr<Device>*)dev, *(RegionSet*)source, (OverlapperType)kind);
    }, nullptr);
}
void gth_mco_free(void* m) { delete (MultiChromOverlapper*)m; }
int gth_mco_count(void* m, void* query, int32_t min_overlap, uint64_t* out) {
    return guard([&]() -> int {
        auto v = ((MultiChromOverlapper*)m)->count_overlaps(*(RegionSet*)query, min_overlap);
        std::copy(v.begin(), v.end(), out);
        return 0;
    }, 1);
}
int gth_mco_any(void* m, void* query, int32_t min_overlap, uint8_t* out) {
    return guard([&]() -> int {
        auto v = ((MultiChromOverlapper*)m)->any_overlaps(*(RegionSet*)query, min_overlap);
        for (size_t i = 0; i < v.size(); ++i) out[i] = v[i];
        return 0;
    }, 1);
}
void* gth_mco_find(void* m, void* query, int32_t min_overlap) {
    return guard([&]() -> void* {
        Lists* l = new Lists();
        l->lists = ((MultiChromOverlapper*)m)->find_overlaps_indices(*(RegionSet*)query, min_overlap);
        return l;
    }, nullptr);
}
void* gth_mco_subset_by(void* m, void* query, int32_t min_overlap) {
    return guard([&]() -> void* { return new RegionSet(((MultiChromOverlapper*)m)->subset_by(*(RegionSet*)query, min_overlap)); },
                 nullptr);
}

// ---- IndexedRegionSet ---------------------------------------------------------------------------------------------------------
void* gth_irs_new(void* dev, void* regions, int kind) {
    return guard([&]() -> void* {
        return new IndexedRegionSet(*(std::shared_ptr<Device>*)dev, *(RegionSet*)regions, (OverlapperType)kind);
    }, nullptr);
}
void gth_irs_free(void* r) { delete (IndexedRegionSet*)r; }
void* gth_irs_find(void* r, void* query, int32_t min_overlap) {
    return guard([&]() -> void* {
        Lists* l = new Lists();
        l->lists = ((IndexedRegionSet*)r)->find_overlaps(*(RegionSet*)query, min_overlap);
        return l;
    }, nullptr);
}
void* gth_irs_subset_by_overlaps(void* r, void* query, int32_t min_overlap) {
    return guard([&]() -> void* { return new RegionSet(((IndexedRegionSet*)r)->subset_by_overlaps(*(RegionSet*)query, min_overlap)); },
                 nullptr);
}
int gth_irs_count(void* r, void* query, int32_t min_overlap, uint64_t* out) {
    return guard([&]() -> int {
        auto v = ((IndexedRegionSet*)r)->count_overlaps(*(RegionSet*)query, min_overlap);
        std::copy(v.begin(), v.end(), out);
        return 0;
    }, 1);
}
int gth_irs_any(void* r, void* query, int32_t min_overlap, uint8_t* out) {
    return guard([&]() -> int {
        auto v = ((IndexedRegionSet*)r)->any_overlaps(*(RegionSet*)query, min_overlap);
        for (size_t i = 0; i < v.size(); ++i) out[i] = v[i];
        return 0;
    }, 1);
}

// ---- the same over BED files: flat results (one copy into the caller's arrays, no per-element conversion) ----------------------
// gth_mco_overlaps_bed_files (mode COUNT / ANY / FIND) and gth_irs_find_bed_files return a BedFilesOverlaps handle; its arrays
// are read with gth_overlaps_len / gth_overlaps_data, which: 0 file_queries (u64), 1 offsets (u64), 2 values (u32), 3 flags (u8).
void* gth_mco_overlaps_bed_files(void* m, uint64_t n, const char** paths, int mode, int32_t min_overlap) {
    return guard([&]() -> void* {
        return new BedFilesOverlaps(
            ((MultiChromOverlapper*)m)->overlaps_bed_files(std::vector<std::string>(paths, paths + n), mode, min_overlap));
    }, nullptr);
}
void* gth_irs_find_bed_files(void* r, uint64_t n, const char** paths, int32_t min_overlap) {
    return guard([&]() -> void* {
        return new BedFilesOverlaps(((IndexedRegionSet*)r)->find_overlaps_bed_files_flat(std::vector<std::string>(paths, paths + n), min_overlap));
    }, nullptr);
}
void gth_overlaps_free(void* h) { delete (BedFilesOverlaps*)h; }
uint64_t gth_overlaps_len(void* h, int which) {
    const BedFilesOverlaps& o = *(BedFilesOverlaps*)h;
    return which == 0 ? o.file_queries.size() : which == 1 ? o.offsets.size() : which == 2 ? o.values.size() : o.flags.size();
}
const void* gth_overlaps_data(void* h, int which) {
    const BedFilesOverlaps& o = *(BedFilesOverlaps*)h;
    return which == 0 ? (const void*)o.file_queries.data() : which == 1 ? (const void*)o.offsets.data()
                                                           : which == 2 ? (const void*)o.values.data() : (const void*)o.flags.data();
}
// out_sets: n RegionSet handles, one per path
int gth_mco_subset_by_bed_files(void* m, uint64_t n, const char** paths, int32_t min_overlap, void** out_sets) {
    return guard([&]() -> int {
        auto sets = ((MultiChromOverlapper*)m)->subset_by_bed_files(std::vector<std::string>(paths, paths + n), min_overlap);
        for (uint64_t f = 0; f < n; ++f) out_sets[f] = new RegionSet(std::move(sets[f]));
        return 0;
    }, 1);
}
int gth_irs_subset_by_overlaps_bed_files(void* r, uint64_t n, const char** paths, int32_t min_overlap, void** out_sets) {
    return guard([&]() -> int {
        auto sets = ((IndexedRegionSet*)r)->subset_by_overlaps_bed_files(std::vector<std::string>(paths, paths + n), min_overlap);
        for (uint64_t f = 0; f < n; ++f) out_sets[f] = new RegionSet(std::move(sets[f]));
        return 0;
    }, 1);
}

// ---- gtars_scoring ---------------------------------------------------------------------------------------------------------------
void* gth_consensus_new(void* dev, const char* path) {
    return guard([&]() -> void* { return new ConsensusSet(*(std::shared_ptr<Device>*)dev, std::string(path)); }, nullptr);
}
void gth_consensus_free(void* c) { delete (ConsensusSet*)c; }
uint64_t gth_consensus_len(void* c) { return ((ConsensusSet*)c)->len(); }
int gth_region_scoring(void* c, uint64_t n_files, const char** paths, int mode, uint32_t* out /* n_files x len */) {
    return guard([&]() -> int {
        std::vector<std::string> files(paths, paths + n_files);
        CountMatrix m = region_scoring_from_fragments(files, *(ConsensusSet*)c, (ScoringMode)mode);
        std::copy(m.data.begin(), m.data.end(), out);
        return 0;
    }, 1);
}
// barcode -> interleaved (peak, count) pairs
void* gth_barcode_scoring(void* c, const char* path) {
    return guard([&]() -> void* {
        Lists* l = new Lists();
        for (auto& kv : barcode_scoring_from_fragments(path, *(ConsensusSet*)c)) {
            l->names.push_back(kv.first);
            std::vector<uint32_t> flat;
            for (auto& pc : kv.second) { flat.push_back(pc.first); flat.push_back(pc.second); }
            l->lists.push_back(std::move(flat));
        }
        return l;
    }, nullptr);
}

// ---- Tokenizer ------------------------------------------------------------------------------------------------------------------
void* gth_tokenizer_new(void* dev, const char* path, int how /*0 auto, 1 bed, 2 config*/) {
    return guard([&]() -> void* {
        auto d = *(std::shared_ptr<Device>*)dev;
        std::unique_ptr<Tokenizer> t = how == 1 ? Tokenizer::from_bed(d, path) : how == 2 ? Tokenizer::from_config(d, path)
                                                                                           : Tokenizer::from_auto(d, path);
        return t.release();
    }, nullptr);
}
void gth_tokenizer_free(void* t) { delete (Tokenizer*)t; }
uint64_t gth_tokenizer_vocab_size(void* t) { return ((Tokenizer*)t)->get_vocab_size(); }
int64_t gth_tokenizer_token_to_id(void* t, const char* tok) { return ((Tokenizer*)t)->convert_token_to_id(tok); }
const char* gth_tokenizer_id_to_token(void* t, uint32_t id) {
    const std::string* s = ((Tokenizer*)t)->convert_id_to_token(id);
    return s ? s->c_str() : nullptr;
}
const char* gth_tokenizer_special(void* t, int which /*0 unk 1 pad 2 mask 3 cls 4 eos 5 bos 6 sep*/) {
    const SpecialTokens& s = ((Tokenizer*)t)->special_tokens();
    const std::string* all[7] = {&s.unk, &s.pad, &s.mask, &s.cls, &s.eos, &s.bos, &s.sep};
    return which >= 0 && which < 7 ? all[which]->c_str() : nullptr;
}
int gth_tokenizer_kind(void* t) { return (int)((Tokenizer*)t)->kind(); }
void* gth_tokenizer_encode_batch(void* t, uint64_t n, void** region_sets) {
    return guard([&]() -> void* {
        std::vector<const std::vector<Region>*> calls(n);
        for (uint64_t i = 0; i < n; ++i) calls[i] = &((RegionSet*)region_sets[i])->regions;
        Lists* l = new Lists();
        l->lists = ((Tokenizer*)t)->encode_batch(calls);
        return l;
    }, nullptr);
}
void* gth_tokenizer_encode_bed_file(void* t, const char* path) {
    return guard([&]() -> void* {
        Lists* l = new Lists();
        l->lists.push_back(((Tokenizer*)t)->encode_bed_file(path));
        return l;
    }, nullptr);
}
void* gth_tokenizer_encode_bed_files(void* t, uint64_t n, const char** paths) {
    return guard([&]() -> void* {
        auto lists = ((Tokenizer*)t)->encode_bed_files(std::vector<std::string>(paths, paths + n));
        Lists* l = new Lists();
        l->lists = std::move(lists);
        return l;
    }, nullptr);
}
// BED text -> (chr ids, starts, ends) through the device parser; chromosome names in `names` (n of them) get ids 0..n-1
void* gth_parse_bed_file(void* dev, const char* path, uint64_t n_names, const char** names) {
    return guard([&]() -> void* {
        ChromMap cmap;
        for (uint64_t i = 0; i < n_names; ++i) cmap.add(names[i]);
        FlatQueries q = parse_bed_text_device(**(std::shared_ptr<Device>*)dev, read_file_bytes(path), cmap);
        Lists* l = new Lists();
        l->lists = {std::move(q.chr), std::move(q.start), std::move(q.end)};
        return l;
    }, nullptr);
}
int gth_gtok_write(const char* path, uint64_t n, const uint32_t* tokens, int mode /*0 write, 1 append, 2 init*/) {
    return guard([&]() -> int {
        std::vector<uint32_t> v(tokens, tokens + n);
        if (mode == 0) write_tokens_to_gtok(path, v);
        else if (mode == 1) append_tokens_to_gtok_file(path, v);
        else init_gtok_file(path);
        return 0;
    }, 1);
}
void* gth_gtok_read(const char* path) {
    return guard([&]() -> void* {
        Lists* l = new Lists();
        l->lists.push_back(read_tokens_from_gtok(path));
        return l;
    }, nullptr);
}
void* gth_tokenizer_fragments_device(void* t, const char* path) {
    return guard([&]() -> void* {
        Lists* l = new Lists();
        for (auto& kv : ((Tokenizer*)t)->tokenize_fragment_file_device(path)) {
            l->names.push_back(kv.first);
            l->lists.push_back(std::move(kv.second));
        }
        return l;
    }, nullptr);
}
int gth_region_scoring_device(void* c, uint64_t n_files, const char** paths, int mode, uint32_t* out /* n_files x len */) {
    return guard([&]() -> int {
        std::vector<std::string> files(paths, paths + n_files);
        CountMatrix m = region_scoring_from_fragments_device(files, *(ConsensusSet*)c, (ScoringMode)mode);
        std::copy(m.data.begin(), m.data.end(), out);
        return 0;
    }, 1);
}
void* gth_barcode_scoring_device(void* c, const char* path) {
    return guard([&]() -> void* {
        Lists* l = new Lists();
        for (auto& kv : barcode_scoring_from_fragments_device(path, *(ConsensusSet*)c)) {
            l->names.push_back(kv.first);
            std::vector<uint32_t> flat;
            for (auto& pc : kv.second) { flat.push_back(pc.first); flat.push_back(pc.second); }
            l->lists.push_back(std::move(flat));
        }
        return l;
    }, nullptr);
}
void* gth_tokenizer_fragments(void* t, const char* path) {
    return guard([&]() -> void* {
        Lists* l = new Lists();
        for (auto& kv : ((Tokenizer*)t)->tokenize_fragment_file(path)) {
            l->names.push_back(kv.first);
            l->lists.push_back(std::move(kv.second));
        }
        return l;
    }, nullptr);
}
// barcode -> interleaved (token id, count) pairs
void* gth_tokenizer_count_fragments(void* t, const char* path) {
    return guard([&]() -> void* { return count_lists(((Tokenizer*)t)->count_fragments_by_barcode(path)); }, nullptr);
}
void* gth_tokenizer_count_fragments_device(void* t, const char* path) {
    return guard([&]() -> void* { return count_lists(((Tokenizer*)t)->count_fragments_by_barcode_device(path)); }, nullptr);
}

// ---- Igd / LOLA -------------------------------------------------------------------------------------------------------------------
void* gth_igd_new(void* dev, uint64_t n, void** region_sets) {
    return guard([&]() -> void* { return new Igd(*(std::shared_ptr<Device>*)dev, as_sets(n, region_sets)); }, nullptr);
}
void* gth_igd_single(void* dev, void* subject) {
    return guard([&]() -> void* { return Igd::from_single_region_set(*(std::shared_ptr<Device>*)dev, *(RegionSet*)subject).release(); },
                 nullptr);
}
// pairs as one flat list [q0, s0, q1, s1, ...]
void* gth_igd_find_pairs(void* g, void* query, int32_t min_overlap) {
    return guard([&]() -> void* {
        Lists* l = new Lists();
        l->lists.emplace_back();
        for (auto& p : ((Igd*)g)->find_overlaps_regionset(*(RegionSet*)query, min_overlap)) {
            l->lists[0].push_back(p.first);
            l->lists[0].push_back(p.second);
        }
        return l;
    }, nullptr);
}
void* gth_igd_count_per_query(void* g, void* query, int32_t min_overlap) {
    return guard([&]() -> void* {
        Lists* l = new Lists();
        l->lists.push_back(((Igd*)g)->count_overlaps_per_query(*(RegionSet*)query, min_overlap));
        return l;
    }, nullptr);
}
int gth_igd_save_sets(uint64_t n, void** region_sets, const char** names, const char* path) {
    return guard([&]() -> int {
        std::vector<std::pair<std::string, const RegionSet*>> sets;
        for (uint64_t i = 0; i < n; ++i) sets.emplace_back(names[i], (const RegionSet*)region_sets[i]);
        Igd::save_named_region_sets(sets, path);
        return 0;
    }, 1);
}
int gth_igd_save(void* g, uint64_t n, const char** names, const char* path) {
    return guard([&]() -> int {
        ((Igd*)g)->save(path, std::vector<std::string>(names, names + n));
        return 0;
    }, 1);
}
void* gth_igd_from_file(void* dev, const char* path) {
    return guard([&]() -> void* { return Igd::from_igd_file(*(std::shared_ptr<Device>*)dev, path).release(); }, nullptr);
}
void* gth_igd_from_bed_files(void* dev, uint64_t n, const char** paths) {
    return guard([&]() -> void* {
        return Igd::from_bed_files(*(std::shared_ptr<Device>*)dev, std::vector<std::string>(paths, paths + n)).release();
    }, nullptr);
}
int gth_igd_info(void* g, uint64_t* out /* 4 */) {
    return guard([&]() -> int {
        auto a = ((Igd*)g)->info();
        std::copy(a.begin(), a.end(), out);
        return 0;
    }, 1);
}
void gth_igd_free(void* g) { delete (Igd*)g; }
uint64_t gth_igd_num_files(void* g) { return ((Igd*)g)->num_files(); }
int gth_igd_count(void* g, uint64_t n_sets, void** region_sets, int32_t min_overlap, int pairwise, uint64_t* out) {
    return guard([&]() -> int {
        auto v = ((Igd*)g)->count_region_hits_batch(as_sets(n_sets, region_sets), min_overlap, pairwise != 0);
        std::copy(v.begin(), v.end(), out);
        return 0;
    }, 1);
}
int gth_lola_contingency(void* g, uint64_t n_user, void** user_sets, void* universe, int32_t min_overlap, int64_t* out) {
    return guard([&]() -> int {
        auto t = lola_contingency(*(Igd*)g, as_sets(n_user, user_sets), *(RegionSet*)universe, min_overlap);
        size_t k = 0;
        for (auto& row : t)
            for (auto& c : row) {
                out[k++] = c.a; out[k++] = c.b; out[k++] = c.c; out[k++] = c.d;
            }
        return 0;
    }, 1);
}
// out: [n_paths x num_files] u64, out_set_regions: n_paths u64
int gth_igd_count_bed_files(void* g, uint64_t n_paths, const char** paths, int32_t min_overlap, int pairwise, uint64_t* out,
                            uint64_t* out_set_regions) {
    return guard([&]() -> int {
        auto r = ((Igd*)g)->count_bed_files(std::vector<std::string>(paths, paths + n_paths), min_overlap, pairwise != 0);
        std::copy(r.matrix.begin(), r.matrix.end(), out);
        std::copy(r.set_regions.begin(), r.set_regions.end(), out_set_regions);
        return 0;
    }, 1);
}
int gth_lola_contingency_bed_files(void* g, uint64_t n_user, const char** user_paths, const char* universe_path, int32_t min_overlap,
                                   int64_t* out) {
    return guard([&]() -> int {
        auto t = lola_contingency_bed_files(*(Igd*)g, std::vector<std::string>(user_paths, user_paths + n_user), universe_path,
                                            min_overlap);
        size_t k = 0;
        for (auto& row : t)
            for (auto& c : row) {
                out[k++] = c.a; out[k++] = c.b; out[k++] = c.c; out[k++] = c.d;
            }
        return 0;
    }, 1);
}

}  // extern "C"
