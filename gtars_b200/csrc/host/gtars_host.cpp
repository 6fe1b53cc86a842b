// gtars_host.cpp — implementation of gtars_host.hpp (host-side mirror of the reference API; all overlap work goes
// through the C ABI of include/gtars_gpu.h).
#include "gtars_host.hpp"

#include <zlib.h>

#include <algorithm>
#include <array>
#include <cstring>
#include <fstream>
#include <set>
#include <sstream>

namespace gtars {

namespace {

[[noreturn]] void throw_gpu(const char* what) { throw Error(std::string(what) + ": " + gtgpu_last_error()); }
void check(int32_t status, const char* what) {
    if (status != GTGPU_OK) throw_gpu(what);
}

// get_dynamic_reader (gtars-core/src/utils.rs:115-126): gzip iff the extension is "gz"; BufRead::lines() semantics.
std::vector<std::string> read_lines(const std::string& path) {
    const std::string data = gtars::read_file_bytes(path);
    std::vector<std::string> lines;
    size_t pos = 0;
    while (pos < data.size()) {
        size_t nl = data.find('\n', pos);
        size_t end = nl == std::string::npos ? data.size() : nl;
        lines.emplace_back(data, pos, end - pos);
        // BufRead::lines: only a '\r' in front of the stripped '\n' goes; a last line without a newline keeps it
        if (nl != std::string::npos && !lines.back().empty() && lines.back().back() == '\r') lines.back().pop_back();
        pos = nl == std::string::npos ? data.size() : nl + 1;
    }
    return lines;
}

std::vector<std::string> split_on(const std::string& s, char sep) {
    std::vector<std::string> out;
    size_t pos = 0;
    for (;;) {
        size_t k = s.find(sep, pos);
        if (k == std::string::npos) {
            out.emplace_back(s, pos);
            return out;
        }
        out.emplace_back(s, pos, k - pos);
        pos = k + 1;
    }
}

std::vector<std::string> split_whitespace(const std::string& s) {
    std::vector<std::string> out;
    size_t i = 0;
    while (i < s.size()) {
        while (i < s.size() && isspace((unsigned char)s[i])) ++i;
        size_t j = i;
        while (j < s.size() && !isspace((unsigned char)s[j])) ++j;
        if (j > i) out.emplace_back(s, i, j - i);
        i = j;
    }
    return out;
}

bool parse_u32(const std::string& s, uint32_t& out) {  // Rust's str::parse::<u32>()
    size_t i = (!s.empty() && s[0] == '+') ? 1 : 0;
    if (i >= s.size()) return false;
    uint64_t v = 0;
    for (; i < s.size(); ++i) {
        if (s[i] < '0' || s[i] > '9') return false;
        v = v * 10 + (uint64_t)(s[i] - '0');
        if (v > 0xFFFFFFFFull) return false;
    }
    out = (uint32_t)v;
    return true;
}

bool has_prefix(const std::string& s, const char* p) { return s.rfind(p, 0) == 0; }

std::string trim(const std::string& s) {
    size_t a = 0, b = s.size();
    while (a < b && isspace((unsigned char)s[a])) ++a;
    while (b > a && isspace((unsigned char)s[b - 1])) --b;
    return s.substr(a, b - a);
}

struct PinnedResult {  // RAII over gtgpu_buf
    gtgpu_buf* buf = nullptr;
    ~PinnedResult() { gtgpu_buf_free(buf); }
    const uint32_t* data() const { return (const uint32_t*)gtgpu_buf_data(buf); }
    uint64_t len() const { return gtgpu_buf_len(buf); }
};

}  // namespace

std::string read_file_bytes(const std::string& path) {
    std::string data;
    const bool gz = path.size() >= 3 && path.compare(path.size() - 3, 3, ".gz") == 0;
    if (gz) {
        gzFile f = gzopen(path.c_str(), "rb");
        if (!f) throw Error("Failed to open file: \"" + path + "\"");
        char buf[1 << 16];
        int n;
        while ((n = gzread(f, buf, sizeof buf)) > 0) data.append(buf, n);
        int zerr = Z_OK;
        const char* zmsg = n < 0 ? gzerror(f, &zerr) : nullptr;  // a truncated / corrupt stream is an error, not an early EOF
        const std::string why = zmsg ? zmsg : "";
        const int closed = gzclose(f);
        if (n < 0 || closed != Z_OK)  // Z_BUF_ERROR from gzclose = the stream ended in the middle of a gzip member (truncated)
            throw Error("Failed to read gzip file: \"" + path + "\"" + (why.empty() ? "" : ": " + why));
    } else {
        std::ifstream f(path, std::ios::binary | std::ios::ate);
        if (!f) throw Error("Failed to open file: \"" + path + "\"");
        const std::streamsize size = f.tellg();
        f.seekg(0);
        data.resize((size_t)std::max<std::streamsize>(size, 0));
        if (size > 0 && !f.read(&data[0], size)) throw Error("Failed to read file: \"" + path + "\"");
    }
    return data;
}

namespace {
struct NameBlob {
    std::string blob;
    std::vector<uint32_t> offsets{0};
    explicit NameBlob(const ChromMap& cmap) {
        for (uint32_t i = 0; i < cmap.size(); ++i) {
            blob += cmap.name(i);
            offsets.push_back((uint32_t)blob.size());
        }
    }
};
}  // namespace

FlatQueries parse_bed_text_device(const Device& dev, const std::string& text, const ChromMap& cmap) {
    NameBlob nb(cmap);
    uint64_t n = 0;
    PinnedResult c, s, e;
    check(gtgpu_parse_bed(dev.ctx(), text.data(), text.size(), (uint32_t)cmap.size(), nb.blob.data(), nb.offsets.data(), &n, &c.buf,
                          &s.buf, &e.buf),
          "gtgpu_parse_bed");
    FlatQueries q;
    q.chr.assign(c.data(), c.data() + n);
    q.start.assign(s.data(), s.data() + n);
    q.end.assign(e.data(), e.data() + n);
    return q;
}

// ---- gtok ------------------------------------------------------------------------------------------------------------------
namespace {
void put_tokens(std::ofstream& f, const std::vector<uint32_t>& tokens, bool small) {
    std::string b;
    b.reserve(tokens.size() * (small ? 2 : 4));
    for (uint32_t t : tokens) {
        b.push_back((char)(t & 0xFF));
        b.push_back((char)((t >> 8) & 0xFF));
        if (!small) {
            b.push_back((char)((t >> 16) & 0xFF));
            b.push_back((char)((t >> 24) & 0xFF));
        }
    }
    f.write(b.data(), (std::streamsize)b.size());
}
}  // namespace

void write_tokens_to_gtok(const std::string& filename, const std::vector<uint32_t>& tokens) {
    std::ofstream f(filename, std::ios::binary);
    if (!f) throw Error("Failed to create gtok file!");
    const bool small = std::all_of(tokens.begin(), tokens.end(), [](uint32_t x) { return x <= 0xFFFFu; });
    f.write("GTOK", 4);
    f.put(small ? (char)0x01 : (char)0x02);
    put_tokens(f, tokens, small);
}
void init_gtok_file(const std::string& filename) {
    std::ofstream f(filename, std::ios::binary);
    if (!f) throw Error("Failed to create gtok file!");
    f.write("GTOK", 4);
    f.put((char)0x02);  // assume large (gtok.rs:238-240)
}
std::vector<uint32_t> read_tokens_from_gtok(const std::string& filename) {
    std::ifstream f(filename, std::ios::binary);
    if (!f) throw Error("Failed to open gtok file!");
    std::stringstream ss;
    ss << f.rdbuf();
    const std::string d = ss.str();
    if (d.size() < 5 || d.compare(0, 4, "GTOK") != 0) throw Error("File doesn't appear to be a valid .gtok file.");
    const unsigned char flag = (unsigned char)d[4];
    if (flag != 0x01 && flag != 0x02) throw Error("Invalid data format flag found in gtok file");
    const size_t w = flag == 0x01 ? 2 : 4;
    std::vector<uint32_t> tokens;
    for (size_t pos = 5; pos + w <= d.size(); pos += w) {  // a trailing partial token is dropped, like read_exact failing
        uint32_t v = 0;
        for (size_t k = 0; k < w; ++k) v |= (uint32_t)(unsigned char)d[pos + k] << (8 * k);
        tokens.push_back(v);
    }
    return tokens;
}
void append_tokens_to_gtok_file(const std::string& filename, const std::vector<uint32_t>& tokens) {
    unsigned char flag;
    {
        std::ifstream f(filename, std::ios::binary);
        if (!f) throw Error("Failed to open gtok file!");
        char h[5];
        if (!f.read(h, 5) || std::string(h, 4) != "GTOK") throw Error("File doesn't appear to be a valid .gtok file.");
        flag = (unsigned char)h[4];
    }
    if (flag != 0x01 && flag != 0x02) throw Error("Invalid data format flag found in gtok file");
    std::ofstream f(filename, std::ios::binary | std::ios::app);
    if (!f) throw Error("Failed to open gtok file for appending");
    put_tokens(f, tokens, flag == 0x01);  // tokens are truncated to u16 when the file says so (gtok.rs:278-284)
}

// ---- RegionSet ---------------------------------------------------------------------------------------------------------
namespace {
// str::parse::<u32>() over [a, b): optional '+', at least one digit, digits only, no overflow
bool parse_u32_range(const char* a, const char* b, uint32_t& out) {
    if (a < b && *a == '+') ++a;
    if (a >= b) return false;
    uint64_t v = 0;
    for (; a < b; ++a) {
        if (*a < '0' || *a > '9') return false;
        v = v * 10 + (uint64_t)(*a - '0');
        if (v > 0xFFFFFFFFull) return false;
    }
    out = (uint32_t)v;
    return true;
}
bool starts_with(const char* a, const char* b, const char* p) {
    const size_t n = strlen(p);
    return (size_t)(b - a) >= n && memcmp(a, p, n) == 0;
}
}  // namespace

RegionSet RegionSet::from_file(const std::string& path) {
    // One pass over the file's bytes (no per-line strings): BufRead::lines() splitting, then region_set.rs:60-185.
    RegionSet rs;
    const std::string data = read_file_bytes(path);
    const char* p = data.data();
    const char* const end = p + data.size();
    bool first_line = true;
    while (p < end) {
        const char* nl = (const char*)memchr(p, '\n', (size_t)(end - p));
        const char* le = nl ? nl : end;              // line = [p, le)
        const char* next = nl ? nl + 1 : end;
        if (le > p && le[-1] == '\r') --le;
        if (starts_with(p, le, "browser") || starts_with(p, le, "track") || starts_with(p, le, "#")) {
            rs.header.append(p, le);
            first_line = false;
            p = next;
            continue;
        }
        const char* t1 = (const char*)memchr(p, '\t', (size_t)(le - p));
        const char* t2 = t1 ? (const char*)memchr(t1 + 1, '\t', (size_t)(le - t1 - 1)) : nullptr;
        const char* t3 = t2 ? (const char*)memchr(t2 + 1, '\t', (size_t)(le - t2 - 1)) : nullptr;
        const bool three = t1 && t2;
        Region r;
        const bool s_ok = three && parse_u32_range(t1 + 1, t2, r.start);
        if (first_line) {
            first_line = false;
            if (three && !s_ok) {  // column header row without '#'
                rs.header.append(p, le);
                p = next;
                continue;
            }
        }
        if (!s_ok) throw Error("Error in parsing start position: " + std::string(p, le));
        if (!parse_u32_range(t2 + 1, t3 ? t3 : le, r.end)) throw Error("Error in parsing end position: " + std::string(p, le));
        r.chr.assign(p, t1);
        if (t3) r.rest.assign(t3 + 1, le);  // parts[3..].join("\t") is the remainder of the line as written
        rs.regions.push_back(std::move(r));
        p = next;
    }
    if (rs.regions.empty()) throw Error("Corrupted file. 0 regions found in the file: " + path);
    rs.sort();
    return rs;
}

void RegionSet::sort() {
    // region_set.rs:502-505: stable, by (chromosome string, start).  Chromosome names repeat millions of times, so they
    // are ranked once and the sort runs on (rank, start, original position) integers.
    const size_t n = regions.size();
    std::unordered_map<std::string, uint32_t> ids;
    std::vector<uint32_t> cid(n);
    std::vector<const std::string*> names;
    for (size_t i = 0; i < n; ++i) {
        auto it = ids.find(regions[i].chr);
        if (it == ids.end()) {
            it = ids.emplace(regions[i].chr, (uint32_t)names.size()).first;
            names.push_back(&it->first);
        }
        cid[i] = it->second;
    }
    std::vector<uint32_t> by_name(names.size()), rank(names.size());
    for (uint32_t k = 0; k < by_name.size(); ++k) by_name[k] = k;
    std::sort(by_name.begin(), by_name.end(), [&](uint32_t a, uint32_t b) { return *names[a] < *names[b]; });
    for (uint32_t r = 0; r < by_name.size(); ++r) rank[by_name[r]] = r;
    struct Key {
        uint64_t k;   // rank << 32 | start
        uint64_t pos; // original position: the tie-break that makes the sort stable
    };
    std::vector<Key> keys(n);
    bool sorted = true;
    for (size_t i = 0; i < n; ++i) {
        keys[i] = Key{((uint64_t)rank[cid[i]] << 32) | regions[i].start, i};
        if (i && keys[i].k < keys[i - 1].k) sorted = false;
    }
    if (sorted) return;
    std::sort(keys.begin(), keys.end(), [](const Key& a, const Key& b) { return a.k != b.k ? a.k < b.k : a.pos < b.pos; });
    std::vector<Region> out;
    out.reserve(n);
    for (const Key& key : keys) out.push_back(std::move(regions[key.pos]));
    regions = std::move(out);
}

// ---- Device / ChromMap -----------------------------------------------------------------------------------------------------
Device::Device(int device) { check(gtgpu_init(device, nullptr, &ctx_), "gtgpu_init"); }
Device::~Device() { gtgpu_shutdown(ctx_); }

uint32_t ChromMap::add(const std::string& name) {
    auto it = ids_.find(name);
    if (it != ids_.end()) return it->second;
    uint32_t id = (uint32_t)names_.size();
    ids_.emplace(name, id);
    names_.push_back(name);
    return id;
}
uint32_t ChromMap::get(const std::string& name) const {
    auto it = ids_.find(name);
    return it == ids_.end() ? GTGPU_UNKNOWN_CHROM : it->second;
}

FlatQueries flatten(const std::vector<Region>& regions, const ChromMap& cmap) {
    FlatQueries q;
    q.chr.reserve(regions.size());
    q.start.reserve(regions.size());
    q.end.reserve(regions.size());
    for (const auto& r : regions) {
        q.chr.push_back(cmap.get(r.chr));
        q.start.push_back(r.start);
        q.end.push_back(r.end);
    }
    return q;
}

namespace {

// Intervals in insertion order -> chromosome-grouped arrays (insertion order kept inside a chromosome).
struct Grouped {
    std::vector<uint64_t> offsets;
    std::vector<uint32_t> start, end, val;
};
Grouped group_by_chrom(const std::vector<uint32_t>& chr, const std::vector<uint32_t>& start, const std::vector<uint32_t>& end,
                       const std::vector<uint32_t>& val, size_t n_chroms) {
    Grouped g;
    g.offsets.assign(n_chroms + 1, 0);
    for (uint32_t c : chr) g.offsets[c + 1]++;
    for (size_t c = 0; c < n_chroms; ++c) g.offsets[c + 1] += g.offsets[c];
    std::vector<uint64_t> cursor(g.offsets.begin(), g.offsets.end() - 1);
    g.start.resize(chr.size());
    g.end.resize(chr.size());
    g.val.resize(chr.size());
    for (size_t i = 0; i < chr.size(); ++i) {
        uint64_t p = cursor[chr[i]]++;
        g.start[p] = start[i];
        g.end[p] = end[i];
        g.val[p] = val[i];
    }
    return g;
}

}  // namespace

// ---- MultiChromOverlapper ---------------------------------------------------------------------------------------------------
MultiChromOverlapper::MultiChromOverlapper(std::shared_ptr<Device> dev, const RegionSet& source, OverlapperType kind)
    : dev_(std::move(dev)) {
    std::vector<uint32_t> chr, start, end, val;
    for (size_t i = 0; i < source.regions.size(); ++i) {
        const Region& r = source.regions[i];
        chr.push_back(cmap_.add(r.chr));
        start.push_back(r.start);
        end.push_back(r.end);
        val.push_back((uint32_t)i);
        source_.push_back(Region{r.chr, r.start, r.end, ""});
    }
    Grouped g = group_by_chrom(chr, start, end, val, cmap_.size());
    check(gtgpu_index_build(dev_->ctx(), (int32_t)kind, (uint32_t)cmap_.size(), g.offsets.data(), g.start.data(), g.end.data(),
                            g.val.data(), &index_),
          "gtgpu_index_build");
}
MultiChromOverlapper::~MultiChromOverlapper() { gtgpu_index_free(index_); }

std::vector<uint64_t> MultiChromOverlapper::count_overlaps(const RegionSet& query, int32_t min_overlap) const {
    FlatQueries q = flatten(query.regions, cmap_);
    std::vector<uint32_t> counts(q.chr.size());
    check(gtgpu_count(index_, q.chr.size(), q.chr.data(), q.start.data(), q.end.data(), std::max(min_overlap, 0), counts.data()),
          "gtgpu_count");
    return std::vector<uint64_t>(counts.begin(), counts.end());
}

std::vector<bool> MultiChromOverlapper::any_overlaps(const RegionSet& query, int32_t min_overlap) const {
    FlatQueries q = flatten(query.regions, cmap_);
    std::vector<uint8_t> any(q.chr.size());
    check(gtgpu_any(index_, q.chr.size(), q.chr.data(), q.start.data(), q.end.data(), std::max(min_overlap, 0), any.data()),
          "gtgpu_any");
    return std::vector<bool>(any.begin(), any.end());
}

std::vector<std::vector<uint32_t>> MultiChromOverlapper::find_overlaps_indices(const RegionSet& query, int32_t min_overlap) const {
    FlatQueries q = flatten(query.regions, cmap_);
    std::vector<uint64_t> offsets(q.chr.size() + 1);
    PinnedResult res;
    check(gtgpu_find(index_, q.chr.size(), q.chr.data(), q.start.data(), q.end.data(), std::max(min_overlap, 0), offsets.data(),
                     &res.buf),
          "gtgpu_find");
    std::vector<std::vector<uint32_t>> out(q.chr.size());
    for (size_t i = 0; i < out.size(); ++i) out[i].assign(res.data() + offsets[i], res.data() + offsets[i + 1]);
    return out;
}

std::vector<std::vector<Region>> MultiChromOverlapper::find_overlaps_regions(const RegionSet& query, int32_t min_overlap) const {
    auto idx = find_overlaps_indices(query, min_overlap);
    std::vector<std::vector<Region>> out(idx.size());
    for (size_t i = 0; i < idx.size(); ++i)
        for (uint32_t v : idx[i]) out[i].push_back(Region{query.regions[i].chr, source_[v].start, source_[v].end, ""});
    return out;
}

RegionSet MultiChromOverlapper::subset_by(const RegionSet& query, int32_t min_overlap) const {
    std::set<std::tuple<std::string, uint32_t, uint32_t>> hits;  // BTreeSet<(String, u32, u32)>
    auto idx = find_overlaps_indices(query, min_overlap);
    for (size_t i = 0; i < idx.size(); ++i)
        for (uint32_t v : idx[i]) hits.emplace(query.regions[i].chr, source_[v].start, source_[v].end);
    RegionSet rs;
    for (const auto& h : hits) rs.regions.push_back(Region{std::get<0>(h), std::get<1>(h), std::get<2>(h), ""});
    return rs;
}

// ---- Universe ---------------------------------------------------------------------------------------------------------------
Universe Universe::from_file(const std::string& path) {
    Universe u;
    auto lines = read_lines(path);
    if (lines.empty()) throw Error("Unable to determine universe type");
    int ftype = 0;  // universe/utils.rs:7-19
    if (!has_prefix(lines[0], "track")) {
        size_t nf = split_on(lines[0], '\t').size();
        if (nf == 3) ftype = 3;
        else if (nf >= 5) ftype = 5;
    }
    if (!ftype) throw Error("Unable to determine universe type");
    for (const auto& line : lines) {
        auto parts = ftype == 3 ? split_whitespace(line) : split_on(line, '\t');
        if (ftype == 3 ? parts.size() != 3 : parts.size() < 5) throw Error("Error parsing line: " + line);
        u.regions.push_back(parts[0] + ":" + parts[1] + "-" + parts[2]);
    }
    for (const auto& r : u.regions) u.region_to_id.emplace(r, (uint32_t)u.region_to_id.size());
    for (size_t i = 0; i < u.regions.size(); ++i) u.id_to_region[(uint32_t)i] = u.regions[i];
    return u;
}

void Universe::add_token_to_universe(const std::string& tok) {
    uint32_t id = (uint32_t)region_to_id.size();
    region_to_id[tok] = id;
    id_to_region[id] = tok;
    regions.push_back(tok);
}

// ---- Tokenizer ----------------------------------------------------------------------------------------------------------------
void Tokenizer::build(std::shared_ptr<Device> dev, Universe universe, SpecialTokens special, OverlapperType kind) {
    dev_ = std::move(dev);
    universe_ = std::move(universe);
    special_ = std::move(special);
    kind_ = kind;
    universe_.special_tokens = special_.as_vec();  // universe/mod.rs:114-120
    for (const auto& t : universe_.special_tokens) universe_.add_token_to_universe(t);
    unk_id_ = universe_.region_to_id.at(special_.unk);
    id_to_first_token_.resize(universe_.region_to_id.size());
    for (const auto& kv : universe_.region_to_id) id_to_first_token_[kv.second] = kv.first;

    // create_tokenize_core_from_universe (utils/mod.rs:49-99).  The reference's tokenize() maps each hit's val to a
    // string (id_to_region, positional) and encode() maps that back (region_to_id, first appearance); the composition
    // is folded into val here so the device emits final ids (identity unless the universe has duplicate lines).
    std::vector<uint32_t> chr, start, end, val;
    for (const auto& region : universe_.regions) {
        if (std::find(universe_.special_tokens.begin(), universe_.special_tokens.end(), region) != universe_.special_tokens.end())
            continue;
        auto parts = split_on(region, ':');
        auto se = parts.size() > 1 ? split_on(parts[1], '-') : std::vector<std::string>{};
        uint32_t s, e;
        if (se.size() < 2 || !parse_u32(se[0], s) || !parse_u32(se[1], e)) throw Error("cannot parse universe region " + region);
        uint32_t v = universe_.region_to_id.at(region);
        uint32_t folded = universe_.region_to_id.at(universe_.id_to_region.at(v));
        chr.push_back(cmap_.add(parts[0]));
        start.push_back(s);
        end.push_back(e);
        val.push_back(folded);
    }
    Grouped g = group_by_chrom(chr, start, end, val, cmap_.size());
    check(gtgpu_index_build(dev_->ctx(), (int32_t)kind, (uint32_t)cmap_.size(), g.offsets.data(), g.start.data(), g.end.data(),
                            g.val.data(), &index_),
          "gtgpu_index_build");
}

Tokenizer::~Tokenizer() { gtgpu_index_free(index_); }

std::unique_ptr<Tokenizer> Tokenizer::from_bed(std::shared_ptr<Device> dev, const std::string& path) {
    std::unique_ptr<Tokenizer> t(new Tokenizer());
    t->build(std::move(dev), Universe::from_file(path), SpecialTokens{}, OverlapperType::Bits);
    return t;
}

std::unique_ptr<Tokenizer> Tokenizer::from_config(std::shared_ptr<Device> dev, const std::string& path) {
    // The subset of TOML the reference's TokenizerConfig uses (config.rs:36-41): universe = "...",
    // tokenizer_type = "bits" | "ailist", special_tokens = [ {name="unk", token="..."}, ... ].
    std::ifstream f(path);
    if (!f) throw Error("No such file: " + path);
    std::stringstream ss;
    ss << f.rdbuf();
    const std::string text = ss.str();
    std::string universe_file;
    OverlapperType kind = OverlapperType::Bits;
    SpecialTokens special;
    auto value_of = [&](const std::string& key) -> std::string {
        size_t pos = 0;
        while ((pos = text.find(key, pos)) != std::string::npos) {
            bool at_line_start = pos == 0 || text[pos - 1] == '\n';
            size_t eq = text.find('=', pos);
            if (at_line_start && eq != std::string::npos && trim(text.substr(pos + key.size(), eq - pos - key.size())).empty()) {
                size_t q1 = text.find('"', eq), q2 = q1 == std::string::npos ? q1 : text.find('"', q1 + 1);
                if (q2 != std::string::npos) return text.substr(q1 + 1, q2 - q1 - 1);
            }
            pos += key.size();
        }
        return "";
    };
    universe_file = value_of("universe");
    if (universe_file.empty()) throw Error("missing field `universe` in " + path);
    std::string tt = value_of("tokenizer_type");
    if (!tt.empty()) {
        if (tt == "bits") kind = OverlapperType::Bits;
        else if (tt == "ailist") kind = OverlapperType::AIList;
        else throw Error("unknown variant `" + tt + "`, expected `bits` or `ailist`");
    }
    size_t st = text.find("special_tokens");
    if (st != std::string::npos) {
        size_t pos = st;
        while ((pos = text.find('{', pos)) != std::string::npos) {
            size_t close = text.find('}', pos);
            if (close == std::string::npos) break;
            std::string item = text.substr(pos + 1, close - pos - 1);
            std::string name, token;
            for (const auto& kv : split_on(item, ',')) {
                size_t eq = kv.find('=');
                if (eq == std::string::npos) continue;
                std::string k = trim(kv.substr(0, eq)), v = trim(kv.substr(eq + 1));
                if (v.size() >= 2 && v.front() == '"' && v.back() == '"') v = v.substr(1, v.size() - 2);
                if (k == "name") name = v;
                if (k == "token") token = v;
            }
            if (name == "unk") special.unk = token;
            else if (name == "pad") special.pad = token;
            else if (name == "mask") special.mask = token;
            else if (name == "cls") special.cls = token;
            else if (name == "bos") special.bos = token;
            else if (name == "eos") special.eos = token;
            else if (name == "sep") special.sep = token;
            else throw Error("unknown special token name `" + name + "`");
            pos = close + 1;
        }
    }
    size_t slash = path.find_last_of('/');
    std::string dir = slash == std::string::npos ? "" : path.substr(0, slash + 1);
    std::unique_ptr<Tokenizer> t(new Tokenizer());
    t->build(std::move(dev), Universe::from_file(dir + universe_file), special, kind);
    return t;
}

std::unique_ptr<Tokenizer> Tokenizer::from_auto(std::shared_ptr<Device> dev, const std::string& path) {
    auto ends_with = [&](const char* suf) {
        size_t n = strlen(suf);
        return path.size() >= n && path.compare(path.size() - n, n, suf) == 0;
    };
    if (ends_with(".toml")) return from_config(std::move(dev), path);
    if (ends_with(".bed") || ends_with(".bed.gz")) return from_bed(std::move(dev), path);
    throw Error("Missing or invalid file extension in tokenizer config file. It must be `toml`, `bed` or `bed.gz`");
}

std::vector<std::vector<uint32_t>> Tokenizer::encode_batch(const std::vector<const std::vector<Region>*>& calls) const {
    // Chromosome ids are shipped as runs: region sets read from BED files are sorted by chromosome, so the device
    // rebuilds the per-query chromosome array from a handful of (offset, id) pairs per file.
    std::vector<uint64_t> file_offsets(calls.size() + 1, 0), run_offsets;
    std::vector<uint32_t> run_chr, start, end;
    for (size_t f = 0; f < calls.size(); ++f) {
        const std::string* last = nullptr;  // a run never spans two files
        for (const auto& r : *calls[f]) {
            if (!last || r.chr != *last) {
                run_offsets.push_back(start.size());
                run_chr.push_back(cmap_.get(r.chr));
                last = &r.chr;
            }
            start.push_back(r.start);
            end.push_back(r.end);
        }
        file_offsets[f + 1] = start.size();
    }
    run_offsets.push_back(start.size());  // n_runs + 1 entries, the first one is 0
    std::vector<uint64_t> tok_offsets(calls.size() + 1);
    PinnedResult res;
    check(gtgpu_tokenize_files_runs(index_, calls.size(), file_offsets.data(), run_chr.size(), run_offsets.data(), run_chr.data(),
                                    start.data(), end.data(), unk_id_, tok_offsets.data(), &res.buf),
          "gtgpu_tokenize_files_runs");
    std::vector<std::vector<uint32_t>> out(calls.size());
    for (size_t f = 0; f < calls.size(); ++f) out[f].assign(res.data() + tok_offsets[f], res.data() + tok_offsets[f + 1]);
    return out;
}

std::vector<uint32_t> Tokenizer::encode(const std::vector<Region>& regions) const { return encode_batch({&regions})[0]; }

// A `.gz` input made of many gzip members (bgzip / BGZF, or concatenated gzips) is inflated on the device, one warp per
// member, and parsed there; a single-member stream is sequential, so it stays with zlib on the host (get_dynamic_reader's
// MultiGzDecoder semantics either way: the text is the concatenation of the members).
static bool ends_with_gz(const std::string& path) { return path.size() >= 3 && path.compare(path.size() - 3, 3, ".gz") == 0; }

// the file's bytes as stored (no decompression)
static void read_raw_bytes(const std::string& path, std::string& raw) {
    std::ifstream f(path, std::ios::binary | std::ios::ate);
    if (!f) throw Error("Failed to open file: \"" + path + "\"");
    const std::streamsize size = f.tellg();
    f.seekg(0);
    raw.resize((size_t)std::max<std::streamsize>(size, 0));
    if (size > 0 && !f.read(&raw[0], size)) throw Error("Failed to read file: \"" + path + "\"");
}

static bool gz_members_for_device(const std::string& path, std::string& raw, std::vector<uint64_t>& members) {
    if (!ends_with_gz(path)) return false;
    read_raw_bytes(path, raw);
    uint64_t n = 0;
    gtgpu_gzip_members((const uint8_t*)raw.data(), raw.size(), 0, nullptr, &n);  // count only
    if (n < 16) return false;
    members.resize(n + 1);
    check(gtgpu_gzip_members((const uint8_t*)raw.data(), raw.size(), members.size(), members.data(), &n), "gtgpu_gzip_members");
    return true;
}

namespace {
// The bytes of n BED files for one device call.  When every path ends in ".gz" they stay gzip: every file's bytes back to back
// with their member offsets, for the device inflater.  Otherwise the texts go back to back (".gz" inflated by zlib).
struct BedFilesBytes {
    bool gz = false;
    std::string raw;                                   // gz: the files' gzip bytes
    std::vector<uint64_t> members{0}, file_members{0};  // gz: member offsets in raw; file f = members [file_members[f], [f + 1])
    std::unique_ptr<char[]> text;                      // otherwise: the texts, file f = text[file_offsets[f], file_offsets[f + 1])
    std::vector<uint64_t> file_offsets{0};
};

BedFilesBytes gather_bed_files(const std::vector<std::string>& paths) {
    BedFilesBytes b;
    if (!paths.empty() && std::all_of(paths.begin(), paths.end(), ends_with_gz)) {
        // one-member .bed.gz files are the common case: every member of every file is inflated on the device in parallel
        b.gz = true;
        std::string raw;
        std::vector<uint64_t> m;
        for (const auto& p : paths) {
            read_raw_bytes(p, raw);
            uint64_t n = 0;
            gtgpu_gzip_members((const uint8_t*)raw.data(), raw.size(), 0, nullptr, &n);  // count only
            m.assign(n + 1, 0);
            check(gtgpu_gzip_members((const uint8_t*)raw.data(), raw.size(), m.size(), m.data(), &n), "gtgpu_gzip_members");
            for (uint64_t k = 1; k <= n; ++k) b.members.push_back(b.raw.size() + m[k]);
            b.file_members.push_back(b.members.size() - 1);
            b.raw += raw;
        }
        return b;
    }
    // the texts back to back; the library stages them to the device through its own pinned blocks
    std::vector<std::string> inflated(paths.size());
    for (size_t f = 0; f < paths.size(); ++f) {
        uint64_t size = 0;
        if (ends_with_gz(paths[f])) {
            inflated[f] = read_file_bytes(paths[f]);
            size = inflated[f].size();
        } else {
            std::ifstream in(paths[f], std::ios::binary | std::ios::ate);
            if (!in) throw Error("Failed to open file: \"" + paths[f] + "\"");
            size = (uint64_t)std::max<std::streamsize>(in.tellg(), 0);
        }
        b.file_offsets.push_back(b.file_offsets.back() + size);
    }
    b.text.reset(new char[std::max<uint64_t>(b.file_offsets.back(), 1)]);
    for (size_t f = 0; f < paths.size(); ++f) {
        char* dst = b.text.get() + b.file_offsets[f];
        const uint64_t size = b.file_offsets[f + 1] - b.file_offsets[f];
        if (ends_with_gz(paths[f])) {
            memcpy(dst, inflated[f].data(), size);
            std::string().swap(inflated[f]);
        } else if (size) {
            std::ifstream in(paths[f], std::ios::binary);
            if (!in || !in.read(dst, (std::streamsize)size)) throw Error("Failed to read file: \"" + paths[f] + "\"");
        }
    }
    return b;
}

// The library's last error as "fn: message", "file k" in it replaced by the file's path
[[noreturn]] void throw_naming_path(const char* fn, const std::vector<std::string>& paths) {
    std::string msg = gtgpu_last_error();
    const size_t k = msg.find(": file ");
    size_t b = k == std::string::npos ? k : k + 7;
    if (b != std::string::npos) {
        const size_t a = b;
        while (b < msg.size() && isdigit((unsigned char)msg[b])) ++b;
        if (b > a && std::stoull(msg.substr(a, b - a)) < paths.size())
            msg = msg.substr(0, k) + ": \"" + paths[std::stoull(msg.substr(a, b - a))] + "\"" + msg.substr(b);
    }
    throw Error(std::string(fn) + ": " + msg);
}
}  // namespace

std::vector<uint32_t> Tokenizer::encode_bed_file(const std::string& path) const {
    NameBlob nb(cmap_);
    PinnedResult ids;
    std::string raw;
    std::vector<uint64_t> members;
    if (gz_members_for_device(path, raw, members)) {
        check(gtgpu_tokenize_bed_gz(index_, members.size() - 1, (const uint8_t*)raw.data(), members.data(), (uint32_t)cmap_.size(),
                                    nb.blob.data(), nb.offsets.data(), unk_id_, &ids.buf),
              "gtgpu_tokenize_bed_gz");
        return std::vector<uint32_t>(ids.data(), ids.data() + ids.len());
    }
    const std::string text = read_file_bytes(path);
    check(gtgpu_tokenize_bed(index_, text.data(), text.size(), (uint32_t)cmap_.size(), nb.blob.data(), nb.offsets.data(), unk_id_,
                             &ids.buf),
          "gtgpu_tokenize_bed");
    return std::vector<uint32_t>(ids.data(), ids.data() + ids.len());
}

std::vector<std::vector<uint32_t>> Tokenizer::encode_bed_files(const std::vector<std::string>& paths) const {
    const BedFilesBytes b = gather_bed_files(paths);
    NameBlob nb(cmap_);
    std::vector<uint64_t> tok_offsets(paths.size() + 1);
    PinnedResult ids;
    int32_t status;
    const char* fn;
    if (b.gz) {
        fn = "gtgpu_tokenize_bed_files_gz";
        status = gtgpu_tokenize_bed_files_gz(index_, paths.size(), b.file_members.data(), b.members.size() - 1, (const uint8_t*)b.raw.data(),
                                             b.members.data(), (uint32_t)cmap_.size(), nb.blob.data(), nb.offsets.data(), unk_id_,
                                             tok_offsets.data(), &ids.buf);
    } else {
        fn = "gtgpu_tokenize_bed_files";
        status = gtgpu_tokenize_bed_files(index_, paths.size(), b.text.get(), b.file_offsets.data(), (uint32_t)cmap_.size(),
                                          nb.blob.data(), nb.offsets.data(), unk_id_, tok_offsets.data(), &ids.buf);
    }
    if (status != GTGPU_OK) throw_naming_path(fn, paths);
    std::vector<std::vector<uint32_t>> out(paths.size());
    for (size_t f = 0; f < paths.size(); ++f) out[f].assign(ids.data() + tok_offsets[f], ids.data() + tok_offsets[f + 1]);
    return out;
}

std::vector<std::string> Tokenizer::tokenize(const std::vector<Region>& regions) const {
    std::vector<std::string> out;
    for (uint32_t id : encode(regions)) out.push_back(id_to_first_token_.at(id));
    return out;
}

std::vector<std::string> Tokenizer::decode(const std::vector<uint32_t>& ids) const {
    std::vector<std::string> out;
    for (uint32_t id : ids) {
        auto it = universe_.id_to_region.find(id);
        out.push_back(it == universe_.id_to_region.end() ? special_.unk : it->second);  // tokenizer.rs:173-181
    }
    return out;
}

int64_t Tokenizer::convert_token_to_id(const std::string& tok) const {
    auto it = universe_.region_to_id.find(tok);
    return it == universe_.region_to_id.end() ? -1 : (int64_t)it->second;
}
const std::string* Tokenizer::convert_id_to_token(uint32_t id) const {
    auto it = universe_.id_to_region.find(id);
    return it == universe_.id_to_region.end() ? nullptr : &it->second;
}

std::vector<std::pair<std::string, std::vector<uint32_t>>> Tokenizer::tokenize_fragment_file(const std::string& path) const {
    // parse_fragment_line (fragments.rs:12-56): split_whitespace, >= 5 fields, chr start end barcode
    std::vector<std::string> barcodes;
    std::unordered_map<std::string, uint32_t> bc_ids;
    FlatQueries q;
    std::vector<uint32_t> bc;
    auto lines = read_lines(path);
    for (size_t i = 0; i < lines.size(); ++i) {
        if (has_prefix(lines[i], "#")) continue;
        auto parts = split_whitespace(lines[i]);
        if (parts.size() < 5) throw Error("Invalid fragment file detected at line: " + std::to_string(i));
        uint32_t s, e;
        if (!parse_u32(parts[1], s)) throw Error("Failed to parse start position at line " + std::to_string(i));
        if (!parse_u32(parts[2], e)) throw Error("Failed to parse end position at line " + std::to_string(i));
        auto it = bc_ids.find(parts[3]);
        if (it == bc_ids.end()) {
            it = bc_ids.emplace(parts[3], (uint32_t)barcodes.size()).first;
            barcodes.push_back(parts[3]);
        }
        q.chr.push_back(cmap_.get(parts[0]));
        q.start.push_back(s);
        q.end.push_back(e);
        bc.push_back(it->second);
    }
    std::vector<uint64_t> offsets(barcodes.size() + 1);
    PinnedResult res;
    check(gtgpu_tokenize_fragments(index_, q.chr.size(), q.chr.data(), q.start.data(), q.end.data(), bc.data(),
                                   (uint32_t)barcodes.size(), unk_id_, offsets.data(), &res.buf),
          "gtgpu_tokenize_fragments");
    std::vector<std::pair<std::string, std::vector<uint32_t>>> out;
    for (size_t b = 0; b < barcodes.size(); ++b)
        out.emplace_back(barcodes[b], std::vector<uint32_t>(res.data() + offsets[b], res.data() + offsets[b + 1]));
    return out;
}

std::vector<std::pair<std::string, std::vector<uint32_t>>> Tokenizer::tokenize_fragment_file_device(const std::string& path) const {
    NameBlob nb(cmap_);
    uint32_t n_barcodes = 0;
    PinnedResult names, name_offsets, offs, ids;
    {
        std::string raw;
        std::vector<uint64_t> members;
        if (gz_members_for_device(path, raw, members)) {  // bgzip'ed fragment file: inflated and parsed on the device
            check(gtgpu_tokenize_fragments_file_gz(index_, members.size() - 1, (const uint8_t*)raw.data(), members.data(),
                                                   (uint32_t)cmap_.size(), nb.blob.data(), nb.offsets.data(), unk_id_, &n_barcodes,
                                                   &names.buf, &name_offsets.buf, &offs.buf, &ids.buf),
                  "gtgpu_tokenize_fragments_file_gz");
        } else {
            const std::string text = read_file_bytes(path);
            check(gtgpu_tokenize_fragments_file(index_, text.data(), text.size(), (uint32_t)cmap_.size(), nb.blob.data(),
                                                nb.offsets.data(), unk_id_, &n_barcodes, &names.buf, &name_offsets.buf, &offs.buf,
                                                &ids.buf),
                  "gtgpu_tokenize_fragments_file");
        }
    }
    const char* blob = (const char*)gtgpu_buf_data(names.buf);
    const uint64_t* noff = (const uint64_t*)gtgpu_buf_data(name_offsets.buf);
    const uint64_t* off = (const uint64_t*)gtgpu_buf_data(offs.buf);
    std::vector<std::pair<std::string, std::vector<uint32_t>>> out;
    out.reserve(n_barcodes);
    for (uint32_t b = 0; b < n_barcodes; ++b)
        out.emplace_back(std::string(blob + noff[b], noff[b + 1] - noff[b]),
                         std::vector<uint32_t>(ids.data() + off[b], ids.data() + off[b + 1]));
    return out;
}

std::vector<std::pair<std::string, std::map<uint32_t, uint32_t>>> Tokenizer::count_fragments_by_barcode(const std::string& path) const {
    std::vector<std::pair<std::string, std::map<uint32_t, uint32_t>>> out;
    for (auto& kv : tokenize_fragment_file(path)) {
        std::map<uint32_t, uint32_t> counts;
        for (uint32_t id : kv.second) counts[id]++;
        out.emplace_back(kv.first, std::move(counts));
    }
    return out;
}

// ---- IndexedRegionSet ---------------------------------------------------------------------------------------------------------
IndexedRegionSet::IndexedRegionSet(std::shared_ptr<Device> dev, RegionSet regions, OverlapperType kind)
    : source_(std::move(regions)), index_(new MultiChromOverlapper(std::move(dev), source_, kind)) {}

std::vector<std::vector<uint32_t>> IndexedRegionSet::find_overlaps(const RegionSet& query, int32_t min_overlap) const {
    // The reference maps hit coordinates back through a (chr, start, end) -> [source indices] table, so a hit on
    // one of several identical regions reports all of them; identical regions overlap the same queries, so the
    // union of the per-hit source indices is already that set.  Sorted, de-duplicated (:256-258).
    auto hits = index_->find_overlaps_indices(query, min_overlap);
    for (auto& v : hits) {
        std::sort(v.begin(), v.end());
        v.erase(std::unique(v.begin(), v.end()), v.end());
    }
    return hits;
}
RegionSet IndexedRegionSet::subset_by_overlaps(const RegionSet& query, int32_t min_overlap) const {
    std::set<uint32_t> keep;  // BTreeSet<usize>: ascending source index
    for (const auto& v : find_overlaps(query, min_overlap)) keep.insert(v.begin(), v.end());
    std::vector<Region> out;
    for (uint32_t i : keep) out.push_back(source_.regions[i]);
    return RegionSet::from_regions(std::move(out));
}
RegionSet IndexedRegionSet::intersect_all(const RegionSet& query) const { return subset_by_overlaps(query, -1); }
std::vector<uint64_t> IndexedRegionSet::count_overlaps(const RegionSet& query, int32_t min_overlap) const {
    return index_->count_overlaps(query, min_overlap);
}
std::vector<bool> IndexedRegionSet::any_overlaps(const RegionSet& query, int32_t min_overlap) const {
    return index_->any_overlaps(query, min_overlap);
}

// ---- gtars_scoring ----------------------------------------------------------------------------------------------------------------
ConsensusSet::ConsensusSet(std::shared_ptr<Device> dev, const std::string& path) : dev_(std::move(dev)) {
    build(RegionSet::from_file(path));
}
ConsensusSet::ConsensusSet(std::shared_ptr<Device> dev, const RegionSet& regions) : dev_(std::move(dev)) { build(regions); }
ConsensusSet::~ConsensusSet() { gtgpu_index_free(index_); }

void ConsensusSet::build(const RegionSet& rs) {
    len_ = rs.regions.size();
    std::unordered_map<std::string, uint32_t> ids;  // generate_region_to_id_map (gtars-core utils.rs:202-214)
    std::vector<uint32_t> chr, start, end, val;
    for (const Region& r : rs.regions) {
        std::string key = r.chr + '\x1f' + std::to_string(r.start) + '\x1f' + std::to_string(r.end) + '\x1f' + r.rest;
        auto it = ids.find(key);
        if (it == ids.end()) it = ids.emplace(std::move(key), (uint32_t)ids.size()).first;
        chr.push_back(cmap_.add(r.chr));
        start.push_back(r.start);
        end.push_back(r.end);
        val.push_back(it->second);
    }
    Grouped g = group_by_chrom(chr, start, end, val, cmap_.size());
    check(gtgpu_index_build(dev_->ctx(), GTGPU_KIND_BITS, (uint32_t)cmap_.size(), g.offsets.data(), g.start.data(), g.end.data(),
                            g.val.data(), &index_),
          "gtgpu_index_build");
}

namespace {
struct ParsedFragments {
    FlatQueries q;
    std::vector<std::string> barcode;
};
// Fragment::from_str (gtars-core/src/models/fragments.rs:16-44): split_whitespace; fields 1, 2 and 4 parse as u32.
void parse_fragment_file(const std::string& path, const ChromMap& cmap, ParsedFragments& out) {
    auto lines = read_lines(path);
    for (size_t i = 0; i < lines.size(); ++i) {
        if (has_prefix(lines[i], "#")) continue;
        auto parts = split_whitespace(lines[i]);
        uint32_t s, e, support;
        if (parts.size() < 5 || !parse_u32(parts[1], s) || !parse_u32(parts[2], e) || !parse_u32(parts[4], support))
            throw Error("Failed to parse fragment at line " + std::to_string(i) + " of " + path);
        out.q.chr.push_back(cmap.get(parts[0]));
        out.q.start.push_back(s);
        out.q.end.push_back(e);
        out.barcode.push_back(parts[3]);
    }
}
}  // namespace

CountMatrix region_scoring_from_fragments(const std::vector<std::string>& fragment_files, const ConsensusSet& consensus,
                                          ScoringMode mode) {
    ParsedFragments all;
    std::vector<uint64_t> file_offsets{0};
    for (const auto& path : fragment_files) {
        parse_fragment_file(path, consensus.chroms(), all);
        file_offsets.push_back(all.q.chr.size());
    }
    CountMatrix m;
    m.rows = fragment_files.size();
    m.cols = consensus.len();
    m.data.assign(m.rows * m.cols, 0);
    check(gtgpu_score_matrix(consensus.index(), m.rows, file_offsets.data(), all.q.chr.size(), all.q.chr.data(), all.q.start.data(),
                             all.q.end.data(), (int32_t)mode, m.cols, m.data.data()),
          "gtgpu_score_matrix");
    return m;
}

std::vector<std::pair<std::string, std::map<uint32_t, uint32_t>>> barcode_scoring_from_fragments(const std::string& fragment_file,
                                                                                                 const ConsensusSet& consensus) {
    ParsedFragments pf;
    parse_fragment_file(fragment_file, consensus.chroms(), pf);
    std::vector<std::string> barcodes;
    std::unordered_map<std::string, uint32_t> bc_ids;
    std::vector<uint32_t> bc;
    for (const auto& b : pf.barcode) {
        auto it = bc_ids.find(b);
        if (it == bc_ids.end()) {
            it = bc_ids.emplace(b, (uint32_t)barcodes.size()).first;
            barcodes.push_back(b);
        }
        bc.push_back(it->second);
    }
    std::vector<uint64_t> offsets(barcodes.size() + 1);
    PinnedResult peaks, counts;
    check(gtgpu_score_barcodes(consensus.index(), bc.size(), pf.q.chr.data(), pf.q.start.data(), pf.q.end.data(), bc.data(),
                               (uint32_t)barcodes.size(), offsets.data(), &peaks.buf, &counts.buf),
          "gtgpu_score_barcodes");
    // Key set of the reference: `barcode_counts.entry(barcode).or_default()` runs whenever ConsensusSet::find_overlaps returns
    // Some(..), i.e. whenever the fragment's chromosome has a tree in the consensus — also when nothing overlaps
    // (gtars-scoring/src/files.rs:106-129, fragment_scoring.rs:146-153).  So a barcode seen on a consensus chromosome gets an
    // entry even if its inner map stays empty; only barcodes seen solely on unknown chromosomes are absent.
    std::vector<uint8_t> seen_on_known(barcodes.size(), 0);
    for (size_t i = 0; i < bc.size(); ++i)
        if (pf.q.chr[i] != GTGPU_UNKNOWN_CHROM) seen_on_known[bc[i]] = 1;
    std::vector<std::pair<std::string, std::map<uint32_t, uint32_t>>> out;
    for (size_t b = 0; b < barcodes.size(); ++b) {
        if (!seen_on_known[b]) continue;
        std::map<uint32_t, uint32_t> m;
        for (uint64_t k = offsets[b]; k < offsets[b + 1]; ++k) m[peaks.data()[k]] = counts.data()[k];
        out.emplace_back(barcodes[b], std::move(m));
    }
    return out;
}

// Device parse of one fragment file: a bgzip'ed file goes to the device inflater (gz_members_for_device), any other file is
// read by read_file_bytes (a single-member gzip is inflated by zlib on the host).  Device errors are prefixed with the path.
namespace {
struct FragmentBytes {
    std::string raw, text;
    std::vector<uint64_t> members;
    bool gz = false;
    explicit FragmentBytes(const std::string& path) {
        gz = gz_members_for_device(path, raw, members);
        if (!gz) text = read_file_bytes(path);
    }
};
void check_file(int32_t status, const std::string& path) {
    if (status != GTGPU_OK) throw Error(path + ": " + gtgpu_last_error());
}
}  // namespace

CountMatrix region_scoring_from_fragments_device(const std::vector<std::string>& fragment_files, const ConsensusSet& consensus,
                                                 ScoringMode mode) {
    NameBlob nb(consensus.chroms());
    CountMatrix m;
    m.rows = fragment_files.size();
    m.cols = consensus.len();
    m.data.assign(m.rows * m.cols, 0);
    for (size_t f = 0; f < fragment_files.size(); ++f) {
        const std::string& path = fragment_files[f];
        FragmentBytes fb(path);
        uint32_t* row = m.data.data() + f * m.cols;
        if (fb.gz)
            check_file(gtgpu_score_matrix_gz(consensus.index(), fb.members.size() - 1, (const uint8_t*)fb.raw.data(), fb.members.data(),
                                             (uint32_t)consensus.chroms().size(), nb.blob.data(), nb.offsets.data(), (int32_t)mode, m.cols, row),
                       path);
        else
            check_file(gtgpu_score_matrix_text(consensus.index(), fb.text.data(), fb.text.size(), (uint32_t)consensus.chroms().size(),
                                               nb.blob.data(), nb.offsets.data(), (int32_t)mode, m.cols, row),
                       path);
    }
    return m;
}

std::vector<std::pair<std::string, std::map<uint32_t, uint32_t>>> barcode_scoring_from_fragments_device(const std::string& fragment_file,
                                                                                                        const ConsensusSet& consensus) {
    NameBlob nb(consensus.chroms());
    FragmentBytes fb(fragment_file);
    uint32_t n_barcodes = 0;
    PinnedResult names, name_offsets, offsets, peaks, counts;
    if (fb.gz)
        check_file(gtgpu_score_barcodes_gz(consensus.index(), fb.members.size() - 1, (const uint8_t*)fb.raw.data(), fb.members.data(),
                                           (uint32_t)consensus.chroms().size(), nb.blob.data(), nb.offsets.data(), &n_barcodes, &names.buf,
                                           &name_offsets.buf, &offsets.buf, &peaks.buf, &counts.buf),
                   fragment_file);
    else
        check_file(gtgpu_score_barcodes_text(consensus.index(), fb.text.data(), fb.text.size(), (uint32_t)consensus.chroms().size(),
                                             nb.blob.data(), nb.offsets.data(), &n_barcodes, &names.buf, &name_offsets.buf, &offsets.buf,
                                             &peaks.buf, &counts.buf),
                   fragment_file);
    const char* blob = (const char*)gtgpu_buf_data(names.buf);
    const uint64_t* noff = (const uint64_t*)gtgpu_buf_data(name_offsets.buf);
    const uint64_t* off = (const uint64_t*)gtgpu_buf_data(offsets.buf);
    std::vector<std::pair<std::string, std::map<uint32_t, uint32_t>>> out;
    out.reserve(n_barcodes);
    for (uint32_t b = 0; b < n_barcodes; ++b) {
        std::map<uint32_t, uint32_t> m;
        for (uint64_t k = off[b]; k < off[b + 1]; ++k) m[peaks.data()[k]] = counts.data()[k];
        out.emplace_back(std::string(blob + noff[b], noff[b + 1] - noff[b]), std::move(m));
    }
    return out;
}

// ---- Igd / LOLA -----------------------------------------------------------------------------------------------------------------
Igd::Igd(std::shared_ptr<Device> dev, const std::vector<const RegionSet*>& sets) : dev_(std::move(dev)), n_files_(sets.size()) {
    std::vector<uint64_t> file_offsets(sets.size() + 1, 0);
    FlatQueries r;
    for (size_t f = 0; f < sets.size(); ++f) {
        for (const auto& reg : sets[f]->regions) {
            r.chr.push_back(cmap_.add(reg.chr));
            r.start.push_back(reg.start);
            r.end.push_back(reg.end);
        }
        file_offsets[f + 1] = r.chr.size();
    }
    check(gtgpu_igd_build(dev_->ctx(), sets.size(), file_offsets.data(), (uint32_t)cmap_.size(), r.chr.data(), r.start.data(),
                          r.end.data(), &igd_),
          "gtgpu_igd_build");
}
Igd::~Igd() {
    if (igd_) gtgpu_igd_free(igd_);
}

std::vector<uint64_t> Igd::count_region_hits_batch(const std::vector<const RegionSet*>& sets, int32_t min_overlap, bool pairwise) const {
    std::vector<uint64_t> set_offsets(sets.size() + 1, 0);
    FlatQueries q;
    for (size_t s = 0; s < sets.size(); ++s) {
        for (const auto& reg : sets[s]->regions) {
            q.chr.push_back(cmap_.get(reg.chr));
            q.start.push_back(reg.start);
            q.end.push_back(reg.end);
        }
        set_offsets[s + 1] = q.chr.size();
    }
    std::vector<uint64_t> out(sets.size() * n_files_);
    auto fn = pairwise ? gtgpu_igd_count_set_overlaps : gtgpu_igd_count_region_hits;
    check(fn(igd_, sets.size(), set_offsets.data(), q.chr.data(), q.start.data(), q.end.data(), min_overlap, out.data()),
          pairwise ? "gtgpu_igd_count_set_overlaps" : "gtgpu_igd_count_region_hits");
    return out;
}

// ---- .igd files ---------------------------------------------------------------------------------------------------------------
namespace {
struct IgdRec {
    int32_t file_idx, start, end, value;
};
void put_i32(std::string& b, int32_t v) {
    const unsigned char c[4] = {(unsigned char)v, (unsigned char)(v >> 8), (unsigned char)(v >> 16), (unsigned char)(v >> 24)};
    b.append((const char*)c, 4);
}
std::string with_extension(const std::string& path, const std::string& ext) {  // Path::with_extension
    size_t slash = path.find_last_of('/');
    size_t dot = path.find_last_of('.');
    std::string stem = (dot == std::string::npos || (slash != std::string::npos && dot < slash) || dot == slash + 1) ? path : path.substr(0, dot);
    return stem + "." + ext;
}
// The companion .tsv (igd.rs:470-484): per file its index, name, region count and the average width to two decimals
std::string igd_tsv(const std::vector<std::string>& names, const uint64_t* regions, const uint64_t* width_sums) {
    std::string tsv = "Index\tFile\tNumber of Regions\tAvg size\n";
    for (size_t f = 0; f < names.size(); ++f) {
        char buf[64];
        snprintf(buf, sizeof buf, "%.2f", regions[f] ? (double)width_sums[f] / (double)regions[f] : 0.0);
        tsv += std::to_string(f) + "\t" + names[f] + "\t" + std::to_string(regions[f]) + "\t" + buf + "\n";
    }
    return tsv;
}
void write_igd_files(const std::string& path, const char* igd, size_t igd_bytes, const std::string& tsv) {
    std::ofstream f(path, std::ios::binary);
    if (!f) throw Error("cannot write " + path);
    f.write(igd, (std::streamsize)igd_bytes);
    if (!f) throw Error("cannot write " + path);
    std::ofstream t(with_extension(path, "tsv"), std::ios::binary);
    if (!t) throw Error("cannot write " + with_extension(path, "tsv"));
    t << tsv;
}
}  // namespace

void Igd::save_named_region_sets(const std::vector<std::pair<std::string, const RegionSet*>>& sets, const std::string& path, int32_t nbp) {
    // from_named_region_sets (igd.rs:285-317) + add (:109-153) + finalize (:157-167) + save (:418-486)
    std::vector<std::string> names;                       // contigs in creation order
    std::unordered_map<std::string, size_t> chrom_index;
    std::vector<std::vector<std::vector<IgdRec>>> contigs;  // [contig][tile][record]
    std::vector<std::string> file_names;
    std::vector<uint64_t> regions(sets.size(), 0), width_sums(sets.size(), 0);
    for (size_t f = 0; f < sets.size(); ++f) {
        file_names.push_back(sets[f].first);
        for (const Region& r : sets[f].second->regions) {
            if (!(r.start < r.end)) continue;
            const int32_t start = (int32_t)r.start, end = (int32_t)r.end;  // `as i32` casts (:295-296)
            regions[f] += 1;
            width_sums[f] += (uint64_t)(int64_t)(int32_t)(r.end - r.start);
            if (start < 0 || end < 0 || start >= end) continue;  // Igd::add skips these silently
            auto it = chrom_index.find(r.chr);
            if (it == chrom_index.end()) {
                it = chrom_index.emplace(r.chr, contigs.size()).first;
                names.push_back(r.chr);
                contigs.emplace_back();
            }
            auto& tiles = contigs[it->second];
            const int32_t n1 = start / nbp, n2 = (end - 1) / nbp;
            if (tiles.size() < (size_t)(n2 + 1)) tiles.resize((size_t)(n2 + 1));
            for (int32_t i = n1; i <= n2; ++i) tiles[i].push_back(IgdRec{(int32_t)f, start, end, 0});
        }
    }
    std::string b;
    put_i32(b, nbp);
    put_i32(b, 1);  // gType 1: 16-byte records
    put_i32(b, (int32_t)contigs.size());
    for (auto& tiles : contigs) put_i32(b, (int32_t)tiles.size());
    for (auto& tiles : contigs)
        for (auto& t : tiles) {
            std::stable_sort(t.begin(), t.end(), [](const IgdRec& a, const IgdRec& c) { return a.start < c.start; });
            put_i32(b, (int32_t)t.size());
        }
    for (const auto& nm : names) {
        std::string padded = nm;
        padded.resize(40, '\0');
        b += padded;
    }
    for (auto& tiles : contigs)
        for (auto& t : tiles)
            for (const IgdRec& r : t) { put_i32(b, r.file_idx); put_i32(b, r.start); put_i32(b, r.end); put_i32(b, r.value); }
    write_igd_files(path, b.data(), b.size(), igd_tsv(file_names, regions.data(), width_sums.data()));
}

void Igd::save(const std::string& path, const std::vector<std::string>& names) const {
    if (!igd_) throw Error("save needs a database Igd (not from_single_region_set)");
    if (names.size() != n_files_)
        throw Error("save: " + std::to_string(names.size()) + " names for " + std::to_string(n_files_) + " files");
    NameBlob nb(cmap_);
    PinnedResult bytes;
    std::vector<uint64_t> regions(n_files_), width_sums(n_files_);
    check(gtgpu_igd_serialize(igd_, (uint32_t)cmap_.size(), nb.blob.data(), nb.offsets.data(), &bytes.buf, regions.data(),
                              width_sums.data()),
          "gtgpu_igd_serialize");
    write_igd_files(path, (const char*)gtgpu_buf_data(bytes.buf), gtgpu_buf_len(bytes.buf), igd_tsv(names, regions.data(), width_sums.data()));
}

std::unique_ptr<Igd> Igd::from_igd_file(std::shared_ptr<Device> dev, const std::string& path) {
    std::ifstream f(path, std::ios::binary);
    if (!f) throw Error("Failed to open file: " + path);
    std::stringstream ss;
    ss << f.rdbuf();
    const std::string d = ss.str();
    size_t pos = 0;
    auto rd = [&]() -> int32_t {
        if (pos + 4 > d.size()) throw Error("truncated .igd file: " + path);
        const unsigned char* c = (const unsigned char*)d.data() + pos;
        pos += 4;
        return (int32_t)((uint32_t)c[0] | ((uint32_t)c[1] << 8) | ((uint32_t)c[2] << 16) | ((uint32_t)c[3] << 24));
    };
    const int32_t nbp = rd(), g_type = rd(), n_ctg = rd();
    if (nbp <= 0 || n_ctg < 0) throw Error("not an .igd file: " + path);
    std::vector<int32_t> n_tiles((size_t)n_ctg);
    for (auto& x : n_tiles) x = rd();
    std::vector<std::vector<int32_t>> n_cnt((size_t)n_ctg);
    for (int32_t i = 0; i < n_ctg; ++i) {
        if (n_tiles[i] < 0) throw Error("not an .igd file: " + path);
        n_cnt[i].resize((size_t)n_tiles[i]);
        for (auto& x : n_cnt[i]) x = rd();
    }
    std::unique_ptr<Igd> g(new Igd());
    g->dev_ = dev;
    for (int32_t i = 0; i < n_ctg; ++i) {
        if (pos + 40 > d.size()) throw Error("truncated .igd file: " + path);
        std::string nm = d.substr(pos, 40);
        pos += 40;
        while (!nm.empty() && nm.back() == '\0') nm.pop_back();
        while (!nm.empty() && nm.front() == '\0') nm.erase(nm.begin());
        g->cmap_.add(nm);
    }
    // records: an interval sits in every tile it spans; its copy in the tile of its start is the one kept
    std::vector<std::vector<std::array<uint32_t, 3>>> per_file;
    for (int32_t i = 0; i < n_ctg; ++i)
        for (int32_t j = 0; j < n_tiles[i]; ++j)
            for (int32_t k = 0; k < n_cnt[i][j]; ++k) {
                const int32_t idx = rd(), start = rd(), end = rd();
                if (g_type != 0) rd();
                if (idx < 0 || start < 0 || start / nbp != j) continue;
                if ((size_t)idx >= per_file.size()) per_file.resize((size_t)idx + 1);
                per_file[idx].push_back({(uint32_t)i, (uint32_t)start, (uint32_t)end});
            }
    size_t n_files = per_file.size();
    {   // companion .tsv (igd.rs:870-893): one line per file after the header
        std::ifstream t(with_extension(path, "tsv"));
        if (t) {
            std::string line;
            size_t lines = 0, rows = 0;
            while (std::getline(t, line))
                if (lines++ > 0 && std::count(line.begin(), line.end(), '\t') >= 3) ++rows;
            n_files = std::max(n_files, rows);
        }
    }
    per_file.resize(n_files);
    g->n_files_ = n_files;
    std::vector<uint64_t> file_offsets(n_files + 1, 0);
    FlatQueries r;
    for (size_t fidx = 0; fidx < n_files; ++fidx) {
        for (const auto& rec : per_file[fidx]) {
            r.chr.push_back(rec[0]);
            r.start.push_back(rec[1]);
            r.end.push_back(rec[2]);
        }
        file_offsets[fidx + 1] = r.chr.size();
    }
    check(gtgpu_igd_build(dev->ctx(), n_files, file_offsets.data(), (uint32_t)g->cmap_.size(), r.chr.data(), r.start.data(), r.end.data(),
                          &g->igd_),
          "gtgpu_igd_build");
    return g;
}

std::unique_ptr<Igd> Igd::from_bed_files(std::shared_ptr<Device> dev, const std::vector<std::string>& paths) {
    std::unique_ptr<Igd> g(new Igd());
    g->dev_ = dev;
    g->n_files_ = paths.size();
    uint32_t n_chroms = 0;
    PinnedResult names, name_offsets;
    int32_t status;
    const char* fn;
    const BedFilesBytes b = gather_bed_files(paths);
    if (b.gz) {
        fn = "gtgpu_igd_build_bed_gz";
        status = gtgpu_igd_build_bed_gz(dev->ctx(), paths.size(), b.file_members.data(), b.members.size() - 1, (const uint8_t*)b.raw.data(),
                                        b.members.data(), &n_chroms, &names.buf, &name_offsets.buf, &g->igd_);
    } else {
        fn = "gtgpu_igd_build_bed";
        status = gtgpu_igd_build_bed(dev->ctx(), paths.size(), b.text.get(), b.file_offsets.data(), &n_chroms, &names.buf,
                                     &name_offsets.buf, &g->igd_);
    }
    if (status != GTGPU_OK) throw_naming_path(fn, paths);
    const char* blob = (const char*)gtgpu_buf_data(names.buf);
    const uint64_t* noff = (const uint64_t*)gtgpu_buf_data(name_offsets.buf);
    for (uint32_t c = 0; c < n_chroms; ++c) g->cmap_.add(std::string(blob + noff[c], noff[c + 1] - noff[c]));
    return g;
}

Igd::BedCounts Igd::count_bed_files(const std::vector<std::string>& paths, int32_t min_overlap, bool pairwise) const {
    if (!igd_) throw Error("count_bed_files needs a database Igd (not from_single_region_set)");
    BedCounts r;
    r.matrix.assign(paths.size() * n_files_, 0);
    r.set_regions.assign(paths.size(), 0);
    const BedFilesBytes b = gather_bed_files(paths);
    NameBlob nb(cmap_);
    int32_t status;
    const char* fn;
    if (b.gz) {
        fn = "gtgpu_igd_count_bed_gz";
        status = gtgpu_igd_count_bed_gz(igd_, pairwise ? 0 : 1, paths.size(), b.file_members.data(), b.members.size() - 1,
                                        (const uint8_t*)b.raw.data(), b.members.data(), (uint32_t)cmap_.size(), nb.blob.data(),
                                        nb.offsets.data(), min_overlap, r.matrix.data(), r.set_regions.data());
    } else {
        fn = "gtgpu_igd_count_bed";
        status = gtgpu_igd_count_bed(igd_, pairwise ? 0 : 1, paths.size(), b.text.get(), b.file_offsets.data(), (uint32_t)cmap_.size(),
                                     nb.blob.data(), nb.offsets.data(), min_overlap, r.matrix.data(), r.set_regions.data());
    }
    if (status != GTGPU_OK) throw_naming_path(fn, paths);
    return r;
}

std::array<uint64_t, 4> Igd::info() const {
    if (!igd_) throw Error("info needs a database Igd (not from_single_region_set)");
    std::array<uint64_t, 4> a{};
    check(gtgpu_igd_info(igd_, a.data()), "gtgpu_igd_info");
    return a;
}

std::unique_ptr<Igd> Igd::from_single_region_set(std::shared_ptr<Device> dev, const RegionSet& subject) {
    std::unique_ptr<Igd> g(new Igd());
    g->dev_ = dev;
    g->n_files_ = 1;
    RegionSet kept;
    for (size_t i = 0; i < subject.regions.size(); ++i) {
        const Region& r = subject.regions[i];
        const int32_t s = (int32_t)r.start, e = (int32_t)r.end;  // igd.rs:623-629 casts, Igd::add drops the rest
        if (s < 0 || e < 0 || s >= e) continue;
        kept.regions.push_back(Region{r.chr, r.start, r.end, ""});
        g->single_src_.push_back((uint32_t)i);
    }
    g->single_.reset(new MultiChromOverlapper(dev, kept, OverlapperType::Bits));
    return g;
}

std::vector<std::pair<uint32_t, uint32_t>> Igd::find_overlaps_regionset(const RegionSet& query, int32_t min_overlap) const {
    if (!single_) throw Error("find_overlaps_regionset needs an Igd built with from_single_region_set");
    if (min_overlap < 1) throw Error("min_overlap < 1 depends on the reference's tile layout and is not supported");
    std::vector<std::pair<uint32_t, uint32_t>> pairs;
    auto idx = single_->find_overlaps_indices(query, min_overlap);
    for (size_t q = 0; q < idx.size(); ++q)
        for (uint32_t v : idx[q]) pairs.emplace_back((uint32_t)q, single_src_[v]);
    std::sort(pairs.begin(), pairs.end());
    return pairs;
}

std::vector<uint32_t> Igd::count_overlaps_per_query(const RegionSet& query, int32_t min_overlap) const {
    if (!single_) throw Error("count_overlaps_per_query needs an Igd built with from_single_region_set");
    if (min_overlap < 1) throw Error("min_overlap < 1 depends on the reference's tile layout and is not supported");
    auto c = single_->count_overlaps(query, min_overlap);
    return std::vector<uint32_t>(c.begin(), c.end());
}

std::vector<uint64_t> Igd::count_set_overlaps(const RegionSet& regions, int32_t min_overlap) const {
    return count_region_hits_batch({&regions}, min_overlap, true);
}
std::vector<uint64_t> Igd::count_region_hits(const RegionSet& regions, int32_t min_overlap) const {
    return count_region_hits_batch({&regions}, min_overlap, false);
}

namespace {
// run_lola's tables (enrichment.rs:198-220) from the hit matrix of the user sets with the universe as its last row
std::vector<std::vector<ContingencyCounts>> contingency_tables(const std::vector<uint64_t>& hits, size_t nf,
                                                               const std::vector<uint64_t>& user_sizes, uint64_t universe_size) {
    const uint64_t* universe_hits = hits.data() + user_sizes.size() * nf;
    std::vector<std::vector<ContingencyCounts>> out(user_sizes.size(), std::vector<ContingencyCounts>(nf));
    for (size_t u = 0; u < user_sizes.size(); ++u)
        for (size_t f = 0; f < nf; ++f) {
            int64_t a = (int64_t)hits[u * nf + f];
            int64_t b = (int64_t)universe_hits[f] - a;
            int64_t c = (int64_t)user_sizes[u] - a;
            int64_t d = (int64_t)universe_size - a - b - c;
            out[u][f] = ContingencyCounts{a, b, c, d};
        }
    return out;
}
}  // namespace

std::vector<std::vector<ContingencyCounts>> lola_contingency(const Igd& igd, const std::vector<const RegionSet*>& user_sets,
                                                             const RegionSet& universe, int32_t min_overlap) {
    if (igd.num_files() == 0) throw Error("Database is empty");       // LolaError::EmptyDatabase, enrichment.rs:189-191
    if (universe.regions.empty()) throw Error("Universe is empty");   // LolaError::EmptyUniverse, enrichment.rs:194-196
    std::vector<const RegionSet*> all(user_sets);
    all.push_back(&universe);
    std::vector<uint64_t> hits = igd.count_region_hits_batch(all, min_overlap, false);  // one device pass
    std::vector<uint64_t> user_sizes(user_sets.size());
    for (size_t u = 0; u < user_sets.size(); ++u) user_sizes[u] = user_sets[u]->regions.size();
    return contingency_tables(hits, igd.num_files(), user_sizes, universe.regions.size());
}

std::vector<std::vector<ContingencyCounts>> lola_contingency_bed_files(const Igd& igd, const std::vector<std::string>& user_paths,
                                                                       const std::string& universe_path, int32_t min_overlap) {
    if (igd.num_files() == 0) throw Error("Database is empty");  // LolaError::EmptyDatabase; an empty universe fails in the parse
    std::vector<std::string> all(user_paths);
    all.push_back(universe_path);
    Igd::BedCounts h = igd.count_bed_files(all, min_overlap, false);  // one device pass
    const uint64_t universe_size = h.set_regions.back();
    h.set_regions.pop_back();
    return contingency_tables(h.matrix, igd.num_files(), h.set_regions, universe_size);
}

}  // namespace gtars
