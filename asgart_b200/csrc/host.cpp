// host.cpp — host side of the path above the C ABI, in C++ because the reference's host is compiled code (Rust) and no
// Rust toolchain exists in this image. It mirrors, for the duplication-search path only:
//   prepare_data            src/bin/asgart.rs:273-471   (FASTA -> normalised strand + fragment map + chunks + '$')
//   ProtoSD -> SD + JSON    src/bin/asgart.rs:770-821, src/structs.rs:36-98,471-493, src/exporters.rs:12-25
//   output file naming      src/bin/asgart.rs:642-654,695-719, src/utils.rs:30-49
//   the step pipeline       src/bin/asgart.rs:731-757 (driven through the device operator of api.cu)
// plus the deterministic synthetic-genome generator used by bench.py and the tests (DESIGN.md "Synthetic inputs").
#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <functional>
#include <map>
#include <regex>
#include <sstream>
#include <string>
#include <thread>
#include <vector>

#include <new>

#include "../../include/asgart_b200.h"
#include "host_internal.h"

namespace {

struct Fragment {
    std::string name;
    uint64_t position, length;
};

}  // namespace

struct asgart_b200_prepared {
    std::string file_names;
    std::vector<uint8_t> data;  // incl. '$'; empty when the strand lives only on the device (GPU-side ingest)
    uint64_t n_plus_1 = 0;
    std::vector<Fragment> map;
    std::vector<asgart_b200_chunk> chunks;
};

namespace {

thread_local std::string g_err;

bool is_base(uint8_t c) { return c == 'A' || c == 'T' || c == 'G' || c == 'C' || c == 'N'; }
bool is_masked_base(uint8_t c) { return c == 'a' || c == 't' || c == 'g' || c == 'c' || c == 'n'; }

// bin/asgart.rs:291-301
void normalise(uint8_t* seq, size_t n, bool skip_masked) {
    for (size_t i = 0; i < n; ++i) {
        uint8_t c = seq[i];
        if (!skip_masked && c >= 'a' && c <= 'z') c = uint8_t(c - 32);
        if (skip_masked && is_masked_base(c)) c = 'N';
        else if (!is_base(c)) c = 'N';
        seq[i] = c;
    }
}

// bin/asgart.rs:317-366 — maximal regions split at N-runs longer than 5000; coordinates relative to the fragment
void find_chunks(const uint8_t* s, uint64_t len, uint64_t global_off, std::vector<asgart_b200_chunk>& out) {
    const uint64_t threshold = 5000;
    const size_t first = out.size();
    uint64_t start = 0, count = 0, i = 0;
    while (i < len) {
        if (s[i] == 'N' || s[i] == 'n') {
            uint64_t run = 0;
            while (i + run < len && (s[i + run] == 'N' || s[i + run] == 'n')) ++run;
            if (run > threshold) {
                if (count > 0) { out.push_back({global_off + start, count}); count = 0; }
                start = i + run;
            } else {
                count += run;
            }
            i += run;
        } else {
            if (count == 0) { count = 1; start = i; } else { ++count; }
            ++i;
        }
    }
    if (count != 0) out.push_back({global_off + start, count});
    if (out.size() == first) out.push_back({global_off, len});
}

size_t rtrim_len(const std::string& s) {
    size_t e = s.size();
    while (e > 0 && isspace((unsigned char)s[e - 1])) --e;
    return e;
}

// bin/asgart.rs:278-313 with the bio FASTA reader's semantics (id = header up to first whitespace; lines trimmed)
bool read_fasta(const std::string& path, bool skip_masked, uint64_t offset, asgart_b200_prepared* p) {
    std::ifstream in(path, std::ios::binary);
    if (!in) { g_err = "Unable to read FASTA file `" + path + "`"; return false; }
    std::string line, name;
    bool have = false, blank_header = false;
    size_t rec_start = p->data.size();
    // false: the record is empty (no id, no description, no sequence) — the bio reader's iterator ends there and the rest
    // of the file is never looked at (bio io/fasta.rs Records::next / Record::is_empty)
    auto close_record = [&]() {
        const size_t len = p->data.size() - rec_start;
        if (blank_header && len == 0) return false;
        normalise(p->data.data() + rec_start, len, skip_masked);
        p->map.push_back(Fragment{name, uint64_t(rec_start), uint64_t(len)});
        find_chunks(p->data.data() + rec_start, len, rec_start, p->chunks);
        return true;
    };
    (void)offset;
    while (std::getline(in, line)) {
        if (!line.empty() && line[0] == '>') {
            if (have && !close_record()) return true;
            const size_t e = rtrim_len(line);
            size_t sp = 1;
            while (sp < e && !isspace((unsigned char)line[sp])) ++sp;
            name = line.substr(1, sp - 1);
            blank_header = e <= 1;
            rec_start = p->data.size();
            have = true;
        } else {
            if (!have) { g_err = "Unable to parse `" + path + "`"; return false; }   // "Expected > at record start."
            const size_t e = rtrim_len(line);
            p->data.insert(p->data.end(), line.begin(), line.begin() + e);
        }
    }
    if (have) close_record();
    return true;
}

std::vector<std::string> split_lines(const char* s) {
    std::vector<std::string> out;
    if (!s) return out;
    std::stringstream ss(s);
    std::string f;
    while (std::getline(ss, f, '\n')) if (!f.empty()) out.push_back(f);
    return out;
}

// ------------------------------------------------------------------------------------------------ JSON
void jstr(std::string& o, const std::string& s) {
    o += '"';
    for (unsigned char c : s) {
        switch (c) {
            case '"': o += "\\\""; break;
            case '\\': o += "\\\\"; break;
            case '\n': o += "\\n"; break;
            case '\r': o += "\\r"; break;
            case '\t': o += "\\t"; break;
            case '\b': o += "\\b"; break;
            case '\f': o += "\\f"; break;
            default:
                if (c < 0x20) { char b[8]; snprintf(b, sizeof b, "\\u%04x", c); o += b; }
                else o += char(c);
        }
    }
    o += '"';
}

// f32 the way serde_json (ryu) prints it: shortest digits that round-trip, ".0" appended to integral values
std::string jf32(float v) {
    if (v == 0.f) return std::signbit(v) ? "-0.0" : "0.0";
    char b[64];
    for (int prec = 1; prec <= 9; ++prec) {
        snprintf(b, sizeof b, "%.*g", prec, double(v));
        if (strtof(b, nullptr) == v) break;
    }
    std::string s(b);
    if (s.find_first_of(".eni") == std::string::npos) s += ".0";
    return s;
}

const Fragment* chr_by_pos(const std::vector<Fragment>& map, uint64_t pos) {  // structs.rs:86-90
    for (const Fragment& c : map)
        if (pos >= c.position && pos < c.position + c.length) return &c;
    return nullptr;
}

struct Ind {  // serde_json PrettyFormatter: two spaces per level
    std::string& o;
    void nl(int level) { o += '\n'; o.append(size_t(level) * 2, ' '); }
};

// ------------------------------------------------------------------------------------------------ synthetic genomes
inline uint64_t splitmix64(uint64_t x) {
    uint64_t z = x + 0x9E3779B97F4A7C15ull;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}
struct Rng {  // splitmix64 stream keyed by (seed, stream id)
    uint64_t s;
    Rng(uint64_t seed, uint64_t stream) : s(splitmix64(seed ^ splitmix64(stream * 0xD1B54A32D192ED03ull + 0x8CB92BA72F3D8DD7ull))) {}
    uint64_t next() { s += 0x9E3779B97F4A7C15ull; uint64_t z = s; z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull; z = (z ^ (z >> 27)) * 0x94D049BB133111EBull; return z ^ (z >> 31); }
    double uniform() { return double(next() >> 11) * (1.0 / 9007199254740992.0); }  // [0,1)
    uint64_t below(uint64_t n) { return n ? uint64_t(uniform() * double(n)) % n : 0; }
};

const uint64_t kHg38[24] = {248956422, 242193529, 198295559, 190214555, 181538259, 170805979, 159345973, 145138636,
                            138394717, 133797422, 135086622, 133275309, 114364328, 107043718, 101991189, 90338345,
                            83257441,  80373285,  58617616,  64444167,  46709983,  50818468,  156040895, 57227415};
const char* kHg38Names[24] = {"chr1", "chr2", "chr3", "chr4", "chr5", "chr6", "chr7", "chr8", "chr9", "chr10", "chr11", "chr12",
                              "chr13", "chr14", "chr15", "chr16", "chr17", "chr18", "chr19", "chr20", "chr21", "chr22", "chrX", "chrY"};

struct Interval { uint64_t b, e; };

struct SynthSpec {
    uint64_t seed = 1;
    uint64_t n = 0;
    std::vector<Fragment> frags;
    std::vector<Interval> nruns;      // stamped last; planted pairs avoid them
    uint64_t n_pairs = 0;
    int rc_percent = 0;               // share of planted pairs that are reverse-complemented
    int inter_percent = 0;            // share of pairs whose copy lands in another fragment
    bool softmask = false;            // ~15 % lower-case, applied before planting
    uint64_t element_copies = 0;      // C3: 300 bp element, <=10 % divergence
    double scale = 1.0;
};

uint64_t scaled(uint64_t v, double sc, uint64_t lo) { return std::max<uint64_t>(lo, uint64_t(double(v) * sc)); }

bool make_spec(int config, int part, int64_t scale_n, uint64_t seed, int64_t n_pairs, int rc_percent, SynthSpec& sp) {
    auto single = [&](const char* name, uint64_t full_n) {
        sp.n = scale_n > 0 ? uint64_t(scale_n) : full_n;
        sp.scale = double(sp.n) / double(full_n);
        sp.frags = {Fragment{name, 0, sp.n}};
    };
    switch (config) {
        case 0:
            if (scale_n <= 0) return false;
            sp.seed = seed; sp.n = uint64_t(scale_n); sp.frags = {Fragment{"synth", 0, sp.n}};
            sp.n_pairs = uint64_t(std::max<int64_t>(0, n_pairs)); sp.rc_percent = rc_percent;
            return true;
        case 1:
            sp.seed = 101; single("synth10m", 10000000ull);
            sp.n_pairs = scaled(40, sp.scale, 2); sp.rc_percent = 0;
            return true;
        case 2: {
            sp.seed = 202; single("synthY", 57227415ull);
            sp.n_pairs = scaled(240, sp.scale, 4); sp.rc_percent = 50; sp.softmask = true;
            const uint64_t tel = scaled(10000, sp.scale, 5001);
            sp.nruns.push_back({0, tel});
            sp.nruns.push_back({sp.n - tel, sp.n});
            const uint64_t big = scaled(3000000, sp.scale, 6000), at = scaled(10000000, sp.scale, tel + 1000);
            sp.nruns.push_back({at, std::min(sp.n - tel, at + big)});
            Rng r(sp.seed, 7001);
            for (int i = 0; i < 20; ++i) {
                const uint64_t len = 10 + r.below(1991), pos = r.below(sp.n - len);
                sp.nruns.push_back({pos, pos + len});
            }
            return true;
        }
        case 3: {
            sp.seed = 303; single("synth1", 248956422ull);
            sp.n_pairs = scaled(1000, sp.scale, 4); sp.rc_percent = 50;
            sp.element_copies = scaled(1500, sp.scale, 600);
            const uint64_t big = scaled(18000000, sp.scale, 6000), at = scaled(121700000, sp.scale, 1000);
            sp.nruns.push_back({at, std::min(sp.n, at + big)});
            Rng r(sp.seed, 7001);
            for (int i = 0; i < 30; ++i) {
                const uint64_t len = 10 + r.below(1991), pos = r.below(sp.n - len);
                sp.nruns.push_back({pos, pos + len});
            }
            return true;
        }
        case 4: {
            sp.seed = 404;
            sp.scale = scale_n > 0 ? double(scale_n) / 3088269832.0 : 1.0;
            uint64_t pos = 0;
            for (int f = 0; f < 24; ++f) {
                const uint64_t len = scaled(kHg38[f], sp.scale, 20000);
                sp.frags.push_back(Fragment{kHg38Names[f], pos, len});
                const uint64_t tel = std::min<uint64_t>(len / 8, scaled(10000, sp.scale, 5001));
                sp.nruns.push_back({pos, pos + tel});
                sp.nruns.push_back({pos + len - tel, pos + len});
                const uint64_t cen = std::max<uint64_t>(5001, len / 50), cat = pos + len * 2 / 5;
                sp.nruns.push_back({cat, cat + cen});
                pos += len;
            }
            sp.n = pos;
            sp.n_pairs = scaled(8000, sp.scale, 8); sp.rc_percent = 50; sp.inter_percent = 30;
            return true;
        }
        case 5: {
            sp.seed = part == 0 ? 505 : 506;
            sp.scale = scale_n > 0 ? double(scale_n) / 1000000000.0 : 1.0;
            uint64_t pos = 0;
            for (int f = 0; f < 10; ++f) {
                const uint64_t len = scaled(100000000ull, sp.scale, 20000);
                char nm[32];
                snprintf(nm, sizeof nm, "%c%d", part == 0 ? 'A' : 'B', f + 1);
                sp.frags.push_back(Fragment{nm, pos, len});
                pos += len;
            }
            sp.n = pos;
            sp.n_pairs = scaled(500, sp.scale, 2); sp.rc_percent = 50;
            return true;
        }
        default: return false;
    }
}

bool hits_nrun(const std::vector<Interval>& nr, uint64_t b, uint64_t e) {
    for (const Interval& r : nr) if (b < r.e && r.b < e) return true;
    return false;
}
int frag_of(const std::vector<Fragment>& fr, uint64_t pos) {
    for (size_t f = 0; f < fr.size(); ++f) if (pos >= fr[f].position && pos < fr[f].position + fr[f].length) return int(f);
    return -1;
}
inline uint8_t comp_keep_case(uint8_t c) {
    switch (c) {
        case 'A': return 'T'; case 'T': return 'A'; case 'C': return 'G'; case 'G': return 'C';
        case 'a': return 't'; case 't': return 'a'; case 'c': return 'g'; case 'g': return 'c';
        default: return c;
    }
}
inline uint8_t other_base(uint8_t c, Rng& r) {
    const bool lower = c >= 'a';
    const char* up = "ACGT";
    uint8_t u = lower ? uint8_t(c - 32) : c;
    int k = int(r.below(3));
    for (int i = 0; i < 4; ++i) if (uint8_t(up[i]) != u) { if (k-- == 0) { u = uint8_t(up[i]); break; } }
    return lower ? uint8_t(u + 32) : u;
}

// mutated copy of src[0..L): divergence d, events 80 % substitutions / 20 % indels of 1-3 bp, output length fixed at L
void mutate_copy(const uint8_t* src, uint64_t avail, uint64_t L, double d, Rng& r, std::vector<uint8_t>& out) {
    out.clear();
    out.reserve(L);
    uint64_t cur = 0;
    while (out.size() < L) {
        if (cur >= avail) { out.push_back(uint8_t("ACGT"[r.below(4)])); continue; }
        if (r.uniform() < d) {
            const double ev = r.uniform();
            if (ev < 0.8) { out.push_back(other_base(src[cur], r)); ++cur; }
            else {
                const uint64_t len = 1 + r.below(3);
                if (ev < 0.9) { for (uint64_t j = 0; j < len && out.size() < L; ++j) out.push_back(uint8_t("ACGT"[r.below(4)])); }
                else cur += len;
            }
        } else { out.push_back(src[cur]); ++cur; }
    }
}

void plant_pairs(std::vector<uint8_t>& g, uint64_t off, const SynthSpec& sp, const uint8_t* donor, uint64_t donor_n, uint64_t n_pairs,
                 uint64_t stream_base) {
    // g = this genome (absolute coordinates start at `off` inside it == 0 here), donor = genome the source is cut from
    (void)off;
    std::vector<uint8_t> buf;
    for (uint64_t j = 0; j < n_pairs; ++j) {
        Rng r(sp.seed, stream_base + j);
        const double lmin = std::log(2000.0), lmax = std::log(50000.0);
        uint64_t L = uint64_t(std::exp(lmin + r.uniform() * (lmax - lmin)));
        L = std::min<uint64_t>(L, std::max<uint64_t>(200, sp.n / 40));
        const double d = r.uniform() * 0.02;
        const bool rc = int(r.below(100)) < sp.rc_percent;
        const bool inter = int(r.below(100)) < sp.inter_percent;
        for (int attempt = 0; attempt < 200; ++attempt) {
            const uint64_t src = r.below(donor_n - L), dst = r.below(sp.n - L);
            const int fd = frag_of(sp.frags, dst);
            if (fd < 0 || dst + L > sp.frags[fd].position + sp.frags[fd].length) continue;
            if (hits_nrun(sp.nruns, dst, dst + L)) continue;
            if (donor == g.data()) {
                const int fs = frag_of(sp.frags, src);
                if (fs < 0 || src + L > sp.frags[fs].position + sp.frags[fs].length) continue;
                if (hits_nrun(sp.nruns, src, src + L)) continue;
                if (src < dst + L && dst < src + L) continue;
                if (sp.frags.size() > 1 && (inter ? fs == fd : fs != fd)) continue;
            }
            mutate_copy(donor + src, donor_n - src, L, d, r, buf);
            if (rc) {
                std::reverse(buf.begin(), buf.end());
                for (auto& c : buf) c = comp_keep_case(c);
            }
            memcpy(g.data() + dst, buf.data(), L);
            break;
        }
    }
}

void generate(const SynthSpec& sp, std::vector<uint8_t>& g, int threads, const std::vector<uint8_t>* donor_a, uint64_t shared_segments) {
    g.resize(sp.n);
    const uint64_t key = sp.seed * 0x9E3779B97F4A7C15ull;
    const int nt = std::max(1, threads);
    std::vector<std::thread> pool;
    auto fill = [&](uint64_t b, uint64_t e) {
        for (uint64_t i = b; i < e; ++i) g[i] = uint8_t("ACGT"[splitmix64(key + i) >> 62]);
    };
    const uint64_t per = (sp.n + nt - 1) / nt;
    for (int t = 0; t < nt; ++t) {
        const uint64_t b = std::min(sp.n, t * per), e = std::min(sp.n, b + per);
        if (b < e) pool.emplace_back(fill, b, e);
    }
    for (auto& th : pool) th.join();
    if (sp.softmask) {  // ~15 % lower-case in intervals of mean 300 bp (mean gap 1700 bp)
        Rng r(sp.seed, 9001);
        uint64_t pos = 0;
        for (;;) {
            pos += uint64_t(-std::log(1.0 - r.uniform()) * 1700.0) + 1;
            const uint64_t len = uint64_t(-std::log(1.0 - r.uniform()) * 300.0) + 1;
            if (pos >= sp.n) break;
            const uint64_t e = std::min(sp.n, pos + len);
            for (uint64_t i = pos; i < e; ++i) g[i] = uint8_t(g[i] + 32);
            pos = e;
        }
    }
    plant_pairs(g, 0, sp, g.data(), sp.n, sp.n_pairs, 100000);
    if (donor_a) plant_pairs(g, 0, sp, donor_a->data(), donor_a->size(), shared_segments, 500000);
    if (sp.element_copies) {
        Rng re(sp.seed, 8001);
        uint8_t elem[300];
        for (auto& c : elem) c = uint8_t("ACGT"[re.below(4)]);
        for (uint64_t c = 0; c < sp.element_copies; ++c) {
            Rng r(sp.seed, 800000 + c);
            const double d = r.uniform() * 0.10;
            for (int attempt = 0; attempt < 100; ++attempt) {
                const uint64_t pos = r.below(sp.n - 300);
                if (hits_nrun(sp.nruns, pos, pos + 300)) continue;
                for (int i = 0; i < 300; ++i) g[pos + i] = (r.uniform() < d) ? other_base(elem[i], r) : elem[i];
                break;
            }
        }
    }
    for (const Interval& r : sp.nruns)
        for (uint64_t i = r.b; i < r.e && i < sp.n; ++i) g[i] = 'N';
}

}  // namespace

// ================================================================================================ C ABI
asgart_b200_prepared* ab200_prepared_device_only(const std::string& file_names, uint64_t n, const std::vector<std::string>& names,
                                                 const std::vector<uint64_t>& pos, const std::vector<uint64_t>& len,
                                                 const std::vector<asgart_b200_chunk>& chunks) {
    auto* p = new asgart_b200_prepared();
    p->file_names = file_names;
    p->n_plus_1 = n + 1;
    for (size_t i = 0; i < names.size(); ++i) p->map.push_back(Fragment{names[i], pos[i], len[i]});
    p->chunks = chunks;
    return p;
}

extern "C" {

asgart_b200_prepared* asgart_b200_prepare_files(const char* files, int32_t skip_masked, const char** err) {
    if (err) *err = nullptr;
    auto* p = new asgart_b200_prepared();
    const std::vector<std::string> fl = split_lines(files);
    for (size_t i = 0; i < fl.size(); ++i) {
        if (!read_fasta(fl[i], skip_masked != 0, 0, p)) {
            delete p;
            if (err) *err = g_err.c_str();
            return nullptr;
        }
        p->file_names += (i ? ", " : "") + fl[i];  // bin/asgart.rs:466
    }
    p->data.push_back('$');  // bin/asgart.rs:430
    return p;
}

asgart_b200_prepared* asgart_b200_prepare_memory(const char* file_names, const uint8_t* strand, int64_t n, const char* fragment_names,
                                                 const uint64_t* frag_pos, const uint64_t* frag_len, int64_t n_fragments) {
    if (!strand || n < 0 || !frag_pos || !frag_len) return nullptr;
    auto* p = new asgart_b200_prepared();
    p->file_names = file_names ? file_names : "";
    p->data.assign(strand, strand + n);
    const std::vector<std::string> names = split_lines(fragment_names);
    for (int64_t i = 0; i < n_fragments; ++i) {
        if (frag_pos[i] + frag_len[i] > uint64_t(n)) { delete p; return nullptr; }
        p->map.push_back(Fragment{size_t(i) < names.size() ? names[i] : std::string("fragment") + std::to_string(i), frag_pos[i], frag_len[i]});
        find_chunks(p->data.data() + frag_pos[i], frag_len[i], frag_pos[i], p->chunks);
    }
    p->data.push_back('$');
    return p;
}

const uint8_t* asgart_b200_prepared_strand(const asgart_b200_prepared* p, int64_t* n_plus_1) {
    if (n_plus_1) *n_plus_1 = int64_t(p->data.empty() ? p->n_plus_1 : p->data.size());
    return p->data.empty() ? nullptr : p->data.data();
}
const asgart_b200_chunk* asgart_b200_prepared_chunks(const asgart_b200_prepared* p, int64_t* n_chunks) {
    if (n_chunks) *n_chunks = int64_t(p->chunks.size());
    return p->chunks.data();
}
int64_t asgart_b200_prepared_n_fragments(const asgart_b200_prepared* p) { return int64_t(p->map.size()); }
const char* asgart_b200_prepared_fragment(const asgart_b200_prepared* p, int64_t i, uint64_t* position, uint64_t* length) {
    if (position) *position = p->map[i].position;
    if (length) *length = p->map[i].length;
    return p->map[i].name.c_str();
}
void asgart_b200_prepared_free(asgart_b200_prepared* p) { delete p; }

// ------------------------------------------------------------------------------------------------ RunResult
// The SD-level result of a run (RunResult / StrandResult / SD, src/structs.rs:60-97, 471-493): what JSONExporter writes
// and what asgart-slice reads back, edits and writes again.
extern "C++" {
namespace {
struct SDRec {
    std::string chr_left, chr_right;
    uint64_t global_left, global_right, chr_left_position, chr_right_position, left_length, right_length;
    float identity;
    bool reversed, complemented;
};
}  // namespace

struct asgart_b200_run_result {
    std::string strand_name;
    uint64_t strand_length = 0;
    std::vector<Fragment> map;
    asgart_b200_settings settings{};
    std::vector<std::vector<SDRec>> families;
    std::string error;
};

namespace {
const char* const kCollapsedName = "ASGART_COLLAPSED";   // src/structs.rs:9

const Fragment* find_chr(const std::vector<Fragment>& map, const std::string& name) {   // StrandResult::find_chr, :77-79
    for (const Fragment& c : map) if (c.name == name) return &c;
    return nullptr;
}

// ProtoSD -> SD (src/bin/asgart.rs:776-821): fragment by position, "unknown" outside every fragment
void fill_run_result(asgart_b200_run_result& rr, const asgart_b200_prepared* p, const asgart_b200_settings* st, const uint64_t* fam_off,
                     int64_t n_fam, const asgart_b200_protosd* sds) {
    rr.strand_name = p->file_names;
    rr.strand_length = 0;
    for (const Fragment& f : p->map) rr.strand_length += f.length;   // bin/asgart.rs:772
    rr.map = p->map;
    rr.settings = *st;
    rr.families.assign(size_t(n_fam), {});
    for (int64_t f = 0; f < n_fam; ++f) {
        for (uint64_t j = fam_off[f]; j < fam_off[f + 1]; ++j) {
            const asgart_b200_protosd& sd = sds[j];
            const Fragment* cl = chr_by_pos(p->map, sd.left);
            const Fragment* cr = chr_by_pos(p->map, sd.right);
            SDRec r;
            r.chr_left = cl ? cl->name : "unknown";
            r.chr_right = cr ? cr->name : "unknown";
            r.global_left = sd.left; r.global_right = sd.right;
            r.chr_left_position = sd.left - (cl ? cl->position : 0);
            r.chr_right_position = sd.right - (cr ? cr->position : 0);
            r.left_length = sd.left_length; r.right_length = sd.right_length;
            r.identity = sd.identity;
            r.reversed = sd.reversed != 0; r.complemented = sd.complemented != 0;
            rr.families[size_t(f)].push_back(std::move(r));
        }
    }
}

// JSONExporter::save (src/exporters.rs:12-25): serde_json pretty layout, field order = declaration order
std::string run_result_json(const asgart_b200_run_result& rr) {
    std::string o;
    size_t n_sds = 0;
    for (const auto& f : rr.families) n_sds += f.size();
    o.reserve(4096 + n_sds * 420);
    Ind in{o};
    auto key = [&](int level, const char* k) { in.nl(level); o += '"'; o += k; o += "\": "; };
    auto num = [&](uint64_t v) { o += std::to_string(v); };
    const asgart_b200_settings* st = &rr.settings;
    o += '{';
    key(1, "strand"); o += '{';
    key(2, "name"); jstr(o, rr.strand_name); o += ',';
    key(2, "length"); num(rr.strand_length); o += ',';
    key(2, "map"); o += '[';
    for (size_t i = 0; i < rr.map.size(); ++i) {
        if (i) o += ',';
        in.nl(3); o += '{';
        key(4, "name"); jstr(o, rr.map[i].name); o += ',';
        key(4, "position"); num(rr.map[i].position); o += ',';
        key(4, "length"); num(rr.map[i].length);
        in.nl(3); o += '}';
    }
    if (!rr.map.empty()) in.nl(2);
    o += ']';
    in.nl(1); o += "},";
    key(1, "settings"); o += '{';
    key(2, "probe_size"); num(st->probe_size); o += ',';
    key(2, "max_gap_size"); num(st->max_gap_size); o += ',';
    key(2, "min_duplication_length"); num(st->min_duplication_length); o += ',';
    key(2, "max_cardinality"); num(st->max_cardinality); o += ',';
    key(2, "trim");
    if (st->has_trim) { o += '['; in.nl(3); num(st->trim_a); o += ','; in.nl(3); num(st->trim_b); in.nl(2); o += ']'; }
    else o += "null";
    o += ',';
    key(2, "skip_masked"); o += st->skip_masked ? "true" : "false";
    in.nl(1); o += "},";
    key(1, "families"); o += '[';
    for (size_t f = 0; f < rr.families.size(); ++f) {
        if (f) o += ',';
        in.nl(2); o += '[';
        for (size_t j = 0; j < rr.families[f].size(); ++j) {
            const SDRec& sd = rr.families[f][j];
            if (j) o += ',';
            in.nl(3); o += '{';
            key(4, "chr_left"); jstr(o, sd.chr_left); o += ',';
            key(4, "chr_right"); jstr(o, sd.chr_right); o += ',';
            key(4, "global_left_position"); num(sd.global_left); o += ',';
            key(4, "global_right_position"); num(sd.global_right); o += ',';
            key(4, "chr_left_position"); num(sd.chr_left_position); o += ',';
            key(4, "chr_right_position"); num(sd.chr_right_position); o += ',';
            key(4, "left_length"); num(sd.left_length); o += ',';
            key(4, "right_length"); num(sd.right_length); o += ',';
            key(4, "left_seq"); o += "null,";
            key(4, "right_seq"); o += "null,";
            key(4, "identity"); o += jf32(sd.identity); o += ',';
            key(4, "reversed"); o += sd.reversed ? "true" : "false"; o += ',';
            key(4, "complemented"); o += sd.complemented ? "true" : "false";
            in.nl(3); o += '}';
        }
        if (!rr.families[f].empty()) in.nl(2);
        o += ']';
    }
    if (!rr.families.empty()) in.nl(1);
    o += ']';
    in.nl(0); o += "}\n";  // exporters.rs:15-17: writeln!
    return o;
}

char* dup_string(const std::string& o) {
    char* out = static_cast<char*>(malloc(o.size() + 1));
    if (out) memcpy(out, o.c_str(), o.size() + 1);
    return out;
}

void drop_empty(asgart_b200_run_result& rr) {   // families.retain(|f| !f.is_empty())
    rr.families.erase(std::remove_if(rr.families.begin(), rr.families.end(), [](const std::vector<SDRec>& f) { return f.empty(); }),
                      rr.families.end());
}
template <typename Pred>
void retain_sds(asgart_b200_run_result& rr, Pred keep) {
    for (auto& f : rr.families) f.erase(std::remove_if(f.begin(), f.end(), [&](const SDRec& sd) { return !keep(sd); }), f.end());
}
bool in_list(const std::vector<std::string>& l, const std::string& n) { return std::find(l.begin(), l.end(), n) != l.end(); }

// RunResult::flatten (src/structs.rs:350-416, `--collapse`): fragments no longer than mean + one standard deviation whose
// name is longer than two bytes become one pseudo-fragment. As in the reference: its Start sits at (kept length + 1),
// strand.length and the duplicons' global positions are left alone.
void rr_flatten(asgart_b200_run_result& rr) {
    if (rr.map.size() < 2) return;
    const double n = double(rr.map.size());
    double sum = 0;
    for (const Fragment& c : rr.map) sum += double(c.length);
    const double avg = sum / n;
    double ss = 0;
    for (const Fragment& c : rr.map) ss += std::pow(double(c.length) - avg, 2.0);
    const double sd = std::sqrt(1.0 / (n - 1.0) * ss);
    std::vector<Fragment> to_flatten, to_keep;
    for (const Fragment& c : rr.map) if (double(c.length) <= avg + sd && c.name.size() > 2) to_flatten.push_back(c);
    uint64_t to_flatten_len = 0, to_keep_len = 0;
    for (const Fragment& c : to_flatten) to_flatten_len += c.length;
    for (const Fragment& c : rr.map) {
        bool fl = false;
        for (const Fragment& r : to_flatten) fl = fl || r.name == c.name;
        if (!fl) to_keep.push_back(c);
    }
    for (const Fragment& c : to_keep) to_keep_len += c.length;
    uint64_t i = 0;
    for (Fragment& c : to_keep) { c.position = i; i += c.length; }
    for (Fragment& c : to_flatten) { c.position = i; i += c.length; }
    std::map<std::string, uint64_t> pos;   // HashMap from (name, position): a repeated name keeps its last position
    for (const Fragment& c : to_flatten) pos[c.name] = c.position;
    rr.map = to_keep;
    rr.map.push_back(Fragment{kCollapsedName, to_keep_len + 1, to_flatten_len});
    for (auto& f : rr.families)
        for (SDRec& s2 : f) {
            const bool lm = pos.count(s2.chr_left) != 0, rm = pos.count(s2.chr_right) != 0;
            if (lm) { s2.chr_left_position += pos[s2.chr_left]; s2.chr_left = kCollapsedName; }
            if (rm) { s2.chr_right_position += pos[s2.chr_right]; s2.chr_right = kCollapsedName; }
        }
}

// the common tail of keep/restrict (consolidate_families, src/structs.rs:204-230) and of exclude (:277-298, which unwraps)
bool rr_relayout(asgart_b200_run_result& rr, const std::function<bool(const std::string&)>& keep_fragment, bool unwrap) {
    drop_empty(rr);
    rr.map.erase(std::remove_if(rr.map.begin(), rr.map.end(), [&](const Fragment& c) { return !keep_fragment(c.name); }), rr.map.end());
    rr.strand_length = 0;
    for (const Fragment& c : rr.map) rr.strand_length += c.length;
    uint64_t i = 0;
    for (Fragment& c : rr.map) { c.position = i; i += c.length; }
    for (auto& f : rr.families)
        for (SDRec& sd : f) {
            const Fragment* l = find_chr(rr.map, sd.chr_left);
            const Fragment* r = find_chr(rr.map, sd.chr_right);
            if (unwrap && (!l || !r)) { rr.error = "exclude-fragments: a duplicon stands on a fragment that is not in the map; the reference panics here (Option::unwrap, src/structs.rs:291-294)"; return false; }
            sd.global_left = l ? l->position + sd.chr_left_position : 0;
            sd.global_right = r ? r->position + sd.chr_right_position : 0;
        }
    return true;
}
}  // namespace
}  // extern "C++"

char* asgart_b200_to_json(const asgart_b200_prepared* p, const asgart_b200_settings* st, const uint64_t* fam_off, int64_t n_fam,
                          const asgart_b200_protosd* sds) {
    asgart_b200_run_result rr;
    fill_run_result(rr, p, st, fam_off, n_fam, sds);
    return dup_string(run_result_json(rr));
}

asgart_b200_run_result* asgart_b200_run_result_new(const asgart_b200_prepared* p, const asgart_b200_settings* st, const uint64_t* fam_off,
                                                   int64_t n_fam, const asgart_b200_protosd* sds) {
    if (!p || !st || !fam_off || n_fam < 0 || (fam_off[n_fam] && !sds)) return nullptr;
    auto* rr = new (std::nothrow) asgart_b200_run_result();
    if (rr) fill_run_result(*rr, p, st, fam_off, n_fam, sds);
    return rr;
}
void asgart_b200_run_result_free(asgart_b200_run_result* rr) { delete rr; }
char* asgart_b200_run_result_to_json(const asgart_b200_run_result* rr) { return rr ? dup_string(run_result_json(*rr)) : nullptr; }
const char* asgart_b200_run_result_error(const asgart_b200_run_result* rr) { return rr ? rr->error.c_str() : ""; }

// asgart-slice's options in ITS order (src/bin/asgart-slice.rs:126-191)
int32_t asgart_b200_run_result_slice(asgart_b200_run_result* rr, const asgart_b200_slice_options* op) {
    if (!rr || !op) return ASGART_B200_EINVAL;
    const uint32_t fl = op->flags;
    if (fl & ASGART_B200_SLICE_COLLAPSE) rr_flatten(*rr);
    auto filter = [&](auto keep) { retain_sds(*rr, keep); drop_empty(*rr); };
    if (fl & ASGART_B200_SLICE_NO_DIRECT) filter([](const SDRec& sd) { return sd.reversed; });
    if (fl & ASGART_B200_SLICE_NO_REVERSED) filter([](const SDRec& sd) { return !sd.reversed; });
    if (fl & ASGART_B200_SLICE_NO_UNCOMPLEMENTED) filter([](const SDRec& sd) { return sd.complemented; });
    if (fl & ASGART_B200_SLICE_NO_COMPLEMENTED) filter([](const SDRec& sd) { return !sd.complemented; });
    if (fl & ASGART_B200_SLICE_NO_INTER) filter([](const SDRec& sd) { return sd.chr_left == sd.chr_right; });
    if (fl & ASGART_B200_SLICE_NO_INTER_RELAXED)
        filter([](const SDRec& sd) { return sd.chr_left == sd.chr_right || sd.chr_left == kCollapsedName || sd.chr_right == kCollapsedName; });
    if (fl & ASGART_B200_SLICE_NO_INTRA) filter([](const SDRec& sd) { return sd.chr_left != sd.chr_right; });
    if (fl & ASGART_B200_SLICE_MIN_LENGTH) { const uint64_t m = op->min_length; filter([m](const SDRec& sd) { return std::min(sd.left_length, sd.right_length) >= m; }); }
    if (op->max_family_members >= 0) {
        const size_t m = size_t(op->max_family_members);
        rr->families.erase(std::remove_if(rr->families.begin(), rr->families.end(), [m](const std::vector<SDRec>& f) { return f.size() > m; }),
                           rr->families.end());
    }
    const bool re_mode = (fl & ASGART_B200_SLICE_REGEXP) != 0;
    // 0 keep (a leg on a listed fragment), 1 restrict (both legs), 2 exclude (neither leg)
    auto select = [&](const char* arg, int mode) -> int32_t {
        if (!arg) return ASGART_B200_OK;
        const std::vector<std::string> items = split_lines(arg);
        if (re_mode) {
            for (const std::string& pat : items) {   // one call of the *_regexp method per pattern, like the reference's loop
                std::regex re;
                try { re.assign(pat, std::regex::ECMAScript); }
                catch (const std::regex_error& e) { rr->error = "Error while compiling `" + pat + "`: " + e.what(); return ASGART_B200_EINVAL; }
                auto m = [&](const std::string& n) { return std::regex_search(n, re); };
                if (mode == 0) retain_sds(*rr, [&](const SDRec& sd) { return m(sd.chr_left) || m(sd.chr_right); });
                else if (mode == 1) retain_sds(*rr, [&](const SDRec& sd) { return m(sd.chr_left) && m(sd.chr_right); });
                else retain_sds(*rr, [&](const SDRec& sd) { return !m(sd.chr_left) && !m(sd.chr_right); });
                if (!rr_relayout(*rr, [&](const std::string& n) { return mode == 2 ? !m(n) : m(n); }, mode == 2)) return ASGART_B200_EPANIC;
            }
        } else {
            auto m = [&](const std::string& n) { return in_list(items, n); };
            if (mode == 0) retain_sds(*rr, [&](const SDRec& sd) { return m(sd.chr_left) || m(sd.chr_right); });
            else if (mode == 1) retain_sds(*rr, [&](const SDRec& sd) { return m(sd.chr_left) && m(sd.chr_right); });
            else retain_sds(*rr, [&](const SDRec& sd) { return !m(sd.chr_left) && !m(sd.chr_right); });
            if (!rr_relayout(*rr, [&](const std::string& n) { return mode == 2 ? !m(n) : m(n); }, mode == 2)) return ASGART_B200_EPANIC;
        }
        return ASGART_B200_OK;
    };
    int32_t rc = select(op->keep_fragments, 0);
    if (!rc) rc = select(op->restrict_fragments, 1);
    if (!rc) rc = select(op->exclude_fragments, 2);
    return rc;
}

void asgart_b200_free_string(char* s) { free(s); }

// asgart-slice's filters (bin/asgart-slice.rs:126-160 over structs.rs:143-198) on families in memory
int32_t asgart_b200_slice_families(const asgart_b200_prepared* p, const uint64_t* fam_off, int64_t n_fam, const asgart_b200_protosd* sds,
                                   uint32_t flags, uint64_t min_length, int64_t max_family_members, asgart_b200_result** out) {
    if (!p || !out || !fam_off || n_fam < 0 || (fam_off[n_fam] && !sds)) return ASGART_B200_EINVAL;
    *out = nullptr;
    static const std::string unknown = "unknown";   // bin/asgart.rs:784-800
    auto chr = [&](uint64_t pos) -> const std::string& {
        const Fragment* f = chr_by_pos(p->map, pos);
        return f ? f->name : unknown;
    };
    auto keep = [&](const asgart_b200_protosd& sd) {
        if ((flags & ASGART_B200_SLICE_NO_DIRECT) && !sd.reversed) return false;            // remove_direct keeps reversed ones
        if ((flags & ASGART_B200_SLICE_NO_REVERSED) && sd.reversed) return false;
        if ((flags & ASGART_B200_SLICE_NO_UNCOMPLEMENTED) && !sd.complemented) return false;
        if ((flags & ASGART_B200_SLICE_NO_COMPLEMENTED) && sd.complemented) return false;
        if (flags & (ASGART_B200_SLICE_NO_INTER | ASGART_B200_SLICE_NO_INTRA)) {
            const bool same = chr(sd.left) == chr(sd.right);
            if ((flags & ASGART_B200_SLICE_NO_INTER) && !same) return false;
            if ((flags & ASGART_B200_SLICE_NO_INTRA) && same) return false;
        }
        if ((flags & ASGART_B200_SLICE_MIN_LENGTH) && std::min(sd.left_length, sd.right_length) < min_length) return false;
        return true;
    };
    const bool drops_empty = flags != 0;   // every duplicon-level filter ends with families.retain(|f| !f.is_empty())
    auto* r = new (std::nothrow) asgart_b200_result();
    if (!r) return ASGART_B200_ENOMEM;
    r->fam_off.push_back(0);
    for (int64_t f = 0; f < n_fam; ++f) {
        const size_t before = r->sds.size();
        for (uint64_t j = fam_off[f]; j < fam_off[f + 1]; ++j) if (keep(sds[j])) r->sds.push_back(sds[j]);
        const size_t members = r->sds.size() - before;
        if (members == 0 && drops_empty) continue;
        if (max_family_members >= 0 && members > size_t(max_family_members)) { r->sds.resize(before); continue; }
        r->fam_off.push_back(r->sds.size());
    }
    *out = r;
    return ASGART_B200_OK;
}

// bin/asgart.rs:642-654 (radix = file stems joined by '-'), :695-719, utils.rs:30-49 (extension forced to json)
char* asgart_b200_out_filename(const char* files, const char* prefix, const char* out, const asgart_b200_settings* st) {
    std::string name;
    if (out && *out) {
        name = out;
    } else {
        std::string radix;
        const std::vector<std::string> fl = split_lines(files);
        for (size_t i = 0; i < fl.size(); ++i) {
            std::string base = fl[i];
            const size_t slash = base.find_last_of('/');
            if (slash != std::string::npos) base = base.substr(slash + 1);
            const size_t dot = base.find_last_of('.');
            if (dot != std::string::npos && dot != 0) base = base.substr(0, dot);  // Path::file_stem
            radix += (i ? "-" : "") + base;
        }
        name = std::string(prefix ? prefix : "") + radix + ((st->reverse || st->complement) ? "_" : "") + (st->reverse ? "R" : "") +
               (st->complement ? "C" : "");
        if (st->has_trim) name += "_" + std::to_string(st->trim_a) + "-" + std::to_string(st->trim_b);
        name += ".json";
    }
    // PathBuf::set_extension("json") on the file name component
    const size_t slash = name.find_last_of('/');
    const size_t start = slash == std::string::npos ? 0 : slash + 1;
    const size_t dot = name.find_last_of('.');
    if (dot != std::string::npos && dot > start) name = name.substr(0, dot);
    name += ".json";
    char* r = static_cast<char*>(malloc(name.size() + 1));
    if (r) memcpy(r, name.c_str(), name.size() + 1);
    return r;
}

// bin/asgart.rs:731-822: prepare_data -> SearchDuplications -> FilterNs -> ReOrder -> ReduceOverlap -> Sort -> JSON,
// for one or several passes over ONE index. prepare_data runs on the device too (GPU-side FASTA ingest): the files'
// bytes go to HBM as they are read. Several passes combine as RunResult::from_files does for their JSON files
// (structs.rs:114-141): strand and settings of the first, families concatenated in pass order. With several devices,
// member 0 ingests, the others copy its strand, and the group builds the index and searches every pass.
static char* run_files_impl(const char* files, const asgart_b200_settings* passes, int32_t n_passes, const int32_t* devices,
                            int32_t n_devices, const asgart_b200_slice_options* slice, const char** err) {
    static thread_local std::string msg;
    if (err) *err = nullptr;
    auto failf = [&](const std::string& m) -> char* { msg = m; if (err) *err = msg.c_str(); return nullptr; };
    if (!passes || n_passes < 1) return failf("no passes");
    if (!devices || n_devices < 1) return failf("no devices");
    for (int32_t i = 1; i < n_passes; ++i)
        if ((passes[i].skip_masked != 0) != (passes[0].skip_masked != 0))
            return failf("passes over one index must agree on skip_masked (it changes the strand)");
    for (int32_t i = 1; i < n_passes; ++i)
        if (passes[i].has_trim != passes[0].has_trim || passes[i].trim_a != passes[0].trim_a || passes[i].trim_b != passes[0].trim_b)
            return failf("passes over one index must agree on trim (it changes the index)");
    if (passes[0].has_trim && n_devices > 1) return failf("--trim builds its index on one device: give one device, not " + std::to_string(n_devices));
    const std::vector<std::string> fl = split_lines(files);
    if (fl.empty()) return failf("no input files");
    std::vector<asgart_b200_ctx*> ctxs(size_t(n_devices), nullptr);
    int rc = 0;
    for (int32_t i = 0; !rc && i < n_devices; ++i) {
        rc = asgart_b200_ctx_create(devices[i], &ctxs[size_t(i)]);
        if (rc && n_devices == 1) failf("no usable CUDA device (code " + std::to_string(rc) + "); this build has no CPU path");
        else if (rc) failf("cannot use CUDA device " + std::to_string(devices[i]) + " (code " + std::to_string(rc) + "); this build has no CPU path");
    }
    asgart_b200_ctx* ctx = ctxs[0];
    auto last_error = [&]() -> std::string {   // the first member that says why it failed
        for (asgart_b200_ctx* c : ctxs)
            if (c && *asgart_b200_ctx_last_error(c)) return asgart_b200_ctx_last_error(c);
        return "code " + std::to_string(rc);
    };
    asgart_b200_prepared* p = nullptr;
    char* js = nullptr;
    if (!rc) {
        rc = asgart_b200_ctx_ingest_begin(ctx);
        for (size_t i = 0; !rc && i < fl.size(); ++i) rc = asgart_b200_ctx_ingest_file(ctx, fl[i].c_str(), int32_t(passes[0].skip_masked));
        if (!rc) rc = asgart_b200_ctx_ingest_finish(ctx, files, &p);
        if (rc) failf(asgart_b200_ctx_last_error(ctx));
    }
    if (!rc) {
        std::vector<uint64_t> fam_off{0};
        std::vector<asgart_b200_protosd> sds;
        // --trim (bin/asgart.rs:432-463 validation, :142-147 index); the raw values stay in the settings block of the JSON
        uint64_t ta = 0, tb = 0;
        int64_t n_plus_1 = 0;
        asgart_b200_prepared_strand(p, &n_plus_1);
        if (n_devices > 1) {
            for (int32_t i = 1; !rc && i < n_devices; ++i) rc = asgart_b200_ctx_copy_strand(ctxs[size_t(i)], ctx);
            if (!rc) rc = asgart_b200_build_index_group(ctxs.data(), n_devices);
        } else if (passes[0].has_trim && asgart_b200_effective_trim(passes[0].trim_a, passes[0].trim_b, n_plus_1, &ta, &tb)) {
            rc = asgart_b200_ctx_build_index_trim(ctx, ta, tb);
        } else {
            rc = asgart_b200_ctx_build_index(ctx);
        }
        for (int32_t i = 0; !rc && i < n_passes; ++i) {
            asgart_b200_result* res = nullptr;
            const uint32_t post = ASGART_B200_POST_ALL | (passes[i].compute_score ? ASGART_B200_POST_COMPUTE_SCORE : 0u);
            const int64_t nc = int64_t(p->chunks.size());
            rc = n_devices > 1 ? asgart_b200_search_group(ctxs.data(), n_devices, p->chunks.data(), nc, &passes[i], post, &res)
                               : asgart_b200_ctx_search(ctx, p->chunks.data(), nc, &passes[i], post, &res);
            if (!rc) {
                const int64_t nf = asgart_b200_result_n_families(res);
                const uint64_t* off = asgart_b200_result_family_offsets(res);
                const asgart_b200_protosd* r = asgart_b200_result_sds(res);
                for (int64_t f = 0; f < nf; ++f) fam_off.push_back(sds.size() + off[f + 1]);
                sds.insert(sds.end(), r, r + off[nf]);
            }
            asgart_b200_result_free(res);
        }
        if (rc) failf("device pipeline failed: " + last_error());
        else if (!slice) js = asgart_b200_to_json(p, &passes[0], fam_off.data(), int64_t(fam_off.size()) - 1, sds.data());
        else {
            asgart_b200_run_result* rr = asgart_b200_run_result_new(p, &passes[0], fam_off.data(), int64_t(fam_off.size()) - 1, sds.data());
            if (!rr) failf("out of memory");
            else if (asgart_b200_run_result_slice(rr, slice) != ASGART_B200_OK) failf(std::string("asgart-slice options: ") + asgart_b200_run_result_error(rr));
            else js = asgart_b200_run_result_to_json(rr);
            asgart_b200_run_result_free(rr);
        }
    }
    for (asgart_b200_ctx* c : ctxs) asgart_b200_ctx_destroy(c);
    if (p) asgart_b200_prepared_free(p);
    return js;
}

char* asgart_b200_run_files_passes(const char* files, const asgart_b200_settings* passes, int32_t n_passes, int32_t device,
                                   const char** err) {
    return run_files_impl(files, passes, n_passes, &device, 1, nullptr, err);
}

char* asgart_b200_run_files_sliced(const char* files, const asgart_b200_settings* passes, int32_t n_passes, int32_t device,
                                   uint32_t slice_flags, uint64_t min_length, int64_t max_family_members, const char** err) {
    asgart_b200_slice_options op{};
    op.flags = slice_flags; op.min_length = min_length; op.max_family_members = max_family_members;
    return run_files_impl(files, passes, n_passes, &device, 1, &op, err);
}

char* asgart_b200_run_files_sliced_ex(const char* files, const asgart_b200_settings* passes, int32_t n_passes, int32_t device,
                                      const asgart_b200_slice_options* options, const char** err) {
    return run_files_impl(files, passes, n_passes, &device, 1, options, err);
}

char* asgart_b200_run_files_devices(const char* files, const asgart_b200_settings* passes, int32_t n_passes, const int32_t* devices,
                                    int32_t n_devices, const asgart_b200_slice_options* options, const char** err) {
    return run_files_impl(files, passes, n_passes, devices, n_devices, options, err);
}

char* asgart_b200_run_files(const char* files, const asgart_b200_settings* st, int32_t device, const char** err) {
    return asgart_b200_run_files_passes(files, st, 1, device, err);
}

// ---- synthetic genomes ---------------------------------------------------------------------------------
int64_t asgart_b200_synth_length(int32_t config, int32_t part, int64_t scale_n) {
    SynthSpec sp;
    if (!make_spec(config, part, scale_n, 1, 0, 0, sp)) return -1;
    return int64_t(sp.n);
}

int64_t asgart_b200_synth_fragments(int32_t config, int32_t part, int64_t scale_n, char* names_buf, int64_t names_cap, uint64_t* pos,
                                    uint64_t* len, int64_t cap) {
    SynthSpec sp;
    if (!make_spec(config, part, scale_n, 1, 0, 0, sp)) return -1;
    std::string names;
    for (size_t i = 0; i < sp.frags.size(); ++i) {
        names += (i ? "\n" : "") + sp.frags[i].name;
        if (int64_t(i) < cap) { if (pos) pos[i] = sp.frags[i].position; if (len) len[i] = sp.frags[i].length; }
    }
    if (names_buf && names_cap > 0) { strncpy(names_buf, names.c_str(), size_t(names_cap - 1)); names_buf[names_cap - 1] = 0; }
    return int64_t(sp.frags.size());
}

int64_t asgart_b200_synth_fill(int32_t config, int32_t part, int64_t scale_n, uint64_t seed, int64_t n_pairs, int32_t rc_percent,
                               uint8_t* out, int64_t cap, int32_t threads) {
    SynthSpec sp;
    if (!make_spec(config, part, scale_n, seed, n_pairs, rc_percent, sp)) return -1;
    if (!out || cap < int64_t(sp.n)) return -1;
    std::vector<uint8_t> g;
    if (config == 5 && part == 1) {
        SynthSpec sa;
        make_spec(5, 0, scale_n, seed, n_pairs, rc_percent, sa);
        std::vector<uint8_t> a;
        generate(sa, a, threads, nullptr, 0);
        generate(sp, g, threads, &a, scaled(3000, sp.scale, 4));
    } else {
        generate(sp, g, threads, nullptr, 0);
    }
    memcpy(out, g.data(), sp.n);
    return int64_t(sp.n);
}

}  // extern "C"
