// cli.cpp — `asgart-b200 FILES... [flags]`: the command line of src/bin/asgart.rs:564-631 for the duplication-search
// path, driving the device operator through the C ABI and writing the same JSON file the reference writes
// (naming rule src/bin/asgart.rs:695-719).
#include <cstdio>
#include <cstdlib>
#include <algorithm>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/asgart_b200.h"

static void usage() {
    fprintf(stderr,
            "Usage: asgart-b200 [OPTIONS] [STRANDS]...\n"
            "  -k, --probe-size <N>        Probing k-mers size [default: 20]\n"
            "  -g, --gap-size <N>          Maximum length of a gap [default: 100]\n"
            "      --min-length <N>        Minimal length (in bp) of the duplications to be reported [default: 1000]\n"
            "      --max-cardinality <N>   maximal cardinality of duplication families [default: 500]\n"
            "  -R, --reverse               Search for reversed duplications\n"
            "  -C, --complement            Search for complemented duplications\n"
            "  -S, --skip-masked           Ignore soft-masked repeated zones (lowercased regions)\n"
            "      --trim <START> <STOP>   Trim the first strand: only duplications whose right arm lies in [START, STOP) are searched\n"
            "      --prefix <P>            prefix to prepend to the default output file name\n"
            "      --out <FILE>            set the output file name\n"
            "      --no-direct --no-reversed --no-uncomplemented --no-complemented --no-inter --no-intra\n"
            "      --slice-min-length <N> --max-family-members <N>\n"
            "                              asgart-slice's duplicon filters, applied before the file is written\n"
            "      --collapse --no-inter-relaxed\n"
            "      --keep-fragments <A,B,..> --restrict-fragments <A,B,..> --exclude-fragments <A,B,..> [--regexp]\n"
            "                              asgart-slice's fragment options (they rewrite the fragment map)\n"
            "      --device <N>            CUDA device [default: 0]\n"
            "      --devices <A,B,..>      run on several CUDA devices at once (a device may repeat); not with --device or --trim\n"
            "      --with-direct           (with -R/-C) also run the direct pass on the same index and write both, combined as\n"
            "                              `asgart-slice` combines the two runs' files\n"
            "      --threads, --chunk-size accepted and ignored (the reference ignores --chunk-size too)\n"
            "  -v                          verbose\n");
}

int main(int argc, char** argv) {
    asgart_b200_settings st{};
    st.probe_size = 20; st.min_duplication_length = 1000; st.max_cardinality = 500;
    uint64_t gap = 100;
    std::string prefix, out;
    std::vector<std::string> files;
    int device = 0, verbose = 0, with_direct = 0;
    bool have_device = false;
    std::vector<int32_t> devices;
    uint32_t slice_flags = 0;
    uint64_t slice_min = 0;
    long long slice_max = -1;
    bool slice = false;
    std::string keep_f, restrict_f, exclude_f;
    bool have_keep = false, have_restrict = false, have_exclude = false;
    auto commas = [](std::string v) { for (char& c : v) if (c == ',') c = '\n'; return v; };
    auto need = [&](int& i) -> const char* { if (i + 1 >= argc) { usage(); exit(2); } return argv[++i]; };
    for (int i = 1; i < argc; ++i) {
        std::string a = argv[i];
        if (a == "-k" || a == "--probe-size") st.probe_size = strtoull(need(i), nullptr, 10);
        else if (a == "-g" || a == "--gap-size") gap = strtoull(need(i), nullptr, 10);
        else if (a == "--min-length") st.min_duplication_length = strtoull(need(i), nullptr, 10);
        else if (a == "--max-cardinality") st.max_cardinality = strtoull(need(i), nullptr, 10);
        else if (a == "--prefix") prefix = need(i);
        else if (a == "--out") out = need(i);
        else if (a == "--device") { device = atoi(need(i)); have_device = true; }
        else if (a == "--devices") {
            devices.clear();
            const std::string v = need(i);
            for (size_t b = 0; b <= v.size();) {
                const size_t e = std::min(v.find(',', b), v.size());
                const std::string d = v.substr(b, e - b);
                char* end = nullptr;
                const long n = strtol(d.c_str(), &end, 10);
                if (d.empty() || *end || n < 0) { usage(); return 2; }
                devices.push_back(int32_t(n));
                b = e + 1;
            }
        }
        else if (a == "--threads" || a == "--chunk-size") need(i);
        else if (a == "--compute-score") st.compute_score = 1;
        else if (a == "--with-direct") with_direct = 1;
        else if (a == "--no-direct") { slice = true; slice_flags |= ASGART_B200_SLICE_NO_DIRECT; }
        else if (a == "--no-reversed") { slice = true; slice_flags |= ASGART_B200_SLICE_NO_REVERSED; }
        else if (a == "--no-uncomplemented") { slice = true; slice_flags |= ASGART_B200_SLICE_NO_UNCOMPLEMENTED; }
        else if (a == "--no-complemented") { slice = true; slice_flags |= ASGART_B200_SLICE_NO_COMPLEMENTED; }
        else if (a == "--no-inter") { slice = true; slice_flags |= ASGART_B200_SLICE_NO_INTER; }
        else if (a == "--no-intra") { slice = true; slice_flags |= ASGART_B200_SLICE_NO_INTRA; }
        else if (a == "--slice-min-length") { slice = true; slice_flags |= ASGART_B200_SLICE_MIN_LENGTH; slice_min = strtoull(need(i), nullptr, 10); }
        else if (a == "--max-family-members") { slice = true; slice_max = atoll(need(i)); }
        else if (a == "--collapse") { slice = true; slice_flags |= ASGART_B200_SLICE_COLLAPSE; }
        else if (a == "--no-inter-relaxed") { slice = true; slice_flags |= ASGART_B200_SLICE_NO_INTER_RELAXED; }
        else if (a == "--regexp") { slice_flags |= ASGART_B200_SLICE_REGEXP; }
        else if (a == "--keep-fragments") { slice = true; have_keep = true; keep_f = commas(need(i)); }
        else if (a == "--restrict-fragments") { slice = true; have_restrict = true; restrict_f = commas(need(i)); }
        else if (a == "--exclude-fragments") { slice = true; have_exclude = true; exclude_f = commas(need(i)); }
        else if (a == "--trim") { st.has_trim = 1; st.trim_a = strtoull(need(i), nullptr, 10); st.trim_b = strtoull(need(i), nullptr, 10); }
        else if (a == "-h" || a == "--help") { usage(); return 0; }
        else if (a == "--reverse") st.reverse = 1;
        else if (a == "--complement") st.complement = 1;
        else if (a == "--skip-masked") st.skip_masked = 1;
        else if (a.size() > 1 && a[0] == '-' && a[1] != '-') {  // clustered short flags: -RCSv
            for (size_t j = 1; j < a.size(); ++j) {
                if (a[j] == 'R') st.reverse = 1; else if (a[j] == 'C') st.complement = 1; else if (a[j] == 'S') st.skip_masked = 1;
                else if (a[j] == 'v') ++verbose; else { usage(); return 2; }
            }
        }
        else if (a[0] == '-') { usage(); return 2; }
        else files.push_back(a);
    }
    if (files.empty() || (have_device && !devices.empty())) { usage(); return 2; }
    if (devices.empty()) devices.push_back(device);
    st.max_gap_size = uint32_t(gap + st.probe_size);  // src/bin/asgart.rs:681
    std::string joined;
    for (size_t i = 0; i < files.size(); ++i) joined += (i ? "\n" : "") + files[i];
    const char* err = nullptr;
    asgart_b200_settings passes[2] = {st, st};
    passes[1].reverse = passes[1].complement = 0;
    const int n_passes = (with_direct && (st.reverse || st.complement)) ? 2 : 1;
    asgart_b200_slice_options op{};
    op.flags = slice_flags; op.min_length = slice_min; op.max_family_members = slice_max;
    op.keep_fragments = have_keep ? keep_f.c_str() : nullptr;
    op.restrict_fragments = have_restrict ? restrict_f.c_str() : nullptr;
    op.exclude_fragments = have_exclude ? exclude_f.c_str() : nullptr;
    char* js = asgart_b200_run_files_devices(joined.c_str(), passes, n_passes, devices.data(), int32_t(devices.size()),
                                             slice ? &op : nullptr, &err);
    if (!js) { fprintf(stderr, "asgart-b200: %s\n", err ? err : "failed"); return 1; }
    char* name = asgart_b200_out_filename(joined.c_str(), prefix.c_str(), out.empty() ? nullptr : out.c_str(), &st);
    FILE* f = fopen(name, "wb");
    if (!f) { fprintf(stderr, "Unable to create `%s`\n", name); return 1; }
    fwrite(js, 1, strlen(js), f);
    fclose(f);
    if (verbose) fprintf(stderr, "Result written to %s\n", name);
    asgart_b200_free_string(js);
    asgart_b200_free_string(name);
    return 0;
}
