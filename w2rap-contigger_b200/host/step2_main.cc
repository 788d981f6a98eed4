// step2_main.cc — file-level drop-in for step 2: `step2 <out_dir> <prefix> [--min_freq F[,F2,...]] [--min_qual Q] [--device D] [--gfa]`
// reads <out_dir>/frag_reads_orig.fastb/.qualp (what `w2rap-contigger --to_step 1` leaves, w2rap-contigger.cc:315-316),
// writes <out_dir>/<prefix>.small_K.hbv, .small_K.paths (post-FixPaths) and small_K.freqs, after which
// `w2rap-contigger -o <out_dir> -p <prefix> --from_step 3` continues (w2rap-contigger.cc:352-358).
// With a list of min_freq values the reads are read, uploaded and counted once (keep floor = the smallest value,
// include/w2rap_step2_counts.h), small_K.freqs is written once, and every value F gets its own graph and paths,
// <prefix>_mf<F>.small_K.hbv / .small_K.paths, continued by `w2rap-contigger -o <out_dir> -p <prefix>_mf<F> --from_step 3`.
// --gfa: also the graph as GFA with per-edge k-mer coverage (include/w2rap_coverage.h) next to each .hbv, <prefix>.small_K.gfa or
// <prefix>_mf<F>.small_K.gfa.  The counts must stay resident for that, so even one value goes through one count and one build.
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "w2rap_step2.h"
#include "w2rap_coverage.h"

// "3,4,5" -> {3, 4, 5}; false on anything that is not a comma-separated list of integers in 1..255
static bool parse_min_freqs(const char* s, std::vector<uint32_t>* out) {
    out->clear();
    while (*s) {
        char* end = nullptr;
        const long v = strtol(s, &end, 10);
        if (end == s || v < 1 || v > 255 || (*end && *end != ',')) return false;
        out->push_back((uint32_t)v);
        s = *end ? end + 1 : end;
        if (*end && !*s) return false;
    }
    return !out->empty();
}

// The graph as GFA, KC/DP from the coverage of its edges in the counts.
static int write_gfa(const std::string& path, const w2rap_counts* counts, const w2rap_graph& g, char* err, size_t errlen) {
    const w2rap_seqs edges = {g.n_edges, g.edge_bases, g.edge_off, g.edge_len};
    std::vector<w2rap_seq_cov> cov(g.n_edges);
    int rc = w2rap_counts_coverage(counts, &edges, cov.data(), nullptr, err, errlen);
    if (rc == W2RAP_OK) rc = w2rap_write_gfa(path.c_str(), &g, cov.data(), err, errlen);
    return rc;
}

// one count, one build per value of `freqs` (in the order given); `gfa`: also <base>.gfa
static int run_sweep(const char* dir, const char* prefix, w2rap_params p, const std::vector<uint32_t>& freqs, bool gfa, char* err, size_t errlen) {
    const std::string d(dir);
    w2rap_reads r;
    int rc = w2rap_read_fastb_qualp((d + "/frag_reads_orig.fastb").c_str(), (d + "/frag_reads_orig.qualp").c_str(), &r, err, errlen);
    if (rc) return rc;
    w2rap_device_reads* reads = nullptr;
    rc = w2rap_step2_upload(&r, p.device, &reads, err, errlen);
    // w2rap_reads from w2rap_read_fastb_qualp are malloc'ed
    free((void*)r.bases); free((void*)r.quals); free((void*)r.base_off); free((void*)r.qual_off); free((void*)r.len);
    if (rc) return rc;
    p.want_paths = 1; p.apply_fixpaths = 1;        // the files hold post-FixPaths paths (w2rap-contigger.cc:340-346)
    p.min_freq = *std::min_element(freqs.begin(), freqs.end());
    p.workdir = dir;                               // small_K.freqs, once
    w2rap_counts* counts = nullptr;
    w2rap_graph spectrum;
    rc = w2rap_step2_count(reads, &p, &counts, &spectrum, err, errlen);
    if (rc == W2RAP_OK) {
        printf("TIME, count (B200), %.3f\n", spectrum.timings.total_ms * 1e-3);
        w2rap_step2_free(&spectrum);
    }
    p.workdir = nullptr;
    for (size_t i = 0; i < freqs.size() && rc == W2RAP_OK; ++i) {
        p.min_freq = freqs[i];
        w2rap_graph g;
        rc = w2rap_step2_build(reads, counts, &p, &g, err, errlen);
        if (rc) break;
        const std::string base = d + "/" + prefix + (freqs.size() > 1 ? "_mf" + std::to_string(freqs[i]) : std::string()) + ".small_K";
        rc = w2rap_write_hbv((base + ".hbv").c_str(), &g, err, errlen);
        if (rc == W2RAP_OK) rc = w2rap_write_paths((base + ".paths").c_str(), &g, err, errlen);
        if (rc == W2RAP_OK && gfa) rc = write_gfa(base + ".gfa", counts, g, err, errlen);
        if (rc == W2RAP_OK) printf("TIME, build min_freq %u +FixPaths (B200), %.3f\n", freqs[i], g.timings.total_ms * 1e-3);
        w2rap_step2_free(&g);
    }
    w2rap_step2_counts_release(counts);
    w2rap_step2_release(reads);
    return rc;
}

int main(int argc, char** argv) {
    if (argc < 3) { fprintf(stderr, "usage: %s <out_dir> <prefix> [--min_freq F[,F2,...]] [--min_qual Q] [--device D] [--gfa] [--quiet]\n", argv[0]); return 2; }
    w2rap_params p;
    memset(&p, 0, sizeof p);
    p.abi_version = W2RAP_STEP2_ABI_VERSION; p.K = W2RAP_K; p.min_qual = 7; p.min_freq = 4; p.device = -1; p.verbose = 1;
    std::vector<uint32_t> freqs = {4};
    bool gfa = false;
    for (int i = 3; i < argc; ++i) {
        if (!strcmp(argv[i], "--min_freq") && i + 1 < argc) {
            ++i;
            if (!strchr(argv[i], ',')) freqs.assign(1, (uint32_t)atoi(argv[i]));        // one value: checked by the library, as always
            else if (!parse_min_freqs(argv[i], &freqs)) { fprintf(stderr, "--min_freq takes integers in 1..255, separated by commas: %s\n", argv[i]); return 2; }
        }
        else if (!strcmp(argv[i], "--min_qual") && i + 1 < argc) p.min_qual = (uint32_t)atoi(argv[++i]);
        else if (!strcmp(argv[i], "--device") && i + 1 < argc) p.device = atoi(argv[++i]);
        else if (!strcmp(argv[i], "--gfa")) gfa = true;
        else if (!strcmp(argv[i], "--quiet")) p.verbose = 0;
        else { fprintf(stderr, "unknown argument %s\n", argv[i]); return 2; }
    }
    char err[1024] = {0};
    if (freqs.size() > 1 || gfa) {
        int rc = run_sweep(argv[1], argv[2], p, freqs, gfa, err, sizeof err);
        if (rc) { fprintf(stderr, "step2 failed (%d): %s\n", rc, err); return 1; }
        return 0;
    }
    p.min_freq = freqs[0];
    w2rap_graph g;
    int rc = w2rap_step2_run_files(argv[1], argv[2], &p, &g, err, sizeof err);
    if (rc) { fprintf(stderr, "step2 failed (%d): %s\n", rc, err); return 1; }   // the reference exits non-zero on any failure
    printf("TIME, buildReadQGraph+FixPaths (B200), %.3f\n", g.timings.total_ms * 1e-3);
    w2rap_step2_free(&g);
    return 0;
}
