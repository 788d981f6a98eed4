// coverage.cpp — TEST INFRASTRUCTURE (never linked into the product library).
//
// Runs the per-tile functions of the coverage kernels (csrc/coverage.cuh) serially: the index as k_insert_counts fills it, the
// tile list as the scan makes it, every tile's owner by the kernel's binary search, and the 32 lanes of a warp one after the other,
// merged as the warp reduction and the atomics merge them.
#include <stdint.h>
#include <string.h>

#include <vector>

#include "../../include/w2rap_coverage.h"
#include "../../w2rap-contigger_b200/csrc/coverage.cuh"

using namespace w2r;

extern "C" {

// recs: distinct canonical k-mers with their counts (the level-2 dump); those with count >= f0 are the kept ones.
int hc_coverage(const w2rap_kmer_rec* recs, uint64_t n_recs, uint32_t f0, const w2rap_seqs* s, w2rap_seq_cov* out) {
    uint64_t n_kept = 0;
    for (uint64_t i = 0; i < n_recs; ++i) n_kept += recs[i].count >= f0;
    std::vector<SolidSlot> slots(solid_table_slots(n_kept));
    memset(slots.data(), 0xff, slots.size() * sizeof(SolidSlot));
    const SolidTable st{slots.data(), slots.size()};
    for (uint64_t i = 0; i < n_recs; ++i) {
        if (recs[i].count < f0) continue;
        const Kmer k{recs[i].w0, recs[i].w1};
        uint64_t h = st.home(k);
        while (slots[h].w0 != EMPTY_W0) h = st.next(h);
        slots[h] = SolidSlot{k.w0, k.w1, recs[i].count, NIL, 0, 0};
    }
    const uint64_t n = s->n;
    std::vector<uint64_t> tile_base(n + 1, 0);
    for (uint64_t i = 0; i < n; ++i) {
        tile_base[i + 1] = tile_base[i] + cov_tiles_of(s->len[i]);
        const uint64_t nk = cov_kmers_of(s->len[i]);
        out[i] = w2rap_seq_cov{nk, 0, 0, nk ? 0xffffffffu : 0u, 0};
    }
    for (uint64_t t = 0; t < tile_base[n]; ++t) {
        const uint64_t i = cov_tile_owner(tile_base.data(), n, t);
        if (i >= n || t < tile_base[i] || t >= tile_base[i + 1]) return 1;
        const uint64_t lo = (t - tile_base[i]) * COV_TILE, nk = cov_kmers_of(s->len[i]);
        const uint64_t hi = lo + COV_TILE < nk ? lo + COV_TILE : nk;
        CovAcc a = cov_empty();
        for (uint32_t lane = 0; lane < 32; ++lane) cov_merge(&a, cov_tile_lane(st, s->bases + s->base_off[i], lo, hi, lane));
        out[i].sum += a.sum; out[i].n_absent += a.absent;
        if (a.mn < out[i].min) out[i].min = a.mn;
        if (a.mx > out[i].max) out[i].max = a.mx;
    }
    return 0;
}

}  // extern "C"
