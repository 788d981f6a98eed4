// coverage_sharded.cpp — TEST INFRASTRUCTURE (never linked into the product library).
//
// The coverage lookup of a sharded count (csrc/coverage.cuh) with W ranks simulated serially: the kept k-mers split by owner into W
// indexes as W sharded counts hold them, every rank's tiles run over the positions it owns (the 32 lanes one after the other), and
// the W partial totals merged as the all-reduces merge them.  Also the owner of a sequence position against the owner of its
// canonical k-mer, the function the map and the sharded graph stage route by.
#include <stdint.h>
#include <string.h>

#include <vector>

#include "../../include/w2rap_coverage.h"
#include "../../w2rap-contigger_b200/csrc/coverage.cuh"

using namespace w2r;

static uint32_t owner_of_kmer(Kmer canon, uint32_t logP, uint32_t world) {
    return owner_of_partition(mini_part(mini_mix(kmer_minimizer_hash_words(canon)), logP), logP, world);
}

extern "C" {

// For every k-mer position of every sequence, in order: at[j] = cov_owner_at, of_kmer[j] = the owner of its canonical k-mer.
int hc_owners(const w2rap_seqs* s, uint32_t logP, uint32_t world, uint32_t* at, uint32_t* of_kmer) {
    uint64_t j = 0;
    for (uint64_t i = 0; i < s->n; ++i) {
        const uint8_t* seq = s->bases + s->base_off[i];
        for (uint64_t p = 0; p < cov_kmers_of(s->len[i]); ++p, ++j) {
            Kmer f, r;
            kmer_pair_at(seq, p, &f, &r);
            at[j] = cov_owner_at(seq, p, logP, world);
            of_kmer[j] = owner_of_kmer(kmer_less(r, f) ? r : f, logP, world);
        }
    }
    return 0;
}

// recs: distinct canonical k-mers with their counts (the level-2 dump); those with count >= f0 are kept, each on its owner.
int hc_coverage_sharded(const w2rap_kmer_rec* recs, uint64_t n_recs, uint32_t f0, uint32_t logP, uint32_t world, const w2rap_seqs* s, w2rap_seq_cov* out) {
    std::vector<std::vector<SolidSlot>> slots(world);
    std::vector<uint64_t> n_kept(world, 0);
    for (uint64_t i = 0; i < n_recs; ++i)
        if (recs[i].count >= f0) ++n_kept[owner_of_kmer(Kmer{recs[i].w0, recs[i].w1}, logP, world)];
    for (uint32_t r = 0; r < world; ++r) {
        slots[r].resize(solid_table_slots(n_kept[r]));
        memset(slots[r].data(), 0xff, slots[r].size() * sizeof(SolidSlot));
    }
    for (uint64_t i = 0; i < n_recs; ++i) {
        if (recs[i].count < f0) continue;
        const Kmer k{recs[i].w0, recs[i].w1};
        std::vector<SolidSlot>& sl = slots[owner_of_kmer(k, logP, world)];
        const SolidTable st{sl.data(), sl.size()};
        uint64_t h = st.home(k);
        while (sl[h].w0 != EMPTY_W0) h = st.next(h);
        sl[h] = SolidSlot{k.w0, k.w1, recs[i].count, NIL, 0, 0};
    }
    const uint64_t n = s->n;
    std::vector<uint64_t> tile_base(n + 1, 0);
    for (uint64_t i = 0; i < n; ++i) tile_base[i + 1] = tile_base[i] + cov_tiles_of(s->len[i]);
    // per rank: k_cov_init's totals, then its owned positions tile by tile
    std::vector<w2rap_seq_cov> part((size_t)world * n);
    for (uint32_t r = 0; r < world; ++r) {
        const SolidTable st{slots[r].data(), slots[r].size()};
        w2rap_seq_cov* o = part.data() + (size_t)r * n;
        for (uint64_t i = 0; i < n; ++i) {
            const uint64_t nk = cov_kmers_of(s->len[i]);
            o[i] = w2rap_seq_cov{nk, 0, 0, nk ? 0xffffffffu : 0u, 0};
        }
        for (uint64_t t = 0; t < tile_base[n]; ++t) {
            const uint64_t i = cov_tile_owner(tile_base.data(), n, t);
            const uint64_t lo = (t - tile_base[i]) * COV_TILE, nk = cov_kmers_of(s->len[i]);
            const uint64_t hi = lo + COV_TILE < nk ? lo + COV_TILE : nk;
            CovAcc a = cov_empty();
            for (uint32_t lane = 0; lane < 32; ++lane) cov_merge(&a, cov_tile_lane_owned(st, s->bases + s->base_off[i], lo, hi, lane, logP, world, r));
            o[i].sum += a.sum; o[i].n_absent += a.absent;
            if (a.mn < o[i].min) o[i].min = a.mn;
            if (a.mx > o[i].max) o[i].max = a.mx;
        }
    }
    // the merge: sum and n_absent summed, min by min, max by max
    for (uint64_t i = 0; i < n; ++i) {
        out[i] = part[i];
        for (uint32_t r = 1; r < world; ++r) {
            const w2rap_seq_cov& b = part[(size_t)r * n + i];
            if (b.n_kmers != out[i].n_kmers) return 1;
            out[i].sum += b.sum; out[i].n_absent += b.n_absent;
            if (b.min < out[i].min) out[i].min = b.min;
            if (b.max > out[i].max) out[i].max = b.max;
        }
    }
    return 0;
}

}  // extern "C"
