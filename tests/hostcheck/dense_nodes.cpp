// dense_nodes.cpp — TEST INFRASTRUCTURE (never linked into the product library).
//
// The single-GPU graph stage numbers its nodes by the dense array of solid k-mers the reduce emits (unipath.cuh: DenseNodes), in
// minimiser order.  These drivers run that stage serially through the same device functions, on top of hostcheck.cpp (included
// whole: its counting, list ranking and graph finishing are reused as they are).
#include "hostcheck.cpp"

namespace {
// The order the reduce emits solid k-mers in (count_part.cuh: k_count_smem): grouped by minimiser partition, inside a partition
// sorted by the sort word's (minimiser bits, offset) — the kernel breaks ties by its shared-memory slot, here by the k-mer.
// Partitions leave in whatever order their CTAs finish: a fixed shuffle of them stands for that.
std::vector<w2rap_kmer_rec> reduce_order(const w2rap_kmer_rec* all, uint64_t n_all, uint32_t min_freq, uint32_t logP) {
    struct Key { uint32_t part, word; uint64_t i; };
    std::vector<Key> keys;
    for (uint64_t i = 0; i < n_all; ++i) {
        if (all[i].count < min_freq) continue;
        uint32_t off;
        const uint32_t mh = kmer_minimizer_offset_words(Kmer{all[i].w0, all[i].w1}, &off);
        const uint32_t part = mini_part(mini_mix(mh), logP);
        keys.push_back(Key{(part * 0x9e3779b1u) ^ (part >> 3), (mh & 0x1fffu) << 6 | off, i});
    }
    std::sort(keys.begin(), keys.end(), [&](const Key& a, const Key& b) {
        if (a.part != b.part) return a.part < b.part;
        if (a.word != b.word) return a.word < b.word;
        return kmer_less(Kmer{all[a.i].w0, all[a.i].w1}, Kmer{all[b.i].w0, all[b.i].w1});
    });
    std::vector<w2rap_kmer_rec> out;
    for (const Key& k : keys) out.push_back(all[k.i]);
    return out;
}
}  // namespace

extern "C" {

// hc_graph with dense node ids: k_insert_solid (+ dense array), k_adjacency_dense, k_links .. k_emit_edges over DenseNodes,
// k_backfill_slots, then the rest exactly as hc_graph.  shuffle != 0: the solid k-mers in a scrambled order instead of the reduce's
// (the order is a locality hint only).  *n_links / *n_near: successor links, and those within +-64 ids of their node.
int hc_graph_dense(const w2rap_kmer_rec* all, uint64_t n_all, uint32_t min_freq, uint32_t logP, int shuffle, const w2rap_reads* in, int want_paths,
                   int apply_fixpaths, uint32_t cap, uint32_t left_cap, w2rap_graph* out, uint64_t* n_links, uint64_t* n_near) {
    memset(out, 0, sizeof(*out));
    std::vector<w2rap_kmer_rec> solid = reduce_order(all, n_all, min_freq, logP);
    if (shuffle)
        for (uint64_t i = solid.size(); i > 1; --i) std::swap(solid[i - 1], solid[(i * 0x9e3779b97f4a7c15ull >> 17) % i]);
    const uint64_t n_solid = solid.size();
    // ---- k_insert_solid
    std::vector<SolidSlot> slots(table_slots_for(n_solid)), dense(n_solid);
    memset(slots.data(), 0xff, slots.size() * sizeof(SolidSlot));
    SolidTable st{slots.data(), slots.size()};
    for (uint64_t i = 0; i < n_solid; ++i) {
        const Kmer k{solid[i].w0, solid[i].w1};
        uint64_t h = st.home(k);
        while (slots[h].w0 != EMPTY_W0) h = st.next(h);
        slots[h] = SolidSlot{k.w0, k.w1, solid[i].ctx, NIL, (uint32_t)i, 0};
        dense[i] = SolidSlot{k.w0, k.w1, solid[i].ctx, NIL, 0, 0};
    }
    out->n_solid = n_solid; out->n_distinct = n_all;
    const DenseNodes dn{st, dense.data(), n_solid};
    const uint64_t nn = 2 * n_solid;
    // ---- k_adjacency_dense
    for (uint64_t i = 0; i < n_solid; ++i) dense[i].ctx = pruned_context(st, Kmer{dense[i].w0, dense[i].w1}, dense[i].ctx & 0xff);
    // ---- k_links, k_rank_*
    std::vector<uint32_t> next0(nn);
    int missing = 0;
    *n_links = 0; *n_near = 0;
    for (uint64_t x = 0; x < nn; ++x) {
        next0[x] = unipath_succ_link(dn, (uint32_t)x, &missing);
        if (next0[x] < EMPTY_NODE) { ++*n_links; const int64_t d = (int64_t)(next0[x] >> 1) - (int64_t)(x >> 1); *n_near += d >= -64 && d <= 64; }
    }
    if (missing) return 101;
    std::vector<RankState> Rv;
    const int64_t ncyc = rank_local(SolidTable{dense.data(), n_solid}, next0, nullptr, Rv);   // (the circle step only reads entries by id)
    if (ncyc < 0) return 102;
    out->timings.count_passes = (uint32_t)ncyc;
    const RankState* R = Rv.data();
    // ---- k_strand_decide, k_collect_heads, sort, k_assign_edges, k_emit_edges
    std::vector<uint8_t> keep(nn, 0);
    for (uint64_t x = 0; x < nn; ++x) if (strand_decide_node(dn, R, (uint32_t)x, keep.data())) return 103;
    struct Head { Kmer k; uint32_t node, n; };
    std::vector<Head> heads;
    for (uint64_t x = 0; x < nn; ++x) if (head_is_kept(dn, R, keep.data(), (uint32_t)x)) heads.push_back(Head{node_kmer(dn, (uint32_t)x), (uint32_t)x, (R[x].y & ~RANK_RESOLVED) + 1u});
    std::sort(heads.begin(), heads.end(), [](const Head& a, const Head& b) { return kmer_less(a.k, b.k); });
    EdgeSet es;
    es.E = heads.size();
    const uint64_t E = es.E;
    std::vector<uint32_t> edge_of_head(nn, NIL);
    es.edge_len.resize(E); es.edge_off.assign(E + 1, 0);
    for (uint64_t i = 0; i < E; ++i) { edge_of_head[heads[i].node] = (uint32_t)i; es.edge_len[i] = heads[i].n + K - 1; es.edge_off[i + 1] = es.edge_off[i] + (es.edge_len[i] + 3) / 4; }
    es.edge_bases.assign(es.edge_off[E] + 32, 0);
    PutBase put{es.edge_bases.data()};
    for (uint64_t x = 0; x < nn; ++x) emit_node(dn, R, edge_of_head.data(), es.edge_off.data(), (uint32_t)x, put);
    // ---- k_backfill_slots
    for (SolidSlot& s : slots)
        if (s.w0 != EMPTY_W0) { const SolidSlot& d = dense[s.off]; s.ctx = d.ctx; s.edge = d.edge; s.off = d.off; }
    return finish_graph(std::vector<PathSlice>{PathSlice{slots.data(), st.size()}}, es, n_solid, in, want_paths, apply_fixpaths, cap, left_cap, out);
}

// The strand-normalised minimiser offset (extract.cuh: kmer_minimizer_offset_words) along every read: a k-mer and its reverse
// complement get the same hash and offset, the hash is kmer_minimizer_hash's, and while the minimiser holds (and occurs once in
// both k-mers) the offset steps by exactly one.  Returns the number of violations; *n_checked / *n_steps: k-mers and steps checked.
uint64_t hc_minimizer_offsets(const w2rap_reads* in, uint64_t* n_checked, uint64_t* n_steps) {
    uint64_t bad = 0, n = 0, ns = 0;
    auto occurrences = [](Kmer k, uint32_t h) {
        const uint64_t lo = rev2(k.w0), hi = rev2(k.w1);
        int c = 0;
        for (int t = 0; t < MINI_W; ++t) {
            const int bit = 2 * t;
            const uint64_t w = bit == 0 ? lo : (bit < 64 ? (lo >> bit) | (hi << (64 - bit)) : hi >> (bit - 64));
            c += mmer_hash_of((uint32_t)w & ((1u << (2 * MINI_M)) - 1u)) == h;
        }
        return c;
    };
    for (uint64_t r = 0; r < in->n_reads; ++r) {
        const uint32_t len = in->len[r];
        if (len < (uint32_t)K) continue;
        const uint8_t* b = in->bases + in->base_off[r];
        uint32_t prev_h = 0, prev_off = 0;
        bool prev_once = false;
        for (uint32_t j = 0; j + K <= len; ++j) {
            const Kmer f = kmer_at(b, j), rc = kmer_rc(f);
            uint32_t of, orc;
            const uint32_t hf = kmer_minimizer_offset_words(f, &of), hr = kmer_minimizer_offset_words(rc, &orc);
            if (hf != hr || of != orc || hf != kmer_minimizer_hash(b, j) || of >= (uint32_t)MINI_W) ++bad;
            const bool once = occurrences(f, hf) == 1;
            if (j > 0 && hf == prev_h && once && prev_once) {
                ++ns;
                if (of + 1 != prev_off && prev_off + 1 != of) ++bad;
            }
            prev_h = hf; prev_off = of; prev_once = once;
            ++n;
        }
    }
    *n_checked = n; *n_steps = ns;
    return bad;
}

}  // extern "C"
