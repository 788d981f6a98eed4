// dense_window.cpp — TEST INFRASTRUCTURE (never linked into the product library).
//
// The single-GPU graph stage as k_adjacency_dense and k_links run it: every neighbour is looked for through the hinted node_find
// (unipath.cuh), first within NODE_WINDOW ids of the node that asks, then in the table.  Built on dense_nodes.cpp (included whole:
// its reduce order and, through it, hostcheck.cpp's list ranking and graph finishing are reused as they are).
#include "dense_nodes.cpp"

namespace {
// DenseNodes as the kernels see it, counting the neighbour lookups and those the window resolves.
struct CountingNodes {
    DenseNodes d;
    uint64_t* n_find;      // [2]: lookups, of which resolved in the window
    uint64_t size() const { return d.n; }
};
SolidSlot& node_entry(const CountingNodes& v, uint64_t id) { return v.d.nodes[id]; }
int64_t node_find(const CountingNodes& v, Kmer k, uint64_t hint) {
    ++v.n_find[0];
    v.n_find[1] += node_find_near(v.d, k, hint) >= 0;
    return node_find(v.d, k, hint);
}
}  // namespace

extern "C" {

// hc_graph_dense with k_adjacency_dense's form of the pruning (pruned_context over the node view, not the table).  win[4]: neighbour
// lookups of the adjacency pruning, of which resolved in the window; the same for the successor links.
int hc_graph_dense_window(const w2rap_kmer_rec* all, uint64_t n_all, uint32_t min_freq, uint32_t logP, int shuffle, const w2rap_reads* in,
                          int want_paths, int apply_fixpaths, uint32_t cap, uint32_t left_cap, w2rap_graph* out, uint64_t* win) {
    memset(out, 0, sizeof(*out));
    win[0] = win[1] = win[2] = win[3] = 0;
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
    const CountingNodes adj{dn, win}, links{dn, win + 2};
    const uint64_t nn = 2 * n_solid;
    // ---- k_adjacency_dense
    for (uint64_t i = 0; i < n_solid; ++i) dense[i].ctx = pruned_context(adj, i, Kmer{dense[i].w0, dense[i].w1}, dense[i].ctx & 0xff);
    // ---- k_links, k_rank_*
    std::vector<uint32_t> next0(nn);
    int missing = 0;
    for (uint64_t x = 0; x < nn; ++x) next0[x] = unipath_succ_link(links, (uint32_t)x, &missing);
    if (missing) return 101;
    std::vector<RankState> Rv;
    const int64_t ncyc = rank_local(SolidTable{dense.data(), n_solid}, next0, nullptr, Rv);
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

}  // extern "C"
