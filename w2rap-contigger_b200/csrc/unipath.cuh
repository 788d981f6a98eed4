// unipath.cuh — unipath (edge) structure over the solid k-mer table, restated for data-parallel execution.
//
// The reference walks edges serially from their ends (EdgeBuilder, paths/long/BuildReadQGraph.cc:99-339).  Here every
// solid k-mer is two ORIENTED nodes, node id = 2*id + o (o = 1: the node spells rc(key[id]); DenseNodes below says what an id is).  A successor link
// x -> n exists iff the reference's walk would step from x to n:
//     x is not a palindrome, x has exactly one successor n, n is not a palindrome, n has exactly one predecessor
//     (extend(): :234-246; the same test seen from n is upstreamExtensionPossible(): :192-202).
// Links pair up under reverse complement (x -> n  <=>  rc(n) -> rc(x)), so the oriented nodes form disjoint simple paths
// and cycles; each unipath appears twice (once per strand) and the strand whose sequence is FWD/PALINDROME under
// dna/CanonicalForm.h:34-46 is the one the reference keeps (:247-258).  Pure cycles are the reference's "smooth circles"
// (:126-180): cut so that the strand through the minimum canonical k-mer in FWD orientation starts there, then treated
// exactly like a path (addEdge() re-applies the canonical-form flip, :278-281).
#pragma once
#include "kmer.cuh"

namespace w2r {

constexpr uint32_t RANK_RESOLVED = 0x80000000u;
constexpr uint32_t EMPTY_NODE = 0xfffffffeu;   // next0[] of a node whose slot holds no k-mer
constexpr uint32_t GHOST_TAIL = 0xfffffffdu;   // next0[] of a GHOST node (sharded graph stage, shardgraph.cuh): a copy of a k-mer another
                                               // rank owns.  A node whose successor is a ghost is the tail of its LOCAL chain piece.
W2R_HD bool slot_is_ghost(const SolidSlot& s) { return s.pad != 0; }      // pad = owner rank + 1, edge = slot on the owner

// How nodes are numbered: oriented node = 2*id + o, and a node view maps an id to its entry (k-mer, context, edge, offset) and a
// canonical k-mer to its id.  Both views probe the same hash table for neighbours.
//   SolidTable : id = slot of the table.  The sharded graph stage numbers its nodes so (its ghosts live in the local table).
//   DenseNodes : id = index in the dense array of solid k-mers, in the order the reduce emitted them: grouped by minimiser and
//                sorted by the minimiser's place (count_part.cuh), so the k-mers of a chain mostly get neighbouring ids and a chain
//                step stays inside a sector or two.  The table's `off` field holds every key's id until the graph stage ends.
// node_find(view, canonical k-mer, hint) -> id or -1.  `hint` is the id of the node asking.  DenseNodes first compares the keys within
// NODE_WINDOW ids of it, nearest first: a neighbour along a chain mostly sits there, in lines the warp has just read, and only a miss
// pays the dependent probe chain in the table plus the read of the slot's `off`.  A window hit is a full key comparison, so the answer
// is the same in any id order.  SolidTable ignores the hint (its ids are hash-placed slots).
constexpr int NODE_WINDOW = 4;
struct DenseNodes {
    SolidTable t;
    SolidSlot* nodes;
    uint64_t n;
    W2R_HD uint64_t size() const { return n; }
};
W2R_HD SolidSlot& node_entry(const SolidTable& t, uint64_t id) { return t.slots[id]; }
W2R_HD SolidSlot& node_entry(const DenseNodes& d, uint64_t id) { return d.nodes[id]; }
W2R_HD int64_t node_find(const SolidTable& t, Kmer k, uint64_t) { return solid_find(t, k); }
W2R_HD bool node_key_is(const DenseNodes& d, uint64_t j, Kmer k) {
#if defined(__CUDA_ARCH__)
    const ulonglong2 kk = __ldg(reinterpret_cast<const ulonglong2*>(d.nodes + j));
    return kk.x == k.w0 && kk.y == k.w1;
#else
    return d.nodes[j].w0 == k.w0 && d.nodes[j].w1 == k.w1;
#endif
}
// The window part alone: id of k within NODE_WINDOW ids of hint (hint itself included: a k-mer can be its own neighbour), or -1.
W2R_HD int64_t node_find_near(const DenseNodes& d, Kmer k, uint64_t hint) {
    if (node_key_is(d, hint, k)) return (int64_t)hint;
#pragma unroll
    for (int r = 1; r <= NODE_WINDOW; ++r) {
        if (hint + r < d.n && node_key_is(d, hint + r, k)) return (int64_t)(hint + r);
        if (hint >= (uint64_t)r && node_key_is(d, hint - r, k)) return (int64_t)(hint - r);
    }
    return -1;
}
W2R_HD int64_t node_find(const DenseNodes& d, Kmer k, uint64_t hint) {
    const int64_t j = node_find_near(d, k, hint);
    if (j >= 0) return j;
    const int64_t s = solid_find(d.t, k);
    return s < 0 ? -1 : (int64_t)d.t.slots[s].off;
}

template <class V>
W2R_HD Kmer node_kmer(const V& v, uint32_t x) {
    const SolidSlot& s = node_entry(v, x >> 1);
    Kmer k{s.w0, s.w1};
    return (x & 1u) ? kmer_rc(k) : k;
}

// Successor link of oriented node x, or NIL.  *missing is set if a neighbour that the pruned context promises is absent
// (the reference would ForceAssert, :265).
// *to_ghost (optional) is set if the successor is a ghost node.
template <class V>
W2R_HD uint32_t unipath_succ_link(const V& t, uint32_t x, int* missing, bool* to_ghost = nullptr) {
    const SolidSlot& s = node_entry(t, x >> 1);
    if (to_ghost) *to_ghost = false;
    if (s.w0 == EMPTY_W0) return EMPTY_NODE;
    if (slot_is_ghost(s)) return GHOST_TAIL;
    Kmer k{s.w0, s.w1};
    Kmer rc = kmer_rc(k);
    if (rc == k) return NIL;                                   // :105 palindromes are one-k-mer edges
    const bool o = x & 1u;
    Kmer xk = o ? rc : k;
    uint32_t c = o ? ctx_rc(s.ctx & 0xffu) : (s.ctx & 0xffu);
    if (nib_count(c) != 1) return NIL;                          // :236
    Kmer n = kmer_succ(xk, nib_single(c));
    Kmer nrc = kmer_rc(n);
    if (nrc == n) return NIL;                                   // :239
    bool rev = kmer_less(nrc, n);
    int64_t ts = node_find(t, rev ? nrc : n, x >> 1);
    if (ts < 0) { if (missing) *missing = 1; return NIL; }
    uint32_t c2 = node_entry(t, ts).ctx & 0xffu;
    if (rev) c2 = ctx_rc(c2);
    if (nib_count(c2 >> 4) != 1) return NIL;                    // :242
    if (to_ghost) *to_ghost = slot_is_ghost(node_entry(t, ts));
    return (uint32_t)(2 * ts) + (rev ? 1u : 0u);
}

// kmers/ReadPather.h:317-346 AdjProc for one entry: clear every context bit whose neighbour k-mer is not in the dictionary.
// id = the entry's node id (the hint of node_find).
template <class V>
W2R_HD bool node_has(const V& v, Kmer k, uint64_t id) {
    const Kmer r = kmer_rc(k);
    return node_find(v, kmer_less(r, k) ? r : k, id) >= 0;
}
template <class V>
W2R_HD uint32_t pruned_context(const V& v, uint64_t id, Kmer k, uint32_t c) {
    for (uint32_t b = 0; b < 4; ++b)
        if (c & (1u << b)) { if (!node_has(v, kmer_succ(k, b), id)) c &= ~(1u << b); }
    for (uint32_t b = 0; b < 4; ++b)
        if (c & (16u << b)) { if (!node_has(v, kmer_pred(k, b), id)) c &= ~(16u << b); }
    return c;
}
W2R_HD uint32_t pruned_context(const SolidTable& t, Kmer k, uint32_t c) { return pruned_context(t, 0, k, c); }


// ---------------------------------------------------------------- list ranking by pointer jumping
// Rank state per oriented node: x = pointer, y = distance | RANK_RESOLVED.  A tail (no successor) is a resolved fixed point
// (x = itself, distance 0); a resolved node points at its tail with its exact distance.
struct alignas(8) RankState { uint32_t x, y; };

W2R_HD RankState rank_init_node(const uint32_t* next0, uint32_t x) {
    uint32_t nx = next0[x];
    return nx >= GHOST_TAIL ? RankState{x, RANK_RESOLVED} : RankState{nx, 1u};
}

// ---- list ranking with splitters (Helman-JaJa): O(N) work instead of O(N log N) pointer jumping over every node.
// A node is a splitter if it heads a strand path or if a hash of its id says so (about 1 in 64).  Each splitter walks
// its successors up to the next splitter, labelling every node it passes with (splitter, steps from it); the splitters
// alone are then ranked by pointer jumping; finally every node derives (tail, distance to tail) from its splitter's.
// Nodes of cycles that contain no splitter stay unlabelled; splitters on a cycle never resolve: both are "circle" nodes.
constexpr uint32_t SPLITTER_MASK = 63u;
W2R_HD bool hash_splitter(uint32_t x) { uint32_t h = x * 0x9e3779b1u; h ^= h >> 15; h *= 0x85ebca77u; h ^= h >> 13; return (h & SPLITTER_MASK) == 0; }
// ghead (may be null): ghead[x] != 0 marks a node whose PREDECESSOR is a ghost: the head of a local chain piece.
W2R_HD bool node_is_splitter(const uint32_t* next0, const uint8_t* ghead, uint32_t x) {
    const uint32_t nx = next0[x];
    if (nx == EMPTY_NODE || nx == GHOST_TAIL) return false;
    return next0[x ^ 1u] == NIL || (ghead && ghead[x]) || hash_splitter(x);
}
// label[] must be initialised to {NIL, 0}.  Writes label[y] for every node of the segment and the splitter's own state S[s].
// A chain ends at a node without successor or at a node whose successor is a ghost (next0[next0[y]] == GHOST_TAIL).
W2R_HD void splitter_walk(const uint32_t* next0, uint32_t s, RankState* label, RankState* S) {
    uint32_t y = s, o = 0, ny = next0[s];
    for (;;) {
        label[y] = RankState{s, o};
        if (ny == NIL) { S[s] = RankState{y, o | RANK_RESOLVED}; return; }          // reached the tail: resolved
        const uint32_t nny = next0[ny];
        if (nny == GHOST_TAIL) { S[s] = RankState{y, o | RANK_RESOLVED}; return; }  // the chain goes on on another rank: local tail
        ++o;
        if (hash_splitter(ny) || ny == s) { S[s] = RankState{ny, o}; return; }       // next splitter (ny == s: a cycle with one splitter)
        y = ny; ny = nny;
    }
}
// After the splitters are ranked: node y -> (tail, distance to tail | RESOLVED), or unresolved if y lies on a circle.
W2R_HD RankState splitter_finish_node(const uint32_t* next0, const RankState* label, const RankState* S, uint32_t y) {
    if (next0[y] == EMPTY_NODE || next0[y] == GHOST_TAIL) return RankState{y, RANK_RESOLVED};
    RankState l = label[y];
    if (l.x == NIL) return RankState{y, 0};                                          // never labelled: a circle without splitter
    RankState st = S[l.x];
    if (!(st.y & RANK_RESOLVED)) return RankState{y, 0};                             // its splitter sits on a circle
    return RankState{st.x, ((st.y & ~RANK_RESOLVED) - l.y) | RANK_RESOLVED};
}
W2R_HD RankState rank_step_node(const RankState* A, uint32_t x, bool* unresolved) {
    RankState a = A[x];
    *unresolved = false;
    if (!(a.y & RANK_RESOLVED)) {
        RankState b = A[a.x];
        a = RankState{b.x, (a.y + (b.y & ~RANK_RESOLVED)) | (b.y & RANK_RESOLVED)};
        *unresolved = !(a.y & RANK_RESOLVED);
    }
    return a;
}
// Smooth circles: state = (jump pointer, id of the minimum canonical k-mer seen so far).
template <class V>
W2R_HD RankState cycle_step_node(const V& t, const RankState* A, uint32_t x, bool* changed) {
    RankState a = A[x], b = A[a.x];
    uint32_t best = a.y;
    if (b.y != a.y) {
        const SolidSlot& sa = node_entry(t, a.y); const SolidSlot& sb = node_entry(t, b.y);
        if (kmer_less(Kmer{sb.w0, sb.w1}, Kmer{sa.w0, sa.w1})) best = b.y;
    }
    *changed = best != a.y;
    return RankState{b.x, best};
}
// Cut both strand cycles at the minimum k-mer (BuildReadQGraph.cc:156-180): (kmin,+) becomes a head, (kmin,-) a tail.
W2R_HD void cycle_cut_node(const RankState* A, uint32_t* next0, uint32_t x) {
    if ((x & 1u) == 0 && A[x].y == (x >> 1)) {
        uint32_t y = next0[x ^ 1u];          // successor of (kmin,-); its flip is the predecessor of (kmin,+)
        next0[y ^ 1u] = NIL;
        next0[x ^ 1u] = NIL;
    }
}
// Strand selection (dna/CanonicalForm.h:34-46, BuildReadQGraph.cc:247-258): R[x] = (tail, distance to tail); keep[] is indexed
// by the head node of a strand path.  Returns true if the strand is longer than KDef's 24-bit offset allows.
template <class V>
W2R_HD bool strand_decide_node(const V& t, const RankState* R, uint32_t x, uint8_t* keep) {
    if (node_entry(t, x >> 1).w0 == EMPTY_W0) return false;
    RankState a = R[x], f = R[x ^ 1u];
    uint32_t d = a.y & ~RANK_RESOLVED, off = f.y & ~RANK_RESOLVED;
    uint64_t n = (uint64_t)d + off + 1;
    uint32_t head = f.x ^ 1u;
    uint64_t L = n + K - 1;
    if (L & 1) {                                         // odd length: the middle base alone decides
        uint64_t m = L / 2, ostar = m < n - 1 ? m : n - 1;
        if (off == ostar) keep[head] = (kmer_base(node_kmer(t, x), (int)(m - off)) & 2u) ? 0 : 1;
    } else if (off == 0) {                               // even length: compare with the reverse complement, outside in;
        Kmer hk = node_kmer(t, x);                       // the first 60 bases always differ unless it is a palindromic 1-k-mer edge
        Kmer ok = node_kmer(t, a.x ^ 1u);
        keep[x] = (kmer_less(hk, ok) || (hk == ok && (x & 1u) == 0)) ? 1 : 0;
    }
    return off == 0 && n > 0x1000000ull;                 // offsets must fit KDef's 24 bits (kmers/ReadPather.h:121-122,144)
}
template <class V>
W2R_HD bool head_is_kept(const V& t, const RankState* R, const uint8_t* keep, uint32_t x) {
    return node_entry(t, x >> 1).w0 != EMPTY_W0 && (R[x ^ 1u].y & ~RANK_RESOLVED) == 0 && keep[x];
}
// Edge emission + KDef back-fill for one node (BuildReadQGraph.cc:287-301).  put(edge byte offset, base position, base code).
template <class V, class Put>
W2R_HD void emit_node(const V& t, const RankState* R, const uint32_t* edge_of_head, const uint64_t* edge_off, uint32_t x, Put& put) {
    SolidSlot* s = &node_entry(t, x >> 1);
    if (s->w0 == EMPTY_W0) return;
    RankState f = R[x ^ 1u];
    uint32_t e = edge_of_head[f.x ^ 1u];
    if (e == NIL) return;
    uint32_t off = f.y & ~RANK_RESOLVED;
    s->edge = e; s->off = off;
    Kmer k = node_kmer(t, x);
    uint64_t bo = edge_off[e];
    put(bo, (uint64_t)off, kmer_first(k));
    if ((R[x].y & ~RANK_RESOLVED) == 0)
        for (int i = 1; i < K; ++i) put(bo, (uint64_t)off + i, kmer_base(k, i));
}

// ---------------------------------------------------------------- HBV end keys (paths/long/HBVFromEdges.cc:18-49)
// End w of an edge: 0 fwd-left, 1 fwd-right, 2 rc-left, 3 rc-right.  Key order = (FNV-1a 64 over the 59 base codes as bytes
// (math/Hash.h:26-35), then the bases).  Returns false for the rc ends of a palindromic edge (they do not exist, :91-97).
struct EndKey { uint64_t h, k0, k1; };
W2R_HD bool edge_end_key(const uint8_t* p, uint32_t len, uint32_t w, bool* is_pal, EndKey* out) {
    bool pal = false;
    if (len == (uint32_t)K) {                                  // only a 1-k-mer edge can be a palindrome
        uint64_t w0 = 0, w1 = 0;
        for (int i = 0; i < 32; ++i) w0 = (w0 << 2) | packed_base(p, i);
        for (int i = 32; i < K; ++i) w1 = (w1 << 2) | packed_base(p, i);
        pal = kmer_is_palindrome(Kmer{w0, w1 << 8});
    }
    *is_pal = pal;
    if (pal && w >= 2) { *out = EndKey{~0ull, ~0ull, ~0ull}; return false; }
    bool rc = w >= 2, distal = w & 1u;
    uint64_t start = distal ? len - (K - 1) : 0;
    uint64_t h = 14695981039346656037ull, a = 0, b = 0;
    for (int i = 0; i < K - 1; ++i) {
        uint64_t pos = start + i;
        uint32_t c = rc ? 3u - packed_base(p, len - 1 - pos) : packed_base(p, pos);
        h = 1099511628211ull * (h ^ (uint64_t)c);
        if (i < 32) a = (a << 2) | c; else b = (b << 2) | c;
    }
    *out = EndKey{h, a, b << 10};
    return true;
}

}  // namespace w2r
