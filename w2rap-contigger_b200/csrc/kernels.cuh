// kernels.cuh — the sm_100a kernels of the step-2 path (device code only).
//
// K1 k_good_len                    : PQVec quality floor (count_part.cuh: k_minimizer_map = k-mer extraction + partition by minimiser)
// K2 k_count_smem, k_count_region / k_scan_region (count_part.cuh) : count per partition in shared memory / in an L2-resident
//    region, histogram, min-frequency filter; k_insert_solid
// K3 k_adjacency_dense / k_adjacency : recomputeAdjacencies (over the dense nodes of one GPU / the local table of a sharded run)
// K4 k_links / k_rank_* / k_cycle_* / k_strand_decide / k_collect_heads / k_assign_edges / k_emit_edges / k_backfill_slots : unipaths
// K5 k_edge_ends / k_vertex_* / k_hbv_edges / k_adj_* : HBV vertices + incidence
// K6 k_path_reads / k_path_gather : read pathing (+FixPaths)
#pragma once
#include "extract.cuh"
#include "kmer.cuh"
#include "path.cuh"
#include "pqvec.cuh"
#include "rt.cuh"
#include "unipath.cuh"

namespace w2r {

struct ReadsView {
    uint64_t n;
    const uint8_t* bases;
    const uint64_t* base_off;
    const uint32_t* len;
    const uint8_t* quals;
    const uint64_t* qual_off;
};

struct U128 { uint64_t lo, hi; };

// 128-bit compare-and-swap on a 16-byte aligned global address (ATOMG.E.CAS.128 on sm_100a).
__device__ __forceinline__ U128 cas128(void* addr, uint64_t cmp_lo, uint64_t cmp_hi, uint64_t val_lo, uint64_t val_hi) {
    U128 old;
    asm volatile(
        "{\n\t.reg .b128 c, v, o;\n\t"
        "mov.b128 c, {%2, %3};\n\t"
        "mov.b128 v, {%4, %5};\n\t"
        "atom.global.relaxed.gpu.cas.b128 o, [%6], c, v;\n\t"
        "mov.b128 {%0, %1}, o;\n\t}"
        : "=l"(old.lo), "=l"(old.hi)
        : "l"(cmp_lo), "l"(cmp_hi), "l"(val_lo), "l"(val_hi), "l"(addr)
        : "memory");
    return old;
}

__device__ __forceinline__ unsigned lane_id() { return threadIdx.x & 31u; }

// Warp-aggregated append: every thread of the (converged) warp calls it; returns the slot index for threads with want.
__device__ __forceinline__ uint64_t warp_append(unsigned long long* cursor, bool want) {
    unsigned active = __activemask();
    unsigned m = __ballot_sync(active, want);
    if (!want) return 0;
    int leader = __ffs(m) - 1;
    unsigned long long base = 0;
    if ((int)lane_id() == leader) base = atomicAdd(cursor, (unsigned long long)__popc(m));
    base = __shfl_sync(m, base, leader);
    return base + __popc(m & ((1u << lane_id()) - 1u));
}
// Warp-reduced counter add (all threads of the converged warp call it).
__device__ __forceinline__ void warp_add(unsigned long long* counter, unsigned long long v) {
    unsigned active = __activemask();
    for (int d = 16; d > 0; d >>= 1) v += __shfl_down_sync(active, v, d);
    // with a partial mask the shuffle of an inactive lane returns the caller's own value, so only use this from full warps
    if (lane_id() == 0 && v) atomicAdd(counter, v);
}

// ================================================================ K1: quality floor, extraction, counting

__global__ void k_init_count_table(CountSlot* tab, uint64_t T) {
    const uint4 key = make_uint4(0xffffffffu, 0xffffffffu, 0xffffffffu, 0xffffffffu), zero = make_uint4(0, 0, 0, 0);
    uint4* p = reinterpret_cast<uint4*>(tab);
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < 2 * T; i += (uint64_t)gridDim.x * blockDim.x) p[i] = (i & 1) ? zero : key;
}

// paths/long/BuildReadQGraph.cc:962-987: one thread decodes one read's PQVec stream and finds its good length.
__global__ void k_good_len(ReadsView r, uint64_t first, uint64_t count, uint32_t min_qual, uint16_t* __restrict__ good, unsigned long long* __restrict__ n_inst,
                           int* __restrict__ bad) {
    const uint64_t end = first + count;
    for (uint64_t base = first + (uint64_t)blockIdx.x * blockDim.x; base < end; base += (uint64_t)gridDim.x * blockDim.x) {
        uint64_t i = base + threadIdx.x;
        unsigned long long mine = 0;
        if (i < end) {
            uint32_t nq = 0;
            uint32_t gl = pq_good_length(r.quals + r.qual_off[i], r.quals + r.qual_off[i + 1], min_qual, &nq);
            if (nq != r.len[i]) atomicExch(bad, 1);              // a valid store has one quality per base, framed inside its stream
            if (gl > r.len[i]) gl = r.len[i];
            good[i] = (uint16_t)gl;
            if (gl > (uint32_t)K) mine = gl - K + 1;
        }
        unsigned active = __activemask();
        for (int d = 16; d > 0; d >>= 1) mine += __shfl_down_sync(active, mine, d);
        if (lane_id() == 0 && mine) atomicAdd(n_inst, mine);
    }
}

// ================================================================ K2: dictionary (the counting kernels live in count_part.cuh)
// Test hooks: dump records (level 2 = every distinct k-mer with saturated count and raw context; level 1 = the dictionary).
struct DumpRec { uint64_t w0, w1; uint32_t count, ctx, edge, off; };
__global__ void k_dump_solid(SolidTable st, DumpRec* __restrict__ out, unsigned long long* cursor) {
    const uint64_t T = st.size();
    for (uint64_t base = (uint64_t)blockIdx.x * blockDim.x; base < T; base += (uint64_t)gridDim.x * blockDim.x) {
        uint64_t i = base + threadIdx.x;
        bool want = i < T && st.slots[i].w0 != EMPTY_W0;
        uint64_t pos = warp_append(cursor, want);
        if (want) { const SolidSlot& s = st.slots[i]; out[pos] = DumpRec{s.w0, s.w1, 0, s.ctx & 0xffu, s.edge, s.off}; }
    }
}

// Dictionary build (BuildReadQGraph.cc:1096-1104 insertEntryNoLocking, in parallel): keys are unique, so a successful CAS owns the slot.
// bloom (optional): the pathing filter's bits are set on the way (kmer.cuh: PathDict), which saves a sweep over the finished table.
// dense (optional, one GPU): record i also becomes node i of the graph stage (unipath.cuh: DenseNodes), and its slot's `off` holds i.
__global__ void k_insert_solid(const ulonglong2* __restrict__ recs, uint64_t n, SolidTable st, uint32_t* __restrict__ bloom, uint32_t bloom_W, uint32_t slice_words,
                               SolidSlot* __restrict__ dense) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        ulonglong2 rec = __ldcs(recs + i);
        Kmer k{rec.x, rec.y & ~0xffull};
        uint32_t ctx = (uint32_t)rec.y & 0xffu;
        if (bloom) { const uint32_t bh = bloom_hash(k); atomicOr(bloom + pd_bloom_word(bloom_W, slice_words, bh), bloom_mask(bh)); }
        uint64_t h = st.home(k);
        for (;;) {
            SolidSlot* p = st.slots + h;
            U128 old = cas128(p, ~0ull, ~0ull, k.w0, k.w1);
            if (old.lo == ~0ull && old.hi == ~0ull) { p->ctx = ctx; p->edge = NIL; p->off = dense ? (uint32_t)i : 0u; p->pad = 0; break; }
            h = st.next(h);
        }
        if (dense) dense[i] = SolidSlot{k.w0, k.w1, ctx, NIL, 0, 0};
    }
}
// The same from whole entries (k-mer, pruned context, edge, offset): the pathing dictionary of a sharded run is built from the
// entries the owner ranks finished (shardgraph.cuh), gathered from all ranks.
__global__ void k_insert_entries(const SolidSlot* __restrict__ recs, uint64_t n, SolidTable st, uint32_t* __restrict__ bloom, uint32_t bloom_W, uint32_t slice_words) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        const SolidSlot e = recs[i];
        if (bloom) { const uint32_t bh = bloom_hash(Kmer{e.w0, e.w1}); atomicOr(bloom + pd_bloom_word(bloom_W, slice_words, bh), bloom_mask(bh)); }
        uint64_t h = st.home(Kmer{e.w0, e.w1});
        for (;;) {
            SolidSlot* p = st.slots + h;
            U128 old = cas128(p, ~0ull, ~0ull, e.w0, e.w1);
            if (old.lo == ~0ull && old.hi == ~0ull) { p->ctx = e.ctx; p->edge = e.edge; p->off = e.off; p->pad = 0; break; }
            h = st.next(h);
        }
    }
}

// ================================================================ K3: adjacency pruning (kmers/ReadPather.h:307-346)
__global__ void k_adjacency(SolidTable st) {
    const uint64_t T = st.size();
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < T; i += (uint64_t)gridDim.x * blockDim.x) {
        SolidSlot* s = st.slots + i;
        if (s->w0 == EMPTY_W0 || slot_is_ghost(*s)) continue;      // (ghosts: copies of k-mers other ranks own; they only answer membership)
        uint32_t c = s->ctx & 0xffu;
        uint32_t c2 = pruned_context(st, Kmer{s->w0, s->w1}, c);
        if (c2 != c) s->ctx = c2;     // other threads only test membership (keys), never contexts, during this kernel
    }
}
// The same over the dense nodes (one GPU): a sequential sweep; a neighbour is looked for next to its node first (unipath.cuh: node_find),
// then probed in the table.  Other threads only read the keys of entries here, never their contexts.
__global__ void k_adjacency_dense(DenseNodes d) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < d.n; i += (uint64_t)gridDim.x * blockDim.x) {
        SolidSlot* s = d.nodes + i;
        const uint32_t c = s->ctx & 0xffu, c2 = pruned_context(d, i, Kmer{s->w0, s->w1}, c);
        if (c2 != c) s->ctx = c2;
    }
}

// ================================================================ K4: unipaths
template <class V>
__global__ void k_links(V st, uint32_t* __restrict__ next0, int* __restrict__ missing) {
    const uint64_t nn = 2 * st.size();
    for (uint64_t x = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; x < nn; x += (uint64_t)gridDim.x * blockDim.x) {
        int miss = 0;
        next0[x] = unipath_succ_link(st, (uint32_t)x, &miss);
        if (miss) atomicExch(missing, 1);
    }
}
// Rank state per node: .x = pointer, .y = distance | RANK_RESOLVED.  Tails (no successor) are resolved fixed points.
__global__ void k_rank_init(const uint32_t* __restrict__ next0, uint64_t nn, RankState* __restrict__ A) {
    for (uint64_t x = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; x < nn; x += (uint64_t)gridDim.x * blockDim.x) A[x] = rank_init_node(next0, (uint32_t)x);
}
__global__ void k_rank_init_list(const uint32_t* __restrict__ list, uint64_t n, const uint32_t* __restrict__ next0, RankState* __restrict__ A) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) { uint32_t x = list[i]; A[x] = rank_init_node(next0, x); }
}
// One pointer-jumping round A -> B over all nodes (list == nullptr) or over a node list; counts unresolved nodes.
__global__ void k_rank_step(const uint32_t* __restrict__ list, uint64_t n, const RankState* __restrict__ A, RankState* __restrict__ B, unsigned long long* __restrict__ unresolved) {
    for (uint64_t base = (uint64_t)blockIdx.x * blockDim.x; base < n; base += (uint64_t)gridDim.x * blockDim.x) {
        uint64_t i = base + threadIdx.x;
        bool un = false;
        if (i < n) {
            uint32_t x = list ? list[i] : (uint32_t)i;
            B[x] = rank_step_node(A, x, &un);
        }
        unsigned m = __ballot_sync(__activemask(), un);
        if (lane_id() == 0 && m) atomicAdd(unresolved, (unsigned long long)__popc(m));
    }
}
// In-place pointer jumping over a node list (used for the splitters): every state (p, d) says "p is d steps ahead of me";
// composing it with ANY valid state of p (old or new) gives a valid state, so no double buffer is needed as long as the
// 8-byte state is read and written in one transaction (L2-coherent __ldcg/__stcg).
__global__ void k_rank_step_inplace(const uint32_t* __restrict__ list, uint64_t n, unsigned long long* S, unsigned long long* __restrict__ unresolved) {
    for (uint64_t base = (uint64_t)blockIdx.x * blockDim.x; base < n; base += (uint64_t)gridDim.x * blockDim.x) {
        uint64_t i = base + threadIdx.x;
        bool un = false;
        if (i < n) {
            uint32_t x = list[i];
            unsigned long long a = __ldcg(S + x);
            uint32_t ax = (uint32_t)a, ay = (uint32_t)(a >> 32);
            if (!(ay & RANK_RESOLVED)) {
                unsigned long long b = __ldcg(S + ax);
                uint32_t bx = (uint32_t)b, by = (uint32_t)(b >> 32);
                ay = (ay + (by & ~RANK_RESOLVED)) | (by & RANK_RESOLVED);
                __stcg(S + x, (unsigned long long)bx | ((unsigned long long)ay << 32));
                un = !(ay & RANK_RESOLVED);
            }
        }
        unsigned m = __ballot_sync(__activemask(), un);
        if (lane_id() == 0 && m) atomicAdd(unresolved, (unsigned long long)__popc(m));
    }
}
// Splitter-based list ranking (see unipath.cuh).
__global__ void k_count_splitters(const uint32_t* __restrict__ next0, const uint8_t* __restrict__ ghead, uint64_t nn, unsigned long long* __restrict__ count) {
    for (uint64_t base = (uint64_t)blockIdx.x * blockDim.x; base < nn; base += (uint64_t)gridDim.x * blockDim.x) {
        uint64_t x = base + threadIdx.x;
        const unsigned m = __ballot_sync(__activemask(), x < nn && node_is_splitter(next0, ghead, (uint32_t)x));
        if (lane_id() == 0 && m) atomicAdd(count, (unsigned long long)__popc(m));
    }
}
// The splitters are listed first and walked from the list: a warp then drives 32 independent chains (walking straight off the node
// sweep kept ~4 of 32 lanes busy, and this kernel lives on memory-level parallelism: every step is a dependent random fetch).
__global__ void k_list_splitters(const uint32_t* __restrict__ next0, const uint8_t* __restrict__ ghead, uint64_t nn, uint32_t* __restrict__ list, uint64_t list_cap,
                                 unsigned long long* cursor) {
    for (uint64_t base = (uint64_t)blockIdx.x * blockDim.x; base < nn; base += (uint64_t)gridDim.x * blockDim.x) {
        uint64_t x = base + threadIdx.x;
        bool sp = x < nn && node_is_splitter(next0, ghead, (uint32_t)x);
        uint64_t pos = warp_append(cursor, sp);
        if (sp && pos < list_cap) list[pos] = (uint32_t)x;
    }
}
__global__ void k_splitter_walk(const uint32_t* __restrict__ next0, const uint32_t* __restrict__ list, uint64_t n, RankState* __restrict__ label, RankState* __restrict__ S) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) splitter_walk(next0, list[i], label, S);
}
__global__ void k_splitter_finish(const uint32_t* __restrict__ next0, uint64_t nn, RankState* __restrict__ label_then_rank, const RankState* __restrict__ S,
                                  unsigned long long* __restrict__ unresolved) {
    for (uint64_t base = (uint64_t)blockIdx.x * blockDim.x; base < nn; base += (uint64_t)gridDim.x * blockDim.x) {
        uint64_t x = base + threadIdx.x;
        bool un = false;
        if (x < nn) { RankState r = splitter_finish_node(next0, label_then_rank, S, (uint32_t)x); label_then_rank[x] = r; un = !(r.y & RANK_RESOLVED); }
        unsigned m = __ballot_sync(__activemask(), un);
        if (lane_id() == 0 && m) atomicAdd(unresolved, (unsigned long long)__popc(m));
    }
}
__global__ void k_copy_list(const uint32_t* __restrict__ list, uint64_t n, const RankState* __restrict__ src, RankState* __restrict__ dst) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) dst[list[i]] = src[list[i]];
}
__global__ void k_collect_unresolved(const RankState* __restrict__ A, uint64_t nn, uint32_t* __restrict__ list, unsigned long long* cursor) {
    for (uint64_t base = (uint64_t)blockIdx.x * blockDim.x; base < nn; base += (uint64_t)gridDim.x * blockDim.x) {
        uint64_t x = base + threadIdx.x;
        bool want = x < nn && !(A[x].y & RANK_RESOLVED);
        uint64_t pos = warp_append(cursor, want);
        if (want) list[pos] = (uint32_t)x;
    }
}
// Smooth circles (BuildReadQGraph.cc:126-180): minimum canonical k-mer of every cycle by pointer doubling.
__global__ void k_cycle_init(const uint32_t* __restrict__ list, uint64_t n, const uint32_t* __restrict__ next0, RankState* __restrict__ A) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        uint32_t x = list[i];
        A[x] = RankState{next0[x], x >> 1};
    }
}
template <class V>
__global__ void k_cycle_step(const uint32_t* __restrict__ list, uint64_t n, V st, const RankState* __restrict__ A, RankState* __restrict__ B, int* __restrict__ changed) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        uint32_t x = list[i];
        bool ch;
        B[x] = cycle_step_node(st, A, x, &ch);
        if (ch) *changed = 1;
    }
}
// Cut both strand cycles at the minimum k-mer: (kmin,+) becomes a head, (kmin,-) a tail.
__global__ void k_cycle_cut(const uint32_t* __restrict__ list, uint64_t n, const RankState* __restrict__ A, uint32_t* __restrict__ next0) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        cycle_cut_node(A, next0, list[i]);
    }
}
// Per strand path: keep it iff its sequence is FWD or PALINDROME (dna/CanonicalForm.h:34-46, BuildReadQGraph.cc:247-258).
// R[x] = (tail(x), dist to tail | RESOLVED).  keep[] is indexed by the head node of the strand.
template <class V>
__global__ void k_strand_decide(V st, const RankState* __restrict__ R, uint8_t* __restrict__ keep, int* __restrict__ too_long) {
    const uint64_t nn = 2 * st.size();
    for (uint64_t xi = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; xi < nn; xi += (uint64_t)gridDim.x * blockDim.x) {
        if (strand_decide_node(st, R, (uint32_t)xi, keep)) atomicExch(too_long, 1);
    }
}
template <class V>
__global__ void k_collect_heads(V st, const RankState* __restrict__ R, const uint8_t* __restrict__ keep, uint32_t* __restrict__ h_node,
                                uint64_t* __restrict__ h_w0, uint64_t* __restrict__ h_w1, uint32_t* __restrict__ h_n, unsigned long long* cursor, uint64_t cap) {
    const uint64_t nn = 2 * st.size();
    for (uint64_t base = (uint64_t)blockIdx.x * blockDim.x; base < nn; base += (uint64_t)gridDim.x * blockDim.x) {
        uint64_t xi = base + threadIdx.x;
        bool want = false;
        uint32_t x = (uint32_t)xi;
        if (xi < nn) want = head_is_kept(st, R, keep, x);
        uint64_t pos = warp_append(cursor, want);
        if (want && pos < cap) {
            Kmer k = node_kmer(st, x);
            h_node[pos] = x; h_w0[pos] = k.w0; h_w1[pos] = k.w1; h_n[pos] = (R[x].y & ~RANK_RESOLVED) + 1u;
        }
    }
}
__global__ void k_assign_edges(const uint32_t* __restrict__ perm, uint64_t E, const uint32_t* __restrict__ h_node, const uint32_t* __restrict__ h_n,
                               uint32_t* __restrict__ edge_of_head, uint32_t* __restrict__ edge_len, uint32_t* __restrict__ edge_nbytes) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < E; i += (uint64_t)gridDim.x * blockDim.x) {
        uint32_t j = perm[i];
        edge_of_head[h_node[j]] = (uint32_t)i;
        uint32_t len = h_n[j] + K - 1;
        edge_len[i] = len;
        edge_nbytes[i] = (len + 3) / 4;
    }
}
struct OrBase {
    uint8_t* bases;   // zeroed, 4-byte aligned
    __device__ __forceinline__ void operator()(uint64_t byte_off, uint64_t pos, uint32_t b) const {
        uint64_t addr = byte_off + (pos >> 2);
        atomicOr(reinterpret_cast<uint32_t*>(bases + (addr & ~3ull)), b << (8 * (uint32_t)(addr & 3ull) + 2 * (uint32_t)(pos & 3ull)));
    }
};
// Every k-mer of a kept strand writes its first base (the tail also its other 59) and its KDef (edge id, offset).
template <class V>
__global__ void k_emit_edges(V st, const RankState* __restrict__ R, const uint32_t* __restrict__ edge_of_head, const uint64_t* __restrict__ edge_off,
                             uint8_t* __restrict__ edge_bases) {
    const uint64_t nn = 2 * st.size();
    OrBase put{edge_bases};
    for (uint64_t xi = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; xi < nn; xi += (uint64_t)gridDim.x * blockDim.x) emit_node(st, R, edge_of_head, edge_off, (uint32_t)xi, put);
}
// After the graph stage over dense nodes: every table slot takes its node's pruned context, edge and offset, so the pathing
// dictionary and the dump see the table they always saw.
__global__ void k_backfill_slots(SolidTable st, const SolidSlot* __restrict__ dense) {
    const uint64_t T = st.size();
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < T; i += (uint64_t)gridDim.x * blockDim.x) {
        SolidSlot* s = st.slots + i;
        if (s->w0 == EMPTY_W0) continue;
        const SolidSlot& d = dense[s->off];
        s->ctx = d.ctx; s->edge = d.edge; s->off = d.off;
    }
}

// Device -> pinned host memory by stores over PCIe instead of the copy engine: the D2H engine is shared by every stream, and the
// small scalar read-backs of the pathing stage would queue behind a gigabyte of graph arrays on it.  A few CTAs are enough to
// keep the link busy.  Both pointers 16-byte aligned.
__global__ void k_copy_to_host(const uint8_t* __restrict__ src, uint8_t* __restrict__ dst, size_t bytes) {
    const size_t n16 = bytes / 16;
    const uint4* s4 = reinterpret_cast<const uint4*>(src);
    uint4* d4 = reinterpret_cast<uint4*>(dst);
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n16; i += (size_t)gridDim.x * blockDim.x) d4[i] = s4[i];
    if (blockIdx.x == 0 && threadIdx.x < (bytes & 15)) dst[n16 * 16 + threadIdx.x] = src[n16 * 16 + threadIdx.x];
}

// ================================================================ K5: HBV vertices (paths/long/HBVFromEdges.cc:76-154)
// End w of edge e: 0 fwd-left, 1 fwd-right, 2 rc-left, 3 rc-right.  Key = (FNV-1a 64 over the 59 base codes as bytes
// (math/Hash.h:26-35), then the bases) — the order EdgeEnd::operator< defines (:34-38).
__global__ void k_edge_ends(const uint8_t* __restrict__ edge_bases, const uint64_t* __restrict__ edge_off, const uint32_t* __restrict__ edge_len, uint64_t E,
                            uint64_t* __restrict__ kh, uint64_t* __restrict__ k0, uint64_t* __restrict__ k1, uint8_t* __restrict__ is_pal) {
    for (uint64_t idx = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < 4 * E; idx += (uint64_t)gridDim.x * blockDim.x) {
        uint64_t e = idx >> 2;
        uint32_t w = (uint32_t)idx & 3u;
        bool pal; EndKey key;
        edge_end_key(edge_bases + edge_off[e], edge_len[e], w, &pal, &key);
        if (w == 0) is_pal[e] = pal ? 1 : 0;
        kh[idx] = key.h; k0[idx] = key.k0; k1[idx] = key.k1;
    }
}
__global__ void k_vertex_flags(const uint32_t* __restrict__ perm, uint64_t n4, const uint64_t* __restrict__ kh, const uint64_t* __restrict__ k0,
                               const uint64_t* __restrict__ k1, uint32_t* __restrict__ flag) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (uint64_t)gridDim.x * blockDim.x) {
        uint32_t j = perm[i];
        bool valid = !(kh[j] == ~0ull && k0[j] == ~0ull && k1[j] == ~0ull);
        uint32_t fl = 0;
        if (valid) {
            if (i == 0) fl = 1;
            else { uint32_t q = perm[i - 1]; fl = (kh[q] != kh[j] || k0[q] != k0[j] || k1[q] != k1[j]) ? 1u : 0u; }
        }
        flag[i] = fl;
    }
}
// After sorting by the hash word alone: do two neighbours share a hash but not the bases?  (Then the order inside that run is
// not EdgeEnd's and the caller sorts by all three words.)
__global__ void k_hash_order_check(const uint32_t* __restrict__ perm, uint64_t n4, const uint64_t* __restrict__ kh, const uint64_t* __restrict__ k0,
                                   const uint64_t* __restrict__ k1, unsigned long long* __restrict__ collisions) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x + 1; i < n4; i += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t j = perm[i], q = perm[i - 1];
        if (kh[q] == kh[j] && (k0[q] != k0[j] || k1[q] != k1[j])) atomicAdd(collisions, 1ull);
    }
}
__global__ void k_scatter_vids(const uint32_t* __restrict__ perm, uint64_t n4, const uint32_t* __restrict__ flag, const uint32_t* __restrict__ excl,
                               const uint64_t* __restrict__ kh, const uint64_t* __restrict__ k0, const uint64_t* __restrict__ k1, int32_t* __restrict__ edge_vertices) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (uint64_t)gridDim.x * blockDim.x) {
        uint32_t j = perm[i];
        bool valid = !(kh[j] == ~0ull && k0[j] == ~0ull && k1[j] == ~0ull);
        edge_vertices[j] = valid ? (int32_t)(excl[i] + flag[i]) - 1 : -1;
    }
}
__global__ void k_pal_widths(const uint8_t* __restrict__ is_pal, uint64_t E, uint32_t* __restrict__ width) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < E; i += (uint64_t)gridDim.x * blockDim.x) width[i] = is_pal[i] ? 1u : 2u;
}
// HBV edge ids: canonical edge i -> fwd id, then rc id (one id for a palindrome) (HBVFromEdges.cc:137-151).
__global__ void k_hbv_edges(uint64_t E, const uint8_t* __restrict__ is_pal, const uint32_t* __restrict__ xl, const int32_t* __restrict__ edge_vertices,
                            int32_t* __restrict__ fwd_xlat, int32_t* __restrict__ rev_xlat, uint32_t* __restrict__ hcanon, int32_t* __restrict__ hleft, int32_t* __restrict__ hright,
                            int32_t* __restrict__ involution) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < E; i += (uint64_t)gridDim.x * blockDim.x) {
        uint32_t f = xl[i];
        fwd_xlat[i] = (int32_t)f;
        hcanon[f] = (uint32_t)(i << 1); hleft[f] = edge_vertices[4 * i]; hright[f] = edge_vertices[4 * i + 1];
        // the involution step 3 asks for (paths/HyperBasevector.cc:648-660) is the fwd/rc pairing itself
        if (is_pal[i]) { rev_xlat[i] = (int32_t)f; involution[f] = (int32_t)f; }
        else {
            rev_xlat[i] = (int32_t)f + 1; hcanon[f + 1] = (uint32_t)(i << 1) | 1u; hleft[f + 1] = edge_vertices[4 * i + 2]; hright[f + 1] = edge_vertices[4 * i + 3];
            involution[f] = (int32_t)f + 1; involution[f + 1] = (int32_t)f;
        }
    }
}
__global__ void k_adj_fill(uint64_t nh, const int32_t* __restrict__ hleft, const int32_t* __restrict__ hright, int32_t* __restrict__ from_e, int32_t* __restrict__ to_e,
                           uint32_t* __restrict__ from_cnt, uint32_t* __restrict__ to_cnt, int* __restrict__ bad) {
    for (uint64_t he = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; he < nh; he += (uint64_t)gridDim.x * blockDim.x) {
        int32_t l = hleft[he], r = hright[he];
        uint32_t a = atomicAdd(&from_cnt[l], 1u);
        if (a < 4) from_e[4 * (int64_t)l + a] = (int32_t)he; else atomicExch(bad, 1);
        uint32_t b = atomicAdd(&to_cnt[r], 1u);
        if (b < 4) to_e[4 * (int64_t)r + b] = (int32_t)he; else atomicExch(bad, 1);
    }
}
// graph/DigraphTemplate.h:1829-1839: lists are ordered by (neighbour vertex, edge id) when edges are added in id order.
__global__ void k_adj_sort(uint64_t nv, const int32_t* __restrict__ hleft, const int32_t* __restrict__ hright, int32_t* __restrict__ from_e, int32_t* __restrict__ to_e,
                           const uint32_t* __restrict__ from_cnt, const uint32_t* __restrict__ to_cnt, uint8_t* __restrict__ from_n, uint8_t* __restrict__ to_n) {
    for (uint64_t v = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; v < nv; v += (uint64_t)gridDim.x * blockDim.x) {
        for (int dir = 0; dir < 2; ++dir) {
            int32_t* lst = (dir ? to_e : from_e) + 4 * v;
            const int32_t* nb = dir ? hleft : hright;
            uint32_t n = dir ? to_cnt[v] : from_cnt[v];
            if (n > 4) n = 4;
            for (uint32_t i = 1; i < n; ++i) {
                int32_t e = lst[i]; int32_t ke = nb[e];
                int j = (int)i - 1;
                while (j >= 0 && (nb[lst[j]] > ke || (nb[lst[j]] == ke && lst[j] > e))) { lst[j + 1] = lst[j]; --j; }
                lst[j + 1] = e;
            }
            (dir ? to_n : from_n)[v] = (uint8_t)n;
        }
    }
}

// ================================================================ K6: read pathing
struct alignas(8) PathMeta { uint32_t x, y; };   // x = first id in the staging row, y = path length | overflow << 31
// One thread per read.  stage: [n_rows][cap] ints; meta: per row (start, len | overflow<<31).
// One thread per read drives a PathWalker.  A k-mer that is not in the dictionary (a sequencing error) is followed by ~60 more
// misses, or misses to the end of the read; a lane walking such a gap alone keeps 31 lanes idle for dozens of dependent
// lookups (measured: 5.9 of 32 lanes active).  Instead the WARP screens the gaps of its lanes: for a requesting lane, every lane
// forms one of its next 32 k-mers and asks the Bloom filter (four requests at a time, so four probes per lane are in flight),
// and the requester gets the 32-bit candidate mask.  Each requester then looks up its own first candidate in the dictionary
// (all requesters at once), and continues along its read.
constexpr int PATH_GAP_BATCH = 4;
constexpr uint32_t PATH_CTAS_PER_SM = 8;          // k_path_reads' register cap and grid (path_stage: why 8)
__global__ void __launch_bounds__(128, PATH_CTAS_PER_SM) k_path_reads(ReadsView r, GraphView g, const uint32_t* __restrict__ list, uint64_t n_rows,
                                                                      int32_t* __restrict__ stage, uint32_t cap, uint32_t left_cap, int32_t* __restrict__ out_offset,
                                                                      PathMeta* __restrict__ out_meta, uint32_t apply_fixpaths) {
    // walker state in shared memory, one slot per thread, padded to an odd number of words (no bank conflicts across lanes)
    struct Slot { PathState st; uint32_t pad[(sizeof(PathState) / 4) % 2 == 0 ? 1 : 2]; };
    __shared__ Slot slots[128];
    PathState& ps = slots[threadIdx.x].st;
    const uint32_t lane = lane_id();
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t row0 = (uint64_t)blockIdx.x * blockDim.x + (threadIdx.x & ~31u); row0 < n_rows; row0 += stride) {   // warp-uniform trip count
        const uint64_t row = row0 + lane;
        const bool live = row < n_rows;
        const uint64_t i = live ? (list ? list[row] : row) : 0;
        PathWalker w(ps);
        w.init(g, r.bases + r.base_off[i], live ? r.len[i] : 0u, stage + (live ? row : 0) * cap, cap, left_cap);
        // scan() and gap_found() have one call site each (the walker's code is large; see PathWalker::scan)
        bool need = false, run = true, have_gap = false;
        uint32_t from = 0, found_p = 0;                            // from: first unscreened position of this lane's gap
        const SolidSlot* found_slot = nullptr;
        for (;;) {
            if (run) {
                if (have_gap) w.gap_found(found_p, found_slot);
                need = w.scan();
                from = ps.itr + 1u;
                run = false; have_gap = false;
            }
            unsigned m = __ballot_sync(0xffffffffu, need);
            if (!m) break;
            uint32_t cand = 0;                                    // candidate mask of positions [from, from + 32)
            while (m) {
                int src[PATH_GAP_BATCH];
                uint32_t word[PATH_GAP_BATCH], bits[PATH_GAP_BATCH];
                int n = 0;
#pragma unroll
                for (int q = 0; q < PATH_GAP_BATCH; ++q) { src[q] = m ? __ffs((int)m) - 1 : -1; if (m) { m &= m - 1; ++n; } }
#pragma unroll
                for (int q = 0; q < PATH_GAP_BATCH; ++q) {
                    word[q] = 0; bits[q] = 1;                     // (word & bits) != bits: not a candidate
                    if (q < n) {
                        const uint8_t* b = reinterpret_cast<const uint8_t*>(__shfl_sync(0xffffffffu, reinterpret_cast<unsigned long long>(ps.bases), src[q]));
                        const uint32_t p = __shfl_sync(0xffffffffu, from, src[q]) + lane, nk = __shfl_sync(0xffffffffu, ps.nk, src[q]);
                        if (p < nk) {
                            Kmer f, rc;
                            kmer_pair_at(b, p, &f, &rc);
                            const uint32_t hh = bloom_hash(kmer_less(rc, f) ? rc : f);
                            if (g.dict.bloom) { word[q] = __ldg(g.dict.bloom + pd_bloom_word(g.dict.W, g.dict.slice_words, hh)); bits[q] = bloom_mask(hh); }
                            else { word[q] = 1; bits[q] = 1; }   // no filter (tiny dictionary): every position is a candidate
                        }
                    }
                }
#pragma unroll
                for (int q = 0; q < PATH_GAP_BATCH; ++q) {
                    if (q < n) {
                        const unsigned mm = __ballot_sync(0xffffffffu, (word[q] & bits[q]) == bits[q]);
                        if ((int)lane == src[q]) cand = mm;
                    }
                }
            }
            if (need) {
                while (cand) {                                    // candidates in read order; the first one is almost always real
                    const uint32_t p = from + (uint32_t)(__ffs((int)cand) - 1);
                    cand &= cand - 1;
                    Kmer f, rc;
                    kmer_pair_at(ps.bases, p, &f, &rc);
                    const Kmer canon = kmer_less(rc, f) ? rc : f;
                    const SolidSlot* s = pd_find(g.dict, canon, bloom_hash(canon));
                    if (s) { found_p = p; found_slot = s; have_gap = true; run = true; break; }
                }
                if (!run) {
                    from += 32;
                    if (from >= ps.nk) { found_p = ps.nk; found_slot = nullptr; have_gap = true; run = true; }
                }
            }
        }
        if (live) {
            PathResult pr = w.finish(r.quals + r.qual_off[i], apply_fixpaths != 0);
            out_offset[row] = pr.offset;
            out_meta[row] = PathMeta{pr.start, pr.overflow ? 0x80000000u : pr.len};
        }
    }
}
// lens[target] = path length (0 for overflowed rows); counters: pathed (>0 edges), multipathed (>2 edges), overflowed rows.
__global__ void k_path_lens(const PathMeta* __restrict__ meta, const uint32_t* __restrict__ list, uint64_t n, uint32_t* __restrict__ lens,
                            unsigned long long* __restrict__ counters /*pathed, multipathed, overflow*/) {
    for (uint64_t base = (uint64_t)blockIdx.x * blockDim.x; base < n; base += (uint64_t)gridDim.x * blockDim.x) {
        uint64_t i = base + threadIdx.x;
        uint32_t len = 0; bool ovf = false;
        if (i < n) { uint32_t m = meta[i].y; ovf = m >> 31; len = ovf ? 0 : m; lens[list ? list[i] : i] = len; }
        unsigned act = __activemask();
        unsigned a = __ballot_sync(act, len > 0), b = __ballot_sync(act, len > 2), c = __ballot_sync(act, ovf);
        if (lane_id() == 0) { if (a) atomicAdd(&counters[0], (unsigned long long)__popc(a)); if (b) atomicAdd(&counters[1], (unsigned long long)__popc(b)); if (c) atomicAdd(&counters[2], (unsigned long long)__popc(c)); }
    }
}
__global__ void k_path_gather(const int32_t* __restrict__ stage, uint32_t cap, const PathMeta* __restrict__ meta, const uint32_t* __restrict__ list,
                              const int32_t* __restrict__ row_offset, const uint64_t* __restrict__ path_off, uint64_t n, int32_t* __restrict__ path_edges,
                              int32_t* __restrict__ path_offset) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        PathMeta m = meta[i];
        if (m.y >> 31) continue;
        uint64_t rd = list ? list[i] : i;
        const int32_t* src = stage + i * cap + m.x;
        int32_t* dst = path_edges + path_off[rd];
        for (uint32_t j = 0; j < m.y; ++j) dst[j] = src[j];
        path_offset[rd] = row_offset[i];
    }
}
// Second-chance pathing for the (rare) reads whose path overflowed the staging row: results are patched into the big arrays.
__global__ void k_collect_overflow(const PathMeta* __restrict__ meta, uint64_t n, uint32_t* __restrict__ list, unsigned long long* cursor) {
    for (uint64_t base = (uint64_t)blockIdx.x * blockDim.x; base < n; base += (uint64_t)gridDim.x * blockDim.x) {
        uint64_t i = base + threadIdx.x;
        bool want = i < n && (meta[i].y >> 31);
        uint64_t pos = warp_append(cursor, want);
        if (want) list[pos] = (uint32_t)i;
    }
}

// ================================================================ result digests (w2rap_graph.digest_*)
__device__ __forceinline__ uint64_t digest_mix(uint64_t x) { x ^= x >> 33; x *= 0xff51afd7ed558ccdull; x ^= x >> 33; x *= 0xc4ceb9fe1a85ec53ull; x ^= x >> 33; return x; }
// *out += sum over i of mix(mix(i + salt) ^ word[i]) for the n_bytes at p (4-byte aligned; the last word is zero-extended)
__global__ void k_digest_words(const uint8_t* __restrict__ p, uint64_t n_bytes, uint64_t salt, unsigned long long* out) {
    const uint64_t nw = (n_bytes + 3) / 4;
    unsigned long long acc = 0;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nw; i += (uint64_t)gridDim.x * blockDim.x) {
        uint32_t w = 0;
        if (4 * i + 4 <= n_bytes) w = reinterpret_cast<const uint32_t*>(p)[i];
        else for (uint64_t b = 4 * i; b < n_bytes; ++b) w |= (uint32_t)p[b] << (8 * (b - 4 * i));
        acc += digest_mix(digest_mix(i + salt) ^ w);
    }
    for (int d = 16; d > 0; d >>= 1) acc += __shfl_down_sync(0xffffffffu, acc, d);
    if (lane_id() == 0 && acc) atomicAdd(out, acc);
}
// one term per read: the read's sequence bound to its path (offset, edges).  A sum, so it does not depend on how the reads are
// sharded over GPUs.
__global__ void k_digest_paths(ReadsView r, const int32_t* __restrict__ path_offset, const uint64_t* __restrict__ path_off, const int32_t* __restrict__ path_edges,
                               unsigned long long* out) {
    unsigned long long acc = 0;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < r.n; i += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t len = r.len[i];
        const uint8_t* b = r.bases + r.base_off[i];
        uint64_t h = digest_mix(len);
        const uint32_t nb = (len + 3) / 4;
        for (uint32_t j = 0; j < nb; ++j) {
            uint32_t v = b[j];
            if (j + 1 == nb && (len & 3u)) v &= (1u << (2u * (len & 3u))) - 1u;      // bits past the last base are not part of the read
            h = digest_mix(h ^ v) + j;
        }
        h = digest_mix(h ^ (uint64_t)(uint32_t)path_offset[i]);
        for (uint64_t e = path_off[i]; e < path_off[i + 1]; ++e) h = digest_mix(h ^ (uint64_t)(uint32_t)path_edges[e]) + 0x9e3779b97f4a7c15ull;
        acc += h;
    }
    for (int d = 16; d > 0; d >>= 1) acc += __shfl_down_sync(0xffffffffu, acc, d);
    if (lane_id() == 0 && acc) atomicAdd(out, acc);
}

}  // namespace w2r
