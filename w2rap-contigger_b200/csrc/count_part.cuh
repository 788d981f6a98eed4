// count_part.cuh — k-mer counting as map (partition) + reduce (count per partition).
//
// A global hash table >> L2 costs one random DRAM sector read and one write-back per k-mer INSTANCE (measured: 13 G inserts/s
// on B200, 0.84 TB/s of 32-byte sector traffic).  Instead, the MapReduceEngine shape (MapReduceEngine.h:288-358) on the device:
//   map     k_minimizer_map     : a warp per read computes the MINIMISER partition of every k-mer; runs of consecutive k-mers in
//                                 the same partition leave as one 32-byte SUPER-K-MER record (extract.cuh: SkmRec, <= 32 k-mers:
//                                 their shared bases + the two context bases) — ~2 bytes per k-mer instance instead of 16.
//                                 Records are built once, into a staging area, while partitions are counted; a scan lays the
//                                 partitions out exactly and a copy kernel (k_scatter_records) moves every record home.
//   reduce  k_count_smem        : one CTA counts one partition (~20 k k-mer instances, a few thousand distinct k-mers) in a
//                                 shared-memory hash table.  The partition's records are staged into shared memory by bulk
//                                 asynchronous copies (cp.async.bulk + mbarrier, double buffered; SASS: UBLKCP/SYNCS), and the
//                                 warps expand them FLAT: lane l takes k-mer t + l of a group of 32 records, so every lane forms and
//                                 inserts a k-mer whatever the record lengths.  Then histogram + solid records, sorted by
//                                 (minimiser, offset of the minimiser) so that the k-mers of a chain leave next to each other:
//                                 their index in the solid array is their node id in the graph stage (unipath.cuh: DenseNodes).
//           k_count_region /    : fallback for partitions whose distinct k-mers do not fit shared memory: inserts into a 32 MB
//           k_scan_region         table region that stays resident in L2 (128-bit CAS, count/context REDs), then scan + reset.
// DRAM traffic: 32 B written + 32 B read per RECORD (~13-18 k-mers) and nothing else; the same records cross NVLink when sharded.
#pragma once
#include "kernels.cuh"
#include "prims.cuh"
#include "shard.cuh"

namespace w2r {

// ---------------------------------------------------------------- map keyed by minimiser
// One WARP per read.  Lane l of step t handles k-mer 32t + l: the window minimum is computed independently per position (no
// rolling state); lanes whose neighbours fall into the same partition form a segment, and every segment becomes one record.
// Window minima: the hashes of all m-mers of a tile live in registers (8 per lane), five doubling steps of shuffles give the
// min over 32 consecutive hashes, the 46-wide window is two overlapping 32-wide ones.  The segments of a tile are listed in
// shared memory and then built one per lane (4 aligned 8-byte loads, 3 funnel shifts, two 16-byte stores).
constexpr uint32_t MINI_TILE = 192;                       // k-mers per tile (a 250-base read is one tile)
constexpr uint32_t MINI_NU = 8;                           // hashes per lane: positions 32u + lane, u < 8, cover the 192 + 45 m-mers of a tile
constexpr uint32_t MAP_CHUNK = 512;                       // records a warp reserves at a time in the staging area (>= MINI_TILE)
constexpr uint32_t MAP_CTAS_PER_SM = 6;                   // k_minimizer_map's occupancy: its register cap, its grid, the staging allowance
struct MiniParams {
    uint32_t logP, npass, pass;
    uint32_t* count;                 // records per partition (this read batch)
    uint32_t* kcount;                // k-mer instances per partition
    SkmRec* tmp;                     // staging area: records in the order the warps produce them ...
    uint32_t* tpart;                 // ... with the partition of each (NIL: unused slot)
    unsigned long long* tmp_cursor;  // slots handed out so far (in chunks of MAP_CHUNK per warp)
    uint64_t tmp_cap;
    int* overflow;
};
// Launch 1 (the expensive one: minimisers): builds every record ONCE, into a staging area in production order, and counts records
// and k-mers per partition.  After an exclusive scan of the counts, launch 2 (k_scatter_records: a copy kernel) moves every record
// to its partition.  Exact sizes mean no capacity guess per partition can overflow, whatever the multiplicity skew of the read set
// (a repeat with 10^4 copies just makes its partitions long).
__global__ void __launch_bounds__(256, MAP_CTAS_PER_SM) k_minimizer_map(ReadsView r, uint64_t first, uint64_t count, const uint16_t* __restrict__ good, MiniParams mp) {
    __shared__ uint32_t wbuf[8][MINI_TILE];
    __shared__ uint32_t sbuf[8][MINI_TILE];               // segment list of the tile: start | n << 16
    uint32_t* wb = wbuf[threadIdx.x >> 5];
    uint32_t* sl = sbuf[threadIdx.x >> 5];
    const uint32_t lane = threadIdx.x & 31u;
    const unsigned upto = (2u << lane) - 1u;                  // lanes 0..lane
    const uint64_t nwarps = ((uint64_t)gridDim.x * blockDim.x) >> 5, end = first + count;
    unsigned long long chunk_pos = 0;                         // this warp's current chunk of the staging area (warp-uniform)
    uint32_t chunk_left = 0;
    for (uint64_t i = first + (((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5); i < end; i += nwarps) {
        const uint32_t gl = good[i];
        if (gl <= (uint32_t)K) continue;
        const uint8_t* bases = r.bases + r.base_off[i];
        const uint32_t nk = gl - K + 1, last = gl - K;
        for (uint32_t j0 = 0; j0 < nk; j0 += MINI_TILE) {
            const uint32_t n_k = nk - j0 < MINI_TILE ? nk - j0 : MINI_TILE, n_h = n_k + MINI_W - 1;
            // window minima in registers: h[u] = hash of the m-mer at tile position 32u + lane; a doubling step with shift s takes
            // position p + s from lane (lane + s) & 31 of the same or the next register
            uint32_t h[MINI_NU + 1];
#pragma unroll
            for (uint32_t u = 0; u < MINI_NU; ++u) { const uint32_t t = 32u * u + lane; h[u] = t < n_h ? mmer_hash_at(bases, (uint64_t)j0 + t) : 0xffffffffu; }
            h[MINI_NU] = 0xffffffffu;
#pragma unroll
            for (uint32_t s = 1; s <= 16; s <<= 1) {                      // after these: h = min over 32 consecutive positions
                const uint32_t src = (lane + s) & 31u;
                const bool wrap = lane + s >= 32u;
                uint32_t x = __shfl_sync(0xffffffffu, h[0], src);
#pragma unroll
                for (uint32_t u = 0; u < MINI_NU; ++u) {
                    const uint32_t y = u + 1 < MINI_NU ? __shfl_sync(0xffffffffu, h[u + 1], src) : 0xffffffffu;
                    const uint32_t o = wrap ? y : x;
                    h[u] = h[u] < o ? h[u] : o;
                    x = y;
                }
            }
            __syncwarp();                                                 // the previous tile's lists have been consumed
            {                                                             // 46-wide window = two 32-wide ones, 14 apart
                const uint32_t src = (lane + (MINI_W - 32)) & 31u;
                const bool wrap = lane + (MINI_W - 32) >= 32u;
                uint32_t x = __shfl_sync(0xffffffffu, h[0], src);
#pragma unroll
                for (uint32_t u = 0; u < MINI_TILE / 32; ++u) {
                    const uint32_t y = __shfl_sync(0xffffffffu, h[u + 1], src);
                    const uint32_t o = wrap ? y : x;
                    // partition of the k-mer at tile position 32u + lane (NIL: not in this counting pass)
                    const uint32_t mh = mini_mix(h[u] < o ? h[u] : o);
                    wb[32u * u + lane] = (mp.npass > 1 && (mh & 0xffffu) % mp.npass != mp.pass) ? NIL : mini_part(mh, mp.logP);
                    x = y;
                }
            }
            uint32_t nseg = 0;
            for (uint32_t t0 = 0; t0 < n_k; t0 += 32) {                   // segments: runs of equal partition inside a 32-lane step
                const uint32_t jj = t0 + lane;
                const uint32_t b = jj < n_k ? wb[jj] : NIL;               // (own entry: written by this lane)
                const bool active = b != NIL;
                const unsigned amask = __ballot_sync(0xffffffffu, active);
                const uint32_t pb = __shfl_up_sync(0xffffffffu, b, 1);
                const bool head = active && (lane == 0 || !((amask >> (lane - 1)) & 1u) || pb != b);
                const unsigned heads = __ballot_sync(0xffffffffu, head);
                if (head) {
                    const unsigned stop = (heads | ~amask) & ~upto;       // next segment head or first idle lane above this one
                    const uint32_t seglen = (stop ? (uint32_t)__ffs((int)stop) - 1u : 32u) - lane;
                    sl[nseg + (uint32_t)__popc(heads & (upto >> 1))] = jj | (seglen << 16);
                }
                nseg += (uint32_t)__popc(heads);
            }
            __syncwarp();
            if (nseg > chunk_left) {                                      // a new chunk of the staging area (the rest of the old one stays NIL)
                if (lane == 0) chunk_pos = atomicAdd(mp.tmp_cursor, (unsigned long long)MAP_CHUNK);
                chunk_pos = __shfl_sync(0xffffffffu, chunk_pos, 0);
                chunk_left = MAP_CHUNK;
            }
            for (uint32_t s = lane; s < nseg; s += 32) {                  // one record per lane
                const uint32_t e = sl[s], jj = e & 0xffffu, n = e >> 16, b = wb[jj];
                atomicAdd(mp.count + b, 1u); atomicAdd(mp.kcount + b, n);
                const unsigned long long pos = chunk_pos + s;
                if (pos < mp.tmp_cap) {
                    const SkmRec rec = skm_build(bases, j0 + jj, n, last);
                    ulonglong2* dst = reinterpret_cast<ulonglong2*>(mp.tmp + pos);
                    dst[0] = make_ulonglong2(rec.q[0], rec.q[1]);
                    dst[1] = make_ulonglong2(rec.q[2], rec.q[3]);
                    mp.tpart[pos] = b;
                } else atomicExch(mp.overflow, 1);
            }
            chunk_pos += nseg; chunk_left -= nseg;
        }
    }
}
// Launch 2: staging slots [range[0], range[1]) -> recs[*batch_off + base[partition] + arrival order]
struct ScatterParams {
    const SkmRec* tmp; const uint32_t* tpart;
    const unsigned long long* range;        // device: first and one-past-last staging slot of this read batch
    const uint64_t* base;                   // first record of every partition, relative to *batch_off
    uint32_t* cursor;                       // records appended so far
    SkmRec* recs;
    const unsigned long long* batch_off;    // where this read batch's records start
    uint64_t recs_cap, tmp_cap;
    int* overflow;
};
__global__ void __launch_bounds__(256) k_scatter_records(ScatterParams sp) {
    const unsigned long long t0 = sp.range[0], t1 = sp.range[1] < sp.tmp_cap ? sp.range[1] : sp.tmp_cap, boff = *sp.batch_off;
    for (unsigned long long i = t0 + (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < t1; i += (unsigned long long)gridDim.x * blockDim.x) {
        const uint32_t b = __ldcs(sp.tpart + i);
        if (b == NIL) continue;
        const ulonglong2* src = reinterpret_cast<const ulonglong2*>(sp.tmp + i);
        const ulonglong2 lo = __ldcs(src), hi = __ldcs(src + 1);
        const unsigned long long pos = boff + sp.base[b] + atomicAdd(sp.cursor + b, 1u);
        if (pos < sp.recs_cap) { ulonglong2* dst = reinterpret_cast<ulonglong2*>(sp.recs + pos); dst[0] = lo; dst[1] = hi; }
        else atomicExch(sp.overflow, 1);
    }
}
__global__ void k_copy_scalar(const unsigned long long* src, unsigned long long* dst) { *dst = *src; }

// batch_off[1] = batch_off[0] + total[0]: chains the record areas of consecutive read batches on the device
__global__ void k_next_batch_off(unsigned long long* batch_off, const uint64_t* total) { batch_off[1] = batch_off[0] + *total; }

// ---------------------------------------------------------------- reduce fallback: the L2-resident counting region
struct RegionParams {
    CountSlot* region;       // 1 << logR slots, resident in L2
    uint32_t logR;
    uint32_t sub_mask, sub_id;   // overflow handling: only k-mers with ((hash >> 3) & sub_mask) == sub_id take part
    int* overflow;
};
constexpr uint32_t REGION_MAX_PROBE = 2048;
constexpr uint32_t COUNT_STOP_REGION = 1u << 24;               // the u32 counter of a region slot stops here (it cannot wrap)

// one 256-bit load of a whole slot (LDG.E.ENL2.256 on sm_100a), L2-coherent
__device__ __forceinline__ void ld_slot(const CountSlot* q, uint64_t& w0, uint64_t& w1, uint64_t& meta) {
    uint64_t pad;
    asm volatile("ld.global.cg.v4.u64 {%0,%1,%2,%3}, [%4];" : "=l"(w0), "=l"(w1), "=l"(meta), "=l"(pad) : "l"(q));
}

__device__ __forceinline__ void region_insert(const RegionParams& rp, Kmer k, uint32_t ctx, uint64_t h) {
    const uint64_t mask = (1ull << rp.logR) - 1;
    uint64_t s = h >> (64 - rp.logR);
    for (uint32_t probe = 0; probe < REGION_MAX_PROBE; ++probe) {
        CountSlot* q = rp.region + s;
        uint64_t w0, w1, meta;
        ld_slot(q, w0, w1, meta);
        bool hit = false;
        uint32_t have = (uint32_t)(meta >> 32);
        if (w0 == k.w0 && w1 == k.w1) hit = true;
        else if (w0 == EMPTY_W0) {
            U128 old = cas128(q, ~0ull, ~0ull, k.w0, k.w1);
            hit = (old.lo == ~0ull && old.hi == ~0ull) || (old.lo == k.w0 && old.hi == k.w1);
            have = 0;
        }
        if (hit) {
            if ((uint32_t)meta < COUNT_STOP_REGION || w0 == EMPTY_W0) atomicAdd(&q->count, 1u);
            if ((have & ctx) != ctx) atomicOr(&q->ctx, ctx);
            return;
        }
        s = (s + 1) & mask;
    }
    atomicExch(rp.overflow, 1);
}

// A partition is, per slab (a read batch on one GPU, a source rank when sharded), one contiguous run of records:
//   recs[slab_off[src] + part_base[src * P + b] .. + sizes[src * P + b]).
// plist (optional): the group is partitions plist[b_first .. b_first + gy) instead of the consecutive range starting at b_first.
struct RunView { const uint64_t* part_base; const unsigned long long* slab_off; uint64_t P; const uint32_t* plist; };
// The "reduce" step (BuildReadQGraph.cc:1081-1082 sort+collapse as a hash count) through the region: a warp per record, lane j
// expands k-mer j.  blockIdx.y = src * gy + partition within the group.
__global__ void __launch_bounds__(256) k_count_region(const SkmRec* __restrict__ recs, const uint32_t* __restrict__ sizes, uint32_t b_first, uint32_t gy, RunView rv,
                                                      RegionParams rp) {
    const uint32_t src = blockIdx.y / gy;
    const uint32_t bi = b_first + (blockIdx.y - src * gy);
    const uint32_t b = rv.plist ? rv.plist[bi] : bi;
    const uint64_t n = sizes[(uint64_t)src * rv.P + b];
    const SkmRec* base = recs + rv.slab_off[src] + rv.part_base[(uint64_t)src * rv.P + b];
    const uint32_t lane = threadIdx.x & 31u;
    const uint64_t nw = ((uint64_t)gridDim.x * blockDim.x) >> 5;
    for (uint64_t i = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; i < n; i += nw) {
        const uint64_t* q = base[i].q;
        if (lane < skm_n(q[3])) {
            Kmer k; uint32_t ctx;
            skm_kmer_at(q, lane, &k, &ctx);
            const uint64_t h = kmer_hash(k);
            if (!rp.sub_mask || (((uint32_t)(h >> 3)) & rp.sub_mask) == rp.sub_id) region_insert(rp, k, ctx, h);
        }
    }
}

// ---------------------------------------------------------------- reduce in SHARED memory
// With ~2^18 partitions a partition holds ~20 k k-mer instances and a few thousand distinct k-mers: one CTA counts it in a
// shared-memory table, so the per-instance atomics are shared-memory atomics instead of L2 atomics (the L2-resident region count
// is limited by L2 atomic throughput, about one k-mer per 30 ps chip-wide).  Partitions whose distinct k-mers do not fit are listed
// in `failed` and go through the region path.
constexpr uint32_t SMEM_LOG_SLOTS_MAX = 13;                    // 8192 slots: 128 KB keys + 32 KB count|ctx = 160 KB
constexpr uint32_t SMEM_MAX_PROBE = 512;
constexpr uint32_t COUNT_STOP = 1u << 16;                      // counters stop here (>= 255 is all anyone asks); + one add per racing thread
constexpr uint32_t SMEM_MAX_BATCH = 16;                        // runs (read batches / source ranks) that make up one partition
constexpr uint32_t SKM_CHUNK = 1024;                           // records per staging buffer (32 KB), two buffers
struct SmemCountParams {
    const SkmRec* recs;
    const uint32_t* cursor;         // [nbatch][P] records of partition p in slab bi
    const uint64_t* part_base;      // partition p is, per slab bi < nbatch, the contiguous run
    const unsigned long long* batch_off;   //   recs[batch_off[bi] + part_base[bi * P + p] .. + cursor[bi * P + p])
    uint32_t nbatch;
    uint32_t P;
    uint32_t min_freq;
    unsigned long long* hist;       // [104]
    ulonglong2* solid_out; unsigned long long* solid_cursor; uint64_t solid_cap; int* solid_overflow;
    DumpRec* dump_out; unsigned long long* dump_cursor;
    uint32_t* failed; unsigned long long* failed_cursor;       // partitions that did not fit the table
    uint32_t log_slots;                                        // log2 of the table's slots: SMEM_LOG_SLOTS_MAX, less under the table_slots test hook
    uint8_t* count_out;                                        // k_count_smem<true>: min(255, count) of solid_out[i] at count_out[i]
};

// --- mbarrier + bulk-copy wrappers (PTX; SASS: SYNCS.*, UBLKCP)
__device__ __forceinline__ uint32_t smem_addr(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) { asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_addr(bar)), "r"(count)); }
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) { asm volatile("mbarrier.expect_tx.relaxed.cta.shared::cta.b64 [%0], %1;" ::"r"(smem_addr(bar)), "r"(bytes) : "memory"); }
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) { asm volatile("{\n\t.reg .b64 st;\n\tmbarrier.arrive.shared::cta.b64 st, [%0];\n\t}" ::"r"(smem_addr(bar)) : "memory"); }
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE_%=;\n\t"
        "bra WAIT_%=;\n\t"
        "DONE_%=:\n\t}" ::"r"(smem_addr(bar)), "r"(parity) : "memory");
}
// global -> shared bulk copy (bytes a multiple of 16, both addresses 16-byte aligned), completion counted on `bar`
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_addr(dst)), "l"(src), "r"(bytes), "r"(smem_addr(bar)) : "memory");
}

// 32-bit slot hash for the shared-memory table.  All k-mers of a partition share a minimiser, i.e. 15 bases somewhere inside; the
// other 45 bases vary freely, so folding the words and two multiplies mix well enough for a few thousand keys in 8192 slots.
__device__ __forceinline__ uint32_t smem_slot_hash(Kmer k) {
    uint32_t x = (uint32_t)k.w0 * 0x9e3779b1u + (uint32_t)(k.w0 >> 32) * 0x85ebca77u;
    x ^= x >> 15;
    x += (uint32_t)(k.w1 >> 8) * 0xc2b2ae3du + (uint32_t)(k.w1 >> 40) * 0x27d4eb2fu;
    x ^= x >> 13; x *= 0x165667b1u; x ^= x >> 16;
    return x;
}

// 128-bit compare-and-swap on a 16-byte aligned shared-memory slot (ATOMS.CAS.128 on sm_100a): a 120-bit k-mer is claimed whole
__device__ __forceinline__ U128 cas128_shared(void* addr, uint64_t cmp_lo, uint64_t cmp_hi, uint64_t val_lo, uint64_t val_hi) {
    U128 old;
    asm volatile(
        "{\n\t.reg .b128 c, v, o;\n\t"
        "mov.b128 c, {%2, %3};\n\t"
        "mov.b128 v, {%4, %5};\n\t"
        "atom.shared.relaxed.cta.cas.b128 o, [%6], c, v;\n\t"
        "mov.b128 {%0, %1}, o;\n\t}"
        : "=l"(old.lo), "=l"(old.hi)
        : "l"(cmp_lo), "l"(cmp_hi), "l"(val_lo), "l"(val_hi), "r"(smem_addr(addr))
        : "memory");
    return old;
}
__device__ __forceinline__ ulonglong2 lds128_volatile(const void* addr) {
    ulonglong2 v;
    asm volatile("ld.volatile.shared.v2.u64 {%0, %1}, [%2];" : "=l"(v.x), "=l"(v.y) : "r"(smem_addr(addr)) : "memory");
    return v;
}

// KEEP_COUNTS (w2rap_step2_count): also write min(255, count) of every emitted record to sp.count_out, parallel to solid_out.
template <bool KEEP_COUNTS>
__global__ void __launch_bounds__(1024, 1) k_count_smem(SmemCountParams sp) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const uint32_t SMEM_SLOTS = 1u << sp.log_slots;
    ulonglong2* keys = reinterpret_cast<ulonglong2*>(smem_raw);             // {w0, w1}; empty = all ones (a canonical 60-mer never starts with 32 T's)
    uint32_t* ccs = reinterpret_cast<uint32_t*>(keys + SMEM_SLOTS);         // count (low 24 bits) | ctx << 24
    SkmRec* stage = reinterpret_cast<SkmRec*>(smem_raw + (size_t)20 * SMEM_SLOTS);   // [2][SKM_CHUNK]
    __shared__ __align__(8) uint64_t mbar[2];
    __shared__ unsigned int sh_hist[104];
    __shared__ int sh_fail;
    __shared__ uint32_t sh_tot[2], sh_cnt[2];                   // per staging buffer: records of the whole partition / of the staged chunk
    __shared__ uint32_t sh_nsolid;                              // solid k-mers of the partition
    __shared__ unsigned long long sh_solid_base;                // where they go in solid_out
    const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5, nwarp = blockDim.x >> 5;
    const unsigned le_mask = (2u << lane) - 1u;                 // lanes 0..lane
    for (int j = threadIdx.x; j < 104; j += blockDim.x) sh_hist[j] = 0;
    if (threadIdx.x == 0) { mbar_init(&mbar[0], 1); mbar_init(&mbar[1], 1); asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
    __syncthreads();
    // Warp 0 stages the records: lane bi owns run bi of a partition (a read batch / source rank).  The run descriptors of the NEXT
    // partition are loaded a whole partition ahead and sit in registers, so that issuing a chunk is a few shuffles and one bulk copy
    // per lane (one thread walking the runs with dependent global loads made warp 0 late at every chunk barrier: ~20 % of the
    // kernel's stall samples).
    uint32_t cu_cnt = 0, nx_cnt = 0;                             // records of my run in the current / next partition
    const SkmRec* cu_src = nullptr; const SkmRec* nx_src = nullptr;
    auto load_desc = [&](uint32_t p, uint32_t& cnt, const SkmRec*& src) {
        cnt = 0; src = nullptr;
        if (p < sp.P && lane < sp.nbatch) {
            cnt = sp.cursor[(uint64_t)lane * sp.P + p];
            src = sp.recs + sp.batch_off[lane] + sp.part_base[(uint64_t)lane * sp.P + p];
        }
    };
    // all lanes of warp 0: stage chunk c of the partition described by (cnt, src) into buffer bf
    auto issue = [&](uint32_t cnt, const SkmRec* src, uint32_t c, uint32_t bf) {
        const uint32_t lo = c * SKM_CHUNK, hi = lo + SKM_CHUNK;
        uint32_t incl = cnt;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) { const uint32_t t = __shfl_up_sync(0xffffffffu, incl, d); if ((int)lane >= d) incl += t; }
        const uint32_t acc = incl - cnt, tot = __shfl_sync(0xffffffffu, incl, 31);
        const uint32_t s = acc > lo ? acc : lo, e = acc + cnt < hi ? acc + cnt : hi;
        if (s < e) {
            mbar_expect_tx(&mbar[bf], (e - s) * (uint32_t)sizeof(SkmRec));
            bulk_g2s(stage + (size_t)bf * SKM_CHUNK + (s - lo), src + (s - acc), (e - s) * (uint32_t)sizeof(SkmRec), &mbar[bf]);
        }
        __syncwarp();                                            // every expect_tx precedes the arrival
        if (lane == 0) {
            sh_tot[bf] = tot;
            sh_cnt[bf] = (tot < hi ? tot : hi) - (tot < lo ? tot : lo);
            mbar_arrive(&mbar[bf]);
        }
    };
    uint32_t it = 0;                                             // staged chunks so far: buffer = it & 1, parity = (it >> 1) & 1
    if (warp == 0) {
        load_desc(blockIdx.x, cu_cnt, cu_src);
        load_desc(blockIdx.x + gridDim.x, nx_cnt, nx_src);
        if (blockIdx.x < sp.P) issue(cu_cnt, cu_src, 0, 0);
    }
    for (uint32_t p = blockIdx.x; p < sp.P; p += gridDim.x) {
        {   // empty table (16-byte stores)
            const ulonglong2 ff = make_ulonglong2(~0ull, ~0ull);
            for (uint32_t j = threadIdx.x; j < SMEM_SLOTS; j += blockDim.x) keys[j] = ff;
            uint4* cw = reinterpret_cast<uint4*>(ccs);
            for (uint32_t j = threadIdx.x; j < SMEM_SLOTS / 4; j += blockDim.x) cw[j] = make_uint4(0, 0, 0, 0);
        }
        if (threadIdx.x == 0) { sh_fail = 0; sh_nsolid = 0; }
        __syncthreads();
        auto insert = [&](const Kmer k, const uint32_t ctx) {
            uint32_t s = smem_slot_hash(k) >> (32 - sp.log_slots);
            bool done = false;
            for (uint32_t probe = 0; probe < SMEM_MAX_PROBE && !done; ++probe) {
                ulonglong2 cur = lds128_volatile(keys + s);
                while (cur.x != ~0ull && cur.y == ~0ull) cur = lds128_volatile(keys + s);      // (a slot caught half-written: no key has an all-ones second word)
                bool mine = cur.x == k.w0 && cur.y == k.w1;
                if (!mine && cur.x == ~0ull) {
                    const U128 old = cas128_shared(keys + s, ~0ull, ~0ull, k.w0, k.w1);
                    mine = (old.lo == ~0ull && old.hi == ~0ull) || (old.lo == k.w0 && old.hi == k.w1);
                }
                if (mine) {
                    // counts saturate at 255 downstream; the 24-bit field must not run into the context bits however many
                    // instances a k-mer has (a poly-G artefact can have 10^8): take the add back once the counter is far beyond 255
                    const uint32_t old = atomicAdd(ccs + s, 1u);
                    if ((old & 0xffffffu) >= COUNT_STOP) atomicSub(ccs + s, 1u);
                    if ((((old >> 24) & ctx) != ctx)) atomicOr(ccs + s, ctx << 24);
                    done = true;
                } else s = (s + 1u) & (SMEM_SLOTS - 1u);
            }
            if (!done) sh_fail = 1;
        };
        for (uint32_t c = 0;; ++c, ++it) {
            const uint32_t bf = it & 1u;
            mbar_wait(&mbar[bf], (it >> 1) & 1u);
            const uint32_t tot = sh_tot[bf], cnt = sh_cnt[bf];
            const bool more = (uint64_t)(c + 1) * SKM_CHUNK < tot;
            // the other buffer is free: everyone left it at the barrier that ended the previous chunk
            if (warp == 0) {
                if (more) issue(cu_cnt, cu_src, c + 1, bf ^ 1u);
                else {
                    if (p + gridDim.x < sp.P) issue(nx_cnt, nx_src, 0, bf ^ 1u);
                    cu_cnt = nx_cnt; cu_src = nx_src;
                    load_desc(p + 2 * gridDim.x, nx_cnt, nx_src);   // (in flight while this chunk and the next partition are counted)
                }
            }
            const SkmRec* st = stage + (size_t)bf * SKM_CHUNK;
            // Every warp takes an equal share of the chunk's records, in groups of <= 32 (a fixed deal of 32-record groups left most
            // warps idle in a partition's short last chunk: 24 % of all stall samples sat at the barrier below).  Inside a group the
            // k-mers are numbered consecutively across the records and lane l takes k-mer t + l.  Which record that is: the records that
            // START inside the 32-k-mer window are ORed into a bit mask (one REDUX), a population count of the mask below the lane gives
            // the record.
            const uint32_t share = (cnt + nwarp - 1) / nwarp;                       // records per warp
            const uint32_t w_end = (warp + 1) * share < cnt ? (warp + 1) * share : cnt;
            for (uint32_t g0 = warp * share; g0 < w_end; g0 += 32u) {
                const uint32_t gn = w_end - g0 < 32u ? w_end - g0 : 32u;            // records in this group
                const bool have = lane < gn;
                const uint64_t hdr = have ? st[g0 + lane].q[3] : 0ull;
                const uint32_t nr = have ? skm_n(hdr) : 0u;
                uint32_t incl = nr;
#pragma unroll
                for (int d = 1; d < 32; d <<= 1) { const uint32_t t = __shfl_up_sync(0xffffffffu, incl, d); if ((int)lane >= d) incl += t; }
                const uint32_t total = __shfl_sync(0xffffffffu, incl, 31), excl = incl - nr;
                uint32_t before_window = 0;                      // records that start before the window
                for (uint32_t t = 0; t < total; t += 32) {
                    const uint32_t rel = excl - t;               // (unsigned: records that start before the window wrap to huge values)
                    const unsigned starts = __reduce_or_sync(0xffffffffu, (nr && rel < 32u) ? 1u << rel : 0u);
                    const uint32_t rr = before_window + (uint32_t)__popc(starts & le_mask) - 1u;
                    const uint32_t r_excl = __shfl_sync(0xffffffffu, excl, rr & 31u);
                    const uint64_t r_hdr = __shfl_sync(0xffffffffu, hdr, rr & 31u);
                    if (t + lane < total) {
                        Kmer k; uint32_t ctx;
                        skm_kmer_at(st[g0 + rr].q, r_hdr, t + lane - r_excl, &k, &ctx);
                        insert(k, ctx);
                    }
                    before_window += (uint32_t)__popc(starts);
                }
            }
            __syncthreads();                                     // chunk consumed (and, after the last one, every insert has landed)
            if (!more) { ++it; break; }
        }
        // KEEP_COUNTS: the count of slot j is stashed at kept[j] from step 1 to step 5, because the sort word of step 3
        // (minimiser 13 | offset 6 | slot 13) has no room for it and the key's spare byte holds the context.  kept[] is the staging
        // buffer this partition's last chunk came through (buffer (it - 1) & 1): the barrier above was the last read of it, the
        // bulk copy into it has completed (waited on), and the next partition's chunk 0 is already in flight into the OTHER buffer.
        // Nothing is issued into this one before the next partition's first chunk has been waited for, which is after the barrier
        // that ends this partition.  It holds SKM_CHUNK * 32 = 32 KB; the counts take SMEM_SLOTS <= 8 KB.
        uint8_t* kept = reinterpret_cast<uint8_t*>(stage + (size_t)((it - 1u) & 1u) * SKM_CHUNK);
        const bool failed = sh_fail != 0;
        if (failed) {
            if (threadIdx.x == 0) sp.failed[atomicAdd(sp.failed_cursor, 1ull)] = p;
        } else {
            // 1. histogram and dump; a solid key takes its context into the free low byte of w1, every other key is cleared
            for (uint32_t base = 0; base < SMEM_SLOTS; base += blockDim.x) {
                const uint32_t j = base + threadIdx.x;
                const bool in = j < SMEM_SLOTS;
                const ulonglong2 kk = in ? keys[j] : make_ulonglong2(~0ull, ~0ull);
                const bool occ = kk.x != ~0ull;
                const uint32_t cc = in ? ccs[j] : 0u;
                uint32_t c = cc & 0xffffffu; if (c > 255u) c = 255u;
                const uint32_t ctx = cc >> 24;
                // histogram: the singletons (sequencing errors: most distinct k-mers) are counted per warp, the rest one by one
                const unsigned ones = __ballot_sync(0xffffffffu, occ && c == 1u);
                if (lane == 0 && ones) atomicAdd(&sh_hist[1], (unsigned)__popc(ones));
                if (occ && c != 1u) atomicAdd(&sh_hist[c > 100u ? 100u : c], 1u);
                if (occ) keys[j] = c >= sp.min_freq ? make_ulonglong2(kk.x, kk.y | ctx) : make_ulonglong2(~0ull, ~0ull);
                if (KEEP_COUNTS && in) kept[j] = (uint8_t)c;
                if (sp.dump_out) {
                    const uint64_t dp = warp_append(sp.dump_cursor, occ);
                    if (occ) sp.dump_out[dp] = DumpRec{kk.x, kk.y, c, ctx, NIL, 0};
                }
            }
            __syncthreads();
            // 2. the solid slots, compacted into the (now free) count array
            for (uint32_t base = 0; base < SMEM_SLOTS; base += blockDim.x) {
                const uint32_t j = base + threadIdx.x;
                const bool solid = j < SMEM_SLOTS && keys[j].x != ~0ull;
                const unsigned m = __ballot_sync(0xffffffffu, solid);
                uint32_t first = 0;
                if (lane == 0 && m) first = atomicAdd(&sh_nsolid, (uint32_t)__popc(m));
                first = __shfl_sync(0xffffffffu, first, 0);
                if (solid) ccs[first + __popc(m & (le_mask >> 1))] = j;
            }
            __syncthreads();
            // 3. one sort word per solid k-mer, in place (after the compaction every lane that computes a minimiser has a k-mer):
            // minimiser bits : 13 | offset : 6 | slot : 13
            const uint32_t ns = sh_nsolid, N = ns <= 1u ? ns : 1u << (32 - __clz(ns - 1u));
            for (uint32_t i = threadIdx.x; i < ns; i += blockDim.x) {
                const uint32_t j = ccs[i];
                const ulonglong2 kk = keys[j];
                uint32_t off;
                const uint32_t mh = kmer_minimizer_offset_words(Kmer{kk.x, kk.y & ~0xffull}, &off);
                ccs[i] = (mh & 0x1fffu) << 19 | off << 13 | j;
            }
            // 4. bitonic sort, ascending, over the next power of two (the pad words sort last)
            if (N <= blockDim.x) {
                // one word per thread in a register: pairs less than 32 apart meet by shuffles, wider ones through shared memory
                const uint32_t i = threadIdx.x;
                __syncthreads();
                uint32_t v = i < ns ? ccs[i] : ~0u;
                for (uint32_t kb = 2; kb <= N; kb <<= 1) {
                    for (uint32_t jb = kb >> 1; jb > 0; jb >>= 1) {
                        uint32_t o;
                        if (jb >= 32u) {
                            __syncthreads();
                            if (i < N) ccs[i] = v;
                            __syncthreads();
                            o = i < N ? ccs[i ^ jb] : ~0u;
                        } else o = __shfl_xor_sync(0xffffffffu, v, jb);
                        const bool keep_min = ((i & jb) == 0) == ((i & kb) == 0);
                        v = keep_min ? (v < o ? v : o) : (v < o ? o : v);
                    }
                }
                __syncthreads();
                if (i < N) ccs[i] = v;
            } else {
                // in shared memory: a substage whose pairs are at most 32 apart stays inside one warp's 64 words, so only the wider
                // ones need the whole CTA at a barrier
                for (uint32_t i = ns + threadIdx.x; i < N; i += blockDim.x) ccs[i] = ~0u;
                __syncthreads();
                for (uint32_t kb = 2; kb <= N; kb <<= 1) {
                    for (uint32_t jb = kb >> 1; jb > 0; jb >>= 1) {
                        if (jb > 32u) __syncthreads();
                        for (uint32_t t = threadIdx.x; t < N / 2; t += blockDim.x) {
                            const uint32_t i = 2 * t - (t & (jb - 1u));
                            const uint32_t a = ccs[i], b = ccs[i + jb];
                            if ((a > b) == ((i & kb) == 0)) { ccs[i] = b; ccs[i + jb] = a; }
                        }
                        if (jb > 32u) __syncthreads(); else __syncwarp();
                    }
                }
            }
            // 5. one cursor atomic per partition, the records in sorted order
            if (threadIdx.x == 0 && ns) sh_solid_base = atomicAdd(sp.solid_cursor, (unsigned long long)ns);
            __syncthreads();
            for (uint32_t i = threadIdx.x; i < ns; i += blockDim.x) {
                const uint64_t pos = sh_solid_base + i;
                if (pos < sp.solid_cap) {
                    const uint32_t j = ccs[i] & 0x1fffu;
                    sp.solid_out[pos] = keys[j];
                    if (KEEP_COUNTS) sp.count_out[pos] = kept[j];
                } else atomicExch(sp.solid_overflow, 1);
            }
        }
        __syncthreads();
    }
    __syncthreads();
    for (int j = threadIdx.x; j <= 100; j += blockDim.x) if (sh_hist[j]) atomicAdd(&sp.hist[j], (unsigned long long)sh_hist[j]);
}

struct ScanParams {
    CountSlot* region;
    uint64_t R;
    uint32_t min_freq;
    unsigned long long* hist;        // [104]: bins 1..100
    ulonglong2* solid_out;           // solid records {w0, w1 | ctx}
    unsigned long long* solid_cursor;
    uint64_t solid_cap;
    DumpRec* dump_out;               // test hook (dump level 2) or nullptr
    unsigned long long* dump_cursor;
    const int* overflow;             // if set: the group failed, only reset the region
    int* solid_overflow;
    uint8_t* count_out;              // or nullptr; else min(255, count) of solid_out[i] goes to count_out[i] (w2rap_step2_count)
};
// hist[min(100,min(255,count))]++ (BuildReadQGraph.cc:1094-1097), keep count >= minFreq (:1098), reset the region.
__global__ void __launch_bounds__(256) k_scan_region(ScanParams sp) {
    __shared__ unsigned int sh[104];
    for (int j = threadIdx.x; j < 104; j += blockDim.x) sh[j] = 0;
    __syncthreads();
    const bool failed = *sp.overflow != 0;
    uint4* raw = reinterpret_cast<uint4*>(sp.region);
    const uint4 key_empty = make_uint4(0xffffffffu, 0xffffffffu, 0xffffffffu, 0xffffffffu), zero = make_uint4(0, 0, 0, 0);
    for (uint64_t base = (uint64_t)blockIdx.x * blockDim.x; base < sp.R; base += (uint64_t)gridDim.x * blockDim.x) {
        uint64_t i = base + threadIdx.x;
        bool occ = false, solid = false;
        uint32_t c = 0, ctx = 0;
        ulonglong2 k = make_ulonglong2(0, 0);
        if (i < sp.R) {
            k = __ldcg(reinterpret_cast<const ulonglong2*>(sp.region + i));
            if (k.x != EMPTY_W0) {
                occ = true;
                uint2 m = __ldcg(reinterpret_cast<const uint2*>(&sp.region[i].count));
                c = m.x > 255u ? 255u : m.x; ctx = m.y & 0xffu;
                raw[2 * i] = key_empty; raw[2 * i + 1] = zero;
            }
        }
        if (failed) continue;
        uint32_t bin = occ ? (c > 100u ? 100u : c) : 103u;
        unsigned peers = __match_any_sync(0xffffffffu, bin);
        if (occ && (peers & ((1u << lane_id()) - 1u)) == 0) atomicAdd(&sh[bin], (unsigned)__popc(peers));
        solid = occ && c >= sp.min_freq;
        uint64_t pos = warp_append(sp.solid_cursor, solid);
        if (solid) {
            if (pos < sp.solid_cap) { sp.solid_out[pos] = make_ulonglong2(k.x, k.y | ctx); if (sp.count_out) sp.count_out[pos] = (uint8_t)c; }
            else atomicExch(sp.solid_overflow, 1);
        }
        if (sp.dump_out) {
            uint64_t dp = warp_append(sp.dump_cursor, occ);
            if (occ) sp.dump_out[dp] = DumpRec{k.x, k.y, c, ctx, NIL, 0};
        }
    }
    __syncthreads();
    if (!failed) {
        for (int j = threadIdx.x; j <= 100; j += blockDim.x) if (sh[j]) atomicAdd(&sp.hist[j], (unsigned long long)sh[j]);
    }
}

// ---------------------------------------------------------------- selection from kept counts (w2rap_step2_build)
// The records a count kept (every k-mer seen >= f0 times, in the reduce's order) with count >= min_freq, compacted STABLY into
// the solid array: the reduce emits each partition's records sorted by minimiser and offset, and that order gives the k-mers of a
// chain neighbouring node ids in the graph stage (unipath.cuh: DenseNodes).  An append by warp aggregation would scramble it.
// Tile t = records [t * SCAN_TILE, +SCAN_TILE), thread i of it holds the SCAN_ITEMS consecutive records from i * SCAN_ITEMS (one
// 8-byte load of their counts): selected per tile, an exclusive scan of the tile sums (prims.cuh), then an in-order scatter.
static_assert(SCAN_ITEMS == 8, "one 8-byte load of counts per thread");
__device__ __forceinline__ uint32_t select_mask(const uint8_t* __restrict__ count, uint64_t n, uint64_t base, uint32_t min_freq) {
    uint32_t m = 0;
    if (base + SCAN_ITEMS <= n) {
        const uint64_t w = *reinterpret_cast<const uint64_t*>(count + base);
#pragma unroll
        for (int i = 0; i < SCAN_ITEMS; ++i) if (((w >> (8 * i)) & 0xffu) >= min_freq) m |= 1u << i;
    } else {
        for (int i = 0; base + i < n; ++i) if (count[base + i] >= min_freq) m |= 1u << i;
    }
    return m;
}
__global__ void __launch_bounds__(SCAN_THREADS) k_select_tile_counts(const uint8_t* __restrict__ count, uint64_t n, uint32_t min_freq, uint32_t* __restrict__ tile_n) {
    __shared__ uint32_t sm[33];
    const uint64_t base = (uint64_t)blockIdx.x * SCAN_TILE + (uint64_t)threadIdx.x * SCAN_ITEMS;
    uint32_t total;
    block_exclusive_scan<uint32_t>((uint32_t)__popc(select_mask(count, n, base, min_freq)), &total, sm);
    if (threadIdx.x == 0) tile_n[blockIdx.x] = total;
}
__global__ void __launch_bounds__(SCAN_THREADS) k_select_solid(const ulonglong2* __restrict__ kept, const uint8_t* __restrict__ count, uint64_t n, uint32_t min_freq,
                                                               const uint64_t* __restrict__ tile_base, ulonglong2* __restrict__ solid) {
    __shared__ uint32_t sm[33];
    const uint64_t base = (uint64_t)blockIdx.x * SCAN_TILE + (uint64_t)threadIdx.x * SCAN_ITEMS;
    uint32_t m = select_mask(count, n, base, min_freq), total;
    uint64_t pos = tile_base[blockIdx.x] + block_exclusive_scan<uint32_t>((uint32_t)__popc(m), &total, sm);
    for (; m; m &= m - 1u) solid[pos++] = kept[base + (uint32_t)(__ffs((int)m) - 1)];
}

}  // namespace w2r
