// coverage.cuh — k-mer coverage of packed sequences from the counts a w2rap_step2_count kept (include/w2rap_coverage.h).
//
// Index: the dictionary's own open-addressing table (kmer.cuh: SolidTable), one slot per kept k-mer, whose `ctx` word holds the
// kept count instead of a context.  Lookups: every sequence is cut into tiles of COV_TILE k-mer positions; a warp takes one tile,
// lane j the positions j, j+32, ... of it, so that one long edge (up to 2^24 k-mers) spreads over many warps and a read is one
// tile.  Each lane accumulates in registers, the warp reduces, and one lane adds the tile into the sequence's totals with atomics.
// The per-tile body is host/device code, so tests/hostcheck/coverage.cpp runs it serially against the oracle's counts.
// Sharded counts: k_cov_tiles_owned looks up only the positions whose k-mer this rank owns; the ranks' totals are then merged.
#pragma once
#include <stdint.h>

#include "extract.cuh"                // minimisers: the owner of a k-mer in a sharded count
#include "kmer.cuh"
#include "shard.cuh"
#if defined(__CUDACC__)
#include "kernels.cuh"              // cas128
#endif

namespace w2r {

constexpr uint32_t COV_TILE = 512;          // k-mer positions per tile (16 per lane)

struct CovAcc { uint64_t sum; uint32_t absent, mn, mx; };
W2R_HD CovAcc cov_empty() { return CovAcc{0, 0, 0xffffffffu, 0}; }
W2R_HD void cov_merge(CovAcc* a, const CovAcc& b) {
    a->sum += b.sum; a->absent += b.absent;
    if (b.mn < a->mn) a->mn = b.mn;
    if (b.mx > a->mx) a->mx = b.mx;
}

W2R_HD uint64_t cov_kmers_of(uint32_t len) { return len >= (uint32_t)K ? (uint64_t)len - (K - 1) : 0; }
W2R_HD uint32_t cov_tiles_of(uint32_t len) { return (uint32_t)((cov_kmers_of(len) + COV_TILE - 1) / COV_TILE); }

// The sequence tile t belongs to: the last i with tile_base[i] <= t (tile_base = exclusive scan of cov_tiles_of; sequences without
// k-mers share their successor's base and are never chosen).
W2R_HD uint64_t cov_tile_owner(const uint64_t* tile_base, uint64_t n, uint64_t t) {
    uint64_t lo = 0, hi = n;                // first index with tile_base > t lies in [lo, hi]
    while (lo < hi) {
        const uint64_t mid = lo + (hi - lo) / 2;
        if (tile_base[mid] <= t) lo = mid + 1; else hi = mid;
    }
    return lo - 1;
}

// The kept count of a canonical k-mer, 0 if it was not kept.
W2R_HD uint32_t cov_count(const SolidTable& t, Kmer canon) {
    const int64_t h = solid_find(t, canon);
    return h < 0 ? 0u : t.slots[h].ctx;
}

// Adds the k-mer at position p of a sequence.  The canonical k-mer is the smaller of the k-mer and its reverse complement (a
// palindrome is its own), the form the reduce stored.
W2R_HD void cov_add_at(CovAcc* a, const SolidTable& t, const uint8_t* seq, uint64_t p) {
    Kmer f, r;
    kmer_pair_at(seq, p, &f, &r);
    const uint32_t c = cov_count(t, kmer_less(r, f) ? r : f);
    a->sum += c; a->absent += c == 0;
    if (c < a->mn) a->mn = c;
    if (c > a->mx) a->mx = c;
}

// Lane `lane` of the tile [lo, hi) of a sequence's k-mer positions: positions lo + lane, lo + lane + 32, ...
W2R_HD CovAcc cov_tile_lane(const SolidTable& t, const uint8_t* seq, uint64_t lo, uint64_t hi, uint32_t lane) {
    CovAcc a = cov_empty();
    for (uint64_t p = lo + lane; p < hi; p += 32) cov_add_at(&a, t, seq, p);
    return a;
}

// ---- sharded counts (include/w2rap_step2_counts_sharded.h).  Every rank holds the kept k-mers of the minimiser partitions it owns,
// so a k-mer position is looked up on its owner only, and every position has exactly one.  The owner is the rank the map routes the
// k-mer to (count_part.cuh): the minimum of its 46 m-mer hashes, re-mixed, gives the partition.  That minimum is the same for a k-mer
// and its reverse complement, so the strand a query holds does not matter.  Reference form; k_cov_tiles_owned gets the same minima
// for 32 positions at a time from shuffles.
W2R_HD uint32_t cov_owner_at(const uint8_t* seq, uint64_t p, uint32_t logP, uint32_t world) {
    return owner_of_partition(mini_part(mini_mix(kmer_minimizer_hash(seq, p)), logP), logP, world);
}

// Lane `lane` of the tile [lo, hi), positions rank `me` owns only: what k_cov_tiles_owned adds up on that rank, serially.
W2R_HD CovAcc cov_tile_lane_owned(const SolidTable& t, const uint8_t* seq, uint64_t lo, uint64_t hi, uint32_t lane, uint32_t logP, uint32_t world,
                                  uint32_t me) {
    CovAcc a = cov_empty();
    for (uint64_t p = lo + lane; p < hi; p += 32)
        if (cov_owner_at(seq, p, logP, world) == me) cov_add_at(&a, t, seq, p);
    return a;
}

#if defined(__CUDACC__)
// Index build: keys are unique, so a successful CAS owns the slot (as k_insert_solid).  Records are {w0, w1 | raw ctx}.
__global__ void k_insert_counts(const ulonglong2* __restrict__ recs, const uint8_t* __restrict__ count, uint64_t n, SolidTable st) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        const ulonglong2 rec = __ldcs(recs + i);
        const Kmer k{rec.x, rec.y & ~0xffull};
        uint64_t h = st.home(k);
        for (;;) {
            SolidSlot* p = st.slots + h;
            const U128 old = cas128(p, ~0ull, ~0ull, k.w0, k.w1);
            if (old.lo == ~0ull && old.hi == ~0ull) { p->ctx = count[i]; p->edge = NIL; p->off = 0; p->pad = 0; break; }
            h = st.next(h);
        }
    }
}

// The device image of w2rap_seq_cov.
struct SeqCov { unsigned long long n_kmers, sum, n_absent; uint32_t mn, mx; };

// Per sequence: its tile count (for the scan) and its initial totals.
__global__ void k_cov_init(const uint32_t* __restrict__ len, uint64_t n, uint32_t* __restrict__ tiles, SeqCov* __restrict__ out) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t L = len[i];
        const uint64_t nk = cov_kmers_of(L);
        tiles[i] = cov_tiles_of(L);
        out[i] = SeqCov{nk, 0, 0, nk ? 0xffffffffu : 0u, 0};
    }
}

// One warp per tile (grid-stride over the tiles).
__global__ void k_cov_tiles(SolidTable st, const uint8_t* __restrict__ bases, const uint64_t* __restrict__ base_off, const uint32_t* __restrict__ len,
                            const uint64_t* __restrict__ tile_base, uint64_t n, uint64_t n_tiles, SeqCov* __restrict__ out) {
    const uint32_t lane = threadIdx.x & 31u;
    const uint64_t warps = (uint64_t)gridDim.x * (blockDim.x >> 5);
    for (uint64_t t = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; t < n_tiles; t += warps) {
        const uint64_t i = cov_tile_owner(tile_base, n, t);
        const uint64_t lo = (t - tile_base[i]) * COV_TILE;
        const uint64_t nk = cov_kmers_of(len[i]);
        const uint64_t hi = lo + COV_TILE < nk ? lo + COV_TILE : nk;
        CovAcc a = cov_tile_lane(st, bases + base_off[i], lo, hi, lane);
        unsigned long long sum = a.sum;
        uint32_t absent = a.absent;
#pragma unroll
        for (int d = 16; d; d >>= 1) { sum += __shfl_xor_sync(0xffffffffu, sum, d); absent += __shfl_xor_sync(0xffffffffu, absent, d); }
        const uint32_t mn = __reduce_min_sync(0xffffffffu, a.mn), mx = __reduce_max_sync(0xffffffffu, a.mx);
        if (lane == 0) {
            atomicAdd(&out[i].sum, sum);
            if (absent) atomicAdd(&out[i].n_absent, (unsigned long long)absent);
            atomicMin(&out[i].mn, mn);
            atomicMax(&out[i].mx, mx);
        }
    }
}

// Per-rank partial totals of a sharded lookup, laid out for the merge: sum[0..n) and absent[0..n) are one array of 2n words
// (all-reduce sum), mn[0..n) (all-reduce min) and mx[0..n) (all-reduce max) are two more.
struct CovParts { unsigned long long *sum, *absent; uint32_t *mn, *mx; };

// k_cov_tiles over a sharded count: one warp per tile, as there, but only positions this rank owns are looked up.  A step covers the
// 32 consecutive positions p0 + lane.  The window minima come from the m-mer hashes of the step's 77-position span in three registers
// per lane (positions p0 + lane, + 32, + 64; two carry over to the next step, so a lane hashes one m-mer per step), five doubling
// steps of shuffles (min over 32 consecutive hashes) and the 46-wide window as two overlapping 32-wide ones, 14 apart, as in
// k_minimizer_map.  About 1/world of the positions are owned: the owned ones of the whole tile are compacted into a shared-memory
// list by ballot, so that the probes then run 32 per round instead of on 1/world of the lanes of every step.
constexpr uint32_t COV_OWNED_THREADS = 256;
__global__ void __launch_bounds__(COV_OWNED_THREADS) k_cov_tiles_owned(SolidTable st, const uint8_t* __restrict__ bases, const uint64_t* __restrict__ base_off,
                                                                     const uint32_t* __restrict__ len, const uint64_t* __restrict__ tile_base, uint64_t n,
                                                                     uint64_t n_tiles, uint32_t logP, uint32_t world, uint32_t me, CovParts out) {
    __shared__ uint16_t owned_buf[COV_OWNED_THREADS / 32][COV_TILE];     // tile offsets of this warp's owned positions
    uint16_t* owned = owned_buf[threadIdx.x >> 5];
    const uint32_t lane = threadIdx.x & 31u;
    const unsigned below = (1u << lane) - 1u;
    const uint64_t warps = (uint64_t)gridDim.x * (blockDim.x >> 5);
    for (uint64_t t = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; t < n_tiles; t += warps) {
        const uint64_t i = cov_tile_owner(tile_base, n, t);
        const uint64_t lo = (t - tile_base[i]) * COV_TILE;
        const uint64_t nk = cov_kmers_of(len[i]);
        const uint64_t hi = lo + COV_TILE < nk ? lo + COV_TILE : nk;
        const uint8_t* seq = bases + base_off[i];
        const uint64_t n_h = nk + MINI_W - 1;                       // m-mers of the sequence: the windows of positions < nk
        uint32_t r0 = lo + lane < n_h ? mmer_hash_at(seq, lo + lane) : 0xffffffffu;
        uint32_t r1 = lo + 32 + lane < n_h ? mmer_hash_at(seq, lo + 32 + lane) : 0xffffffffu;
        uint32_t n_owned = 0;
        for (uint64_t p0 = lo; p0 < hi; p0 += 32) {
            const uint32_t r2 = p0 + 64 + lane < n_h ? mmer_hash_at(seq, p0 + 64 + lane) : 0xffffffffu;
            uint32_t m0 = r0, m1 = r1, m2 = r2;
#pragma unroll
            for (uint32_t s = 1; s <= 16; s <<= 1) {                 // after these: m_u = min of the 32 hashes from p0 + 32u + lane
                const uint32_t src = (lane + s) & 31u;
                const bool wrap = lane + s >= 32u;
                const uint32_t x0 = __shfl_sync(0xffffffffu, m0, src), x1 = __shfl_sync(0xffffffffu, m1, src), x2 = __shfl_sync(0xffffffffu, m2, src);
                m0 = min(m0, wrap ? x1 : x0);
                m1 = min(m1, wrap ? x2 : x1);
                m2 = min(m2, wrap ? 0xffffffffu : x2);
            }
            const uint32_t src = (lane + (MINI_W - 32)) & 31u;
            const bool wrap = lane + (MINI_W - 32) >= 32u;
            const uint32_t y0 = __shfl_sync(0xffffffffu, m0, src), y1 = __shfl_sync(0xffffffffu, m1, src);
            const uint32_t wmin = min(m0, wrap ? y1 : y0);           // the minimiser hash of the k-mer at p0 + lane
            const bool mine = p0 + lane < hi && owner_of_partition(mini_part(mini_mix(wmin), logP), logP, world) == me;
            const unsigned b = __ballot_sync(0xffffffffu, mine);
            if (mine) owned[n_owned + __popc(b & below)] = (uint16_t)(p0 - lo + lane);
            n_owned += __popc(b);
            r0 = r1; r1 = r2;
        }
        if (!n_owned) continue;                                     // (warp-uniform)
        __syncwarp();
        CovAcc a = cov_empty();
        for (uint32_t j = lane; j < n_owned; j += 32) cov_add_at(&a, st, seq, lo + owned[j]);
        unsigned long long sum = a.sum;
        uint32_t absent = a.absent;
#pragma unroll
        for (int d = 16; d; d >>= 1) { sum += __shfl_xor_sync(0xffffffffu, sum, d); absent += __shfl_xor_sync(0xffffffffu, absent, d); }
        const uint32_t mn = __reduce_min_sync(0xffffffffu, a.mn), mx = __reduce_max_sync(0xffffffffu, a.mx);
        if (lane == 0) {
            atomicAdd(&out.sum[i], sum);
            if (absent) atomicAdd(&out.absent[i], (unsigned long long)absent);
            atomicMin(&out.mn[i], mn);
            atomicMax(&out.mx[i], mx);
        }
        __syncwarp();                                               // the list is read before the next tile overwrites it
    }
}

// The merged partials into the totals k_cov_init made.  Its min, 0xffffffff for a sequence with k-mers and 0 without, takes the
// merged min; every position of a sequence with k-mers has one owner, so that min is a kept count or 0.
__global__ void k_cov_gather(const unsigned long long* __restrict__ sum_absent, const uint32_t* __restrict__ mn, const uint32_t* __restrict__ mx, uint64_t n,
                             SeqCov* __restrict__ out) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        out[i].sum = sum_absent[i];
        out[i].n_absent = sum_absent[n + i];
        if (mn[i] < out[i].mn) out[i].mn = mn[i];
        out[i].mx = mx[i];
    }
}
#endif

}  // namespace w2r
