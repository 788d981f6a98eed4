// coverage.cuh — k-mer coverage of packed sequences from the counts a w2rap_step2_count kept (include/w2rap_coverage.h).
//
// Index: the dictionary's own open-addressing table (kmer.cuh: SolidTable), one slot per kept k-mer, whose `ctx` word holds the
// kept count instead of a context.  Lookups: every sequence is cut into tiles of COV_TILE k-mer positions; a warp takes one tile,
// lane j the positions j, j+32, ... of it, so that one long edge (up to 2^24 k-mers) spreads over many warps and a read is one
// tile.  Each lane accumulates in registers, the warp reduces, and one lane adds the tile into the sequence's totals with atomics.
// The per-tile body is host/device code, so tests/hostcheck/coverage.cpp runs it serially against the oracle's counts.
#pragma once
#include <stdint.h>

#include "kmer.cuh"
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

// Lane `lane` of the tile [lo, hi) of a sequence's k-mer positions: positions lo + lane, lo + lane + 32, ...  The canonical
// k-mer is the smaller of the k-mer and its reverse complement (a palindrome is its own), the form the reduce stored.
W2R_HD CovAcc cov_tile_lane(const SolidTable& t, const uint8_t* seq, uint64_t lo, uint64_t hi, uint32_t lane) {
    CovAcc a = cov_empty();
    for (uint64_t p = lo + lane; p < hi; p += 32) {
        Kmer f, r;
        kmer_pair_at(seq, p, &f, &r);
        const uint32_t c = cov_count(t, kmer_less(r, f) ? r : f);
        a.sum += c; a.absent += c == 0;
        if (c < a.mn) a.mn = c;
        if (c > a.mx) a.mx = c;
    }
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
#endif

}  // namespace w2r
