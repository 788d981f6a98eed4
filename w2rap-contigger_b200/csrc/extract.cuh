// extract.cuh — per-read canonical 60-mer + context extraction (the leaf loop of createDictOMPRecursive,
// paths/long/BuildReadQGraph.cc:1062-1080) as a host/device function over a packed read.
#pragma once
#include "kmer.cuh"

namespace w2r {

// Resumable form of the extraction loop: open() a read, then next() yields one (canonical k-mer, context) at a time.
//   - only reads with good_len > K contribute (BuildReadQGraph.cc:1064)
//   - first k-mer: successor bit only; last: predecessor bit only (:1066-1078)
//   - REV k-mers are stored reverse-complemented with the context bit-reversed (:1069,1074,1078); palindromes as seen.
struct KmerCursor {
    const uint8_t* bases;
    Kmer f, r;
    uint64_t buf;             // the next bases of the read, 32 at a time (one pair of 8-byte loads per 32 k-mers)
    uint32_t j, last, prev_first;
    bool live;
    W2R_HD KmerCursor() : bases(nullptr), f{0, 0}, r{0, 0}, buf(0), j(0), last(0), prev_first(0), live(false) {}
    W2R_HD void open(const uint8_t* b, uint32_t good_len) {
        live = good_len > (uint32_t)K;
        if (!live) return;
        bases = b; f = kmer_at(b, 0); r = kmer_rc(f); last = good_len - K; j = 0; prev_first = 0; buf = 0;
    }
    W2R_HD bool next(Kmer* canon, uint32_t* ctx) {
        if (!live) return false;
        uint32_t nxt = 0, c = 0;
        if ((j & 31u) == 0) buf = bases32_at(bases, (uint64_t)j + K);
        if (j < last) { nxt = (uint32_t)buf & 3u; c |= 1u << nxt; }
        buf >>= 2;
        if (j > 0) c |= 16u << prev_first;
        const bool rev = kmer_less(r, f);       // select first, emit once: no divergent copies of the consumer
        *canon = Kmer{rev ? r.w0 : f.w0, rev ? r.w1 : f.w1};
        *ctx = rev ? ctx_rc(c) : c;
        if (j == last) live = false;
        else { prev_first = kmer_first(f); f = kmer_succ(f, nxt); r = kmer_pred(r, 3u - nxt); ++j; }
        return true;
    }
};

// Calls emit(canonical k-mer, context byte) for every k-mer of the quality-floored read prefix [0, good_len).
template <class Emit>
W2R_HD void extract_read_kmers(const uint8_t* bases, uint32_t good_len, Emit& emit) {
    KmerCursor cur;
    cur.open(bases, good_len);
    Kmer k; uint32_t ctx;
    while (cur.next(&k, &ctx)) emit(k, ctx);
}

// ---------------------------------------------------------------- super-k-mer records (the unit the map hands to the reduce)
// Consecutive k-mers of a read that fall into the same partition are shipped as ONE 32-byte record instead of one 16-byte
// record each: the n <= 32 k-mers share n + 59 bases, plus one base on either side when the read has one there (it carries the
// predecessor context of the first k-mer / the successor context of the last; BuildReadQGraph.cc:1066-1078).  Layout:
//   q[0..2]  bases, 2 bits each, LSB-first exactly as in the packed read (base i of the record in bits 2i..2i+1), <= 93 bases
//   q[3]     header: bits 56-60 n-1, bit 61 hp (a base precedes the first k-mer), bit 62 hs (a base follows the last k-mer)
// ~13-18 k-mers per record on 250-base reads: ~2 bytes per k-mer instance instead of 16, through HBM and through NVLink.
constexpr uint32_t SKM_MAX = 32;
struct alignas(16) SkmRec { uint64_t q[4]; };
W2R_HD uint32_t skm_n(uint64_t hdr) { return (uint32_t)((hdr >> 56) & 31u) + 1u; }
// Record for the n k-mers starting at k-mer position j_first of a read whose last k-mer position is `last` (= good_len - K).
W2R_HD SkmRec skm_build(const uint8_t* bases, uint32_t j_first, uint32_t n, uint32_t last) {
    const uint32_t hp = j_first > 0 ? 1u : 0u, hs = j_first + n - 1u < last ? 1u : 0u;
    const uint64_t p0 = (uint64_t)j_first - hp;
    const uint32_t bits = 2u * (n + (uint32_t)K - 1u + hp + hs);                 // 120 .. 186
    const uintptr_t addr = (uintptr_t)bases + (uintptr_t)(p0 >> 2);
    const uint64_t* w = (const uint64_t*)(addr & ~(uintptr_t)7);
    const uint32_t sh = (uint32_t)(addr & 7u) * 8u + (uint32_t)(p0 & 3u) * 2u;  // 0..62
    const uint64_t a = w[0], b = w[1], c = w[2], d = w[3];
    SkmRec r;
    r.q[0] = sh ? (a >> sh) | (b << (64u - sh)) : a;
    r.q[1] = sh ? (b >> sh) | (c << (64u - sh)) : b;
    r.q[2] = sh ? (c >> sh) | (d << (64u - sh)) : c;
    if (bits < 128u) { r.q[1] &= (1ull << (bits - 64u)) - 1ull; r.q[2] = 0; }
    else if (bits < 192u) r.q[2] = bits > 128u ? r.q[2] & ((1ull << (bits - 128u)) - 1ull) : 0ull;
    r.q[3] = ((uint64_t)(n - 1u) << 56) | ((uint64_t)hp << 61) | ((uint64_t)hs << 62);
    return r;
}
// K-mer j (< n) of a record: canonical form and context byte, exactly what extract_read_kmers emits for that read position.
// `q` may point to global, shared or host memory.
W2R_HD void skm_kmer_at(const uint64_t* q, uint64_t hdr /* = q[3] */, uint32_t j, Kmer* canon, uint32_t* ctx) {
    const uint32_t n = skm_n(hdr), hp = (uint32_t)(hdr >> 61) & 1u, hs = (uint32_t)(hdr >> 62) & 1u;
    const uint32_t b = 2u * (hp + j), wo = b >> 6, sh = b & 63u;                // b <= 66: wo is 0 or 1
    const uint64_t A = q[wo], B = q[wo + 1], C = wo ? 0ull : q[2];              // wo == 1: C only reaches bits that are masked off
    const uint64_t lo = sh ? (A >> sh) | (B << (64u - sh)) : A;
    const uint64_t hi = sh ? (B >> sh) | (C << (64u - sh)) : B;
    const Kmer f{rev2(lo), rev2(hi) & ~0xffull};
    const Kmer rc{(~hi << 8) | (~lo >> 56), ~lo << 8};                           // as in kmer_pair_at
    uint32_t c = 0;
    if (j + 1u < n || hs) c |= 1u << ((uint32_t)(hi >> 56) & 3u);                // the base after the k-mer
    if (j > 0u || hp) c |= 16u << (sh ? (uint32_t)(A >> (sh - 2u)) & 3u : (uint32_t)(q[wo - 1] >> 62));   // sh == 0 here means b == 64
    const bool rev = kmer_less(rc, f);
    *canon = Kmer{rev ? rc.w0 : f.w0, rev ? rc.w1 : f.w1};
    *ctx = rev ? ctx_rc(c) : c;
}
W2R_HD void skm_kmer_at(const uint64_t* q, uint32_t j, Kmer* canon, uint32_t* ctx) { skm_kmer_at(q, q[3], j, canon, ctx); }

// ---------------------------------------------------------------- minimisers (partition key of the single-GPU count)
// The partition of a k-mer is derived from its MINIMISER: the canonical 15-mer with the smallest hash among the 46 inside the
// k-mer.  It is strand-symmetric (a k-mer and its reverse complement contain the same canonical m-mers), so every instance of a
// canonical k-mer lands in the same partition, and consecutive k-mers of a read share it for ~24 positions on average: a read
// appends RUNS of records to a partition (one cursor atomic per run, contiguous stores) instead of scattering single records.
// The counts do not depend on the partition function; this is purely a data-movement choice (the reference's own bucketing,
// MapReduceEngine.h:288-358, hashes whole k-mers).
constexpr int MINI_M = 15;
constexpr int MINI_W = K - MINI_M + 1;     // m-mers per k-mer
// hash of the canonical m-mer starting at base `pos` (a bijection of its 30-bit value, so equal hash <=> equal canonical m-mer)
W2R_HD uint32_t mmer_rc(uint32_t v) { return rev2_32(~v) >> (32 - 2 * MINI_M); }             // reverse complement, same encoding
W2R_HD uint32_t mmer_mix(uint32_t c) { c ^= c >> 16; c *= 0x85ebca6bu; c ^= c >> 13; c *= 0xc2b2ae35u; c ^= c >> 16; return c; }
W2R_HD uint32_t mmer_hash_of(uint32_t v) {                                                   // v: the m-mer, first base in bits 1:0
    const uint32_t rc = mmer_rc(v);
    return mmer_mix(v < rc ? v : rc);
}
W2R_HD uint32_t mmer_hash_at(const uint8_t* bases, uint64_t pos) { return mmer_hash_of(bases16_at(bases, pos) & ((1u << (2 * MINI_M)) - 1u)); }
// window minima are biased towards 0: re-mix before taking partition bits (top) and pass bits (low 16)
W2R_HD uint32_t mini_mix(uint32_t wmin) {
    uint32_t x = wmin * 0x9e3779b1u;
    x ^= x >> 15; x *= 0x2c1b3c6du; x ^= x >> 13;
    return x;
}
W2R_HD uint32_t mini_part(uint32_t mixed, uint32_t logP) { return logP ? mixed >> (32u - logP) : 0u; }
// the minimiser hash of a k-mer given as words (either orientation gives the same value): the graph stage of a sharded run asks
// "which rank owns this neighbour k-mer" (shardgraph.cuh)
W2R_HD uint32_t kmer_minimizer_hash_words(Kmer k) {
    const uint64_t lo = rev2(k.w0), hi = rev2(k.w1);          // LSB-first like a packed read: base i in bits 2i.. of hi:lo
    uint32_t m = 0xffffffffu;
    for (int t = 0; t < MINI_W; ++t) {
        const int bit = 2 * t;
        const uint64_t w = bit == 0 ? lo : (bit < 64 ? (lo >> bit) | (hi << (64 - bit)) : hi >> (bit - 64));
        const uint32_t h = mmer_hash_of((uint32_t)w & ((1u << (2 * MINI_M)) - 1u));
        if (h < m) m = h;
    }
    return m;
}
// The same minimiser hash, and in *offset where the minimiser sits, normalised for strand: q if the canonical m-mer occurs forward
// at base q of k, MINI_W - 1 - q if it occurs reverse-complemented there.  A k-mer and its reverse complement get the same offset,
// and along a stretch of genome that keeps its minimiser the offset steps by exactly one per k-mer, whichever strand each k-mer is
// stored in: sorting a partition's k-mers by (minimiser, offset) puts the k-mers of a chain next to each other (the reduce does
// that, count_part.cuh).  A minimiser that occurs twice takes the smaller offset, which keeps the offset strand-symmetric.
W2R_HD uint32_t mmer_bits_at(uint64_t lo, uint64_t hi, int bit) {        // the 15 bases from 2-bit group bit/2 of hi:lo
    const uint64_t w = bit == 0 ? lo : (bit < 64 ? (lo >> bit) | (hi << (64 - bit)) : hi >> (bit - 64));
    return (uint32_t)w & ((1u << (2 * MINI_M)) - 1u);
}
W2R_HD uint32_t kmer_minimizer_offset_words(Kmer k, uint32_t* offset) {
    const uint64_t lo = rev2(k.w0), hi = rev2(k.w1);                  // the k-mer LSB-first (base i in bits 2i..2i+1 of hi:lo)
    const uint64_t rlo = (~k.w1 >> 8) | (~k.w0 << 56), rhi = ~k.w0 >> 8; // its reverse complement LSB-first: the complement moved down 8
    uint32_t m = 0xffffffffu, off = 0;
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for (int t = 0; t < MINI_W; ++t) {
        const uint32_t v = mmer_bits_at(lo, hi, 2 * t), rc = mmer_bits_at(rlo, rhi, 2 * (MINI_W - 1 - t));   // rc == mmer_rc(v)
        const uint32_t h = mmer_mix(v < rc ? v : rc), o = v < rc ? (uint32_t)t : (uint32_t)(MINI_W - 1 - t);
        if (h < m || (h == m && o < off)) { m = h; off = o; }
    }
    *offset = off;
    return m;
}
// reference form for tests: the minimiser hash of the k-mer starting at base j
W2R_HD uint32_t kmer_minimizer_hash(const uint8_t* bases, uint64_t j) {
    uint32_t m = 0xffffffffu;
    for (int t = 0; t < MINI_W; ++t) { const uint32_t h = mmer_hash_at(bases, j + t); if (h < m) m = h; }
    return m;
}

}  // namespace w2r
