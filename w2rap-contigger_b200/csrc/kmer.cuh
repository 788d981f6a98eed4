// kmer.cuh — 60-mer arithmetic, context bytes, hashing and the two open-addressing tables.
//
// Everything here is W2R_HD (host + device) so that the same code the kernels run can be unit-tested on the host
// (tests/hostcheck) against the oracle.  The product library only ever runs it on the device.
//
// K-mer layout = the reference's KMer<60> (kmers/KMer.h:155-162): two u64 words, base 0 in bits 63-62 of w0,
// bases 32..59 in bits 63..8 of w1, low 8 bits of w1 zero.  Unsigned (w0,w1) order == the reference's operator<
// (kmers/KMer.h:312-319) == lexicographic order with A<C<G<T.
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define W2R_HD __host__ __device__ __forceinline__
#else
#define W2R_HD inline
#endif

namespace w2r {

constexpr int K = 60;
constexpr uint32_t NIL = 0xffffffffu;
constexpr uint64_t EMPTY_W0 = ~0ull;   // a canonical 60-mer never has 32 leading T's (its RC would start with 28+ A's and be smaller)

struct Kmer { uint64_t w0, w1; };

W2R_HD bool operator==(Kmer a, Kmer b) { return a.w0 == b.w0 && a.w1 == b.w1; }
W2R_HD bool kmer_less(Kmer a, Kmer b) { return a.w0 < b.w0 || (a.w0 == b.w0 && a.w1 < b.w1); }

// kmers/KMer.h:191-203 toSuccessor / :176-189 toPredecessor
W2R_HD Kmer kmer_succ(Kmer k, uint32_t b) { return Kmer{(k.w0 << 2) | (k.w1 >> 62), (k.w1 << 2) | ((uint64_t)b << 8)}; }
W2R_HD Kmer kmer_pred(Kmer k, uint32_t b) { return Kmer{(k.w0 >> 2) | ((uint64_t)b << 62), ((k.w1 >> 2) | (k.w0 << 62)) & ~0xffull}; }

// reverse the order of the 32 two-bit groups of a word
W2R_HD uint64_t rev2(uint64_t x) {
#if defined(__CUDA_ARCH__)
    x = __brevll(x);
    return ((x & 0xaaaaaaaaaaaaaaaaull) >> 1) | ((x & 0x5555555555555555ull) << 1);
#else
    x = ((x >> 2) & 0x3333333333333333ull) | ((x & 0x3333333333333333ull) << 2);
    x = ((x >> 4) & 0x0f0f0f0f0f0f0f0full) | ((x & 0x0f0f0f0f0f0f0f0full) << 4);
    x = ((x >> 8) & 0x00ff00ff00ff00ffull) | ((x & 0x00ff00ff00ff00ffull) << 8);
    x = ((x >> 16) & 0x0000ffff0000ffffull) | ((x & 0x0000ffff0000ffffull) << 16);
    return (x >> 32) | (x << 32);
#endif
}
// kmers/KMer.h:205-227 rc(): complement, reverse the 60 bases, re-align to the top.
W2R_HD Kmer kmer_rc(Kmer k) {
    // 128-bit value V = w0:w1 holds 60 bases then 8 zero bits.  Reverse all 64 groups of ~V: the 4 pad groups come first.
    uint64_t a = rev2(~k.w1);          // groups 63..32 reversed -> becomes the high word of the reversed value
    uint64_t b = rev2(~k.w0);
    // reversed value R = a:b, whose top 4 groups are the complemented padding (all ones); shift left by 8 bits.
    return Kmer{(a << 8) | (b >> 56), b << 8};
}
// dna/CanonicalForm.h:51-63, K even: FWD (0) iff kmer < rc, REV (1) iff rc < kmer, PALINDROME (2)
W2R_HD int kmer_form(Kmer k, Kmer rc) { return kmer_less(k, rc) ? 0 : (kmer_less(rc, k) ? 1 : 2); }
W2R_HD bool kmer_is_palindrome(Kmer k) { return kmer_rc(k) == k; }
W2R_HD uint32_t kmer_base(Kmer k, int i) { return i < 32 ? (uint32_t)(k.w0 >> (62 - 2 * i)) & 3u : (uint32_t)(k.w1 >> (62 - 2 * (i - 32))) & 3u; }
W2R_HD uint32_t kmer_first(Kmer k) { return (uint32_t)(k.w0 >> 62); }
W2R_HD uint32_t kmer_last(Kmer k) { return (uint32_t)(k.w1 >> 8) & 3u; }

// kmers/KMerContext.h: high nibble = predecessor mask, low nibble = successor mask; RC = bit reversal (KMerContext.cc:19-37)
W2R_HD uint32_t ctx_rc(uint32_t c) {
#if defined(__CUDA_ARCH__)
    return __brev(c) >> 24;
#else
    c = ((c >> 4) | (c << 4)) & 0xff; c = ((c & 0xcc) >> 2) | ((c & 0x33) << 2); c = ((c & 0xaa) >> 1) | ((c & 0x55) << 1);
    return c & 0xff;
#endif
}
W2R_HD int nib_count(uint32_t m) {
#if defined(__CUDA_ARCH__)
    return __popc(m & 15u);
#else
    m &= 15u; return (int)((m & 1) + ((m >> 1) & 1) + ((m >> 2) & 1) + ((m >> 3) & 1));
#endif
}
W2R_HD uint32_t nib_single(uint32_t m) { m &= 15u; return m == 1 ? 0u : (m == 2 ? 1u : (m == 4 ? 2u : 3u)); }

// 64-bit mixing hash of a k-mer (any mixing hash will do; the reference's FNV over the k-mer bytes is only used for
// its own HashSet placement, kmers/KMer.h:229-232).  Low 16 bits select the counting pass / owner GPU, the slot comes
// from the high bits.
W2R_HD uint64_t kmer_hash(Kmer k) {
    uint64_t a = k.w0 * 0x9e3779b97f4a7c15ull;
    a ^= a >> 32;
    a += k.w1 * 0xc2b2ae3d27d4eb4full;
    a ^= a >> 29;
    a *= 0xbf58476d1ce4e5b9ull;
    a ^= a >> 32;
    a *= 0x94d049bb133111ebull;
    a ^= a >> 31;
    return a;
}
W2R_HD int ctz64(uint64_t x) {
#if defined(__CUDA_ARCH__)
    return __ffsll((long long)x) - 1;
#else
    return __builtin_ctzll(x);
#endif
}
W2R_HD uint64_t mulhi64(uint64_t a, uint64_t b) {
#if defined(__CUDA_ARCH__)
    return __umul64hi(a, b);
#else
    return (uint64_t)(((unsigned __int128)a * b) >> 64);
#endif
}

// ---------------------------------------------------------------- packed reads / edges (feudal/FieldVec.h:765-769)
W2R_HD uint32_t packed_base(const uint8_t* p, uint64_t i) { return (p[i >> 2] >> ((i & 3) * 2)) & 3u; }

// 32 consecutive bases starting at base index i of a packed sequence (any byte alignment), LSB-first: base i in bits 1:0.
// Two aligned 8-byte loads + a funnel shift instead of up to 32 byte loads; may touch up to 15 bytes past the last base
// needed, so every packed store (reads, edges) carries >= 16 bytes of padding.
W2R_HD uint64_t bases32_at(const uint8_t* p, uint64_t i) {
    const uintptr_t addr = (uintptr_t)p + (uintptr_t)(i >> 2);
    const uint64_t* q = (const uint64_t*)(addr & ~(uintptr_t)7);
    const uint32_t sh = (uint32_t)(addr & 7u) * 8u + (uint32_t)(i & 3u) * 2u;   // 0..62
    const uint64_t lo = q[0], hi = q[1];
    return sh ? (lo >> sh) | (hi << (64u - sh)) : lo;
}
// The k-mer starting at base `pos` of a packed sequence.
W2R_HD Kmer kmer_at(const uint8_t* bases, uint64_t pos) {
    return Kmer{rev2(bases32_at(bases, pos)), rev2(bases32_at(bases, pos + 32)) & ~0xffull};
}

// The k-mer starting at base `pos` AND its reverse complement, from three aligned 8-byte loads.  In the packed store a base sits
// LSB-first, in the Kmer layout MSB-first: the reverse complement of the k-mer is therefore just the complement of the packed
// bits moved up by 8 (no bit reversal); only the forward k-mer needs rev2.
W2R_HD void kmer_pair_at(const uint8_t* bases, uint64_t pos, Kmer* f, Kmer* rc) {
    const uintptr_t addr = (uintptr_t)bases + (uintptr_t)(pos >> 2);
    const uint64_t* q = (const uint64_t*)(addr & ~(uintptr_t)7);
    const uint32_t sh = (uint32_t)(addr & 7u) * 8u + (uint32_t)(pos & 3u) * 2u;   // 0..62
    const uint64_t a = q[0], b = q[1], c = q[2];
    const uint64_t lo = sh ? (a >> sh) | (b << (64u - sh)) : a;                    // bases pos .. pos+31
    const uint64_t hi = sh ? (b >> sh) | (c << (64u - sh)) : b;                    // bases pos+32 .. pos+63
    *f = Kmer{rev2(lo), rev2(hi) & ~0xffull};
    *rc = Kmer{(~hi << 8) | (~lo >> 56), ~lo << 8};
}
// 16 consecutive bases starting at base i, LSB-first (two aligned 4-byte loads + a funnel shift; may touch 7 bytes past the end)
W2R_HD uint32_t bases16_at(const uint8_t* p, uint64_t i) {
    const uintptr_t addr = (uintptr_t)p + (uintptr_t)(i >> 2);
    const uint32_t* q = (const uint32_t*)(addr & ~(uintptr_t)3);
    const uint32_t sh = (uint32_t)(addr & 3u) * 8u + (uint32_t)(i & 3u) * 2u;     // 0..30
    const uint32_t lo = q[0], hi = q[1];
#if defined(__CUDA_ARCH__)
    return __funnelshift_r(lo, hi, sh);
#else
    return sh ? (lo >> sh) | (hi << (32u - sh)) : lo;
#endif
}
// reverse the order of the 16 two-bit groups of a 32-bit word
W2R_HD uint32_t rev2_32(uint32_t x) {
#if defined(__CUDA_ARCH__)
    x = __brev(x);
    return ((x & 0xaaaaaaaau) >> 1) | ((x & 0x55555555u) << 1);
#else
    x = ((x >> 2) & 0x33333333u) | ((x & 0x33333333u) << 2);
    x = ((x >> 4) & 0x0f0f0f0fu) | ((x & 0x0f0f0f0fu) << 4);
    x = ((x >> 8) & 0x00ff00ffu) | ((x & 0x00ff00ffu) << 8);
    return (x >> 16) | (x << 16);
#endif
}

// ---------------------------------------------------------------- tables
// Counting table slot: one 32-byte sector.  {w0,w1} is claimed with a single 128-bit CAS.
struct __attribute__((aligned(32))) CountSlot { uint64_t w0, w1; uint32_t count, ctx; uint64_t pad; };
// Solid (dictionary) slot = the reference's KmerDictEntry (kmers/ReadPather.h:149-169): k-mer + KDef{edge, offset, context}.
struct __attribute__((aligned(32))) SolidSlot { uint64_t w0, w1; uint32_t ctx, edge, off, pad; };

struct SolidTable {
    SolidSlot* slots;
    uint64_t nslots;           // any size (not only powers of two): the home slot is the hash scaled to [0, nslots).  Tables whose slots
                               // become 32-bit oriented node ids (2*slot+o: the sharded graph stage) hold <= 2^31 slots; the pathing table any number
    W2R_HD uint64_t size() const { return nslots; }
    W2R_HD uint64_t home_of_hash(uint64_t h) const { return mulhi64(h, nslots); }
    W2R_HD uint64_t home(Kmer k) const { return home_of_hash(kmer_hash(k)); }
    W2R_HD uint64_t next(uint64_t h) const { return h + 1 == nslots ? 0 : h + 1; }
};

// slots for n keys: load ~0.6 (linear probing: ~1.8 probes per hit, ~3.6 per miss; pathing screens misses with the Bloom filter)
// (beyond 2^29 keys the table is what decides whether a genome fits the device: load ~0.77 there)
W2R_HD uint64_t solid_table_slots(uint64_t n) { return n < (1ull << 29) ? n + (n >> 1) + (n >> 3) + 1024 : n + (n >> 2) + (n >> 4); }

// Canonical lookup with the k-mer's hash already known; returns slot or -1.
W2R_HD int64_t solid_find_hashed(const SolidTable& t, Kmer k, uint64_t hh) {
    uint64_t h = t.home_of_hash(hh);
    for (;;) {
        const SolidSlot* s = t.slots + h;
#if defined(__CUDA_ARCH__)
        ulonglong2 kk = __ldg(reinterpret_cast<const ulonglong2*>(s));
        uint64_t a = kk.x, b = kk.y;
#else
        uint64_t a = s->w0, b = s->w1;
#endif
        if (a == k.w0 && b == k.w1) return (int64_t)h;
        if (a == EMPTY_W0) return -1;
        h = t.next(h);
    }
}
W2R_HD int64_t solid_find(const SolidTable& t, Kmer k) { return solid_find_hashed(t, k, kmer_hash(k)); }
// ---------------------------------------------------------------- the dictionary the reads are pathed against
// W slices keyed by a hash of the k-mer.  One GPU: one slice = the graph stage's own table.  Sharded: slice r is BUILT by GPU r (1/W of
// the insert work each) and the finished slices are replicated with one bulk all-gather, so every path kernel probes local memory.
// In front of it a blocked Bloom filter (two bits in one 32-bit word per key), sliced and gathered the same way: read pathing
// looks up every k-mer of a read's error-laden tail, almost all of them absent, and a negative answer then costs one sector instead
// of a probe chain in the multi-GB table.  No false negatives.
// The filter has its own cheap 32-bit hash (two multiply-adds per word half): gap screening hashes ~100 k-mers per read, and the
// 64-bit table hash (four 64-bit multiplies) is only worth computing for the few candidates that pass.
struct PathSlice { const SolidSlot* tab; uint64_t nslots; };
struct PathDict {
    const PathSlice* slices;   // [W] (device memory)
    uint32_t W;
    const uint32_t* bloom;     // W consecutive filter slices of slice_words words; nullptr = no filter
    uint32_t slice_words;
};
W2R_HD uint32_t bloom_hash(Kmer k) {
    uint32_t x = (uint32_t)k.w0 * 0x9e3779b1u + (uint32_t)(k.w0 >> 32) * 0x85ebca77u;
    x ^= x >> 15;
    x += (uint32_t)(k.w1 >> 8) * 0xc2b2ae3du + (uint32_t)(k.w1 >> 40) * 0x27d4eb2fu;
    x ^= x >> 13; x *= 0x165667b1u; x ^= x >> 16;
    return x;
}
W2R_HD uint32_t pd_slice_of(uint32_t W, uint32_t bh) { return W == 1 ? 0u : (uint32_t)(((uint64_t)bh * W) >> 32); }
W2R_HD uint64_t pd_bloom_word(uint32_t W, uint32_t slice_words, uint32_t bh) {
    uint32_t y = bh * 0x9e3779b1u; y ^= y >> 15;                               // (re-mixed: the top bits of bh chose the slice)
    return (uint64_t)pd_slice_of(W, bh) * slice_words + (((uint64_t)y * slice_words) >> 32);
}
W2R_HD uint32_t bloom_mask(uint32_t h) { const uint32_t y = h * 0x2c1b3c6du; return (1u << (y >> 27)) | (1u << ((y >> 22) & 31u)); }
W2R_HD bool pd_may_contain(const PathDict& d, uint32_t bh) {
    if (!d.bloom) return true;
    const uint32_t m = bloom_mask(bh);
#if defined(__CUDA_ARCH__)
    return (__ldg(d.bloom + pd_bloom_word(d.W, d.slice_words, bh)) & m) == m;
#else
    return (d.bloom[pd_bloom_word(d.W, d.slice_words, bh)] & m) == m;
#endif
}
// Canonical lookup (bh = bloom_hash(k)); returns the entry or nullptr.  The probe sequence inside a slice is SolidTable's.
W2R_HD const SolidSlot* pd_find(const PathDict& d, Kmer k, uint32_t bh) {
    const PathSlice sl = d.slices[pd_slice_of(d.W, bh)];
    uint64_t h = mulhi64(kmer_hash(k), sl.nslots);
    for (;;) {
        const SolidSlot* s = sl.tab + h;
#if defined(__CUDA_ARCH__)
        const ulonglong2 kk = __ldg(reinterpret_cast<const ulonglong2*>(s));
        const uint64_t a = kk.x, b = kk.y;
#else
        const uint64_t a = s->w0, b = s->w1;
#endif
        if (a == k.w0 && b == k.w1) return s;
        if (a == EMPTY_W0) return nullptr;
        h = h + 1 == sl.nslots ? 0 : h + 1;
    }
}
W2R_HD const SolidSlot* pd_find_filtered(const PathDict& d, Kmer k) {
    const uint32_t bh = bloom_hash(k);
    if (!pd_may_contain(d, bh)) return nullptr;
    return pd_find(d, k, bh);
}

// kmers/ReadPather.h:196-199 findEntry: canonicalise then look up.  *rev = query was in REV form (rc < query).
W2R_HD int64_t solid_find_any(const SolidTable& t, Kmer k, bool* rev) {
    Kmer r = kmer_rc(k);
    bool isrev = kmer_less(r, k);
    if (rev) *rev = isrev;
    return solid_find(t, isrev ? r : k);
}

}  // namespace w2r
