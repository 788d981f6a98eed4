// coverage.cu — w2rap_counts_coverage (include/w2rap_coverage.h): index over the kept counts, then one lookup per k-mer position
// of every sequence (coverage.cuh).  Part of the library's single translation unit, after pipeline.cu (check_device, SlabLease, SBuf).
#include "../../include/w2rap_coverage.h"
#include "coverage.cuh"

static_assert(sizeof(w2rap_seq_cov) == sizeof(w2r::SeqCov), "w2rap_seq_cov is the host image of SeqCov");

namespace w2r {

// The checks of upload(): every sequence's bases fit between its offsets.
static void validate_seqs(const w2rap_seqs* s, const w2rap_seq_cov* out) {
    if (!s) W2R_FAIL(W2RAP_ERR_BAD_ARG, "null sequence set");
    if (!s->n) return;
    if (!out) W2R_FAIL(W2RAP_ERR_BAD_ARG, "null output");
    if (!s->bases || !s->base_off || !s->len) W2R_FAIL(W2RAP_ERR_BAD_ARG, "null pointer in sequence set");
    for (uint64_t i = 0; i < s->n; ++i)
        if (s->base_off[i + 1] < s->base_off[i] || s->base_off[i + 1] - s->base_off[i] < ((uint64_t)s->len[i] + 3) / 4)
            W2R_FAIL(W2RAP_ERR_BAD_ARG, "sequence %llu: base offsets do not hold its bases", (unsigned long long)i);
}

static void counts_coverage(const w2rap_counts& h, const w2rap_seqs& s, w2rap_seq_cov* out, float* device_ms) {
    Ctx c;
    check_device(h.device, c);
    W2R_CUDA(cudaStreamCreateWithFlags(&c.stream, cudaStreamNonBlocking));
    struct StreamGuard { cudaStream_t s; ~StreamGuard() { cudaStreamSynchronize(s); cudaStreamDestroy(s); } } sg{c.stream};
    SlabLease lease(h.device);              // declared before the buffers: they go back before the lease does
    c.slab = lease.slab;
    const uint64_t n = s.n;
    const uint64_t nbytes = n ? s.base_off[n] : 0;
    SBuf<uint8_t> bases(c, nbytes + 32);
    SBuf<uint64_t> base_off(c, n + 1);
    SBuf<uint32_t> len(c, n + 1), tiles(c, n + 1);
    SBuf<uint64_t> tile_base(c, n + 1), total(c, 1);
    SBuf<SeqCov> cov(c, n + 1);
    W2R_CUDA(cudaMemsetAsync(bases.p + nbytes, 0, 32, c.stream));     // kmer_pair_at may read a few bytes past the last base
    if (n) {
        W2R_CUDA(cudaMemcpyAsync(bases.p, s.bases, nbytes, cudaMemcpyHostToDevice, c.stream));
        W2R_CUDA(cudaMemcpyAsync(base_off.p, s.base_off, (n + 1) * 8, cudaMemcpyHostToDevice, c.stream));
        W2R_CUDA(cudaMemcpyAsync(len.p, s.len, n * 4, cudaMemcpyHostToDevice, c.stream));
    }
    EventTimer et(c.stream);
    et.start();
    // the index: the kept k-mers in a SolidTable whose slots hold their counts
    const uint64_t nslots = solid_table_slots(h.n_kept);
    SBuf<SolidSlot> slots(c, nslots);
    slots.fill_ff();
    const SolidTable st{slots.p, nslots};
    if (h.n_kept) W2R_LAUNCH(c, k_insert_counts, grid_for(c, h.n_kept, 256), 256, 0, (const ulonglong2*)h.solid, (const uint8_t*)h.count, h.n_kept, st);
    uint64_t n_tiles = 0;
    if (n) {
        W2R_LAUNCH(c, k_cov_init, grid_for(c, n, 256), 256, 0, (const uint32_t*)len.p, n, tiles.p, cov.p);
        exclusive_scan<uint32_t, uint64_t>(c, tiles.p, n, tile_base.p, total.p);
        n_tiles = d2h_scalar(c, total.p);
    }
    if (n_tiles)
        W2R_LAUNCH(c, k_cov_tiles, grid_for(c, n_tiles * 32, 256), 256, 0, st, (const uint8_t*)bases.p, (const uint64_t*)base_off.p, (const uint32_t*)len.p,
                   (const uint64_t*)tile_base.p, n, n_tiles, cov.p);
    const float ms = et.stop();
    if (device_ms) *device_ms = ms;
    if (n) W2R_CUDA(cudaMemcpyAsync(out, cov.p, n * sizeof(SeqCov), cudaMemcpyDeviceToHost, c.stream));
    W2R_CUDA(cudaStreamSynchronize(c.stream));
}

}  // namespace w2r

extern "C" {

int w2rap_counts_coverage(const w2rap_counts* counts, const w2rap_seqs* seqs, w2rap_seq_cov* out, float* device_ms, char* err, size_t errlen) {
    W2R_API_BEGIN
    if (!counts) W2R_FAIL(W2RAP_ERR_BAD_ARG, "null counts handle");
    validate_seqs(seqs, out);
    counts_coverage(*counts, *seqs, out, device_ms);
    W2R_API_END
}

}  // extern "C"
