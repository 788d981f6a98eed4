// coverage.cu — w2rap_counts_coverage (include/w2rap_coverage.h) and w2rap_counts_coverage_sharded
// (include/w2rap_step2_counts_sharded.h): index over the kept counts, then one lookup per k-mer position of every sequence
// (coverage.cuh).  Part of the library's single translation unit, after pipeline.cu (check_device, SlabLease, SBuf, w2rap_comm).
#include "../../include/w2rap_step2_counts_sharded.h"
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

// Sharded: rank 0's set goes to every rank, each rank looks up the positions it owns against its own kept k-mers, and the
// per-rank totals are merged by all-reduce.
static void counts_coverage_sharded(const w2rap_counts& h, const w2rap_comm& cm, const w2rap_seqs* s, w2rap_seq_cov* out, float* device_ms) {
    Ctx c;
    check_device(h.device, c);
    W2R_CUDA(cudaStreamCreateWithFlags(&c.stream, cudaStreamNonBlocking));
    struct StreamGuard { cudaStream_t s; ~StreamGuard() { cudaStreamSynchronize(s); cudaStreamDestroy(s); } } sg{c.stream};
    SlabLease lease(h.device);
    c.slab = lease.slab;
    NcclApi& nc = NcclApi::get();
    auto nccl = [](ncclResult_t r, const char* what) {
        if (r != ncclSuccess) W2R_FAIL(W2RAP_ERR_CUDA, "NCCL %s failed: %s", what, NcclApi::get().GetErrorString(r));
    };
    // rank 0's verdict on its set and the set's size, first: a refused set makes every rank return, none waits in a collective
    unsigned long long hdr[3] = {0, 0, 0};                  // status, n, bytes
    Error refused{0, ""};
    if (cm.rank == 0) {
        try {
            validate_seqs(s, out);
            hdr[1] = s->n; hdr[2] = s->n ? s->base_off[s->n] : 0;
        } catch (const Error& e) { refused = e; hdr[0] = (unsigned long long)e.code; }
    }
    SBuf<unsigned long long> dhdr(c, 3);
    W2R_CUDA(cudaMemcpyAsync(dhdr.p, hdr, sizeof hdr, cudaMemcpyHostToDevice, c.stream));
    nccl(nc.Broadcast(dhdr.p, dhdr.p, 3, ncclUint64, 0, cm.comm, c.stream), "broadcast");
    W2R_CUDA(cudaMemcpyAsync(hdr, dhdr.p, sizeof hdr, cudaMemcpyDeviceToHost, c.stream));
    W2R_CUDA(cudaStreamSynchronize(c.stream));
    if (hdr[0]) {
        if (cm.rank == 0) throw refused;
        W2R_FAIL(W2RAP_ERR_BAD_ARG, "rank 0 refused its sequence set");
    }
    const uint64_t n = hdr[1], nbytes = hdr[2];
    SBuf<uint8_t> bases(c, nbytes + 32);
    SBuf<uint64_t> base_off(c, n + 1);
    SBuf<uint32_t> len(c, n + 1), tiles(c, n + 1), mn(c, n + 1), mx(c, n + 1);
    SBuf<uint64_t> tile_base(c, n + 1), total(c, 1);
    SBuf<unsigned long long> sum_absent(c, 2 * n + 1);
    SBuf<SeqCov> cov(c, n + 1);
    W2R_CUDA(cudaMemsetAsync(bases.p + nbytes, 0, 32, c.stream));     // kmer_pair_at may read a few bytes past the last base
    if (n) {
        if (cm.rank == 0) {
            W2R_CUDA(cudaMemcpyAsync(bases.p, s->bases, nbytes, cudaMemcpyHostToDevice, c.stream));
            W2R_CUDA(cudaMemcpyAsync(base_off.p, s->base_off, (n + 1) * 8, cudaMemcpyHostToDevice, c.stream));
            W2R_CUDA(cudaMemcpyAsync(len.p, s->len, n * 4, cudaMemcpyHostToDevice, c.stream));
        }
        nccl(nc.GroupStart(), "group start");
        nccl(nc.Broadcast(bases.p, bases.p, nbytes, ncclUint8, 0, cm.comm, c.stream), "broadcast");
        nccl(nc.Broadcast(base_off.p, base_off.p, n + 1, ncclUint64, 0, cm.comm, c.stream), "broadcast");
        nccl(nc.Broadcast(len.p, len.p, n, ncclUint32, 0, cm.comm, c.stream), "broadcast");
        nccl(nc.GroupEnd(), "group end");
    }
    EventTimer et(c.stream);
    et.start();
    // the index over this rank's kept k-mers
    const uint64_t nslots = solid_table_slots(h.n_kept);
    SBuf<SolidSlot> slots(c, nslots);
    slots.fill_ff();
    const SolidTable st{slots.p, nslots};
    if (h.n_kept) W2R_LAUNCH(c, k_insert_counts, grid_for(c, h.n_kept, 256), 256, 0, (const ulonglong2*)h.solid, (const uint8_t*)h.count, h.n_kept, st);
    if (n) {
        W2R_LAUNCH(c, k_cov_init, grid_for(c, n, 256), 256, 0, (const uint32_t*)len.p, n, tiles.p, cov.p);
        exclusive_scan<uint32_t, uint64_t>(c, tiles.p, n, tile_base.p, total.p);
        const uint64_t n_tiles = d2h_scalar(c, total.p);
        sum_absent.zero(); mn.fill_ff(); mx.zero();
        const CovParts parts{sum_absent.p, sum_absent.p + n, mn.p, mx.p};
        if (n_tiles)
            W2R_LAUNCH(c, k_cov_tiles_owned, grid_for(c, n_tiles * 32, COV_OWNED_THREADS), COV_OWNED_THREADS, 0, st, (const uint8_t*)bases.p, (const uint64_t*)base_off.p,
                       (const uint32_t*)len.p, (const uint64_t*)tile_base.p, n, n_tiles, h.logP, (uint32_t)cm.world, (uint32_t)cm.rank, parts);
        nccl(nc.GroupStart(), "group start");
        nccl(nc.AllReduce(sum_absent.p, sum_absent.p, 2 * n, ncclUint64, ncclSum, cm.comm, c.stream), "all-reduce");
        nccl(nc.AllReduce(mn.p, mn.p, n, ncclUint32, ncclMin, cm.comm, c.stream), "all-reduce");
        nccl(nc.AllReduce(mx.p, mx.p, n, ncclUint32, ncclMax, cm.comm, c.stream), "all-reduce");
        nccl(nc.GroupEnd(), "group end");
        W2R_LAUNCH(c, k_cov_gather, grid_for(c, n, 256), 256, 0, (const unsigned long long*)sum_absent.p, (const uint32_t*)mn.p, (const uint32_t*)mx.p, n, cov.p);
    }
    const float ms = et.stop();
    if (device_ms) *device_ms = ms;
    if (n && out) W2R_CUDA(cudaMemcpyAsync(out, cov.p, n * sizeof(SeqCov), cudaMemcpyDeviceToHost, c.stream));
    W2R_CUDA(cudaStreamSynchronize(c.stream));
}

}  // namespace w2r

extern "C" {

int w2rap_counts_coverage(const w2rap_counts* counts, const w2rap_seqs* seqs, w2rap_seq_cov* out, float* device_ms, char* err, size_t errlen) {
    W2R_API_BEGIN
    if (!counts) W2R_FAIL(W2RAP_ERR_BAD_ARG, "null counts handle");
    validate_seqs(seqs, out);
    check_counts_comm(counts, nullptr);
    counts_coverage(*counts, *seqs, out, device_ms);
    W2R_API_END
}

int w2rap_counts_coverage_sharded(const w2rap_counts* counts, w2rap_comm* comm, const w2rap_seqs* seqs, w2rap_seq_cov* out, float* device_ms, char* err,
                                  size_t errlen) {
    W2R_API_BEGIN
    if (!counts || !comm) W2R_FAIL(W2RAP_ERR_BAD_ARG, "null counts handle or communicator");
    check_counts_comm(counts, comm);
    counts_coverage_sharded(*counts, *comm, seqs, out, device_ms);
    W2R_API_END
}

}  // extern "C"
