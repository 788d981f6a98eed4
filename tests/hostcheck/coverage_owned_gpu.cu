// coverage_owned_gpu.cu — TEST INFRASTRUCTURE (never linked into the product library; compiled by the test with nvcc for sm_100a).
//
// Runs the sharded lookup kernel k_cov_tiles_owned (csrc/coverage.cuh) for W simulated ranks on ONE device: the kept k-mers split
// by owner into W indexes (built by k_insert_counts), one launch per rank with that rank's index and number, and the W partial
// totals merged on the host as the all-reduces merge them.  So the shuffle window minima and the ballot compaction of the kernel
// are checked for W > 1 where only one GPU is available.
#include <stdint.h>
#include <string.h>

#include <vector>

#include "../../include/w2rap_coverage.h"
#include "../../w2rap-contigger_b200/csrc/coverage.cuh"

using namespace w2r;

#define CK(x) do { if ((x) != cudaSuccess) return 2; } while (0)

extern "C" int gc_coverage_owned(const w2rap_kmer_rec* recs, uint64_t n_recs, uint32_t f0, uint32_t logP, uint32_t world, const w2rap_seqs* s,
                                 w2rap_seq_cov* out) {
    const uint64_t n = s->n, nbytes = n ? s->base_off[n] : 0;
    std::vector<uint64_t> tile_base(n + 1, 0);
    for (uint64_t i = 0; i < n; ++i) tile_base[i + 1] = tile_base[i] + cov_tiles_of(s->len[i]);
    const uint64_t n_tiles = tile_base[n];
    uint8_t* d_bases; uint64_t *d_off, *d_tb; uint32_t* d_len;
    CK(cudaMalloc(&d_bases, nbytes + 32)); CK(cudaMemset(d_bases, 0, nbytes + 32));
    CK(cudaMalloc(&d_off, (n + 1) * 8)); CK(cudaMalloc(&d_tb, (n + 1) * 8)); CK(cudaMalloc(&d_len, (n + 1) * 4));
    CK(cudaMemcpy(d_bases, s->bases, nbytes, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(d_off, s->base_off, (n + 1) * 8, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(d_len, s->len, n * 4, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(d_tb, tile_base.data(), (n + 1) * 8, cudaMemcpyHostToDevice));
    for (uint64_t i = 0; i < n; ++i) {
        const uint64_t nk = cov_kmers_of(s->len[i]);
        out[i] = w2rap_seq_cov{nk, 0, 0, nk ? 0xffffffffu : 0u, 0};
    }
    std::vector<unsigned long long> sa(2 * n + 1);
    std::vector<uint32_t> mn(n + 1), mx(n + 1);
    for (uint32_t r = 0; r < world; ++r) {
        std::vector<ulonglong2> mine;
        std::vector<uint8_t> cnt;
        for (uint64_t i = 0; i < n_recs; ++i) {
            const Kmer k{recs[i].w0, recs[i].w1};
            if (recs[i].count < f0 || owner_of_partition(mini_part(mini_mix(kmer_minimizer_hash_words(k)), logP), logP, world) != r) continue;
            mine.push_back(make_ulonglong2(k.w0, k.w1 | (recs[i].ctx & 0xffu)));
            cnt.push_back((uint8_t)(recs[i].count < 255 ? recs[i].count : 255));
        }
        const uint64_t nk = mine.size(), nslots = solid_table_slots(nk);
        ulonglong2* d_recs; uint8_t* d_cnt; SolidSlot* d_slots; unsigned long long* d_sa; uint32_t *d_mn, *d_mx;
        CK(cudaMalloc(&d_recs, (nk + 1) * 16)); CK(cudaMalloc(&d_cnt, nk + 1)); CK(cudaMalloc(&d_slots, nslots * sizeof(SolidSlot)));
        CK(cudaMalloc(&d_sa, (2 * n + 1) * 8)); CK(cudaMalloc(&d_mn, (n + 1) * 4)); CK(cudaMalloc(&d_mx, (n + 1) * 4));
        CK(cudaMemcpy(d_recs, mine.data(), nk * 16, cudaMemcpyHostToDevice));
        CK(cudaMemcpy(d_cnt, cnt.data(), nk, cudaMemcpyHostToDevice));
        CK(cudaMemset(d_slots, 0xff, nslots * sizeof(SolidSlot)));
        CK(cudaMemset(d_sa, 0, (2 * n + 1) * 8)); CK(cudaMemset(d_mn, 0xff, (n + 1) * 4)); CK(cudaMemset(d_mx, 0, (n + 1) * 4));
        const SolidTable st{d_slots, nslots};
        if (nk) k_insert_counts<<<64, 256>>>(d_recs, d_cnt, nk, st);
        if (n_tiles)
            k_cov_tiles_owned<<<(unsigned)((n_tiles * 32 + COV_OWNED_THREADS - 1) / COV_OWNED_THREADS), COV_OWNED_THREADS>>>(
                st, d_bases, d_off, d_len, d_tb, n, n_tiles, logP, world, r, CovParts{d_sa, d_sa + n, d_mn, d_mx});
        CK(cudaGetLastError());
        CK(cudaDeviceSynchronize());
        CK(cudaMemcpy(sa.data(), d_sa, (2 * n + 1) * 8, cudaMemcpyDeviceToHost));
        CK(cudaMemcpy(mn.data(), d_mn, (n + 1) * 4, cudaMemcpyDeviceToHost));
        CK(cudaMemcpy(mx.data(), d_mx, (n + 1) * 4, cudaMemcpyDeviceToHost));
        for (uint64_t i = 0; i < n; ++i) {
            out[i].sum += sa[i]; out[i].n_absent += sa[n + i];
            if (mn[i] < out[i].min) out[i].min = mn[i];
            if (mx[i] > out[i].max) out[i].max = mx[i];
        }
        cudaFree(d_recs); cudaFree(d_cnt); cudaFree(d_slots); cudaFree(d_sa); cudaFree(d_mn); cudaFree(d_mx);
    }
    cudaFree(d_bases); cudaFree(d_off); cudaFree(d_tb); cudaFree(d_len);
    return 0;
}
