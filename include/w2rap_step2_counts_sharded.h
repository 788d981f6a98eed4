/*
 * w2rap_step2_counts_sharded.h — count once, build per min_freq and look up k-mer coverage with the read set sharded over GPUs.
 *
 * The collective forms of w2rap_step2_count / w2rap_step2_build (include/w2rap_step2_counts.h) and w2rap_counts_coverage
 * (include/w2rap_coverage.h), for jobs that run as w2rap_step2_run_sharded does: one rank per GPU, reads sharded by index, every
 * k-mer counted on the rank that owns its minimiser partition.  Each rank's handle keeps the k-mers of the partitions it owns,
 * so comparing min_freq values on a genome too large for one GPU costs one sharded count and one build per value, not one
 * sharded run per value.
 *
 * All three calls are collective: every rank calls them with the same parameters (its own shard and handle), in the same order,
 * as with w2rap_step2_run_sharded.  w2rap_step2_counts_release stays local.  A handle made with a communicator is used only with
 * that communicator and only through these calls; a handle made by w2rap_step2_count only through the single-GPU calls.  Every
 * refusal below is made before any collective, from arguments alone, so ranks given the same arguments refuse together.
 *
 *   w2rap_step2_upload(&my_shard, device, &reads, err, n);            one shard per rank
 *   p.min_freq = 3;  w2rap_step2_count_sharded(reads, &p, comm, &counts, &spectrum, err, n);
 *   for F in 3, 4, 5:
 *       p.min_freq = F;  w2rap_step2_build_sharded(reads, counts, &p, comm, &g, err, n);
 *       w2rap_seqs edges = {g.n_edges, g.edge_bases, g.edge_off, g.edge_len};          (rank 0; other ranks may pass NULL)
 *       w2rap_counts_coverage_sharded(counts, comm, rank == 0 ? &edges : NULL, cov, NULL, err, n);
 *       w2rap_step2_free(&g);
 *   w2rap_step2_counts_release(counts);  w2rap_step2_free(&spectrum);  w2rap_step2_release(reads);
 */
#ifndef W2RAP_STEP2_COUNTS_SHARDED_H_
#define W2RAP_STEP2_COUNTS_SHARDED_H_

#include "w2rap_coverage.h"

#ifdef __cplusplus
extern "C" {
#endif

/* Quality floor + map + exchange + reduce over this rank's resident shard.  Each rank keeps the k-mers of the partitions it owns
 * that were seen >= f0 = p->min_freq times over the whole job, with their raw context and min(255, count): 17 bytes of device
 * memory per kept k-mer, owned by the handle.  `summary` (may be NULL) carries the whole-job counters, identical on every rank,
 * exactly as w2rap_step2_run_sharded at min_freq = f0 reports them: n_kmer_instances, n_distinct, n_solid (= k-mers kept over all
 * ranks), hist[101] and the count-stage timings; n_reads and n_bases are this rank's shard.  Uses min_qual, min_freq (f0, 1..255),
 * force_passes, table_slots, verbose and workdir; rank 0 writes <workdir>/small_K.freqs.  Refused with W2RAP_ERR_BAD_ARG: null
 * arguments, dump_kmers != 0, and a shard that does not live on the communicator's device. */
int w2rap_step2_count_sharded(w2rap_device_reads* shard, const w2rap_params* p, w2rap_comm* comm, w2rap_counts** counts,
                              w2rap_graph* summary, char* err, size_t errlen);

/* The rest of step 2 for p->min_freq >= f0 from a sharded count.  On every rank `out` equals w2rap_step2_run_sharded(shard, p,
 * comm) at that min_freq in every field except timings, graph_on_root_only, places_K2 and dump_kmers = 1 included, and both
 * digests.  Does not modify `counts`: any number of builds, in any order.  Refused with W2RAP_ERR_BAD_ARG: null arguments,
 * min_freq < f0, a min_qual other than the count's, dump_kmers == 2, a shard handle other than the one counted, a communicator
 * other than the count's, and a handle made by w2rap_step2_count. */
int w2rap_step2_build_sharded(w2rap_device_reads* shard, const w2rap_counts* counts, const w2rap_params* p, w2rap_comm* comm,
                              w2rap_graph* out, char* err, size_t errlen);

/* Coverage (w2rap_seq_cov, include/w2rap_coverage.h) of the sequence set passed on RANK 0 against the counts kept over all
 * ranks; the other ranks' `seqs` is ignored and may be NULL, so the edges of a graph_on_root_only build can be looked up.  Every
 * rank whose `out` is non-null receives out[0 .. n) for the whole set.  The values equal w2rap_counts_coverage against a
 * single-GPU count of the union of the shards at the same f0 and min_qual: every k-mer position is looked up on the one rank that
 * owns its minimiser partition, and the per-rank totals are merged by all-reduce (sum, n_absent: sum; min: min; max: max).
 * device_ms (may be NULL) is this rank's index build, lookups and merge, not rank 0's upload or the broadcast of the set.
 * Refused with W2RAP_ERR_BAD_ARG on every rank: null counts or comm, a communicator other than the count's, a handle made by
 * w2rap_step2_count, and (after one broadcast of rank 0's verdict) a set rank 0 refuses as w2rap_counts_coverage would. */
int w2rap_counts_coverage_sharded(const w2rap_counts* counts, w2rap_comm* comm, const w2rap_seqs* seqs, w2rap_seq_cov* out,
                                  float* device_ms, char* err, size_t errlen);

#ifdef __cplusplus
}
#endif
#endif /* W2RAP_STEP2_COUNTS_SHARDED_H_ */
