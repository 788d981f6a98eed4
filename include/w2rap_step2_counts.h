/*
 * w2rap_step2_counts.h — count the k-mers of a read set once, then build the step-2 graph for any number of min_freq values.
 *
 * Users choose --min_freq from the 60-mer spectrum (small_K.freqs) and often build and compare several graphs, e.g. at 3, 4
 * and 5.  The counts do not depend on min_freq: only the final `count >= min_freq` test does.  w2rap_step2_count() runs the
 * quality floor, map and reduce of step 2 once and keeps every distinct k-mer seen at least f0 times (the "keep floor",
 * params.min_freq of the count) with its raw context and min(255, count), on the device.  w2rap_step2_build() then selects the
 * k-mers seen >= min_freq times (any min_freq >= f0) and runs the rest of step 2 on them: dictionary, adjacency, unipaths, HBV,
 * paths (+FixPaths) and places.  Its result is identical, in every field except the timings, to w2rap_step2_run_resident() on
 * the same reads with the same min_qual and min_freq.
 *
 * Single GPU (no communicator); the sharded forms are in w2rap_step2_counts_sharded.h.  Exported from libw2rap_step2.so, next to
 * w2rap_step2.h.
 *
 *   w2rap_device_reads* reads;  w2rap_step2_upload(&host_reads, device, &reads, err, n);
 *   w2rap_counts* counts;       p.min_freq = 3;  w2rap_step2_count(reads, &p, &counts, &spectrum, err, n);
 *   for F in 3, 4, 5:           p.min_freq = F;  w2rap_step2_build(reads, counts, &p, &graph, err, n);  ...  w2rap_step2_free(&graph);
 *   w2rap_step2_counts_release(counts);  w2rap_step2_free(&spectrum);  w2rap_step2_release(reads);
 */
#ifndef W2RAP_STEP2_COUNTS_H_
#define W2RAP_STEP2_COUNTS_H_

#include "w2rap_step2.h"

#ifdef __cplusplus
extern "C" {
#endif

typedef struct w2rap_counts w2rap_counts;        /* opaque, device-resident, single GPU */

/* Quality floor + map + reduce over a resident read set; keeps every distinct k-mer seen >= p->min_freq times
 * (the "keep floor" f0) with its raw context and min(255, count): 17 bytes of device memory per kept k-mer, owned by the handle.
 * Uses min_qual, min_freq (as f0, 1..255), force_passes, table_slots, verbose and workdir; dump_kmers may be 0 or 2 (1 is refused:
 * there is no dictionary yet).  `summary` (may be NULL) receives exactly the counters a w2rap_step2_run_resident with
 * min_freq = f0 would report: n_reads, n_bases, n_kmer_instances, n_distinct, n_solid (= k-mers kept), hist[101], the count-stage
 * timings, and the level-2 dump if p->dump_kmers == 2.  Every graph/path array is null, so w2rap_write_freqs() works on it; free it
 * with w2rap_step2_free().  Writes <workdir>/small_K.freqs like a run. */
int  w2rap_step2_count(w2rap_device_reads* reads, const w2rap_params* p, w2rap_counts** counts,
                       w2rap_graph* summary, char* err, size_t errlen);

/* The rest of step 2 for p->min_freq >= f0: selection, dictionary, adjacency, unipaths, HBV, paths (+FixPaths), places.
 * `out` is identical in every field except timings to w2rap_step2_run_resident(reads, p) with the same min_qual.
 * Uses min_freq, want_paths, apply_fixpaths, dump_kmers (0 or 1), places_K2, verbose and workdir.  Refused with
 * W2RAP_ERR_BAD_ARG before any device work: min_freq < f0, a min_qual other than the count's, dump_kmers == 2, and a `reads`
 * handle other than the one counted.  timings.count_ms is the selection (+ the dictionary build, as in a run); the map and reduce
 * timings and count_launches are 0.  Does not modify `counts`: any number of builds, in any order. */
int  w2rap_step2_build(w2rap_device_reads* reads, const w2rap_counts* counts, const w2rap_params* p,
                       w2rap_graph* out, char* err, size_t errlen);

void w2rap_step2_counts_release(w2rap_counts* counts);

#ifdef __cplusplus
}
#endif
#endif /* W2RAP_STEP2_COUNTS_H_ */
