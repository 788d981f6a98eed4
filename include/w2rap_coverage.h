/*
 * w2rap_coverage.h — k-mer coverage of any set of sequences from the counts a w2rap_step2_count() kept, and the step-2 graph
 * written as GFA 1.0 with per-edge coverage.
 *
 * What tells min_freq choices apart is coverage: error tips and bubbles sit at a few x, heterozygous arms at half the coverage,
 * repeats at a multiple of it.  The count handle (include/w2rap_step2_counts.h) holds the exact count, min(255, occurrences), of
 * every 60-mer seen at least f0 times, so the coverage of the graph's edges (or of reads, or of contigs) is a lookup of every
 * k-mer of a sequence in those counts.
 *
 * Single GPU, on the device the counts live on.  Exported from libw2rap_step2.so, next to w2rap_step2.h.
 *
 *   w2rap_step2_count(reads, &p, &counts, NULL, err, n);               p.min_freq = f0
 *   w2rap_step2_build(reads, counts, &p, &g, err, n);                  p.min_freq = F >= f0
 *   w2rap_seqs edges = {g.n_edges, g.edge_bases, g.edge_off, g.edge_len};
 *   w2rap_counts_coverage(counts, &edges, cov, NULL, err, n);          cov: g.n_edges entries
 *   w2rap_write_gfa("x.small_K.gfa", &g, cov, err, n);
 */
#ifndef W2RAP_COVERAGE_H_
#define W2RAP_COVERAGE_H_

#include "w2rap_step2_counts.h"

#ifdef __cplusplus
extern "C" {
#endif

/* Host sequences, packed like reads and edges: 2-bit bases, LSB-first within a byte (A=0 C=1 G=2 T=3), sequence i in
 * bases[base_off[i] .. base_off[i+1]) holding at least ceil(len[i]/4) bytes.  The edge arrays of a w2rap_graph fit as they are. */
typedef struct w2rap_seqs {
    uint64_t n;
    const uint8_t* bases;
    const uint64_t* base_off;   /* n+1 */
    const uint32_t* len;        /* n */
} w2rap_seqs;

/* Coverage of one sequence (32 bytes).  n_kmers = max(0, len - 59); for each of its 60-mers c = the kept count of the canonical
 * form (min(255, occurrences)), or 0 if the k-mer was not kept (seen fewer than f0 times, or never).  sum = sum of c,
 * n_absent = number of k-mers with c = 0, min / max over the c values (both 0 when n_kmers = 0). */
typedef struct w2rap_seq_cov {
    uint64_t n_kmers, sum, n_absent;
    uint32_t min, max;
} w2rap_seq_cov;

/* Fills out[0 .. seqs->n) (caller-owned).  Builds a hash index over the kept k-mers for the call and frees it afterwards (the
 * handle stays at 17 bytes per kept k-mer), then looks up every k-mer of every sequence.  device_ms (may be NULL) receives the
 * device time of the index build and the lookups (CUDA events; without the copies).  The index is built on every call, also for
 * an empty set, whose device_ms is then the index build alone.  Refused with W2RAP_ERR_BAD_ARG before any device work: null
 * pointers, and offsets that do not hold ceil(len/4) bytes.  Without an sm_100 device: W2RAP_ERR_NO_DEVICE (no CPU path).
 * Does not modify `counts`. */
int w2rap_counts_coverage(const w2rap_counts* counts, const w2rap_seqs* seqs, w2rap_seq_cov* out, float* device_ms,
                          char* err, size_t errlen);

/* GFA 1.0 of a step-2 graph (host only).
 *   H  VN:Z:1.0
 *   S  one line per canonical edge i, in edge order: name = its fwd hbv id (fwd_xlat[i]), so that the ids of .paths map directly
 *      (hbv id fwd_xlat[i] is the segment read `+`, its involution the segment read `-`); the canonical sequence; LN:i:<len>, and
 *      with edge_cov (n_edges entries, indexed like the edges; may be NULL) KC:i:<sum> and DP:f:<sum / n_kmers, 3 decimals>.
 *   L  one line for every pair of hbv edges (x, y) with to(x) = from(y), overlap 59M.  A link and its complement
 *      (inv y, inv x) are the same GFA link: only the smaller of the tuples (x, y) and (inv y, inv x) is written.  Lines are
 *      ordered by the shared vertex, then x, then y.
 * Refused with W2RAP_ERR_BAD_ARG: a graph without edge_vertices, fwd_xlat or involution (the non-root result of a
 * graph_on_root_only run), without edge sequences, or with ids out of range.  A graph built without paths is fine. */
int w2rap_write_gfa(const char* path, const w2rap_graph* g, const w2rap_seq_cov* edge_cov, char* err, size_t errlen);

#ifdef __cplusplus
}
#endif
#endif /* W2RAP_COVERAGE_H_ */
