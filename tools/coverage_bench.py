"""K-mer coverage lookups on one B200 (w2rap_counts_coverage, include/w2rap_coverage.h).

Input: bench.py's config 2 (135 Mbp synthetic genome, 2x250 PE at 60x, seed 1000, 32.4 M reads), generated on the device.  One
count at f0 = 3, one build at min_freq 4, then, alternating for --repeats rounds: an empty sequence set (the call then builds the
index and nothing else), the build's edges (~134 M lookups) and all reads (~6 G lookups, downloaded once to pinned host memory).
Reported as medians of device_ms (CUDA events around the index build and the lookups, without copies): the index build, the probe
time (a call's device_ms minus the index build), lookups per second, and the DRAM bytes per lookup estimated from the sectors a
probe touches: one 32-byte slot per probed slot, with the expected linear-probing lengths at the table's load (hits
(1 + 1/(1-a))/2, misses (1 + 1/(1-a)^2)/2), weighted by the measured hit fraction, plus the packed bases of the sequences.
The card's name and power limit are read in the same process.  Prints one JSON line (and writes it to --out).  There is no CPU
path: without a B200 the script fails.

    python tools/coverage_bench.py [--repeats 5] [--out profiles/<name>.json]
"""
import argparse
import ctypes as C
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "tools"))
import numpy as np  # noqa: E402
import w2r_testlib as T  # noqa: E402
from min_freq_sweep import card, median  # noqa: E402


class Seqs(C.Structure):
    _fields_ = [("n", C.c_uint64), ("bases", C.c_void_p), ("base_off", C.c_void_p), ("len", C.c_void_p)]


COV_DTYPE = np.dtype([("n_kmers", "<u8"), ("sum", "<u8"), ("n_absent", "<u8"), ("min", "<u4"), ("max", "<u4")])


def table_slots(n):
    """kmer.cuh: solid_table_slots"""
    return n + (n >> 1) + (n >> 3) + 1024 if n < (1 << 29) else n + (n >> 2) + (n >> 4)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--genome-mbp", type=float, default=135.0)
    ap.add_argument("--coverage", type=int, default=60)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if args.repeats < 3:
        raise SystemExit("--repeats must be at least 3")
    lib = T.product_lib()
    if lib.w2rap_step2_device_count() < 1:
        raise SystemExit("no B200 visible: this measurement has no CPU path")
    name, watts = card()
    if "B200" not in name:
        raise SystemExit("device 0 is %s, not a B200" % name)
    E = [C.c_char_p, C.c_size_t]
    lib.w2rap_step2_count.argtypes = [C.c_void_p, C.POINTER(T.Params), C.POINTER(C.c_void_p), C.POINTER(T.Graph)] + E
    lib.w2rap_step2_build.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(T.Params), C.POINTER(T.Graph)] + E
    lib.w2rap_step2_counts_release.argtypes = [C.c_void_p]
    lib.w2rap_step2_counts_release.restype = None
    lib.w2rap_counts_coverage.argtypes = [C.c_void_p, C.POINTER(Seqs), C.c_void_p, C.POINTER(C.c_float)] + E
    err = C.create_string_buffer(1024)

    def check(rc):
        if rc:
            raise SystemExit("call failed (%d): %s" % (rc, err.value.decode()))

    genome = int(args.genome_mbp * 1e6)
    n_reads = (genome * args.coverage // 250) & ~1
    h = C.c_void_p()
    check(lib.w2rap_step2_synth(C.byref(T.SynthParams(genome, 250, args.coverage, 1000, 0, 0, n_reads, 0)), 0, C.byref(h), err, 1024))
    ch, summ = C.c_void_p(), T.Graph()
    check(lib.w2rap_step2_count(h, C.byref(T.default_params(min_freq=3, device=0)), C.byref(ch), C.byref(summ), err, 1024))
    n_kept = int(summ.n_solid)
    lib.w2rap_step2_free(C.byref(summ))
    g = T.Graph()
    check(lib.w2rap_step2_build(h, ch, C.byref(T.default_params(min_freq=4, want_paths=0, device=0)), C.byref(g), err, 1024))
    hr = T.Reads()
    check(lib.w2rap_step2_download_reads(h, C.byref(hr), err, 1024))
    sets = {"empty": (Seqs(0, None, None, None), 0),
            "edges": (Seqs(g.n_edges, g.edge_bases, g.edge_off, g.edge_len), int(g.n_edges)),
            "reads": (Seqs(hr.n_reads, hr.bases, hr.base_off, hr.len), int(hr.n_reads))}
    outs = {k: np.zeros(max(1, n), COV_DTYPE) for k, (_, n) in sets.items()}
    ms = {k: [] for k in sets}

    def call(k):
        t = C.c_float(0)
        check(lib.w2rap_counts_coverage(ch, C.byref(sets[k][0]), outs[k].ctypes.data, C.byref(t), err, 1024))
        return t.value
    for k in sets:                                       # warm-up
        call(k)
    for _ in range(args.repeats):
        for k in sets:
            ms[k].append(call(k))
    index_ms = median(ms["empty"])
    load = n_kept / table_slots(n_kept)
    hit_slots, miss_slots = (1 + 1 / (1 - load)) / 2, (1 + 1 / (1 - load) ** 2) / 2
    res = {}
    for k in ("edges", "reads"):
        cov = outs[k][:sets[k][1]]
        lookups = int(cov["n_kmers"].sum())
        hits = lookups - int(cov["n_absent"].sum())
        bases = int(np.ctypeslib.as_array(C.cast(sets[k][0].len, C.POINTER(C.c_uint32)), (sets[k][1],)).sum(dtype=np.int64))
        total = median(ms[k])
        probe = total - index_ms
        slots = (hits * hit_slots + (lookups - hits) * miss_slots) / max(1, lookups)
        bpl = 32 * slots + bases / 4 / max(1, lookups)
        res[k] = dict(sequences=sets[k][1], lookups=lookups, hit_fraction=round(hits / max(1, lookups), 4), device_ms=round(total, 2),
                      probe_ms=round(probe, 2), lookups_per_s=float("%.4g" % (lookups / (probe * 1e-3))),
                      est_dram_bytes_per_lookup=round(bpl, 1), est_dram_tb_per_s=round(bpl * lookups / (probe * 1e-3) / 1e12, 2),
                      sum_of_counts=int(cov["sum"].sum()))
    out = {"tool": "coverage_bench", "device": name, "power_limit_w": watts,
           "workload": "config 2: %.1f Mbp synthetic genome, 2x250 PE at %dx, %d reads; count at f0 = 3, build at min_freq 4" % (args.genome_mbp, args.coverage, n_reads),
           "repeats": args.repeats, "statistic": "median device ms per call (CUDA events), calls alternating empty / edges / reads",
           "n_kept": n_kept, "index_slots": table_slots(n_kept), "index_load": round(load, 3), "index_build_ms": round(index_ms, 2),
           "est_slots_per_hit": round(hit_slots, 2), "est_slots_per_miss": round(miss_slots, 2), "edges": res["edges"], "reads": res["reads"]}
    lib.w2rap_step2_free_host_reads(C.byref(hr))
    lib.w2rap_step2_free(C.byref(g))
    lib.w2rap_step2_counts_release(ch)
    lib.w2rap_step2_release(h)
    line = json.dumps(out)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
