"""Count once and build per min_freq with the reads sharded over GPUs, against one sharded run per min_freq
(include/w2rap_step2_counts_sharded.h).

Inputs: bench.py's configs, generated on the devices with w2rap_step2_synth (rank r synthesises the reads [first_read,
first_read + n_reads) of the one read set, as bench.py --gpus does): config 3 (1 Gbp, 60x, 1 % heterozygous) and config 2
(135 Mbp, 60x), both on 8 GPUs.  Ranks are threads of this process, one per GPU.  Per config, alternating for --repeats rounds:
  runs    w2rap_step2_run_sharded_resident at min_freq 3, 4, 5, 6;
  counted w2rap_step2_count_sharded at f0 = 3, then w2rap_step2_build_sharded at 3, 4, 5, 6, then the coverage of the min_freq 4
          edges (passed on rank 0) with w2rap_counts_coverage_sharded, then the handle is released.
Every call's time is timings.total_ms (device time, CUDA events) taken as the largest over the ranks; reported as medians over the
rounds.  Every build's digests must equal the run's at the same min_freq on every rank.  Also recorded: the handle's device bytes
per rank (17 per kept k-mer; the mean over the ranks, whose partition ranges are equal) and the coverage call's device_ms per rank (index build, lookups and merge).  The card's name and
power limit are read in the same process.  Prints one JSON line per config (and writes them to --out).  There is no CPU path.

    python tools/count_once_sharded_bench.py [--gpus 8] [--configs c3,c2] [--repeats 3] [--out profiles/<name>.jsonl]
"""
import argparse
import ctypes as C
import json
import os
import sys
import threading

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "tools"))
import numpy as np  # noqa: E402
import w2r_testlib as T  # noqa: E402
from coverage_bench import COV_DTYPE, Seqs  # noqa: E402
from min_freq_sweep import card, median  # noqa: E402

CONFIGS = {"c2": (135.0, 60, 0), "c3": (1000.0, 60, 100)}      # genome Mbp, coverage, het SNPs per 10 kb (bench.py's presets)
FREQS = (3, 4, 5, 6)
F0 = 3


def bind(lib):
    E = [C.c_char_p, C.c_size_t]
    P = C.POINTER
    lib.w2rap_step2_count_sharded.argtypes = [C.c_void_p, P(T.Params), C.c_void_p, P(C.c_void_p), P(T.Graph)] + E
    lib.w2rap_step2_build_sharded.argtypes = [C.c_void_p, C.c_void_p, P(T.Params), C.c_void_p, P(T.Graph)] + E
    lib.w2rap_counts_coverage_sharded.argtypes = [C.c_void_p, C.c_void_p, P(Seqs), C.c_void_p, P(C.c_float)] + E
    lib.w2rap_step2_counts_release.argtypes = [C.c_void_p]
    lib.w2rap_step2_counts_release.restype = None


def rank_body(lib, uid, world, r, cfg, repeats, res):
    """One rank: synthesise its shard, then the rounds.  Fills res[r] with this rank's times and checks."""
    genome_mbp, coverage, het = CONFIGS[cfg]
    err = C.create_string_buffer(1024)

    def check(rc):
        if rc:
            raise RuntimeError("rank %d: call failed (%d): %s" % (r, rc, err.value.decode(errors="replace")))
    comm, h = C.c_void_p(), C.c_void_p()
    check(lib.w2rap_step2_comm_init(uid, world, r, r, C.byref(comm), err, 1024))
    try:
        genome = int(genome_mbp * 1e6)
        total = (genome * coverage // 250) & ~1
        per = (total // world) & ~1
        mine = per if r < world - 1 else total - per * r
        check(lib.w2rap_step2_synth(C.byref(T.SynthParams(genome, 250, coverage, 1000, het, 0, mine, per * r)), r, C.byref(h), err, 1024))
        p = lambda mf: T.default_params(min_freq=mf, apply_fixpaths=1, device=r)      # noqa: E731

        def graph(call):
            g = T.Graph()
            check(call(g))
            d = dict(total_ms=g.timings.total_ms, digests=(g.digest_graph, g.digest_paths), n_solid=g.n_solid, n_edges=g.n_edges)
            return g, d
        out = dict(runs={f: [] for f in FREQS}, count=[], builds={f: [] for f in FREQS}, coverage_ms=[], digests_equal=True, kept=0,
                   n_solid={}, n_edges={}, edge_lookups=0)
        rounds = [("runs", "counted") if i % 2 == 0 else ("counted", "runs") for i in range(repeats + 1)]     # round 0 is the warm-up
        for i, order in enumerate(rounds):
            digests = {}
            for arm in order:
                if arm == "runs":
                    for f in FREQS:
                        g, d = graph(lambda g: lib.w2rap_step2_run_sharded_resident(h, C.byref(p(f)), comm, C.byref(g), err, 1024))
                        lib.w2rap_step2_free(C.byref(g))
                        digests.setdefault(f, {})["run"] = d["digests"]
                        out["n_solid"][f], out["n_edges"][f] = d["n_solid"], d["n_edges"]
                        if i:
                            out["runs"][f].append(d["total_ms"])
                    continue
                ch, s = C.c_void_p(), T.Graph()
                check(lib.w2rap_step2_count_sharded(h, C.byref(p(F0)), comm, C.byref(ch), C.byref(s), err, 1024))
                if i:
                    out["count"].append(s.timings.total_ms)
                out["kept"] = int(s.n_solid)
                lib.w2rap_step2_free(C.byref(s))
                try:
                    for f in FREQS:
                        g, d = graph(lambda g: lib.w2rap_step2_build_sharded(h, ch, C.byref(p(f)), comm, C.byref(g), err, 1024))
                        digests.setdefault(f, {})["build"] = d["digests"]
                        if i:
                            out["builds"][f].append(d["total_ms"])
                        if f == 4:
                            sv = Seqs(g.n_edges, g.edge_bases, g.edge_off, g.edge_len)
                            cov = np.zeros(max(1, int(g.n_edges)), COV_DTYPE)
                            ms = C.c_float(0)
                            check(lib.w2rap_counts_coverage_sharded(ch, comm, C.byref(sv) if r == 0 else None, cov.ctypes.data, C.byref(ms), err, 1024))
                            bad = int(cov["n_absent"][:int(g.n_edges)].sum()) + int((cov["min"][:int(g.n_edges)] < 4).sum())
                            out["edge_lookups"] = int(cov["n_kmers"][:int(g.n_edges)].sum())
                            if bad or out["edge_lookups"] != int(g.n_solid):
                                raise RuntimeError("rank %d: min_freq 4 edges have absent or rarer k-mers" % r)
                            if i:
                                out["coverage_ms"].append(ms.value)
                        lib.w2rap_step2_free(C.byref(g))
                finally:
                    lib.w2rap_step2_counts_release(ch)
            for f in FREQS:
                if digests[f]["run"] != digests[f]["build"]:
                    out["digests_equal"] = False
        res[r] = out
    finally:
        if h.value:
            lib.w2rap_step2_release(h)
        lib.w2rap_step2_comm_destroy(comm)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=8)
    ap.add_argument("--configs", default="c3,c2")
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if args.repeats < 3:
        raise SystemExit("--repeats must be at least 3")
    lib = T.product_lib()
    if lib.w2rap_step2_device_count() < args.gpus:
        raise SystemExit("%d B200s needed, %d visible: this measurement has no CPU path" % (args.gpus, lib.w2rap_step2_device_count()))
    name, watts = card()
    if "B200" not in name:
        raise SystemExit("device 0 is %s, not a B200" % name)
    bind(lib)
    lines = []
    for cfg in args.configs.split(","):
        err = C.create_string_buffer(512)
        uid = (C.c_uint8 * 128)()
        if lib.w2rap_step2_comm_unique_id(uid, err, 512):
            raise SystemExit(err.value.decode())
        res, errors = [None] * args.gpus, [None] * args.gpus

        def worker(r):
            try:
                rank_body(lib, uid, args.gpus, r, cfg, args.repeats, res)
            except Exception as e:      # noqa: BLE001 — reported below
                errors[r] = repr(e)
        th = [threading.Thread(target=worker, args=(r,), daemon=True) for r in range(args.gpus)]
        [t.start() for t in th]
        [t.join(3000) for t in th]
        if any(t.is_alive() for t in th) or any(errors):
            raise SystemExit("%s: ranks failed or did not finish: %s" % (cfg, errors))
        step = lambda key, f=None: [max(res[r][key][f][i] if f else res[r][key][i] for r in range(args.gpus)) for i in range(args.repeats)]   # noqa: E731
        runs = {f: median(step("runs", f)) for f in FREQS}
        count = median(step("count"))
        builds = {f: median(step("builds", f)) for f in FREQS}
        genome_mbp, coverage, het = CONFIGS[cfg]
        out = {"tool": "count_once_sharded_bench", "device": name, "power_limit_w": watts, "gpus": args.gpus,
               "workload": "config %s: %.0f Mbp synthetic genome%s, 2x250 PE at %dx, seed 1000, sharded by read index over %d GPUs; min_qual 7, FixPaths" % (
                   cfg[1], genome_mbp, (", second haplotype with %d SNPs per 10 kb" % het) if het else "", coverage, args.gpus),
               "repeats": args.repeats, "statistic": "median over rounds of the largest per-rank timings.total_ms (device time) of each call; arms alternate",
               "run_ms": {str(f): round(v, 1) for f, v in runs.items()}, "runs_total_ms": round(sum(runs.values()), 1),
               "count_ms": round(count, 1), "build_ms": {str(f): round(v, 1) for f, v in builds.items()},
               "count_plus_builds_total_ms": round(count + sum(builds.values()), 1),
               "saving_per_extra_graph_ms": round((sum(runs.values()) - count - sum(builds.values())) / (len(FREQS) - 1), 1),
               "digests_equal": all(res[r]["digests_equal"] for r in range(args.gpus)),
               "kept_at_f0": res[0]["kept"], "handle_bytes_per_rank_mean": 17 * res[0]["kept"] // args.gpus,
               "n_solid": {str(f): int(res[0]["n_solid"][f]) for f in FREQS}, "n_edges": {str(f): int(res[0]["n_edges"][f]) for f in FREQS},
               "coverage_mf4_edges": {"lookups": res[0]["edge_lookups"],
                                      "device_ms_per_rank": [round(median(res[r]["coverage_ms"]), 2) for r in range(args.gpus)]}}
        lines.append(json.dumps(out))
        print(lines[-1], flush=True)
        if not out["digests_equal"]:
            raise SystemExit("%s: a build's digests differ from the run's" % cfg)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
