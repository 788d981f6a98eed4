"""min_freq sweep on one B200: four whole runs (w2rap_step2_run_resident at min_freq 3, 4, 5, 6) against one count at f0 = 3 and
four builds from it (w2rap_step2_count + w2rap_step2_build, include/w2rap_step2_counts.h), alternating in one process.

Input: bench.py's config 2 (135 Mbp synthetic genome, 2x250 PE at 60x, seed 1000), generated on the device.  Every call is
repeated --repeats times (the runs, then the count and the builds, per repeat); the medians of the device timings are reported:
total_ms, count_ms and adjacency_ms + unipath_ms.  Each build's digests must equal those of the run at the same min_freq.  The card's
name and power limit are read (read-only NVML query) in the same process.  Prints one JSON line (and writes it to --out).
There is no CPU path: without a B200 the script fails.

    python tools/min_freq_sweep.py [--repeats 5] [--out profiles/<name>.json]
"""
import argparse
import ctypes as C
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import w2r_testlib as T  # noqa: E402


def card():
    """(name, power limit in W) of device 0 from NVML (pynvml, else nvidia-smi's query): reads only."""
    try:
        import pynvml as N
        N.nvmlInit()
        h = N.nvmlDeviceGetHandleByIndex(0)
        name = N.nvmlDeviceGetName(h)
        return (name.decode() if isinstance(name, bytes) else name), N.nvmlDeviceGetPowerManagementLimit(h) / 1000.0
    except Exception:
        import subprocess
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader,nounits", "-i", "0"], capture_output=True, text=True, timeout=30)
        name, watts = [x.strip() for x in r.stdout.strip().splitlines()[0].split(",")]
        return name, float(watts)


def median(v):
    v = sorted(v)
    return v[len(v) // 2] if len(v) % 2 else 0.5 * (v[len(v) // 2 - 1] + v[len(v) // 2])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--genome-mbp", type=float, default=135.0)
    ap.add_argument("--coverage", type=int, default=60)
    ap.add_argument("--freqs", default="3,4,5,6")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if args.repeats < 3:
        raise SystemExit("--repeats must be at least 3")
    freqs = [int(x) for x in args.freqs.split(",")]
    f0 = min(freqs)

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
    err = C.create_string_buffer(1024)

    genome = int(args.genome_mbp * 1e6)
    n_reads = (genome * args.coverage // 250) & ~1
    h = C.c_void_p()
    if lib.w2rap_step2_synth(C.byref(T.SynthParams(genome, 250, args.coverage, 1000, 0, 0, n_reads, 0)), 0, C.byref(h), err, 1024):
        raise SystemExit("synth failed: " + err.value.decode())

    def result(rc, g):
        if rc:
            raise SystemExit("call failed (%d): %s" % (rc, err.value.decode()))
        t = g.timings
        r = dict(total_ms=t.total_ms, count_ms=t.count_ms, graph_ms=t.adjacency_ms + t.unipath_ms, digests=(int(g.digest_graph), int(g.digest_paths)),
                 n_solid=int(g.n_solid), map_ms=t.kernel_ms[1])
        lib.w2rap_step2_free(C.byref(g))
        return r

    def run(mf):
        g = T.Graph()
        return result(lib.w2rap_step2_run_resident(h, C.byref(T.default_params(min_freq=mf, apply_fixpaths=1, device=0)), C.byref(g), err, 1024), g)

    def count():
        ch, g = C.c_void_p(), T.Graph()
        return ch, result(lib.w2rap_step2_count(h, C.byref(T.default_params(min_freq=f0, device=0)), C.byref(ch), C.byref(g), err, 1024), g)

    def build(ch, mf):
        g = T.Graph()
        return result(lib.w2rap_step2_build(h, ch, C.byref(T.default_params(min_freq=mf, apply_fixpaths=1, device=0)), C.byref(g), err, 1024), g)

    for _ in range(args.warmup):
        run(f0)
        ch, _c = count()
        build(ch, f0)
        lib.w2rap_step2_counts_release(ch)
    runs = {mf: [] for mf in freqs}
    builds = {mf: [] for mf in freqs}
    counts = []
    for _ in range(args.repeats):
        for mf in freqs:
            runs[mf].append(run(mf))
        ch, cr = count()
        counts.append(cr)
        for mf in freqs:
            builds[mf].append(build(ch, mf))
        lib.w2rap_step2_counts_release(ch)
    lib.w2rap_step2_release(h)

    def med(rs, key):
        return round(median([r[key] for r in rs]), 2)
    per = {}
    digests_equal = True
    for mf in freqs:
        same = all(b["digests"] == r["digests"] and b["n_solid"] == r["n_solid"] for b in builds[mf] for r in runs[mf])
        digests_equal &= same
        rt, rc, rg = med(runs[mf], "total_ms"), med(runs[mf], "count_ms"), med(runs[mf], "graph_ms")
        bt, bc, bg = med(builds[mf], "total_ms"), med(builds[mf], "count_ms"), med(builds[mf], "graph_ms")
        per[str(mf)] = dict(
            run=dict(total_ms=rt, count_ms=rc, adjacency_plus_unipath_ms=rg),
            build=dict(total_ms=bt, count_ms=bc, adjacency_plus_unipath_ms=bg, map_ms=max(b["map_ms"] for b in builds[mf])),
            n_solid=runs[mf][0]["n_solid"], digests_equal=same,
            build_total_within_run_minus_0p8_count=bool(bt <= rt - 0.8 * rc),
            build_graph_within_5pct_of_run=bool(bg <= 1.05 * rg))
    count_total = med(counts, "total_ms")
    out = {
        "tool": "min_freq_sweep", "device": name, "power_limit_w": watts,
        "workload": "config 2: %.1f Mbp synthetic genome, 2x250 PE at %dx, %d reads, resident; min_qual 7; runs and builds with FixPaths" % (args.genome_mbp, args.coverage, n_reads),
        "repeats": args.repeats, "statistic": "median device ms per call (CUDA events)", "f0": f0,
        "count_call": dict(total_ms=count_total, n_kept=counts[0]["n_solid"]),
        "per_min_freq": per,
        "sweep_total_ms": dict(runs=round(sum(per[str(mf)]["run"]["total_ms"] for mf in freqs), 2),
                               count_plus_builds=round(count_total + sum(per[str(mf)]["build"]["total_ms"] for mf in freqs), 2)),
        "digests_equal": digests_equal,
    }
    line = json.dumps(out)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")
    if not digests_equal:
        raise SystemExit("a build's digests differ from the run at the same min_freq")


if __name__ == "__main__":
    main()
