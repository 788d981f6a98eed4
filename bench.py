#!/usr/bin/env python
"""bench.py — step-2 K=60 graph build throughput (Gbases/s) on N B200s; see DESIGN.md §Measurement.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--genome-mbp G] [--coverage C] [--impl reference] [--dump-outputs DIR]

One step = one whole pass of step 2 (count -> adjacency -> unipaths -> HBV -> read pathing) over one synthetic read set.
`value` = bases / device time with the read stores already resident in HBM; `e2e` = the same through w2rap_step2_run()
with pinned HOST buffers (H2D of the stores and D2H of graph + paths inside the timed region).
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(ROOT, "tests"))

METRIC = "step-2 K=60 graph build Gbases/s"


def clocks_sampler(stop, out):
    """SM clock + throttle reasons during the timed region.  In-process NVML (a few microseconds per sample); spawning nvidia-smi
    five times a second re-initialises NVML every time, which takes driver locks and perturbs the very calls being timed."""
    idx = int(os.environ.get("LOCAL_RANK", "0"))
    try:
        import pynvml as N
        N.nvmlInit()
        h = N.nvmlDeviceGetHandleByIndex(idx)
        mx = N.nvmlDeviceGetMaxClockInfo(h, N.NVML_CLOCK_SM)
        reasons_fn = getattr(N, "nvmlDeviceGetCurrentClocksEventReasons", None) or N.nvmlDeviceGetCurrentClocksThrottleReasons
        while not stop.is_set():
            sm = N.nvmlDeviceGetClockInfo(h, N.NVML_CLOCK_SM)
            r = int(reasons_fn(h))
            act = lambda bit: "Active" if r & bit else "Not Active"
            out.append([str(sm), str(mx), act(0x8), act(0x40), act(0x20), act(0x4)])      # hw_slowdown, hw_thermal, sw_thermal, sw_power_cap
            stop.wait(0.05)
        return
    except Exception:
        pass
    q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
    while not stop.is_set():
        try:
            r = subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader,nounits", "-i", str(idx)], capture_output=True, text=True, timeout=5)
            f = [x.strip() for x in r.stdout.strip().split(",")]
            if len(f) >= 6:
                out.append(f)
        except Exception:
            pass
        stop.wait(1.0)


def summarize_clocks(samples):
    if not samples:
        return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
    sm = sorted(int(s[0]) for s in samples if s[0].isdigit())
    reasons = []
    for i, name in enumerate(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")):
        if any(s[2 + i].lower().startswith("active") for s in samples):
            reasons.append(name)
    return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": int(samples[0][1]) if samples[0][1].isdigit() else None, "reasons": reasons}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return json.load(open(p)).get("hbm_gbs", 6650.0), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def sample_reads(args):
    """The bounded CPU-baseline sample: same read model as the bench workload (2x250 PE, 60x... of a random genome with repeat
    families), sized for ~10-30 s of reference CPU time.  Both arms get exactly these reads."""
    import numpy as np
    import w2r_testlib as T
    genome = int(args.ref_genome_mbp * 1e6)
    rng = np.random.default_rng(1)
    g = T.make_genome(rng, genome, max(1, genome // 50000))
    n_pairs = genome * args.coverage // (2 * args.read_len)
    rs = T.flatten_reads(*T.simulate_reads(rng, [(g, False, 1.0)], n_pairs, args.read_len))
    desc = "%.1f Mbp random genome + repeats, 2x%d PE at %dx (%d reads, %.0f Mbases)" % (args.ref_genome_mbp, args.read_len, args.coverage, rs.n, rs.n_bases / 1e6)
    return rs, desc


def time_reference(rs, cores, binary=None):
    """One run of the reference's own step 2 (oracle/_ref, all host threads) on `rs`; returns (seconds, kind, result dir or None)."""
    import w2r_testlib as T
    if os.path.exists(binary or T.REF_BIN):
        d = tempfile.mkdtemp(prefix="w2rap_ref_")
        T.write_fastb_qualp(d, rs)
        _, perf = T.run_reference_step2(d, threads=cores, binary=binary)
        return perf.get("buildReadQGraph", 0.0) + perf.get("FixPaths", 0.0), "reference", d
    t0 = time.time()
    T.run_oracle(rs, T.default_params(apply_fixpaths=1))
    return time.time() - t0, "port", None


def run_reference_arm(args):
    """The reference's own CPU step 2 (oracle/_ref/w2rap-contigger, all host threads) on a bounded sample of the same workload."""
    import w2r_testlib as T
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    rs, desc = sample_reads(args)
    times, kind = [], "port"
    for it in range(args.warmup + args.steps):
        t, kind, d = time_reference(rs, cores)
        if d:
            subprocess.run(["rm", "-rf", d])
        if it >= args.warmup:
            times.append(t)
    times.sort()
    t = times[len(times) // 2]
    v = rs.n_bases / t / 1e9
    sample = desc + "; " + ("oracle/_ref/w2rap-contigger --from_step 2 --to_step 2, TIME buildReadQGraph+FixPaths" if kind == "reference" else "oracle/step2_oracle.c")
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": "Gbases/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": t * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u64", "data": "synthetic",
            "config": {"workload": "bounded sample of the bench workload: " + sample},
            "cpu_baseline": {"value": v, "unit": "Gbases/s", "cores": cores if kind == "reference" else 1, "kind": kind, "sample": sample},
            "e2e": {"value": v, "unit": "Gbases/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def same_input_comparison(args, lib, local):
    """The bounded sample through BOTH arms on identical reads: the reference binary on the host cores, the product through
    w2rap_step2_run (host buffers, copies inside), and the reference binary with the drop-in translation unit.  Also a cheap
    cross-check of the results (histogram, edge bases, reads pathed)."""
    import numpy as np
    import w2r_testlib as T
    cores = os.cpu_count() or 1
    rs, desc = sample_reads(args)
    t_cpu, kind, d = time_reference(rs, cores)
    out = {"sample": desc, "cpu_s": t_cpu, "cpu_kind": kind, "cpu_cores": cores if kind == "reference" else 1, "cpu_gbases_per_s": rs.n_bases / t_cpu / 1e9}
    p = T.default_params(apply_fixpaths=1, device=local)
    T.run_product(rs, p)                                  # warm-up (pinned pool, device pool)
    walls = []
    got = None
    for _ in range(3):
        got = T.run_product(rs, p)
        walls.append(got["timings"]["wall_ms"])
    walls.sort()
    out["gpu_wall_ms"] = walls[1]
    out["gpu_gbases_per_s"] = rs.n_bases / (walls[1] * 1e-3) / 1e9
    out["vs_cpu_same_input"] = out["gpu_gbases_per_s"] / out["cpu_gbases_per_s"]
    if d:
        try:
            hist = T.parse_freqs(os.path.join(d, "small_K.freqs"))
            hbv = T.parse_hbv(os.path.join(d, "x.small_K.hbv"))
            out["check"] = {"hist_equal": bool(np.array_equal(hist[1:], got["hist"][1:])),
                            "hbv_edges": [len(hbv["edges"]), got["n_hbv_edges"]],
                            "hbv_edge_bases_equal": int(sum(len(e) for e in hbv["edges"])) == int(sum(int(got["edge_len"][i]) * (1 if got["fwd_xlat"][i] == got["rev_xlat"][i] else 2) for i in range(got["n_edges"])))}
        except Exception as e:
            out["check"] = {"error": repr(e)[:200]}
        subprocess.run(["rm", "-rf", d])
    dropin = os.path.join(os.path.dirname(T.REF_BIN), "w2rap-contigger-b200")
    if os.path.exists(dropin):                             # the reference's own main() with the step-2 TU swapped (INTEGRATION.md)
        try:
            t_d, _, d2 = time_reference(rs, cores, binary=dropin)
            d3 = None
            out["dropin_binary_s"] = t_d
            out["dropin_note"] = "TIME buildReadQGraph+FixPaths inside oracle/_ref/w2rap-contigger-b200: flatten of vecbvec/VecPQVec + w2rap_step2_run + HyperBasevector/ReadPathVec rebuild, cold process (CUDA context + pool creation inside)"
            for x in (d2, d3):
                if x:
                    subprocess.run(["rm", "-rf", x])
        except Exception as e:
            out["dropin_binary_s"] = None
            out["dropin_note"] = repr(e)[:200]
    return out


# ncu --set full of the dominant kernels on THIS workload (profiles/r2_ncu_*): dram__bytes_read.sum + dram__bytes_write.sum per launch
NCU_TRAFFIC_BYTES = {}
NCU_TRAFFIC_SOURCE = "profiles/r2_ncu_c2_summary.txt"


def load_ncu_traffic():
    p = os.path.join(ROOT, "profiles", "r2_ncu_traffic.json")
    if os.path.exists(p):
        try:
            return json.load(open(p))
        except Exception:
            pass
    return {}


def digest_reference(key):
    p = os.path.join(ROOT, "tests", "golden", "bench_digests.json")
    if os.path.exists(p):
        try:
            return json.load(open(p)).get(key)
        except Exception:
            pass
    return None


DUMP_ARRAYS = ("hist", "edge_off", "edge_len", "edge_bases", "edge_vertices", "fwd_xlat", "rev_xlat", "involution",
               "path_offset", "path_off", "path_edges", "place_off", "place_edges")
DUMP_COUNTS = ("n_reads", "n_bases", "n_kmer_instances", "n_distinct", "n_solid", "n_edges", "n_edge_bases", "n_vertices", "n_hbv_edges",
               "n_paths", "n_path_edges", "n_pathed", "n_multipathed", "n_places_kept", "n_places")
DUMP_CAP = 1 << 19          # elements kept per array: the 13 arrays and the counters stay under 64 MB in float64


def dump_outputs(d, out_dir):
    """Writes the w2rap_graph `d` (a T.graph_to_dict) as out_dir/<field>.npy in float64, which holds every value exactly (all are
    below 2^53).  An array longer than DUMP_CAP is replaced by its elements at DUMP_CAP sorted positions drawn with a fixed seed, so
    two builds that agree on its length sample the same positions.  An array the step did not fill (the places without --places) is
    not written.  counts.npy holds the counters in DUMP_COUNTS order, then the graph and path digests as 32-bit halves (high, low)."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name in DUMP_ARRAYS:
        a = np.asarray(d[name]).reshape(-1)
        if a.size == 0:
            continue
        if a.size > DUMP_CAP:
            a = a[np.sort(np.random.default_rng(0).choice(a.size, DUMP_CAP, replace=False))]
        np.save(os.path.join(out_dir, name + ".npy"), a.astype(np.float64))
    digests = [x for k in ("digest_graph", "digest_paths") for x in (d[k] >> 32, d[k] & 0xffffffff)]
    np.save(os.path.join(out_dir, "counts.npy"), np.array([d[k] for k in DUMP_COUNTS] + digests, dtype=np.float64))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--config", default="c2", choices=["c1", "c2", "c3", "custom"], help="BASELINE.json configs: c1 = 4.6 Mbp 100x, c2 = 135 Mbp 60x (default, the single-GPU bench), c3 = 1 Gbp 60x 1%% het (8 GPUs)")
    ap.add_argument("--genome-mbp", type=float, default=None)
    ap.add_argument("--coverage", type=int, default=None)
    ap.add_argument("--read-len", type=int, default=250)
    ap.add_argument("--het", type=int, default=None, help="SNPs per 10,000 bases on the second haplotype")
    ap.add_argument("--ref-genome-mbp", type=float, default=2.0, help="size of the bounded CPU-baseline sample")
    ap.add_argument("--places", type=int, default=0, help="also build step 3's places for this large K inside the timed step (SURVEY N1; off by default: not part of the metric)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true", help="skip the host-buffer (e2e) legs: for workloads whose reads do not fit pinned host memory")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the graph and paths the last timed step returned as DIR/<name>.npy (float64; arrays longer than %d elements as a "
                         "fixed seeded sample of that many; the places only with --places; in a sharded run rank 0's: the graph and the paths "
                         "of its reads)" % DUMP_CAP)
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes what the B200 path returns; the reference arm has no such output")
    preset = {"c1": (4.6, 100, 0), "c2": (135.0, 60, 0), "c3": (1000.0, 60, 100), "custom": (135.0, 60, 0)}[args.config]
    if args.genome_mbp is None:
        args.genome_mbp = preset[0]
    else:
        args.config = "custom" if args.genome_mbp != preset[0] else args.config
    if args.coverage is None:
        args.coverage = preset[1]
    if args.het is None:
        args.het = preset[2]
    if args.impl == "reference":
        return run_reference_arm(args)

    import w2r_testlib as T
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    dist = None
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    lib = T.product_lib()
    if lib.w2rap_step2_device_count() <= local:
        raise SystemExit("no B200 visible: this benchmark has no CPU path")
    err = C.create_string_buffer(1024)
    genome = int(args.genome_mbp * 1e6)
    # strong scaling: ONE read set (a function of the seed only); rank r holds the reads [r*n/N, (r+1)*n/N) of it
    total_reads = (genome * args.coverage // args.read_len) & ~1
    per = (total_reads // world) & ~1
    first = per * rank
    mine = per if rank < world - 1 else total_reads - first
    sp = T.SynthParams(genome, args.read_len, args.coverage, 1000, args.het, 0, mine, first)
    h = C.c_void_p()
    comm = C.c_void_p()
    if world > 1:
        import torch
        uid = torch.zeros(128, dtype=torch.uint8)
        if rank == 0:
            buf = (C.c_uint8 * 128)()
            if lib.w2rap_step2_comm_unique_id(buf, err, 1024):
                raise SystemExit("nccl id failed: " + err.value.decode())
            uid = torch.tensor(list(buf), dtype=torch.uint8)
        uid = uid.cuda()
        dist.broadcast(uid, 0)
        buf = (C.c_uint8 * 128)(*uid.cpu().tolist())
        if lib.w2rap_step2_comm_init(buf, world, rank, local, C.byref(comm), err, 1024):
            raise SystemExit("comm init failed: " + err.value.decode())
    if lib.w2rap_step2_synth(C.byref(sp), local, C.byref(h), err, 1024):
        raise SystemExit("synth failed: " + err.value.decode())
    p = T.default_params(apply_fixpaths=1, device=local, graph_on_root_only=1 if world > 1 else 0, places_K2=args.places)      # (the graph arrays go to the one process that would write the .hbv)
    hr = T.Reads()
    do_e2e = not args.no_e2e
    if do_e2e and lib.w2rap_step2_download_reads(h, C.byref(hr), err, 1024):
        raise SystemExit("download failed: " + err.value.decode())
    n_reads = mine
    n_bases = n_reads * args.read_len

    def barrier():
        if dist is not None:
            dist.barrier()

    def timings_of(g):
        return {n: (list(getattr(g.timings, n)) if n == "kernel_ms" else getattr(g.timings, n)) for n, _ in T.Timings._fields_}

    kept = {}

    def step_resident(keep=False):
        g = T.Graph()
        rc = lib.w2rap_step2_run_sharded_resident(h, C.byref(p), comm, C.byref(g), err, 1024) if world > 1 else lib.w2rap_step2_run_resident(h, C.byref(p), C.byref(g), err, 1024)
        if rc:
            raise SystemExit("run failed: " + err.value.decode())
        t = timings_of(g)
        t["n_places_kept"], t["n_places"] = int(g.n_places_kept), int(g.n_places)
        info = (int(g.n_kmer_instances), int(g.n_distinct), int(g.n_solid), int(g.n_edges), int(g.n_edge_bases), int(g.n_pathed), int(g.n_path_edges), int(g.digest_graph), int(g.digest_paths))
        if keep:
            kept["graph"] = T.graph_to_dict(g)      # host copy after the step's own timings were taken
        lib.w2rap_step2_free(C.byref(g))
        return t, info

    def step_e2e(reads):
        g = T.Graph()
        rc = lib.w2rap_step2_run_sharded(C.byref(reads), C.byref(p), comm, C.byref(g), err, 1024) if world > 1 else lib.w2rap_step2_run(C.byref(reads), C.byref(p), C.byref(g), err, 1024)
        if rc:
            raise SystemExit("run failed: " + err.value.decode())
        t = timings_of(g)
        d2h = 8 * (int(g.n_edges) + 1) + 4 * int(g.n_edges) * 7 + int(g.n_edge_bases) // 4 + 4 * int(g.n_hbv_edges) + 4 * int(g.n_paths) + 8 * (int(g.n_paths) + 1) + 4 * int(g.n_path_edges)
        dg = (int(g.digest_graph), int(g.digest_paths))
        lib.w2rap_step2_free(C.byref(g))
        return t, d2h, dg

    def median(v):
        v = sorted(v)
        return v[len(v) // 2] if len(v) % 2 else 0.5 * (v[len(v) // 2 - 1] + v[len(v) // 2])

    for _ in range(args.warmup):
        step_resident()
    stop, samples = threading.Event(), []
    th = threading.Thread(target=clocks_sampler, args=(stop, samples), daemon=True)
    th.start()
    barrier()
    tt, info = [], None
    for i in range(args.steps):
        t, info2 = step_resident(keep=args.dump_outputs is not None and rank == 0 and i == args.steps - 1)
        if info is not None and info2 != info:
            raise SystemExit("non-deterministic result between steps: %r vs %r" % (info, info2))
        info = info2
        tt.append(t)
    barrier()
    if kept:
        dump_outputs(kept.pop("graph"), args.dump_outputs)
    dev_ms = median([t["total_ms"] - t["d2h_ms"] for t in tt])      # device time, results left on the device side of the copy
    full_ms = median([t["total_ms"] for t in tt])
    # end to end through the host-buffer entry point: pinned host buffers, then pageable ones
    e2e_ms, e2e_d2h, e2e_t, e2e_pageable_ms = None, 0, [], None
    if do_e2e:
        _, _, dg = step_e2e(hr)
        if dg != info[7:9]:
            raise SystemExit("host-buffer run and resident run disagree: digests %r vs %r" % (dg, info[7:9]))
        barrier()
        walls = []
        for _ in range(args.steps):
            t0 = time.time()
            tt_e, e2e_d2h, _ = step_e2e(hr)
            walls.append((time.time() - t0) * 1e3)
            e2e_t.append(tt_e)
        barrier()
        e2e_ms = median(walls)
        if world == 1:
            # pageable host memory (what a caller that does not pin its read stores hands over: host/BuildReadQGraph_b200.cc)
            import numpy as np
            nr = int(hr.n_reads)
            boff, qoff = T._arr(hr.base_off, nr + 1, "<u8"), T._arr(hr.qual_off, nr + 1, "<u8")
            pg = T.ReadSet(T._arr(hr.bases, int(boff[-1]), "u1"), boff, T._arr(hr.len, nr, "<u4"), T._arr(hr.quals, int(qoff[-1]), "u1"), qoff)
            pr = pg.c()
            step_e2e(pr)
            walls = []
            for _ in range(max(1, min(args.steps, 3))):
                t0 = time.time()
                step_e2e(pr)
                walls.append((time.time() - t0) * 1e3)
            e2e_pageable_ms = median(walls)
    stop.set()
    th.join(timeout=2)
    total_bases = n_bases
    if dist is not None:
        import torch
        v = torch.tensor([dev_ms, e2e_ms or 0.0, full_ms], device="cuda")
        dist.all_reduce(v, op=dist.ReduceOp.MAX)
        dev_ms, e2e_max, full_ms = [float(x) for x in v.tolist()]
        e2e_ms = e2e_max if do_e2e else None
        nb = torch.tensor([n_bases, int(tt[-1]["exchange_bytes"]), int(tt[-1]["count_exchange_bytes"])], device="cuda", dtype=torch.int64)
        dist.all_reduce(nb)
        total_bases, xbytes_all, xbytes_count = int(nb[0].item()), int(nb[1].item()), int(nb[2].item())
    else:
        xbytes_all = xbytes_count = 0
    if rank != 0:
        if world > 1:
            lib.w2rap_step2_comm_destroy(comm)
            dist.destroy_process_group()
        return
    I_all, D, S, E, EB, pathed, npe, dig_g, dig_p = info
    I = I_all // world                  # this rank's share of the k-mer instances (the counters are whole-job)
    qbytes = int(T._arr(hr.qual_off, n_reads + 1, "<u8")[-1]) if do_e2e else int(0.42 * n_bases)
    b_bases = n_reads * ((args.read_len + 3) // 4)
    b_in = b_bases + qbytes + 12 * n_reads
    b_path = 6 * n_reads + 4 * npe
    alg_bytes_total = 2 * b_in + 34 * I + 48 * S + EB // 2 + b_path                 # SURVEY.md §8(d), per rank
    # per-kernel CUDA-event times (w2rap_timings.kernel_ms) with the SURVEY §8(d) bytes each kernel owns.  The model charges 34 B per
    # k-mer instance for "written once and read once": the map owns the write half, the reduce the read half (the product moves
    # ~2.5 B per instance instead: super-k-mer records; the fractions of these two are quoted against the model's bytes all the
    # same).  k_scatter_records is charged what it really moves: 32 + 4 B read and 32 B written per record.
    km = {T.KERNEL_NAMES[i]: median([t["kernel_ms"][i] for t in tt]) for i in range(len(T.KERNEL_NAMES))}
    S_rank = S // world
    nrec = int(tt[-1]["n_records"])
    alg = {"k_good_len": qbytes + 12 * n_reads, "k_minimizer_map": b_bases + 14 * n_reads + 17 * I, "k_scatter_records": 72 * nrec,
           "k_count_smem": 17 * I, "k_insert_solid": 48 * S_rank // 2, "k_adjacency": 48 * S_rank // 2, "k_links": 24 * S_rank, "k_splitter_walk": 24 * S_rank, "k_splitter_finish": 24 * S_rank,
           "k_emit_edges": EB // 2 // world + 24 * S_rank, "k_path_reads": b_in + b_path}
    launches = {"k_minimizer_map": max(1, tt[-1]["count_launches"]), "k_scatter_records": max(1, tt[-1]["count_launches"]), "k_good_len": max(1, tt[-1]["count_launches"])}
    phases = {k: v for k, v in km.items() if k not in alg and not k.startswith("unused")}      # phase timers of the sharded graph stage: several kernels + exchanges each
    km = {k: v for k, v in km.items() if k in alg}
    dom = max(km, key=lambda k: km[k])
    peak, peak_src = peaks()
    traffic = load_ncu_traffic()
    per_kernel = {k: {"ms": round(km[k], 3), "algorithmic_bytes": int(alg[k]), "GBps": round(alg[k] / (km[k] * 1e-3) / 1e9, 1) if km[k] > 0 else None,
                      "frac": round(alg[k] / (km[k] * 1e-3) / 1e9 / peak, 4) if km[k] > 0 else None} for k in km}
    achieved = alg[dom] / (km[dom] * 1e-3) / 1e9
    nl = launches.get(dom, 1)
    cpu, same = None, None
    if not args.no_cpu_baseline and world == 1:
        try:
            same = same_input_comparison(args, lib, local)
            arm = "oracle/_ref/w2rap-contigger --from_step 2 --to_step 2, TIME buildReadQGraph+FixPaths" if same["cpu_kind"] == "reference" else "oracle/step2_oracle.c"
            cpu = {"value": same["cpu_gbases_per_s"], "unit": "Gbases/s", "cores": same["cpu_cores"], "kind": same["cpu_kind"],
                   "sample": same["sample"] + "; " + arm + " (bounded sample: the ratio to `value` is indicative; `same_input` holds the like-for-like one)"}
        except Exception as e:   # the baseline is reported, never required
            cpu = {"value": None, "unit": "Gbases/s", "cores": os.cpu_count(), "kind": "unavailable", "sample": repr(e)[:200]}
    wkey = "genome%.1fMbp_cov%d_len%d_het%d_seed1000" % (args.genome_mbp, args.coverage, args.read_len, args.het)
    ref_dig = digest_reference(wkey)
    digest = {"graph": "%016x" % dig_g, "paths": "%016x" % dig_p, "workload_key": wkey,
              "check": "no stored digest for this workload" if not ref_dig else ("match" if ref_dig == ["%016x" % dig_g, "%016x" % dig_p] else "MISMATCH vs tests/golden/bench_digests.json")}
    line = {
        "metric": METRIC, "value": total_bases / (dev_ms * 1e-3) / 1e9, "unit": "Gbases/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": dev_ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u64", "data": "synthetic",
        "config": {"workload": "%s: %.1f Mbp synthetic genome + repeat families%s, 2x%d bp PE at %dx (rank 0 shard: %d reads, %.2f Gbases; whole job = n_gpus shards), min_qual 7, min_freq 4; whole step 2 incl. read pathing + FixPaths" % (
                       args.config, args.genome_mbp, (", second haplotype with %d SNPs per 10 kb" % args.het) if args.het else "", args.read_len, args.coverage, n_reads, n_bases / 1e9),
                   "cache": "inputs (%.1f GB) and dictionary larger than the 126 MB L2" % (b_in / 1e9),
                   "statistic": "median over the timed steps",
                   "kmer_instances": I_all, "distinct": D, "solid": S, "edges": E, "reads_pathed": pathed,
                   "parallelism": "one process per GPU; reads sharded by index; super-k-mer records routed to the owner GPU of their minimiser partition (NCCL all-to-all of exactly sized runs); dictionary, adjacency and unipaths sharded by the same owners (neighbour queries + chain-end records exchanged); pathing dictionary built in hash slices (one per GPU) and replicated by one all-gather of table memory; reads pathed by shard; graph arrays returned to rank 0 (graph_on_root_only), paths to the rank of their reads"},
        "e2e": ({"value": total_bases / (e2e_ms * 1e-3) / 1e9, "unit": "Gbases/s", "h2d_bytes_per_step": b_in, "d2h_bytes_per_step": e2e_d2h, "ms_per_step": e2e_ms, "host_memory": "pinned",
                 "inside": {k: median([t[k] for t in e2e_t]) for k in ("h2d_ms", "total_ms", "count_ms", "count_kernel_ms", "region_ms", "path_ms", "d2h_ms", "host_pre_ms", "host_post_ms", "wall_ms")}}
                if do_e2e else {"value": None, "unit": "Gbases/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0, "skipped": "--no-e2e"}),
        "e2e_pageable": ({"value": total_bases / (e2e_pageable_ms * 1e-3) / 1e9, "unit": "Gbases/s", "ms_per_step": e2e_pageable_ms, "host_memory": "pageable (numpy buffers)"} if e2e_pageable_ms else None),
        "gpu_launches": int(tt[-1]["kernel_launches"]) * args.steps,
        "roofline": {"bound": "hbm", "kernel": dom, "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": traffic.get(dom, {}).get("dram_bytes_per_launch"), "traffic_source": traffic.get(dom, {}).get("source"),
                     "peak_source": peak_src, "algorithmic_bytes_per_launch": alg[dom] / nl, "launches_per_step": nl,
                     "kernel_ms_per_step": km[dom], "per_kernel": per_kernel, "sharded_graph_phases_ms": {k: round(v, 3) for k, v in phases.items()} if world > 1 else None,
                     "whole_step_algorithmic_GBps": alg_bytes_total / (dev_ms * 1e-3) / 1e9, "whole_step_frac": alg_bytes_total / (dev_ms * 1e-3) / 1e9 / peak},
        "alloc_host_ms": [round(t["alloc_host_ms"], 1) for t in tt],
        "places": ({"K2": args.places, "ms": median([t["places_ms"] for t in tt]), "paths_kept": tt[-1].get("n_places_kept"), "unique_places": tt[-1].get("n_places"), "note": "inside ms_per_step; RepathInMemory's places built on the device (paths/long/large/Repath.cc:46-72)"} if args.places else None),
        "stage_ms": {k: median([t[k] for t in tt]) for k in ("count_ms", "count_kernel_ms", "region_ms", "dict_ms", "exchange_ms", "graph_exchange_ms", "adjacency_ms", "unipath_ms", "hbv_ms", "path_ms", "d2h_ms", "total_ms")},
        "nvlink": ({"bytes_delivered_all_ranks_per_step": xbytes_all, "of_which_count_records": xbytes_count,
                    "of_which_graph_and_dictionary": xbytes_all - xbytes_count,
                    "count_record_bytes_per_kmer_instance": xbytes_count / max(1, I_all),
                    "count_exchange_GBps_per_gpu": (xbytes_count / world) / max(1e-9, median([t["exchange_ms"] for t in tt]) * 1e-3) / 1e9,
                    "note": "bytes each rank sends to the other ranks (an all-gathered slice counts once per receiver)"} if world > 1 else None),
        "result_digest": digest,
        "clocks": summarize_clocks(samples),
        "per_step": {"resident_ms": [round(t["total_ms"] - t["d2h_ms"], 2) for t in tt], "resident_count_ms": [round(t["count_ms"], 2) for t in tt],
                     "e2e_wall_ms": [round(t["wall_ms"], 2) for t in e2e_t]},
        "cpu_baseline": cpu,
        "same_input": same,
    }
    print(json.dumps(line))
    if digest["check"].startswith("MISMATCH"):
        raise SystemExit("result digest differs from the stored single-GPU digest of this workload")
    if do_e2e:
        lib.w2rap_step2_free_host_reads(C.byref(hr))
    lib.w2rap_step2_release(h)
    if world > 1:
        lib.w2rap_step2_comm_destroy(comm)
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
