"""Count once, build per min_freq and look up k-mer coverage with the reads sharded over GPUs (include/w2rap_step2_counts_sharded.h).

A sharded count keeps, on each rank, the k-mers of the minimiser partitions it owns.  Every build from it is compared with the oracle
and with w2rap_step2_run_sharded at the same min_freq (every field but the timings, on every rank); the count's summary with the
oracle's counters and with a single-GPU count.  Coverage is compared with the numpy expectation of tests/test_coverage.py and with
the single-GPU call.  On the CPU, the lookup is run with W simulated ranks against the oracle's counts.  Ranks are driven from
threads of this process, one per GPU, as in tests/test_gpu_sharded.py; every rank always gets the same arguments.
"""
import ctypes as C
import os
import re
import subprocess
import threading
import time

import numpy as np
import pytest

import w2r_testlib as T
from test_coverage import COV_DTYPE, SeqSet, Seqs, assert_cov_equal, expected_coverage, kept_dict, mixed_sequences, seqs_of_reads

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
HC_SO = os.path.join(ROOT, "oracle", "_build", "libhostcheck_cov_sharded.so")
BAD_ARG = 1
E = [C.c_char_p, C.c_size_t]


def lib():
    lb = T.product_lib()
    P = C.POINTER
    lb.w2rap_step2_count.argtypes = [C.c_void_p, P(T.Params), P(C.c_void_p), P(T.Graph)] + E
    lb.w2rap_step2_build.argtypes = [C.c_void_p, C.c_void_p, P(T.Params), P(T.Graph)] + E
    lb.w2rap_step2_count_sharded.argtypes = [C.c_void_p, P(T.Params), C.c_void_p, P(C.c_void_p), P(T.Graph)] + E
    lb.w2rap_step2_build_sharded.argtypes = [C.c_void_p, C.c_void_p, P(T.Params), C.c_void_p, P(T.Graph)] + E
    lb.w2rap_step2_counts_release.argtypes = [C.c_void_p]
    lb.w2rap_step2_counts_release.restype = None
    lb.w2rap_counts_coverage.argtypes = [C.c_void_p, P(Seqs), C.c_void_p, P(C.c_float)] + E
    lb.w2rap_counts_coverage_sharded.argtypes = [C.c_void_p, C.c_void_p, P(Seqs), C.c_void_p, P(C.c_float)] + E
    for f in ("w2rap_step2_count_sharded", "w2rap_step2_build_sharded", "w2rap_counts_coverage", "w2rap_counts_coverage_sharded"):
        getattr(lb, f).restype = C.c_int
    return lb


# ---------------------------------------------------------------- CPU: interface

def test_declared_symbols_are_exported():
    txt = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "w2rap_step2_counts_sharded.h")).read(), flags=re.S)
    names = sorted(set(re.findall(r"\b(w2rap_[a-z0-9_]+)\s*\(", txt)))
    assert names == ["w2rap_counts_coverage_sharded", "w2rap_step2_build_sharded", "w2rap_step2_count_sharded"]
    lb = lib()
    for n in names:
        assert hasattr(lb, n), "missing export " + n


def test_null_arguments_and_parameters_are_refused_without_a_device():
    lb, err = lib(), C.create_string_buffer(512)
    fake = C.c_void_p(16)          # never dereferenced: every call below is refused before a handle or communicator is used
    p, g, ch = T.default_params(), T.Graph(), C.c_void_p()
    ss = SeqSet([np.zeros(100, np.uint8)])
    out = np.zeros(1, COV_DTYPE)
    assert lb.w2rap_step2_count_sharded(None, C.byref(p), fake, C.byref(ch), None, err, 512) == BAD_ARG
    assert lb.w2rap_step2_count_sharded(fake, None, fake, C.byref(ch), None, err, 512) == BAD_ARG
    assert lb.w2rap_step2_count_sharded(fake, C.byref(p), None, C.byref(ch), None, err, 512) == BAD_ARG
    assert lb.w2rap_step2_count_sharded(fake, C.byref(p), fake, None, None, err, 512) == BAD_ARG
    for bad, word in ((dict(dump_kmers=1), b"dump_kmers"), (dict(dump_kmers=2), b"dump_kmers"), (dict(min_freq=0), b"min_freq"),
                      (dict(min_freq=256), b"min_freq")):
        ch = C.c_void_p()
        assert lb.w2rap_step2_count_sharded(fake, C.byref(T.default_params(**bad)), fake, C.byref(ch), None, err, 512) == BAD_ARG
        assert word in err.value and not ch.value, bad
    assert lb.w2rap_step2_build_sharded(None, fake, C.byref(p), fake, C.byref(g), err, 512) == BAD_ARG
    assert lb.w2rap_step2_build_sharded(fake, None, C.byref(p), fake, C.byref(g), err, 512) == BAD_ARG
    assert lb.w2rap_step2_build_sharded(fake, fake, None, fake, C.byref(g), err, 512) == BAD_ARG
    assert lb.w2rap_step2_build_sharded(fake, fake, C.byref(p), None, C.byref(g), err, 512) == BAD_ARG
    assert lb.w2rap_step2_build_sharded(fake, fake, C.byref(p), fake, None, err, 512) == BAD_ARG
    assert lb.w2rap_step2_build_sharded(fake, fake, C.byref(T.default_params(min_freq=0)), fake, C.byref(g), err, 512) == BAD_ARG
    assert lb.w2rap_counts_coverage_sharded(None, fake, C.byref(ss.c()), out.ctypes.data, None, err, 512) == BAD_ARG
    assert lb.w2rap_counts_coverage_sharded(fake, None, C.byref(ss.c()), out.ctypes.data, None, err, 512) == BAD_ARG


# ---------------------------------------------------------------- CPU: ownership and simulated ranks

@pytest.fixture(scope="module")
def hc():
    src = os.path.join(HERE, "hostcheck", "coverage_sharded.cpp")
    deps = [src, os.path.join(ROOT, "include", "w2rap_coverage.h")]
    deps += [os.path.join(ROOT, "w2rap-contigger_b200", "csrc", f) for f in ("coverage.cuh", "kmer.cuh", "extract.cuh", "shard.cuh")]
    if not os.path.exists(HC_SO) or any(os.path.getmtime(x) > os.path.getmtime(HC_SO) for x in deps):
        os.makedirs(os.path.dirname(HC_SO), exist_ok=True)
        subprocess.run(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-x", "c++", "-o", HC_SO, src], check=True)
    lb = C.CDLL(HC_SO)
    lb.hc_owners.argtypes = [C.POINTER(Seqs), C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p]
    lb.hc_coverage_sharded.argtypes = [C.c_void_p, C.c_uint64, C.c_uint32, C.c_uint32, C.c_uint32, C.POINTER(Seqs), C.c_void_p]
    return lb


@pytest.mark.parametrize("world", [1, 2, 4, 8])
def test_owner_of_a_position_is_the_owner_of_its_canonical_kmer(hc, world):
    rng = np.random.default_rng(world)
    seqs = [rng.integers(0, 4, int(L), dtype=np.uint8) for L in rng.integers(60, 700, 60)]
    seqs += [np.tile(np.array([0, 1], np.uint8), 100), np.zeros(150, np.uint8)]      # repeats: the minimiser occurs many times
    rcs = [T.revcomp(s) for s in seqs]
    for logP in (3, 10, 16):
        owners = []
        for group in (seqs, rcs):
            ss = SeqSet(group)
            nk = int(np.maximum(ss.len.astype(np.int64) - 59, 0).sum())
            at, ref = np.zeros(nk, np.uint32), np.zeros(nk, np.uint32)
            assert hc.hc_owners(C.byref(ss.c()), logP, world, at.ctypes.data, ref.ctypes.data) == 0
            assert np.array_equal(at, ref), (world, logP)
            owners.append(at)
        # the k-mer at position p of a sequence is the reverse complement of the one at len - 60 - p of its reverse complement
        off = np.concatenate([[0], np.cumsum([len(s) - 59 for s in seqs])])
        for i in range(len(seqs)):
            assert np.array_equal(owners[0][off[i]:off[i + 1]], owners[1][off[i]:off[i + 1]][::-1]), (world, logP, i)
        assert set(owners[0].tolist()) == set(range(world)), (world, logP)


@pytest.mark.parametrize("f0", [1, 3])
def test_simulated_ranks_against_the_oracle_counts(hc, f0):
    rs = T.rich_set(seed=9, genome=20000, cov=40, families=2, palindromes=3, plasmid=700)
    dump = T.run_oracle(rs, T.default_params(min_freq=f0, dump_kmers=2, want_paths=0))["dump"]
    seqs = mixed_sequences(rs, np.random.default_rng(f0)) + step_boundary_sequences(rs)
    ss = SeqSet(seqs)
    want = expected_coverage(seqs, kept_dict(dump, f0))
    for world, logP in ((2, 6), (4, 9), (8, 12)):
        got = np.zeros(len(seqs), COV_DTYPE)
        assert hc.hc_coverage_sharded(dump.ctypes.data, len(dump), f0, logP, world, C.byref(ss.c()), got.ctypes.data) == 0
        assert_cov_equal(want, got, "%d simulated ranks, f0=%d" % (world, f0))


@pytest.fixture(scope="module")
def gc():
    """The kernel harness of tests/hostcheck/coverage_owned_gpu.cu, compiled for sm_100a."""
    src = os.path.join(HERE, "hostcheck", "coverage_owned_gpu.cu")
    so = os.path.join(ROOT, "oracle", "_build", "libgpucheck_cov_owned.so")
    deps = [src] + [os.path.join(ROOT, "w2rap-contigger_b200", "csrc", f) for f in ("coverage.cuh", "kmer.cuh", "extract.cuh", "shard.cuh", "kernels.cuh")]
    if not os.path.exists(so) or any(os.path.getmtime(x) > os.path.getmtime(so) for x in deps):
        os.makedirs(os.path.dirname(so), exist_ok=True)
        nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
        subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O2", "-std=c++17", "--expt-relaxed-constexpr", "-Xcompiler", "-fPIC",
                        "-shared", "-o", so, src], check=True)
    lb = C.CDLL(so)
    lb.gc_coverage_owned.argtypes = [C.c_void_p, C.c_uint64, C.c_uint32, C.c_uint32, C.c_uint32, C.POINTER(Seqs), C.c_void_p]
    return lb


@pytest.mark.gpu
@pytest.mark.parametrize("f0", [1, 3])
def test_owned_lookup_kernel_with_simulated_ranks_on_one_device(gc, f0):
    """k_cov_tiles_owned launched once per simulated rank (W = 1, 2, 4, 8) on one B200, each with the k-mers that rank would keep."""
    if lib().w2rap_step2_device_count() < 1:
        pytest.skip("needs a B200")
    rs = T.rich_set(seed=9, genome=20000, cov=40, families=2, palindromes=3, plasmid=700)
    dump = T.run_oracle(rs, T.default_params(min_freq=f0, dump_kmers=2, want_paths=0))["dump"]
    seqs = mixed_sequences(rs, np.random.default_rng(f0)) + step_boundary_sequences(rs) + seqs_of_reads(rs)
    ss = SeqSet(seqs)
    want = expected_coverage(seqs, kept_dict(dump, f0))
    for world, logP in ((1, 4), (2, 6), (4, 9), (8, 12)):
        got = np.zeros(len(seqs), COV_DTYPE)
        assert gc.gc_coverage_owned(dump.ctypes.data, len(dump), f0, logP, world, C.byref(ss.c()), got.ctypes.data) == 0
        assert_cov_equal(want, got, "kernel, %d simulated ranks, f0=%d" % (world, f0))


def step_boundary_sequences(rs):
    """Read prefixes whose k-mer counts end around the 32-position steps of k_cov_tiles_owned, and reverse-complemented reads."""
    seqs = [rs.read_codes(7 + i)[:59 + m] for i, m in enumerate((31, 32, 33, 64, 65))]
    return seqs + [T.revcomp(rs.read_codes(r)) for r in (2, 5, 8, 13)]


# ---------------------------------------------------------------- GPU: ranks on threads

def shards_of(rs, world):
    n = rs.n - (rs.n % (2 * world))
    bounds = [(n // world) * r for r in range(world)] + [rs.n]      # pairs stay together; the last rank takes the remainder
    return [rs.subset(np.arange(bounds[r], bounds[r + 1])) for r in range(world)], bounds


class Rank:
    """What a rank's body calls.  Every call is collective: each rank's body must make the same calls in the same order."""

    def __init__(self, lb, r, world, comm, reads, shard):
        self.lib, self.r, self.world, self.comm, self.h, self.shard = lb, r, world, comm, reads, shard
        self.err = C.create_string_buffer(1024)
        self.counts = []

    def check(self, rc):
        if rc != 0:
            raise RuntimeError("rank %d failed (%d): %s" % (self.r, rc, self.err.value.decode(errors="replace")))

    def params(self, **kw):
        return T.default_params(device=self.r, **kw)

    def count(self, **kw):
        ch, g = C.c_void_p(), T.Graph()
        self.check(self.lib.w2rap_step2_count_sharded(self.h, C.byref(self.params(**kw)), self.comm, C.byref(ch), C.byref(g), self.err, 1024))
        self.counts.append(ch)
        d = T.graph_to_dict(g)
        self.lib.w2rap_step2_free(C.byref(g))
        return ch, d

    def build(self, ch, **kw):
        g = T.Graph()
        self.check(self.lib.w2rap_step2_build_sharded(self.h, ch, C.byref(self.params(**kw)), self.comm, C.byref(g), self.err, 1024))
        d = T.graph_to_dict(g)
        self.lib.w2rap_step2_free(C.byref(g))
        return d

    def run(self, **kw):
        g = T.Graph()
        reads = self.shard.c()
        self.check(self.lib.w2rap_step2_run_sharded(C.byref(reads), C.byref(self.params(**kw)), self.comm, C.byref(g), self.err, 1024))
        d = T.graph_to_dict(g)
        self.lib.w2rap_step2_free(C.byref(g))
        return d

    def coverage(self, ch, ss, n):
        """ss: the set on rank 0 (ignored elsewhere); n: its size, known to every rank for the output array."""
        sv = ss.c() if self.r == 0 else None
        out = np.zeros(max(1, n), COV_DTYPE)
        ms = C.c_float(-1)
        self.check(self.lib.w2rap_counts_coverage_sharded(ch, self.comm, C.byref(sv) if sv is not None else None, out.ctypes.data, C.byref(ms),
                                                          self.err, 1024))
        return out[:n], ms.value


def run_ranks(rs, world, body, timeout=400):
    """body(rank) on `world` ranks, each with a communicator, its device and its shard uploaded; returns the bodies' results."""
    lb = lib()
    if lb.w2rap_step2_device_count() < world:
        pytest.skip("needs %d B200s" % world)
    err0 = C.create_string_buffer(512)
    uid = (C.c_uint8 * 128)()
    assert lb.w2rap_step2_comm_unique_id(uid, err0, 512) == 0, err0.value
    shards, bounds = shards_of(rs, world)
    results, errors = [None] * world, [None] * world

    def worker(r):
        comm, reads = C.c_void_p(), C.c_void_p()
        err = C.create_string_buffer(512)
        if lb.w2rap_step2_comm_init(uid, world, r, r, C.byref(comm), err, 512):
            errors[r] = err.value
            return
        rk = None
        try:
            if lb.w2rap_step2_upload(C.byref(shards[r].c()), r, C.byref(reads), err, 512):
                errors[r] = err.value
                return
            rk = Rank(lb, r, world, comm, reads, shards[r])
            results[r] = body(rk)
        except Exception as e:      # noqa: BLE001 — reported to the main thread
            errors[r] = repr(e)
        finally:
            if rk is not None:
                for ch in rk.counts:
                    lb.w2rap_step2_counts_release(ch)
            if reads.value:
                lb.w2rap_step2_release(reads)
            lb.w2rap_step2_comm_destroy(comm)

    th = [threading.Thread(target=worker, args=(r,), daemon=True) for r in range(world)]      # daemon: a hung rank must not block exit
    [t.start() for t in th]
    deadline = time.time() + timeout
    [t.join(max(0.0, deadline - time.time())) for t in th]
    assert not any(t.is_alive() for t in th), "ranks did not finish within %d s (alive: %s; errors so far: %s)" % (timeout, [t.is_alive() for t in th], errors)
    assert all(e is None for e in errors), errors
    return results, bounds


def single_gpu(rs, f0, body):
    """body(lib, reads handle, counts handle, err) against a single-GPU count of the whole read set on device 0."""
    lb, err = lib(), C.create_string_buffer(1024)
    h, ch, g = C.c_void_p(), C.c_void_p(), T.Graph()
    assert lb.w2rap_step2_upload(C.byref(rs.c()), 0, C.byref(h), err, 1024) == 0, err.value
    try:
        assert lb.w2rap_step2_count(h, C.byref(T.default_params(min_freq=f0, device=0)), C.byref(ch), C.byref(g), err, 1024) == 0, err.value
        summ = T.graph_to_dict(g)
        lb.w2rap_step2_free(C.byref(g))
        return summ, body(lb, h, ch, err)
    finally:
        if ch.value:
            lb.w2rap_step2_counts_release(ch)
        lb.w2rap_step2_release(h)


def single_coverage(lb, ch, ss, err):
    sv = ss.c()
    out = np.zeros(max(1, int(sv.n)), COV_DTYPE)
    assert lb.w2rap_counts_coverage(ch, C.byref(sv), out.ctypes.data, None, err, 1024) == 0, err.value
    return out[:int(sv.n)]


def assert_equal_but_timings(want, got, what):
    for k, v in want.items():
        if k == "timings":
            continue
        if isinstance(v, np.ndarray):
            assert v.dtype == got[k].dtype and np.array_equal(v, got[k]), "%s: array %s differs" % (what, k)
        else:
            assert v == got[k], "%s: %s differs: %s vs %s" % (what, k, v, got[k])


def assert_graph_and_shard_paths(want, got, bounds, r, what):
    """The graph as the oracle's (every rank), and the paths of rank r's shard."""
    T.assert_graph_equal(want, dict(got, n_reads=want["n_reads"], n_bases=want["n_bases"]), what, check_paths=False)
    lo, hi = bounds[r], bounds[r + 1]
    assert got["n_paths"] == hi - lo, what
    assert np.array_equal(got["path_offset"], want["path_offset"][lo:hi]), what
    a, b = int(want["path_off"][lo]), int(want["path_off"][hi])
    assert np.array_equal(got["path_edges"], want["path_edges"][a:b]), what
    assert np.array_equal(got["path_off"], want["path_off"][lo:hi + 1] - want["path_off"][lo]), what


SUMMARY_KEYS = ("n_kmer_instances", "n_distinct", "n_solid")


def freqs_text(hist):
    """small_K.freqs of a histogram, as w2rap_write_freqs writes it."""
    return "".join("%d, %d\n" % (i, hist[i]) for i in range(1, 101))


@pytest.mark.gpu
@pytest.mark.parametrize("world", [1, 2, 4, 8])
def test_count_builds_and_coverage(tmp_path, world):
    """f0 = 3: the summary on every rank; builds at 6, 3, 4 from one count, each equal to the oracle and to a sharded run; the coverage
    of mixed sequences and of every build's edges, passed on rank 0 only."""
    rs = T.rich_set(seed=12, genome=80000, cov=50, families=5, palindromes=3, plasmid=1500)
    f0, mfs = 3, (6, 3, 4)
    counted = T.run_oracle(rs, T.default_params(min_freq=f0, dump_kmers=2, want_paths=0))
    kept = kept_dict(counted["dump"], f0)
    seqs = mixed_sequences(rs, np.random.default_rng(world)) + step_boundary_sequences(rs)
    ss = SeqSet(seqs)
    single_summ, single_cov = single_gpu(rs, f0, lambda lb, h, ch, err: single_coverage(lb, ch, ss, err))
    wd = [tmp_path / ("r%d" % r) for r in range(world)]
    [d.mkdir() for d in wd]

    def body(rk):
        ch, summ = rk.count(min_freq=f0, workdir=str(wd[rk.r]))
        res = dict(summ=summ, builds={}, runs={}, edge_cov={})
        res["cov"], res["ms"] = rk.coverage(ch, ss, len(seqs))
        for mf in mfs:
            b = rk.build(ch, min_freq=mf, dump_kmers=1, apply_fixpaths=1)
            res["builds"][mf] = b
            res["runs"][mf] = rk.run(min_freq=mf, dump_kmers=1, apply_fixpaths=1)
            res["edge_cov"][mf] = rk.coverage(ch, SeqSet(T.unpack_edges(b)), b["n_edges"])[0]
        return res

    res, bounds = run_ranks(rs, world, body)
    want_cov = expected_coverage(seqs, kept)
    assert_cov_equal(want_cov, single_cov, "single GPU")
    for r, got in enumerate(res):
        for k in SUMMARY_KEYS:
            assert got["summ"][k] == counted[k] == single_summ[k], (r, k, got["summ"][k], counted[k], single_summ[k])
        assert np.array_equal(got["summ"]["hist"], counted["hist"]) and np.array_equal(got["summ"]["hist"], single_summ["hist"]), r
        assert_cov_equal(want_cov, got["cov"], "rank %d mixed sequences" % r)
        assert got["ms"] > 0
    assert (wd[0] / "small_K.freqs").read_text() == freqs_text(counted["hist"])
    assert not any((d / "small_K.freqs").exists() for d in wd[1:])
    for mf in mfs:
        want = T.run_oracle(rs, T.default_params(min_freq=mf, dump_kmers=1, apply_fixpaths=1))
        edges = T.unpack_edges(want)
        want_edge_cov = expected_coverage(edges, kept)
        assert (want_edge_cov["n_absent"] == 0).all() and (want_edge_cov["min"] >= mf).all(), mf
        for r, got in enumerate(res):
            what = "world %d rank %d min_freq %d" % (world, r, mf)
            assert_graph_and_shard_paths(want, got["builds"][mf], bounds, r, what + ": build vs oracle")
            assert_equal_but_timings(got["runs"][mf], got["builds"][mf], what + ": build vs sharded run")
            assert got["builds"][mf]["timings"]["count_launches"] == 0, what
            assert_cov_equal(want_edge_cov, got["edge_cov"][mf], what + ": edge coverage")


@pytest.mark.gpu
@pytest.mark.parametrize("world", [1, 2])
def test_keep_floor_one_and_the_spectrum_file(tmp_path, world):
    """f0 = 1 on 1 and 2 GPUs: the summary equals the oracle's and a single-GPU count's, rank 0's small_K.freqs the oracle's, and a build at 1."""
    rs = T.rich_set(seed=2, genome=60000, cov=50, pq_mode=1)
    counted = T.run_oracle(rs, T.default_params(min_freq=1, dump_kmers=2, want_paths=0))
    single_summ, _ = single_gpu(rs, 1, lambda *a: None)
    wd = tmp_path / "count"
    wd.mkdir()

    def body(rk):
        ch, summ = rk.count(min_freq=1, workdir=str(wd) if rk.r == 0 else None)
        return summ, rk.build(ch, min_freq=1, dump_kmers=1, apply_fixpaths=1)

    res, bounds = run_ranks(rs, world, body)
    want = T.run_oracle(rs, T.default_params(min_freq=1, dump_kmers=1, apply_fixpaths=1))
    for r, (summ, b) in enumerate(res):
        for k in SUMMARY_KEYS:
            assert summ[k] == counted[k] == single_summ[k], (r, k)
        assert np.array_equal(summ["hist"], counted["hist"]), r
        assert_graph_and_shard_paths(want, b, bounds, r, "f0=1 rank %d" % r)
    assert (wd / "small_K.freqs").read_text() == freqs_text(counted["hist"])


@pytest.mark.gpu
@pytest.mark.parametrize("world", [1, 2])
def test_build_options_and_count_paths(world):
    """On 1 and 2 GPUs: graph_on_root_only and places_K2 builds equal sharded runs (and the root-only edges' coverage from rank 0);
    counts through forced hash-range passes and through the small L2 region build the oracle's graph."""
    rs = T.rich_set(seed=17, genome=60000, cov=50, families=4, palindromes=2, plasmid=1200)
    kept = kept_dict(T.run_oracle(rs, T.default_params(min_freq=3, dump_kmers=2, want_paths=0))["dump"], 3)

    def body(rk):
        ch, _ = rk.count(min_freq=3)
        out = {}
        for name, kw in (("root_only", dict(min_freq=4, apply_fixpaths=1, graph_on_root_only=1)), ("places", dict(min_freq=4, apply_fixpaths=1, places_K2=200))):
            out[name] = (rk.build(ch, **kw), rk.run(**kw))
        b = out["root_only"][0]
        edges = SeqSet(T.unpack_edges(b) if rk.r == 0 else [])
        out["root_only_cov"] = rk.coverage(ch, edges, b["n_edges"])[0]
        for name, kw in (("passes", dict(force_passes=3)), ("region", dict(table_slots=256))):
            ch2, summ = rk.count(min_freq=3, **kw)
            out[name] = (summ, rk.build(ch2, min_freq=4, dump_kmers=1, apply_fixpaths=1))
        return out

    res, bounds = run_ranks(rs, world, body)
    want = T.run_oracle(rs, T.default_params(min_freq=4, dump_kmers=1, apply_fixpaths=1))
    want_cov = expected_coverage(T.unpack_edges(want), kept)
    places = T.run_oracle(rs, T.default_params(min_freq=4, apply_fixpaths=1, places_K2=200))
    assert places["n_places"] > 0
    for r, got in enumerate(res):
        for name in ("root_only", "places"):
            assert_equal_but_timings(got[name][1], got[name][0], "rank %d %s: build vs sharded run" % (r, name))
        assert_cov_equal(want_cov, got["root_only_cov"], "rank %d root-only edges" % r)
        assert got["places"][0]["n_places"] == places["n_places"] and np.array_equal(got["places"][0]["place_edges"], places["place_edges"]), r
        assert got["passes"][0]["timings"]["count_passes"] >= 3 and got["region"][0]["timings"]["count_passes"] > 1, (r, got["passes"][0]["timings"]["count_passes"], got["region"][0]["timings"]["count_passes"])
        for name in ("passes", "region"):
            assert_graph_and_shard_paths(want, got[name][1], bounds, r, "rank %d %s count" % (r, name))
    T.assert_graph_equal(want, dict(res[0]["root_only"][0], n_reads=want["n_reads"], n_bases=want["n_bases"]), "root-only graph", check_paths=False, check_dump=False)
    assert all(got["root_only"][0]["edge_bases"].size == 0 for got in res[1:])


@pytest.mark.gpu
@pytest.mark.parametrize("world", [1, 2])
def test_refusals_leave_the_counts_usable(world):
    """Every refusal given identically to every rank, each made before any collective; then a build equals the oracle.  A set that rank
    0 refuses makes every rank return BAD_ARG."""
    rs = T.rich_set(seed=8, genome=30000, cov=40, families=3, palindromes=2, plasmid=1000)
    lb = lib()
    other_uid = (C.c_uint8 * 128)()
    err0 = C.create_string_buffer(512)
    if lb.w2rap_step2_device_count() >= world:
        assert lb.w2rap_step2_comm_unique_id(other_uid, err0, 512) == 0, err0.value
    shards, _ = shards_of(rs, world)
    bad_set = SeqSet([np.zeros(100, np.uint8), np.ones(70, np.uint8)])
    bad_set.base_off[1] = 24                                 # 100 bases need 25 bytes

    def refused(rk, call, word):
        rc = call()
        assert rc == BAD_ARG and word in rk.err.value.decode(), (rk.r, rc, rk.err.value)

    def body(rk):
        ch, _ = rk.count(min_freq=3)
        g, p = T.Graph(), rk.params
        other = C.c_void_p()                                 # the same shard uploaded again: another handle
        rk.check(rk.lib.w2rap_step2_upload(C.byref(rk.shard.c()), rk.r, C.byref(other), rk.err, 1024))
        comm2 = C.c_void_p()                                 # a second communicator over the same ranks
        rk.check(rk.lib.w2rap_step2_comm_init(other_uid, world, rk.r, rk.r, C.byref(comm2), rk.err, 1024))
        single = C.c_void_p()                                # a single-GPU count of this rank's shard
        rk.check(rk.lib.w2rap_step2_count(rk.h, C.byref(p(min_freq=3)), C.byref(single), None, rk.err, 1024))
        try:
            L = rk.lib
            for kw, word in ((dict(min_freq=2), "keep floor"), (dict(min_qual=8), "min_qual"), (dict(dump_kmers=2), "dump_kmers 2")):
                refused(rk, lambda: L.w2rap_step2_build_sharded(rk.h, ch, C.byref(p(**kw)), rk.comm, C.byref(g), rk.err, 1024), word)
            refused(rk, lambda: L.w2rap_step2_build_sharded(other, ch, C.byref(p(min_freq=4)), rk.comm, C.byref(g), rk.err, 1024), "reads handle")
            refused(rk, lambda: L.w2rap_step2_build_sharded(rk.h, ch, C.byref(p(min_freq=4)), comm2, C.byref(g), rk.err, 1024), "another communicator")
            refused(rk, lambda: L.w2rap_step2_build_sharded(rk.h, single, C.byref(p(min_freq=4)), rk.comm, C.byref(g), rk.err, 1024), "one GPU")
            refused(rk, lambda: L.w2rap_counts_coverage_sharded(single, rk.comm, C.byref(bad_set.c()), None, None, rk.err, 1024), "one GPU")
            refused(rk, lambda: L.w2rap_counts_coverage_sharded(ch, comm2, C.byref(bad_set.c()), None, None, rk.err, 1024), "another communicator")
            refused(rk, lambda: L.w2rap_step2_build(rk.h, ch, C.byref(p(min_freq=4)), C.byref(g), rk.err, 1024), "sharded")
            out = np.zeros(2, COV_DTYPE)
            refused(rk, lambda: L.w2rap_counts_coverage(ch, C.byref(SeqSet([np.zeros(70, np.uint8)]).c()), out.ctypes.data, None, rk.err, 1024), "sharded")
            ch_bad = C.c_void_p()
            refused(rk, lambda: L.w2rap_step2_count_sharded(rk.h, C.byref(p(min_freq=3, dump_kmers=2)), rk.comm, C.byref(ch_bad), None, rk.err, 1024), "dump_kmers")
            # rank 0 refuses its set (its offsets are too short); the other ranks pass nothing and learn it from the broadcast
            rc = L.w2rap_counts_coverage_sharded(ch, rk.comm, C.byref(bad_set.c()) if rk.r == 0 else None, out.ctypes.data, None, rk.err, 1024)
            assert rc == BAD_ARG and (b"sequence 0" if rk.r == 0 else b"rank 0") in rk.err.value, (rk.r, rc, rk.err.value)
            return rk.build(ch, min_freq=4, dump_kmers=1, apply_fixpaths=1)
        finally:
            rk.lib.w2rap_step2_counts_release(single)
            rk.lib.w2rap_step2_comm_destroy(comm2)
            rk.lib.w2rap_step2_release(other)

    res, bounds = run_ranks(rs, world, body)
    want = T.run_oracle(rs, T.default_params(min_freq=4, dump_kmers=1, apply_fixpaths=1))
    for r, got in enumerate(res):
        assert_graph_and_shard_paths(want, got, bounds, r, "rank %d after refusals" % r)


@pytest.mark.gpu
@pytest.mark.parametrize("world", [1, 2])
def test_config1_scale(world):
    """Config 1 (4.6 Mbp, 100x) on 1 and 2 GPUs, each rank synthesising its share: a build at 4 from a count at 3 has the digests of the
    sharded run and of the single-GPU run."""
    lb, err = lib(), C.create_string_buffer(1024)
    n_reads = 1_840_000
    if lb.w2rap_step2_device_count() < world:
        pytest.skip("needs %d B200s" % world)
    h, g = C.c_void_p(), T.Graph()
    assert lb.w2rap_step2_synth(C.byref(T.SynthParams(4_600_000, 250, 100, 11, 0, 0, 0, 0)), 0, C.byref(h), err, 1024) == 0, err.value
    try:
        assert lb.w2rap_step2_run_resident(h, C.byref(T.default_params(min_freq=4, device=0)), C.byref(g), err, 1024) == 0, err.value
        single = T.graph_to_dict(g)
        lb.w2rap_step2_free(C.byref(g))
    finally:
        lb.w2rap_step2_release(h)
    uid = (C.c_uint8 * 128)()
    assert lb.w2rap_step2_comm_unique_id(uid, err, 1024) == 0, err.value
    results, errors = [None] * world, [None] * world

    def worker(r):
        e = C.create_string_buffer(1024)
        comm, reads, ch = C.c_void_p(), C.c_void_p(), C.c_void_p()
        try:
            if lb.w2rap_step2_comm_init(uid, world, r, r, C.byref(comm), e, 1024):
                raise RuntimeError(e.value)
            part = n_reads // world
            if lb.w2rap_step2_synth(C.byref(T.SynthParams(4_600_000, 250, 100, 11, 0, 0, part, r * part)), r, C.byref(reads), e, 1024):
                raise RuntimeError(e.value)
            out = {}
            for name, call in (("run", lambda gg: lb.w2rap_step2_run_sharded_resident(reads, C.byref(T.default_params(min_freq=4, device=r)), comm, C.byref(gg), e, 1024)),
                               ("count", lambda gg: lb.w2rap_step2_count_sharded(reads, C.byref(T.default_params(min_freq=3, device=r)), comm, C.byref(ch), C.byref(gg), e, 1024)),
                               ("build", lambda gg: lb.w2rap_step2_build_sharded(reads, ch, C.byref(T.default_params(min_freq=4, device=r)), comm, C.byref(gg), e, 1024))):
                gg = T.Graph()
                if call(gg):
                    raise RuntimeError(e.value)
                out[name] = T.graph_to_dict(gg)
                lb.w2rap_step2_free(C.byref(gg))
            results[r] = out
        except Exception as x:      # noqa: BLE001 — reported to the main thread
            errors[r] = repr(x)
        finally:
            if ch.value:
                lb.w2rap_step2_counts_release(ch)
            if reads.value:
                lb.w2rap_step2_release(reads)
            if comm.value:
                lb.w2rap_step2_comm_destroy(comm)

    th = [threading.Thread(target=worker, args=(r,), daemon=True) for r in range(world)]
    [t.start() for t in th]
    deadline = time.time() + 400
    [t.join(max(0.0, deadline - time.time())) for t in th]
    assert not any(t.is_alive() for t in th), "ranks did not finish within 400 s (errors so far: %s)" % errors
    assert all(x is None for x in errors), errors
    for r, out in enumerate(results):
        assert out["count"]["n_solid"] > out["build"]["n_solid"] > 0, r
        for k in ("digest_graph", "n_solid", "n_edges"):
            assert out["build"][k] == out["run"][k] == single[k], (r, k)
        assert out["build"]["digest_paths"] == out["run"]["digest_paths"], r
        assert_equal_but_timings(out["run"], out["build"], "config 1 rank %d" % r)
    assert sum(out["build"]["n_pathed"] for out in results) == single["n_pathed"]
