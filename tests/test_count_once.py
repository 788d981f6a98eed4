"""Count once, build the step-2 graph for several min_freq: w2rap_step2_count + w2rap_step2_build (include/w2rap_step2_counts.h).

A count keeps every distinct k-mer seen >= f0 times with its count; a build selects those seen >= min_freq times and runs the rest
of step 2.  Every build is compared with the oracle and with w2rap_step2_run_resident at the same min_freq: every array, and both
digests.  The count's summary is compared with the oracle's counters, histogram and level-2 dump at min_freq = f0.
"""
import ctypes as C
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

import w2r_testlib as T

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HERE = os.path.dirname(os.path.abspath(__file__))
GOLD = os.path.join(HERE, "golden")
BAD_ARG = 1
MAP = 1                   # W2RAP_KT_MAP
ORACLE_IGNORES = ("table_slots", "force_passes", "device")


def declared_symbols():
    txt = open(os.path.join(ROOT, "include", "w2rap_step2_counts.h")).read()
    txt = re.sub(r"/\*.*?\*/", "", txt, flags=re.S)
    return sorted(set(re.findall(r"\b(w2rap_[a-z0-9_]+)\s*\(", txt)) - set(T.ABI_SYMBOLS))


def lib():
    lb = T.product_lib()
    E = [C.c_char_p, C.c_size_t]
    lb.w2rap_step2_count.argtypes = [C.c_void_p, C.POINTER(T.Params), C.POINTER(C.c_void_p), C.POINTER(T.Graph)] + E
    lb.w2rap_step2_count.restype = C.c_int
    lb.w2rap_step2_build.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(T.Params), C.POINTER(T.Graph)] + E
    lb.w2rap_step2_build.restype = C.c_int
    lb.w2rap_step2_counts_release.argtypes = [C.c_void_p]
    lb.w2rap_step2_counts_release.restype = None
    return lb


class Session:
    """One uploaded read set; count(), build() and run() return w2rap_graph dicts (or raise with the library's message)."""

    def __init__(self, rs):
        self.lib, self.err = lib(), C.create_string_buffer(1024)
        self.h = C.c_void_p()
        self.check(self.lib.w2rap_step2_upload(C.byref(rs.c()), -1, C.byref(self.h), self.err, 1024))
        self.counts = []

    def check(self, rc):
        if rc != 0:
            raise RuntimeError("failed (%d): %s" % (rc, self.err.value.decode(errors="replace")))

    def count(self, **kw):
        ch, g = C.c_void_p(), T.Graph()
        self.check(self.lib.w2rap_step2_count(self.h, C.byref(T.default_params(**kw)), C.byref(ch), C.byref(g), self.err, 1024))
        self.counts.append(ch)
        d = T.graph_to_dict(g)
        self.lib.w2rap_step2_free(C.byref(g))
        return ch, d

    def build(self, ch, reads=None, **kw):
        g = T.Graph()
        self.check(self.lib.w2rap_step2_build(reads if reads is not None else self.h, ch, C.byref(T.default_params(**kw)), C.byref(g), self.err, 1024))
        d = T.graph_to_dict(g)
        self.lib.w2rap_step2_free(C.byref(g))
        return d

    def run(self, **kw):
        g = T.Graph()
        self.check(self.lib.w2rap_step2_run_resident(self.h, C.byref(T.default_params(**kw)), C.byref(g), self.err, 1024))
        d = T.graph_to_dict(g)
        self.lib.w2rap_step2_free(C.byref(g))
        return d

    def close(self):
        for ch in self.counts:
            self.lib.w2rap_step2_counts_release(ch)
        self.lib.w2rap_step2_release(self.h)


def assert_build_matches(s, rs, ch, what, oracle=True, **kw):
    """The build equals run_resident at the same parameters (every array, digests) and, if asked, the oracle."""
    got = s.build(ch, **{k: v for k, v in kw.items() if k not in ("table_slots", "force_passes")})
    run = s.run(**kw)
    T.assert_graph_equal(run, got, what + ": build vs run_resident")
    assert (got["digest_graph"], got["digest_paths"]) == (run["digest_graph"], run["digest_paths"]), what
    assert got["timings"]["kernel_ms"][MAP] == 0 and got["timings"]["count_launches"] == 0, what
    if oracle:
        want = T.run_oracle(rs, T.default_params(**{k: v for k, v in kw.items() if k not in ORACLE_IGNORES}))
        T.assert_graph_equal(want, got, what + ": build vs oracle")
    return got


# ---------------------------------------------------------------- CPU: interface

def test_every_declared_symbol_is_exported():
    names = declared_symbols()
    assert names == ["w2rap_step2_build", "w2rap_step2_count", "w2rap_step2_counts_release"]
    lb = lib()
    for n in names:
        assert hasattr(lb, n), "missing export " + n


def test_null_arguments_and_count_parameters_are_refused_before_device_work():
    lb, err = lib(), C.create_string_buffer(512)
    fake = C.c_void_p(16)          # never dereferenced: every call below is refused before the handles are used
    p, g, ch = T.default_params(), T.Graph(), C.c_void_p()
    assert lb.w2rap_step2_count(None, C.byref(p), C.byref(ch), None, err, 512) == BAD_ARG
    assert lb.w2rap_step2_count(fake, None, C.byref(ch), None, err, 512) == BAD_ARG
    assert lb.w2rap_step2_count(fake, C.byref(p), None, None, err, 512) == BAD_ARG
    assert lb.w2rap_step2_build(None, fake, C.byref(p), C.byref(g), err, 512) == BAD_ARG
    assert lb.w2rap_step2_build(fake, None, C.byref(p), C.byref(g), err, 512) == BAD_ARG
    assert lb.w2rap_step2_build(fake, fake, None, C.byref(g), err, 512) == BAD_ARG
    assert lb.w2rap_step2_build(fake, fake, C.byref(p), None, err, 512) == BAD_ARG
    for bad, word in ((dict(dump_kmers=1), b"dump_kmers"), (dict(min_freq=0), b"min_freq"), (dict(min_freq=256), b"min_freq")):
        ch = C.c_void_p()
        assert lb.w2rap_step2_count(fake, C.byref(T.default_params(**bad)), C.byref(ch), None, err, 512) == BAD_ARG
        assert word in err.value and not ch.value
    lb.w2rap_step2_counts_release(None)


# ---------------------------------------------------------------- GPU

@pytest.mark.gpu
@pytest.mark.parametrize("f0", [1, 2])
def test_spectrum_equals_the_oracle_and_a_run(tmp_path, f0):
    rs = T.rich_set(seed=2, genome=60000, cov=50, pq_mode=1)
    s = Session(rs)
    try:
        wc, wr = tmp_path / "count", tmp_path / "run"
        wc.mkdir(); wr.mkdir()
        _, summ = s.count(min_freq=f0, dump_kmers=2, workdir=str(wc))
        want = T.run_oracle(rs, T.default_params(min_freq=f0, dump_kmers=2, want_paths=0))
        for k in ("n_reads", "n_bases", "n_kmer_instances", "n_distinct", "n_solid"):
            assert summ[k] == want[k], (k, summ[k], want[k])
        assert np.array_equal(summ["hist"], want["hist"])
        assert len(summ["dump"]) == want["n_distinct"]
        for f in ("w0", "w1", "count", "ctx", "edge", "offset"):
            assert np.array_equal(summ["dump"][f], want["dump"][f]), f
        assert summ["n_edges"] == 0 and summ["n_paths"] == 0 and summ["timings"]["count_launches"] == 1
        s.run(min_freq=f0, workdir=str(wr))
        assert (wc / "small_K.freqs").read_bytes() == (wr / "small_K.freqs").read_bytes()
    finally:
        s.close()


@pytest.mark.gpu
def test_sweep_of_builds_from_one_count():
    """f0 = 2, builds at 4, 2, 3, 6 and 4 again (the handle is not consumed); f0 = 1 with a build at 1; places from a build."""
    rs = T.rich_set(seed=2, genome=100000, cov=60, pq_mode=1)
    s = Session(rs)
    try:
        ch, summ = s.count(min_freq=2)
        assert summ["n_solid"] > 0
        first = None
        for mf in (4, 2, 3, 6, 4):
            got = assert_build_matches(s, rs, ch, "f0=2 min_freq=%d" % mf, min_freq=mf, dump_kmers=1, apply_fixpaths=1)
            if mf == 4 and first is None:
                first = got
            elif mf == 4:
                T.assert_graph_equal(first, got, "second build at 4")
        ch1, _ = s.count(min_freq=1)
        assert_build_matches(s, rs, ch1, "f0=1 min_freq=1", min_freq=1, dump_kmers=1, apply_fixpaths=1)
        got = assert_build_matches(s, rs, ch, "places", min_freq=3, apply_fixpaths=1, places_K2=200)
        assert got["n_places"] > 0
    finally:
        s.close()


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["passes2", "passes3", "region", "tiny_region"])
def test_reduce_paths_keep_counts(case):
    """The count-keeping reduce through forced hash-range passes, the L2 region fallback (60000 slots) and the 64-slot region whose
    partitions are split into hash sub-ranges with roll-back; each count built at two min_freq values."""
    if case.startswith("passes"):
        rs, kw, least = T.rich_set(seed=14, genome=60000, cov=40), dict(force_passes=int(case[-1])), int(case[-1])
    elif case == "region":
        rs, kw, least = T.rich_set(seed=6, genome=50000, cov=40), dict(table_slots=60000), 4
    else:
        rs, kw, least = T.rich_set(seed=6, genome=12000, cov=30, families=2, palindromes=1, plasmid=600), dict(table_slots=64), 1001
    s = Session(rs)
    try:
        ch, summ = s.count(min_freq=2, **kw)
        assert summ["timings"]["count_passes"] >= least, summ["timings"]["count_passes"]
        for mf in (2, 5):
            assert_build_matches(s, rs, ch, "%s min_freq=%d" % (case, mf), min_freq=mf, dump_kmers=1, **kw)
    finally:
        s.close()


@pytest.mark.gpu
def test_edge_cases():
    # every read shorter than K: nothing is kept, every build is the empty graph
    rng = np.random.default_rng(4)
    codes = rng.integers(0, 4, (50, 100), dtype=np.uint8)
    short = T.flatten_reads(codes, np.full((50, 100), 30, np.uint8), rng.integers(1, 60, 50).astype(np.uint32))
    s = Session(short)
    try:
        ch, summ = s.count(min_freq=1)
        assert summ["n_kmer_instances"] == 0 and summ["n_solid"] == 0
        for mf in (1, 2):
            got = assert_build_matches(s, short, ch, "short reads min_freq=%d" % mf, min_freq=mf)
            assert got["n_edges"] == 0 and got["n_paths"] == 50 and got["n_pathed"] == 0
    finally:
        s.close()
    # min_freq 200: nothing selected, every path empty
    rs = T.rich_set(seed=7, genome=30000, cov=12, families=4, palindromes=2, plasmid=800)
    s = Session(rs)
    try:
        ch, summ = s.count(min_freq=2)
        assert summ["n_solid"] > 0
        got = assert_build_matches(s, rs, ch, "min_freq=200", min_freq=200, apply_fixpaths=1)
        assert got["n_solid"] == 0 and got["n_edges"] == 0 and got["n_pathed"] == 0 and got["n_path_edges"] == 0
    finally:
        s.close()


@pytest.mark.gpu
def test_refusals_leave_the_counts_usable():
    rs = T.rich_set(seed=8, genome=30000, cov=40, families=3, palindromes=2, plasmid=1000)
    s = Session(rs)
    other = Session(rs)          # the same reads uploaded again: a different handle
    try:
        ch, _ = s.count(min_freq=3)
        for kw, reads, word in ((dict(min_freq=2), None, "keep floor"), (dict(min_qual=8), None, "min_qual"),
                                (dict(dump_kmers=2), None, "dump_kmers 2"), (dict(), other.h, "reads handle")):
            with pytest.raises(RuntimeError, match=r"failed \(1\).*" + word):
                s.build(ch, reads=reads, **kw)
        with pytest.raises(RuntimeError, match=r"failed \(1\).*dump_kmers 1"):
            s.count(min_freq=3, dump_kmers=1)
        assert_build_matches(s, rs, ch, "after refusals", min_freq=4, dump_kmers=1, apply_fixpaths=1)
    finally:
        other.close()
        s.close()


@pytest.mark.gpu
def test_config1_scale():
    """Config 1 (4.6 Mbp, 100x, 1.84 M reads): one count at f0 = 2, builds at 3, 4 and 5 equal to run_resident, every array."""
    lb, err = lib(), C.create_string_buffer(512)
    sp = T.SynthParams(4_600_000, 250, 100, 11, 0, 0, 0, 0)
    s = Session.__new__(Session)
    s.lib, s.err, s.h, s.counts = lb, C.create_string_buffer(1024), C.c_void_p(), []
    assert lb.w2rap_step2_synth(C.byref(sp), -1, C.byref(s.h), err, 512) == 0, err.value
    try:
        ch, summ = s.count(min_freq=2)
        assert summ["n_reads"] == 1_840_000
        for mf in (3, 4, 5):
            assert_build_matches(s, None, ch, "config 1 min_freq=%d" % mf, oracle=False, min_freq=mf, dump_kmers=1, apply_fixpaths=1)
    finally:
        s.close()


@pytest.mark.gpu
def test_cli_min_freq_list(tmp_path):
    exe = os.path.join(T.PKG_DIR, "step2")
    if not os.path.exists(exe):
        pytest.skip("step2 binary not built")
    dirs = {k: tmp_path / k for k in ("sweep", "mf3", "mf4")}
    for d in dirs.values():
        d.mkdir()
        for f in ("frag_reads_orig.fastb", "frag_reads_orig.qualp"):
            shutil.copy(os.path.join(GOLD, "circ", f), d)
    for k, arg in (("sweep", "3,4"), ("mf3", "3"), ("mf4", "4")):
        r = subprocess.run([exe, str(dirs[k]), "x", "--min_freq", arg, "--quiet"], capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stdout + r.stderr
    for mf in (3, 4):
        for ext in ("hbv", "paths"):
            a = (dirs["sweep"] / ("x_mf%d.small_K.%s" % (mf, ext))).read_bytes()
            b = (dirs["mf%d" % mf] / ("x.small_K.%s" % ext)).read_bytes()
            assert a == b, (mf, ext)
    assert not (dirs["sweep"] / "x.small_K.hbv").exists()
    freqs = (dirs["sweep"] / "small_K.freqs").read_bytes()
    assert freqs == (dirs["mf3"] / "small_K.freqs").read_bytes() == (dirs["mf4"] / "small_K.freqs").read_bytes()
