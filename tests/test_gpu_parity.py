"""Parity of the CUDA path (through the C ABI, host buffers) with the oracle — bit-exact, every stage.

Both sides emit canonical edges sorted by sequence, so every array must be identical: counters, histogram, the distinct
k-mer set with counts and contexts (dump level 2), the solid dictionary with pruned contexts and (edge, offset) (level 1),
edge sequences, vertex ids, hbv ids and every read path.
"""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def both(T, rs, **kw):
    got = T.run_product(rs, T.default_params(**kw))
    want = T.run_oracle(rs, T.default_params(**{k: v for k, v in kw.items() if k not in ("table_slots", "device", "force_passes")}))
    return want, got


def test_smoke_set(T):
    want, got = both(T, T.smoke_set(seed=1, genome=20000, cov=40), dump_kmers=1)
    T.assert_graph_equal(want, got)
    assert got["timings"]["kernel_launches"] > 20


def test_distinct_kmers_counts_contexts(T):
    rs = T.rich_set(seed=2, genome=60000, cov=50, pq_mode=1)
    want, got = both(T, rs, dump_kmers=2, want_paths=0)
    T.assert_graph_equal(want, got, check_paths=False)
    assert len(got["dump"]) == got["n_distinct"] and got["dump"]["count"].max() <= 255


def test_rich_set_all_stages(T):
    rs = T.rich_set(seed=2, genome=100000, cov=60, pq_mode=1)
    want, got = both(T, rs, dump_kmers=1)
    T.assert_graph_equal(want, got)
    assert got["n_edges"] > 1000 and got["n_multipathed"] > 1000


def test_varlen_reads_fixpaths(T):
    rs = T.rich_set(seed=5, genome=40000, cov=50, families=5, palindromes=4, plasmid=1500, vary_len=True)
    want, got = both(T, rs, dump_kmers=1, apply_fixpaths=1)
    T.assert_graph_equal(want, got)


def test_long_reads_span_several_map_tiles(T):
    """600-base reads: the map kernel handles a read in tiles of 192 k-mers, the path kernel screens gaps 32 positions at a time."""
    rs = T.rich_set(seed=9, genome=50000, cov=40, read_len=600, families=3, palindromes=2, plasmid=2000, vary_len=True)
    want, got = both(T, rs, dump_kmers=2, apply_fixpaths=1)
    T.assert_graph_equal(want, got)
    assert int(rs.len.max()) > 500 and got["n_pathed"] > 0


@pytest.mark.parametrize("fine_recs", ["300000", "4000000"])
def test_partitions_that_do_not_fit_shared_memory(fine_recs):
    """Oversized partitions: every partition fails the shared-memory count and goes through the L2 region in bulk groups
    (300 k records each), and one partition larger than the region itself is split into hash sub-ranges (4 M)."""
    here = os.path.dirname(os.path.abspath(__file__))
    env = dict(os.environ, W2RAP_FINE_RECS=fine_recs, PYTHONPATH=here)
    r = subprocess.run([sys.executable, os.path.join(here, "env_case_runner.py"), "100000", "60", "21"], env=env, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "OK" in r.stdout, (r.stdout[-2000:], r.stderr[-2000:])
    passes = int(r.stdout.split("passes=")[1].split()[0])
    assert passes >= 2, "the fallback path did not run"


def test_vertex_sort_long_path():
    """HBV vertices: the product sorts the edge ends by their 64-bit hash word and proves the order by a neighbour check; the
    23-pass sort over hash + bases only runs after a hash collision.  W2RAP_HBV_FULL_SORT forces it: same graph."""
    here = os.path.dirname(os.path.abspath(__file__))
    env = dict(os.environ, W2RAP_HBV_FULL_SORT="1", PYTHONPATH=here)
    r = subprocess.run([sys.executable, os.path.join(here, "env_case_runner.py"), "100000", "60", "22"], env=env, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "OK" in r.stdout, (r.stdout[-2000:], r.stderr[-2000:])


@pytest.mark.parametrize("case", ["circ", "rich", "long"])
def test_golden_reference_outputs(T, case):
    """Straight against the files the UNMODIFIED reference wrote (tests/golden): modulo its racy edge numbering."""
    d = os.path.join(GOLD, case)
    rs = T.read_fastb_qualp(d)
    got = T.run_product(rs, T.default_params(apply_fixpaths=1))
    rep = T.compare_with_reference(got, T.graph_from_reference_files(d))
    assert rep["edge_set_equal"] and rep["hist_equal"] and rep["vertices_equal"], rep
    assert rep["path_mismatches"] == [] and rep["path_ties"] <= 3, rep


@pytest.mark.parametrize("npass", [2, 3])
def test_forced_hash_range_passes(T, npass):
    """The replacement of the reference's disk batches (BuildReadQGraph.cc:1120-1250): when the records of the whole job do not fit
    in device memory the k-mer space is counted in hash-range passes.  Forced here: every pass filter, the cross-pass accumulation
    of solid records and the histogram must give the single-pass answer, k-mer for k-mer."""
    rs = T.rich_set(seed=14, genome=60000, cov=40)
    want, got = both(T, rs, dump_kmers=2, force_passes=npass)
    T.assert_graph_equal(want, got)
    assert got["timings"]["count_passes"] >= npass


def test_small_counting_region_many_groups(T):
    """Forced small counting tables: every partition fails the shared-memory count and goes through a small L2 region in groups."""
    rs = T.rich_set(seed=6, genome=50000, cov=40)
    want, got = both(T, rs, dump_kmers=2, table_slots=60000)
    assert got["timings"]["count_passes"] > 3
    T.assert_graph_equal(want, got)


def test_tiny_counting_region_overflow_paths(T):
    """A 4-slot shared-memory table and a 64-slot region: every partition exceeds both, so the per-partition retry and the hash
    sub-range split (with roll-back of partial output) are exercised."""
    rs = T.rich_set(seed=6, genome=12000, cov=30, families=2, palindromes=1, plasmid=600)
    want, got = both(T, rs, dump_kmers=2, table_slots=64)
    assert got["timings"]["count_passes"] > 1000
    T.assert_graph_equal(want, got)


def test_parameters(T):
    rs = T.rich_set(seed=7, genome=30000, cov=12, families=4, palindromes=2, plasmid=800)
    for mq, mf in ((7, 3), (10, 2), (20, 1), (0, 8)):
        want, got = both(T, rs, dump_kmers=1, min_qual=mq, min_freq=mf)
        T.assert_graph_equal(want, got, "min_qual=%d min_freq=%d" % (mq, mf))


def test_edge_cases(T):
    rng = np.random.default_rng(9)
    empty = T.ReadSet(np.zeros(0, np.uint8), np.zeros(1, np.uint64), np.zeros(0, np.uint32), np.zeros(0, np.uint8), np.zeros(1, np.uint64))
    got = T.run_product(empty)
    assert got["n_edges"] == 0 and got["n_paths"] == 0 and got["n_vertices"] == 0
    g = rng.integers(0, 4, 400, dtype=np.uint8)
    codes = np.zeros((40, 250), np.uint8)
    quals = np.full((40, 250), 30, np.uint8)
    lens = np.full(40, 250, np.uint32)
    for i in range(40):
        codes[i] = g[i:i + 250]
    lens[0], lens[1] = 10, 59
    quals[2, :] = 2
    quals[3, 60:] = 2
    quals[4, 61:] = 2
    rs = T.flatten_reads(codes, quals, lens)
    want, got = both(T, rs, dump_kmers=1, min_freq=1)
    T.assert_graph_equal(want, got)
    # nothing solid at all: no edges, every path empty
    want, got = both(T, rs, min_freq=200)
    T.assert_graph_equal(want, got)
    assert got["n_solid"] == 0 and got["n_pathed"] == 0


def test_corrupt_quality_stream_is_rejected(T):
    """A PQVec block whose payload would run past its stream (truncated / corrupted .qualp) is a clean W2RAP_ERR_BAD_ARG, not
    an out-of-bounds walk on the device (the decoders are bounded by qual_off[i+1])."""
    rs = T.smoke_set(seed=3, genome=3000, cov=10)
    o = int(rs.qual_off[rs.n - 1])
    rs.quals[o] = 255                    # the last read's first block claims 255 qualities ...
    rs.quals[o + 1] |= 7                 # ... of 7 bits each: 225 bytes of payload in a ~100-byte stream
    with pytest.raises(RuntimeError, match=r"failed \(1\)"):
        T.run_product(rs)
    got = T.run_product(T.smoke_set(seed=3, genome=3000, cov=10))      # and the library is still usable afterwards
    assert got["n_pathed"] > 0


def test_saturating_counts(T):
    """>255 copies of the same read: counts saturate at 255, histogram bin 100 collects them."""
    rng = np.random.default_rng(10)
    g = rng.integers(0, 4, 300, dtype=np.uint8)
    codes = np.tile(g[:250], (400, 1))
    rs = T.flatten_reads(codes, np.full((400, 250), 35, np.uint8), np.full(400, 250, np.uint32))
    want, got = both(T, rs, dump_kmers=2)
    T.assert_graph_equal(want, got)
    assert got["dump"]["count"].max() == 255 and got["hist"][100] == got["n_distinct"]


def test_resident_and_file_level_entry_points(T, tmp_path):
    lib = T.product_lib()
    rs = T.rich_set(seed=8, genome=30000, cov=40, families=3, palindromes=2, plasmid=1000)
    want = T.run_oracle(rs, T.default_params(apply_fixpaths=1))
    # device-resident variant
    h = C.c_void_p()
    err = C.create_string_buffer(512)
    reads = rs.c()
    assert lib.w2rap_step2_upload(C.byref(reads), -1, C.byref(h), err, 512) == 0, err.value
    p = T.default_params(apply_fixpaths=1)
    for _ in range(2):
        g = T.Graph()
        assert lib.w2rap_step2_run_resident(h, C.byref(p), C.byref(g), err, 512) == 0, err.value
        got = T.graph_to_dict(g)
        lib.w2rap_step2_free(C.byref(g))
        T.assert_graph_equal(want, got, "resident run")
    lib.w2rap_step2_release(h)
    # file-level drop-in: .fastb/.qualp in, .hbv/.paths/.freqs out
    T.write_fastb_qualp(str(tmp_path), rs)
    assert lib.w2rap_step2_run_files(str(tmp_path).encode(), b"x", C.byref(T.default_params()), None, err, 512) == 0, err.value
    ref = T.graph_from_reference_files(str(tmp_path))
    rep = T.compare_with_reference(want, ref)
    assert rep["edge_set_equal"] and rep["vertices_equal"] and rep["hist_equal"] and rep["path_mismatches"] == [] and rep["path_ties"] == 0


def test_device_synth_reads_are_valid_and_path(T):
    """The on-device generator emits valid read stores: the oracle decodes them and both sides agree on the result."""
    lib = T.product_lib()
    sp = T.SynthParams(150000, 250, 30, 42, 50, 0, 0)
    h = C.c_void_p()
    err = C.create_string_buffer(512)
    assert lib.w2rap_step2_synth(C.byref(sp), -1, C.byref(h), err, 512) == 0, err.value
    r = T.Reads()
    assert lib.w2rap_step2_download_reads(h, C.byref(r), err, 512) == 0, err.value
    n = int(r.n_reads)
    assert n == 150000 * 30 // 250
    boff, qoff = T._arr(r.base_off, n + 1, "<u8"), T._arr(r.qual_off, n + 1, "<u8")
    rs = T.ReadSet(T._arr(r.bases, int(boff[-1]), "u1"), boff, T._arr(r.len, n, "<u4"), T._arr(r.quals, int(qoff[-1]), "u1"), qoff)
    lib.w2rap_step2_free_host_reads(C.byref(r))
    want = T.run_oracle(rs)
    g = T.Graph()
    p = T.default_params()
    assert lib.w2rap_step2_run_resident(h, C.byref(p), C.byref(g), err, 512) == 0, err.value
    got = T.graph_to_dict(g)
    lib.w2rap_step2_free(C.byref(g))
    lib.w2rap_step2_release(h)
    T.assert_graph_equal(want, got, "device-generated reads")
    assert got["n_pathed"] > 0.95 * n and 0.9 * 150000 < got["n_solid"] < 2.2 * 150000


def test_size_independent_properties_at_scale(T):
    """A few million reads (too slow for the oracle): structural invariants of the result."""
    lib = T.product_lib()
    sp = T.SynthParams(4_000_000, 250, 40, 7, 0, 0, 0)
    h = C.c_void_p()
    err = C.create_string_buffer(512)
    assert lib.w2rap_step2_synth(C.byref(sp), -1, C.byref(h), err, 512) == 0, err.value
    g = T.Graph()
    p = T.default_params(apply_fixpaths=1, dump_kmers=1)
    assert lib.w2rap_step2_run_resident(h, C.byref(p), C.byref(g), err, 512) == 0, err.value
    d = T.graph_to_dict(g)
    lib.w2rap_step2_free(C.byref(g))
    lib.w2rap_step2_release(h)
    # every solid k-mer lies on exactly one edge at a valid offset, and the edge k-mer count adds up
    assert d["n_solid"] == len(d["dump"]) == int((d["edge_len"].astype(np.int64) - 59).sum())
    assert (d["dump"]["edge"] < d["n_edges"]).all()
    assert (d["dump"]["offset"] + 60 <= d["edge_len"][d["dump"]["edge"]]).all()
    assert int(d["hist"][1:].sum()) == d["n_distinct"] and int(d["hist"][4:].sum()) == d["n_solid"]
    # dump sorted strictly (no duplicate k-mers); edges sorted by sequence; vertex ids dense
    w = d["dump"]
    assert ((w["w0"][1:] > w["w0"][:-1]) | ((w["w0"][1:] == w["w0"][:-1]) & (w["w1"][1:] > w["w1"][:-1]))).all()
    assert set(np.unique(d["edge_vertices"][d["edge_vertices"] >= 0])) == set(range(d["n_vertices"]))
    # post-FixPaths paths are walks in the graph
    seqs, left, right = T.hbv_view(d)
    pe, po = d["path_edges"], d["path_off"]
    inner = np.ones(len(pe), bool)
    inner[(po[1:][po[1:] > po[:-1]] - 1).astype(np.int64)] = False
    idx = np.nonzero(inner)[0]
    assert (right[pe[idx]] == left[pe[idx + 1]]).all()
    assert d["n_pathed"] > 0.97 * d["n_reads"]


def test_reference_binary_with_dropin_translation_unit(T, tmp_path):
    """The reference's own main() with only src/paths/long/BuildReadQGraph.cc swapped for host/BuildReadQGraph_b200.cc
    (oracle/_ref/w2rap-contigger-b200, linked by `make -C oracle dropin`): --from_step 2 --to_step 2 must write the same
    step-2 files as the unmodified reference did for tests/golden (modulo its racy edge numbering).  It links the reference's own
    object files, so no stored output can stand in for it: it skips unless the reference was built from its sources (W2RAP_REFERENCE
    at build time).  The same golden files are compared with the library itself in test_golden_reference_outputs and
    test_standalone_step2_binary, which always run."""
    import shutil
    import subprocess
    exe = os.path.join(os.path.dirname(T.REF_BIN), "w2rap-contigger-b200")
    if not os.path.exists(exe):
        pytest.skip("drop-in binary not built (needs the reference's sources: W2RAP_REFERENCE=<checkout> at build time)")
    for case in ("circ", "rich"):
        d = str(tmp_path / case)
        os.makedirs(d)
        for f in ("frag_reads_orig.fastb", "frag_reads_orig.qualp"):
            shutil.copy(os.path.join(GOLD, case, f), d)
        r = subprocess.run([exe, "-t", "4", "-o", d, "-p", "x", "-r", "dummy", "--from_step", "2", "--to_step", "2"], capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
        mine = T.graph_from_reference_files(d)
        gold = T.graph_from_reference_files(os.path.join(GOLD, case))
        # compare the two file sets through the same relabelling: edges by sequence
        a = {e.tobytes(): i for i, e in enumerate(mine["hbv"]["edges"])}
        assert set(a) == {e.tobytes() for e in gold["hbv"]["edges"]}
        g2m = np.array([a[e.tobytes()] for e in gold["hbv"]["edges"]])
        assert np.array_equal(mine["left"][g2m], gold["left"]) and np.array_equal(mine["right"][g2m], gold["right"])
        assert np.array_equal(mine["hist"], gold["hist"])
        assert np.array_equal(mine["path_offset"], gold["path_offset"])
        diff = [i for i, (p, q) in enumerate(zip(mine["paths"], gold["paths"])) if not np.array_equal(p, g2m[q] if len(q) else q)]
        assert len(diff) <= 3, diff[:10]      # extension ties between parallel edges (SURVEY.md §8c)


def test_standalone_step2_binary(T, tmp_path):
    import shutil
    import subprocess
    exe = os.path.join(T.PKG_DIR, "step2")
    if not os.path.exists(exe):
        pytest.skip("step2 binary not built")
    d = str(tmp_path)
    for f in ("frag_reads_orig.fastb", "frag_reads_orig.qualp"):
        shutil.copy(os.path.join(GOLD, "circ", f), d)
    r = subprocess.run([exe, d, "x", "--quiet"], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    got = T.run_product(T.read_fastb_qualp(d), T.default_params(apply_fixpaths=1))
    rep = T.compare_with_reference(got, T.graph_from_reference_files(d))
    assert rep["edge_set_equal"] and rep["vertices_equal"] and rep["hist_equal"] and rep["path_mismatches"] == [] and rep["path_ties"] == 0


def test_config1_against_the_reference_binary(T, tmp_path):
    """BASELINE.json configs[0] at full size — E. coli-sized 4.6 Mbp genome, 2x250 PE at 100x, 1.84 M reads — through the UNMODIFIED
    reference binary (oracle/_ref/w2rap-contigger, all host threads) and through the B200 path, same reads: histogram, edge set,
    vertices and every read path must agree (modulo the reference's racy edge numbering and its extension ties).  It runs the
    reference itself and skips without it; test_config1_against_the_oracle runs the same reads against the oracle everywhere."""
    if not os.path.exists(T.REF_BIN):
        pytest.skip("oracle/_ref/w2rap-contigger not built (needs the reference's sources: W2RAP_REFERENCE=<checkout> at build time)")
    lib = T.product_lib()
    err = C.create_string_buffer(512)
    sp = T.SynthParams(4_600_000, 250, 100, 11, 0, 0, 0, 0)
    h = C.c_void_p()
    assert lib.w2rap_step2_synth(C.byref(sp), -1, C.byref(h), err, 512) == 0, err.value
    hr = T.Reads()
    assert lib.w2rap_step2_download_reads(h, C.byref(hr), err, 512) == 0, err.value
    assert int(hr.n_reads) == 1_840_000
    d = str(tmp_path)
    assert lib.w2rap_write_fastb(os.path.join(d, "frag_reads_orig.fastb").encode(), C.byref(hr), err, 512) == 0, err.value
    assert lib.w2rap_write_qualp(os.path.join(d, "frag_reads_orig.qualp").encode(), C.byref(hr), err, 512) == 0, err.value
    lib.w2rap_step2_free_host_reads(C.byref(hr))
    g = T.Graph()
    p = T.default_params(apply_fixpaths=1)
    assert lib.w2rap_step2_run_resident(h, C.byref(p), C.byref(g), err, 512) == 0, err.value
    got = T.graph_to_dict(g)
    lib.w2rap_step2_free(C.byref(g))
    lib.w2rap_step2_release(h)
    T.run_reference_step2(d, threads=os.cpu_count() or 1)
    rep = T.compare_with_reference_fast(got, T.graph_from_reference_files(d))
    assert rep["edge_set_equal"] and rep["hist_equal"] and rep["vertices_equal"], {k: v for k, v in rep.items() if k != "path_mismatches"}
    assert rep["path_mismatches"] == [] and rep["path_ties"] <= 50, (rep["path_ties"], rep["path_mismatches"][:10])
    assert got["n_pathed"] > 0.97 * got["n_reads"]


def test_config1_against_the_oracle(T):
    """BASELINE.json configs[0] at full size (the reads of test_config1_against_the_reference_binary: 4.6 Mbp, 100x, 1.84 M reads,
    seed 11) through the B200 path and through the oracle, whose restatement is pinned on the reference's own files
    (test_oracle_golden.py): every array bit for bit, at a size the other parity tests do not reach.  Runs without the reference."""
    lib = T.product_lib()
    err = C.create_string_buffer(512)
    sp = T.SynthParams(4_600_000, 250, 100, 11, 0, 0, 0, 0)
    h = C.c_void_p()
    assert lib.w2rap_step2_synth(C.byref(sp), -1, C.byref(h), err, 512) == 0, err.value
    r = T.Reads()
    assert lib.w2rap_step2_download_reads(h, C.byref(r), err, 512) == 0, err.value
    n = int(r.n_reads)
    assert n == 1_840_000
    boff, qoff = T._arr(r.base_off, n + 1, "<u8"), T._arr(r.qual_off, n + 1, "<u8")
    rs = T.ReadSet(T._arr(r.bases, int(boff[-1]), "u1"), boff, T._arr(r.len, n, "<u4"), T._arr(r.quals, int(qoff[-1]), "u1"), qoff)
    lib.w2rap_step2_free_host_reads(C.byref(r))
    g = T.Graph()
    p = T.default_params(apply_fixpaths=1, dump_kmers=1)
    assert lib.w2rap_step2_run_resident(h, C.byref(p), C.byref(g), err, 512) == 0, err.value
    got = T.graph_to_dict(g)
    lib.w2rap_step2_free(C.byref(g))
    lib.w2rap_step2_release(h)
    want = T.run_oracle(rs, T.default_params(apply_fixpaths=1, dump_kmers=1))
    T.assert_graph_equal(want, got, "config 1")
    assert got["n_pathed"] > 0.97 * got["n_reads"]


@pytest.mark.parametrize("K2", [100, 200])
def test_places_for_step3(T, K2):
    """SURVEY §8 N1: RepathInMemory's places (paths/long/large/Repath.cc:46-72) built on the device from the finished paths, against
    the oracle (whose restatement reproduces the reference's logged counts, tests/test_oracle_golden.py)."""
    rs = T.rich_set(seed=33, genome=120000, cov=60, families=6, palindromes=3, plasmid=2500)
    want = T.run_oracle(rs, T.default_params(apply_fixpaths=1, places_K2=K2))
    got = T.run_product(rs, T.default_params(apply_fixpaths=1, places_K2=K2))
    assert want["n_places"] > 500 and want["n_places_kept"] > want["n_places"] + 1000
    T.assert_graph_equal(want, got, check_dump=False)
    # sorted in std::vector<int> order and unique
    pl = [tuple(int(e) for e in got["place_edges"][int(got["place_off"][i]):int(got["place_off"][i + 1])]) for i in range(got["n_places"])]
    assert pl == sorted(set(pl))


@pytest.mark.parametrize("case", ["circ", "rich", "long"])
def test_places_counts_of_the_reference_on_golden_cases(T, case):
    """The reference prints how many paths pass the K2 test and how many unique places remain (tests/golden/<case>/
    reference_step3_places.txt, from the unmodified binary run on its own step-2 files): the product's counts on the same reads may
    differ only by the <= 3 extension ties its paths differ by."""
    d = os.path.join(GOLD, case)
    rs = T.read_fastb_qualp(d)
    for line in open(os.path.join(d, "reference_step3_places.txt")).read().splitlines():
        K2, n_paths, kept, unique = (int(x) for x in line.split())
        got = T.run_product(rs, T.default_params(apply_fixpaths=1, places_K2=K2))
        assert got["n_paths"] == n_paths
        assert abs(got["n_places_kept"] - kept) <= 3 and abs(got["n_places"] - unique) <= 3, (K2, got["n_places_kept"], got["n_places"], kept, unique)


def test_places_parameter_checks(T):
    rs = T.smoke_set()
    for bad in (dict(apply_fixpaths=0, places_K2=200), dict(apply_fixpaths=1, want_paths=0, places_K2=200), dict(apply_fixpaths=1, places_K2=40)):
        with pytest.raises(RuntimeError, match="places_K2"):
            T.run_product(rs, T.default_params(**bad))
