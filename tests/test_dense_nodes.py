"""The single-GPU graph stage over dense node ids (csrc/unipath.cuh: DenseNodes), driven serially through the device functions
(tests/hostcheck/dense_nodes.cpp) and compared with the oracle; the strand-normalised minimiser offset the reduce sorts by
(csrc/extract.cuh: kmer_minimizer_offset_words); and the locality that sort buys the list ranking."""
import ctypes as C
import os
import subprocess

import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
SO = os.path.join(ROOT, "oracle", "_build", "libhostcheck_dense.so")


@pytest.fixture(scope="module")
def hd(T):
    src = os.path.join(HERE, "hostcheck", "dense_nodes.cpp")
    deps = [src, os.path.join(HERE, "hostcheck", "hostcheck.cpp"), os.path.join(ROOT, "include", "w2rap_step2.h")]
    deps += [os.path.join(ROOT, "w2rap-contigger_b200", "csrc", f) for f in os.listdir(os.path.join(ROOT, "w2rap-contigger_b200", "csrc"))]
    if not os.path.exists(SO) or any(os.path.getmtime(d) > os.path.getmtime(SO) for d in deps):
        os.makedirs(os.path.dirname(SO), exist_ok=True)
        subprocess.run(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-x", "c++", "-o", SO, src], check=True)
    lib = C.CDLL(SO)
    lib.hc_count.argtypes = [C.POINTER(T.Reads), C.c_uint32, C.POINTER(C.c_void_p), C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]
    lib.hc_graph_dense.argtypes = [C.c_void_p, C.c_uint64, C.c_uint32, C.c_uint32, C.c_int, C.POINTER(T.Reads), C.c_int, C.c_int, C.c_uint32, C.c_uint32,
                                   C.POINTER(T.Graph), C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]
    lib.hc_minimizer_offsets.restype = C.c_uint64
    lib.hc_minimizer_offsets.argtypes = [C.POINTER(T.Reads), C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]
    lib.hc_free.argtypes = [C.c_void_p]
    lib.hc_graph_free.argtypes = [C.POINTER(T.Graph)]
    return lib


def dense_graph(T, hd, rs, min_qual=7, min_freq=4, apply_fixpaths=0, logP=7, shuffle=0, cap=24, left_cap=8):
    """Count, then the dense-id graph stage; returns the graph as a dict and (successor links, links within +-64 ids)."""
    ptr, n, ninst = C.c_void_p(), C.c_uint64(), C.c_uint64()
    reads = rs.c()
    assert hd.hc_count(C.byref(reads), min_qual, C.byref(ptr), C.byref(n), C.byref(ninst)) == 0
    g = T.Graph()
    nl, nnear = C.c_uint64(), C.c_uint64()
    rc = hd.hc_graph_dense(ptr, n, min_freq, logP, shuffle, C.byref(reads), 1, apply_fixpaths, cap, left_cap, C.byref(g), C.byref(nl), C.byref(nnear))
    hd.hc_free(ptr)
    assert rc == 0, "dense graph stage failure %d" % rc
    d = T.graph_to_dict(g)
    d["_circle_nodes"] = g.timings.count_passes
    hd.hc_graph_free(C.byref(g))
    return d, nl.value, nnear.value


def check_dense_against_oracle(T, hd, rs, **kw):
    d, nl, nnear = dense_graph(T, hd, rs, **kw)
    pk = {k: v for k, v in kw.items() if k in ("min_qual", "min_freq", "apply_fixpaths")}
    want = T.run_oracle(rs, T.default_params(dump_kmers=1, **pk))
    for k in ("n_kmer_instances", "n_bases", "n_reads", "hist"):      # not produced by the graph stage
        d[k] = want[k]
    circle_nodes = d.pop("_circle_nodes")
    T.assert_graph_equal(want, d, "dense-id graph stage vs oracle")
    return d, nl, nnear, circle_nodes


@pytest.mark.parametrize("name", ["rich", "long", "circ"])
def test_dense_graph_stage_golden(T, hd, name):
    """Graph, dictionary (pruned contexts, edge + offset of every k-mer after the back-fill) and paths equal the oracle's on the
    golden sets; circ has smooth circles of both parities and palindromes, and its tiny staging rows force the overflow path."""
    rs = T.read_fastb_qualp(os.path.join(HERE, "golden", name))
    _, _, _, circle_nodes = check_dense_against_oracle(T, hd, rs, apply_fixpaths=1, cap=3 if name == "circ" else 24, left_cap=1 if name == "circ" else 8)
    if name == "circ":
        assert circle_nodes > 0


def test_dense_graph_stage_palindromes_and_fragments(T, hd):
    """Palindromic k-mers and a plasmid circle; a shattered low-coverage graph with many tips and one-k-mer edges."""
    check_dense_against_oracle(T, hd, T.rich_set(seed=5, genome=40000, cov=50, families=5, palindromes=6, plasmid=1500, vary_len=True), apply_fixpaths=1)
    check_dense_against_oracle(T, hd, T.rich_set(seed=7, genome=30000, cov=12, families=4, palindromes=2, plasmid=800), min_freq=3)


def test_dense_ids_in_any_order(T, hd):
    """The emitted order is a locality hint, never a correctness condition: scrambled ids give the same graph."""
    rs = T.rich_set(seed=2, genome=60000, cov=50, pq_mode=1)
    a, _, _, _ = check_dense_against_oracle(T, hd, rs)
    b, nl, nnear = dense_graph(T, hd, rs, shuffle=1)
    b.pop("_circle_nodes")
    for k in ("n_kmer_instances", "n_bases", "n_reads", "hist"):
        b[k] = a[k]
    T.assert_graph_equal(a, b, "scrambled dense ids vs reduce order")
    assert nnear < 0.2 * nl


def test_minimizer_offset_is_strand_normalised(T, hd):
    """A k-mer and its reverse complement get the same minimiser and offset; along a read the offset steps by one while the
    minimiser holds."""
    rs = T.rich_set(seed=11, genome=20000, cov=8, families=2, palindromes=2, plasmid=500)
    n, ns = C.c_uint64(), C.c_uint64()
    assert hd.hc_minimizer_offsets(C.byref(rs.c()), C.byref(n), C.byref(ns)) == 0
    assert n.value > 10000 and ns.value > 0.8 * n.value


def test_reduce_order_keeps_successor_links_local(T, hd):
    """Locality guard: in the reduce's order (partitions of ~500 solid k-mers, as on the full-size workload) at least 80 % of the
    successor links stay within +-64 ids."""
    rs = T.read_fastb_qualp(os.path.join(HERE, "golden", "rich"))
    d, nl, nnear = dense_graph(T, hd, rs)
    logP = max(0, (int(d["n_solid"]) // 512).bit_length() - 1)
    d, nl, nnear = dense_graph(T, hd, rs, logP=logP)
    assert nl > 1000
    assert nnear >= 0.8 * nl, "%d of %d successor links within 64 ids" % (nnear, nl)
