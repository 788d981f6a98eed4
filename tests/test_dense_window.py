"""The dense-id graph stage as k_adjacency_dense and k_links run it: every neighbour is looked for first within NODE_WINDOW ids of
the node that asks, then in the table (csrc/unipath.cuh: node_find with a hint).  Driven serially through the device functions
(tests/hostcheck/dense_window.cpp) and compared with the oracle; the share of lookups the window answers is guarded."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
SO = os.path.join(ROOT, "oracle", "_build", "libhostcheck_dense_window.so")


@pytest.fixture(scope="module")
def hw(T):
    src = os.path.join(HERE, "hostcheck", "dense_window.cpp")
    deps = [src, os.path.join(HERE, "hostcheck", "dense_nodes.cpp"), os.path.join(HERE, "hostcheck", "hostcheck.cpp"),
            os.path.join(ROOT, "include", "w2rap_step2.h")]
    deps += [os.path.join(ROOT, "w2rap-contigger_b200", "csrc", f) for f in os.listdir(os.path.join(ROOT, "w2rap-contigger_b200", "csrc"))]
    if not os.path.exists(SO) or any(os.path.getmtime(d) > os.path.getmtime(SO) for d in deps):
        os.makedirs(os.path.dirname(SO), exist_ok=True)
        subprocess.run(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-x", "c++", "-o", SO, src], check=True)
    lib = C.CDLL(SO)
    lib.hc_count.argtypes = [C.POINTER(T.Reads), C.c_uint32, C.POINTER(C.c_void_p), C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]
    lib.hc_graph_dense_window.argtypes = [C.c_void_p, C.c_uint64, C.c_uint32, C.c_uint32, C.c_int, C.POINTER(T.Reads), C.c_int, C.c_int,
                                          C.c_uint32, C.c_uint32, C.POINTER(T.Graph), C.POINTER(C.c_uint64 * 4)]
    lib.hc_free.argtypes = [C.c_void_p]
    lib.hc_graph_free.argtypes = [C.POINTER(T.Graph)]
    return lib


def window_graph(T, hw, rs, min_qual=7, min_freq=4, apply_fixpaths=0, logP=7, shuffle=0, cap=24, left_cap=8):
    """Count, then the graph stage; returns the graph as a dict and (adjacency lookups, of which in the window, successor-link
    lookups, of which in the window)."""
    ptr, n, ninst = C.c_void_p(), C.c_uint64(), C.c_uint64()
    reads = rs.c()
    assert hw.hc_count(C.byref(reads), min_qual, C.byref(ptr), C.byref(n), C.byref(ninst)) == 0
    g = T.Graph()
    win = (C.c_uint64 * 4)()
    rc = hw.hc_graph_dense_window(ptr, n, min_freq, logP, shuffle, C.byref(reads), 1, apply_fixpaths, cap, left_cap, C.byref(g), C.byref(win))
    hw.hc_free(ptr)
    assert rc == 0, "dense graph stage failure %d" % rc
    d = T.graph_to_dict(g)
    hw.hc_graph_free(C.byref(g))
    return d, tuple(win)


def check_against_oracle(T, hw, rs, **kw):
    """The graph in the reduce's order and in a scrambled one, each against the oracle."""
    pk = {k: v for k, v in kw.items() if k in ("min_qual", "min_freq", "apply_fixpaths")}
    want = T.run_oracle(rs, T.default_params(dump_kmers=1, **pk))
    for shuffle in (0, 1):
        d, _ = window_graph(T, hw, rs, shuffle=shuffle, **kw)
        for k in ("n_kmer_instances", "n_bases", "n_reads", "hist"):      # not produced by the graph stage
            d[k] = want[k]
        T.assert_graph_equal(want, d, "graph stage with window lookups (shuffle=%d) vs oracle" % shuffle)


def repeat_runs_set(T):
    """A homopolymer run of 80 bases (its k-mer is its own successor: found at its own id) and a 160-base dinucleotide repeat
    (two k-mers that succeed each other: a two-node cycle) in random sequence, error-free reads of both strands."""
    rng = np.random.default_rng(17)
    g = np.concatenate([rng.integers(0, 4, 700), np.zeros(80), rng.integers(0, 4, 500), np.tile([0, 1], 80),
                        rng.integers(0, 4, 700)]).astype(np.uint8)
    codes, quals, lens = T.simulate_reads(rng, [(g, False, 1.0)], 160, read_len=150, frag_mean=300, frag_sd=30, errors=False)
    return T.flatten_reads(codes, quals, lens)


def tiny_set(T, length):
    """One error-free sequence of `length` bases read whole from both strands: a graph of length - 59 k-mers (61, 66: fewer than the
    window holds), so lookups clip at ids 0 and n - 1."""
    rng = np.random.default_rng(length)
    g = rng.integers(0, 4, length).astype(np.uint8)
    codes = np.stack([g, T.revcomp(g)] * 6)
    return T.flatten_reads(codes, np.full(codes.shape, 37, np.uint8), np.full(len(codes), length, np.uint32))


@pytest.mark.parametrize("name", ["rich", "long", "circ", "repeat_runs", "tiny_61", "tiny_66", "tiny_200"])
def test_window_graph_stage(T, hw, name):
    """Graph, dictionary and paths equal the oracle's on the golden sets, on self-neighbours and two-node cycles, and on graphs smaller
    than the window, with ids in the reduce's order and scrambled (where almost every lookup takes the table)."""
    if name in ("rich", "long", "circ"):
        rs = T.read_fastb_qualp(os.path.join(HERE, "golden", name))
    else:
        rs = repeat_runs_set(T) if name == "repeat_runs" else tiny_set(T, int(name.split("_")[1]))
    check_against_oracle(T, hw, rs, apply_fixpaths=1, cap=3 if name == "circ" else 24, left_cap=1 if name == "circ" else 8)


def test_reduce_order_resolves_lookups_in_window(T, hw):
    """Window guard: in the reduce's order, at the partition size of test_reduce_order_keeps_successor_links_local (~500 solid
    k-mers per partition, as on the full-size workload), most neighbour lookups are answered in the window.  On the rich golden set
    the window answers 67 % of the adjacency lookups (the rest are mostly neighbours left by sequencing errors, absent from the
    dictionary) and 69 % of the successor-link lookups; in a scrambled order almost none."""
    rs = T.read_fastb_qualp(os.path.join(HERE, "golden", "rich"))
    d, _ = window_graph(T, hw, rs)
    logP = max(0, (int(d["n_solid"]) // 512).bit_length() - 1)
    _, (adj, adj_near, links, links_near) = window_graph(T, hw, rs, logP=logP)
    assert adj > 10000 and links > 10000
    assert adj_near >= 0.55 * adj, "%d of %d adjacency lookups in the window" % (adj_near, adj)
    assert links_near >= 0.55 * links, "%d of %d successor-link lookups in the window" % (links_near, links)
    _, (adj, adj_near, links, links_near) = window_graph(T, hw, rs, logP=logP, shuffle=1)
    assert adj_near < 0.05 * adj and links_near < 0.05 * links
