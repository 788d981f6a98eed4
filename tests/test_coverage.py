"""K-mer coverage from the kept counts (w2rap_counts_coverage) and the graph as GFA (w2rap_write_gfa), include/w2rap_coverage.h.

Expected coverage comes from the oracle's level-2 dump (every distinct canonical k-mer with min(255, count)), filtered at f0, with
the canonical form of every k-mer of a sequence computed here in numpy: never from the product.  The GFA writer is compared with a
writer in Python, and its links with a derivation from sequences alone: oriented edges whose last 59 bases are the next one's first.
"""
import ctypes as C
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

import w2r_testlib as T

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
GOLD = os.path.join(HERE, "golden")
HC_SO = os.path.join(ROOT, "oracle", "_build", "libhostcheck_cov.so")
BAD_ARG = 1
K = 60


class Seqs(C.Structure):
    _fields_ = [("n", C.c_uint64), ("bases", C.c_void_p), ("base_off", C.c_void_p), ("len", C.c_void_p)]


class SeqCov(C.Structure):
    _fields_ = [("n_kmers", C.c_uint64), ("sum", C.c_uint64), ("n_absent", C.c_uint64), ("min", C.c_uint32), ("max", C.c_uint32)]


COV_DTYPE = np.dtype([("n_kmers", "<u8"), ("sum", "<u8"), ("n_absent", "<u8"), ("min", "<u4"), ("max", "<u4")])


def lib():
    lb = T.product_lib()
    E = [C.c_char_p, C.c_size_t]
    lb.w2rap_step2_count.argtypes = [C.c_void_p, C.POINTER(T.Params), C.POINTER(C.c_void_p), C.POINTER(T.Graph)] + E
    lb.w2rap_step2_build.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(T.Params), C.POINTER(T.Graph)] + E
    lb.w2rap_step2_counts_release.argtypes = [C.c_void_p]
    lb.w2rap_step2_counts_release.restype = None
    lb.w2rap_counts_coverage.argtypes = [C.c_void_p, C.POINTER(Seqs), C.c_void_p, C.POINTER(C.c_float)] + E
    lb.w2rap_counts_coverage.restype = C.c_int
    lb.w2rap_write_gfa.argtypes = [C.c_char_p, C.POINTER(T.Graph), C.c_void_p] + E
    lb.w2rap_write_gfa.restype = C.c_int
    return lb


# ---------------------------------------------------------------- sequences and the expected coverage

class SeqSet:
    """Packed sequences (2-bit, LSB-first, each starting on a byte) with 32 bytes of padding, and the ctypes view."""

    def __init__(self, seqs):
        self.codes = [np.asarray(s, np.uint8) for s in seqs]
        self.len = np.array([len(s) for s in self.codes], np.uint32)
        nb = (self.len.astype(np.int64) + 3) // 4
        self.base_off = np.concatenate([[0], np.cumsum(nb)]).astype(np.uint64)
        self.bases = np.zeros(int(self.base_off[-1]) + 32, np.uint8)
        for s, o in zip(self.codes, self.base_off[:-1]):
            p = np.zeros(((len(s) + 3) // 4) * 4, np.uint8)
            p[:len(s)] = s
            self.bases[int(o):int(o) + len(p) // 4] = (p.reshape(-1, 4) << np.array([0, 2, 4, 6], np.uint8)).sum(axis=1).astype(np.uint8)
        self.len_store = np.concatenate([self.len, np.zeros(1, np.uint32)])

    def c(self):
        return Seqs(len(self.codes), self.bases.ctypes.data, self.base_off.ctypes.data, self.len_store.ctypes.data)


def seqs_of_reads(rs, idx=None):
    return [rs.read_codes(r) for r in (range(rs.n) if idx is None else idx)]


def kmer_words(codes):
    """(w0, w1) of every 60-mer of a code array: base 0 in bits 63-62 of w0, bases 32..59 in bits 63..8 of w1."""
    n = len(codes) - K + 1
    if n <= 0:
        return np.zeros(0, np.uint64), np.zeros(0, np.uint64)
    win = np.lib.stride_tricks.sliding_window_view(codes.astype(np.uint64), K)
    w0 = np.zeros(n, np.uint64)
    w1 = np.zeros(n, np.uint64)
    for i in range(32):
        w0 |= win[:, i] << np.uint64(62 - 2 * i)
    for i in range(32, K):
        w1 |= win[:, i] << np.uint64(62 - 2 * (i - 32))
    return w0, w1


def canonical_kmers(codes):
    f0, f1 = kmer_words(codes)
    r0, r1 = kmer_words(T.revcomp(codes))
    r0, r1 = r0[::-1], r1[::-1]                       # rc of the k-mer at position p = k-mer at L-60-p of the rc sequence
    rev = (r0 < f0) | ((r0 == f0) & (r1 < f1))
    return np.where(rev, r0, f0), np.where(rev, r1, f1)


def kept_dict(dump, f0):
    m = dump["count"] >= f0
    return dict(zip(zip(dump["w0"][m].tolist(), dump["w1"][m].tolist()), dump["count"][m].tolist()))


def expected_coverage(seqs, kept):
    out = np.zeros(len(seqs), COV_DTYPE)
    for i, s in enumerate(seqs):
        w0, w1 = canonical_kmers(s)
        c = np.array([kept.get(k, 0) for k in zip(w0.tolist(), w1.tolist())], np.uint64)
        out[i] = (len(c), c.sum(), (c == 0).sum(), c.min() if len(c) else 0, c.max() if len(c) else 0)
    return out


def assert_cov_equal(want, got, what):
    for f in COV_DTYPE.names:
        bad = np.nonzero(want[f] != got[f])[0]
        assert len(bad) == 0, "%s: field %s differs at sequences %s: %s vs %s" % (what, f, bad[:5], want[f][bad[:5]], got[f][bad[:5]])


def mixed_sequences(rs, rng):
    """Reads, random sequences, lengths 0/59/60/61, palindromic 60-mers inside, long sequences over many tiles, and sequences of
    k-mers seen fewer than f0 times (reads' low-quality tails dominate those; random sequences have none kept)."""
    seqs = seqs_of_reads(rs, range(0, rs.n, 7))
    seqs += [rng.integers(0, 4, int(L), dtype=np.uint8) for L in rng.integers(0, 400, 40)]
    seqs += [rng.integers(0, 4, L, dtype=np.uint8) for L in (0, 59, 60, 61, 0)]
    seqs += [s[:L] for s, L in zip(seqs_of_reads(rs, range(5)), (59, 60, 61, 62, 119))]
    for i in range(6):                                  # palindromic 60-mers, alone and inside reads
        half = rng.integers(0, 4, 30, dtype=np.uint8)
        pal = np.concatenate([half, T.revcomp(half)])
        r = rs.read_codes(3 * i + 1)
        seqs += [pal, np.concatenate([r[:100], pal, r[100:]])]
    long_seq = np.concatenate(seqs_of_reads(rs, range(11, 11 + 240)))   # ~60 k bases: > 100 tiles, mostly kept k-mers
    seqs += [long_seq, long_seq[:512 + 59], long_seq[:512 + 60], long_seq[:1024 + 59]]
    return seqs


# ---------------------------------------------------------------- GFA in Python

def gfa_text(d, cov=None):
    """The GFA w2rap_write_gfa writes for a w2rap_graph dict (header: include/w2rap_coverage.h)."""
    edges = T.unpack_edges(d)
    out = ["H\tVN:Z:1.0\n"]
    for i, e in enumerate(edges):
        line = "S\t%d\t%s\tLN:i:%d" % (d["fwd_xlat"][i], "".join("ACGT"[b] for b in e), len(e))
        if cov is not None:
            line += "\tKC:i:%d" % cov["sum"][i]
            if cov["n_kmers"][i]:
                line += "\tDP:f:%.3f" % (cov["sum"][i] / cov["n_kmers"][i])
        out.append(line + "\n")
    inv = [int(x) for x in d["involution"]]
    seg, minus, left, right = {}, {}, {}, {}
    for i in range(d["n_edges"]):
        fw = int(d["fwd_xlat"][i])
        seg[fw], minus[fw], left[fw], right[fw] = fw, False, d["edge_vertices"][i][0], d["edge_vertices"][i][1]
        if inv[fw] != fw:
            rv = inv[fw]
            seg[rv], minus[rv], left[rv], right[rv] = fw, True, d["edge_vertices"][i][2], d["edge_vertices"][i][3]
    links = sorted((right[x], x, y) for x in range(d["n_hbv_edges"]) for y in range(d["n_hbv_edges"]) if right[x] == left[y])
    for _, x, y in links:
        if (inv[y], inv[x]) < (x, y):
            continue
        out.append("L\t%d\t%s\t%d\t%s\t59M\n" % (seg[x], "-" if minus[x] else "+", seg[y], "-" if minus[y] else "+"))
    return "".join(out)


def parse_gfa(text):
    segs, links = {}, []
    for line in text.splitlines():
        t = line.split("\t")
        if t[0] == "S":
            segs[int(t[1])] = dict(seq=t[2], tags=dict((x.split(":")[0], x.split(":")[2]) for x in t[3:]))
        elif t[0] == "L":
            assert t[5] == "59M"
            links.append((int(t[1]), t[2], int(t[3]), t[4]))
    return segs, links


def derived_links(hbv_seqs):
    """Every pair of oriented edges (hbv ids) whose sequences overlap by 59 bases, one per complementary pair."""
    rc = {s: i for i, s in enumerate(hbv_seqs)}
    inv = [rc[bytes(T.revcomp(np.frombuffer(s, np.uint8)))] for s in hbv_seqs]
    by_head = {}
    for y, s in enumerate(hbv_seqs):
        by_head.setdefault(s[:K - 1], []).append(y)
    pairs = set()
    for x, s in enumerate(hbv_seqs):
        for y in by_head.get(s[-(K - 1):], []):
            pairs.add(min((x, y), (inv[y], inv[x])))
    return pairs, inv


def gfa_links_as_hbv(links, inv):
    return [(a if oa == "+" else inv[a], b if ob == "+" else inv[b]) for a, oa, b, ob in links]


def hand_graph(edge_seqs):
    """A w2rap_graph dict from canonical edge sequences: hbv ids as HBVFromEdges assigns them (edge i: fwd id, then rc id unless
    palindromic), vertices = the distinct (K-1)-mers at edge ends."""
    edge_seqs = sorted((min(bytes(s), bytes(T.revcomp(np.asarray(s, np.uint8)))) for s in edge_seqs))
    nxt, fwd, rev, hseq = 0, [], [], []
    for s in edge_seqs:
        r = bytes(T.revcomp(np.frombuffer(s, np.uint8)))
        fwd.append(nxt); hseq.append(s); nxt += 1
        if r != s:
            rev.append(nxt); hseq.append(r); nxt += 1
        else:
            rev.append(fwd[-1])
    ends = sorted({s[:K - 1] for s in hseq} | {s[-(K - 1):] for s in hseq})
    vid = {e: i for i, e in enumerate(ends)}
    ev = []
    for i, s in enumerate(edge_seqs):
        r = hseq[rev[i]]
        ev.append([vid[s[:K - 1]], vid[s[-(K - 1):]]] + ([vid[r[:K - 1]], vid[r[-(K - 1):]]] if rev[i] != fwd[i] else [-1, -1]))
    inv = np.zeros(nxt, np.int32)
    for f, r in zip(fwd, rev):
        inv[f], inv[r] = r, f
    ss = SeqSet([np.frombuffer(s, np.uint8) for s in edge_seqs])
    return dict(n_edges=len(edge_seqs), n_vertices=len(ends), n_hbv_edges=nxt, edge_len=ss.len, edge_off=ss.base_off,
                edge_bases=ss.bases, edge_vertices=np.array(ev, np.int32).reshape(-1, 4), fwd_xlat=np.array(fwd, np.int32),
                rev_xlat=np.array(rev, np.int32), involution=inv, _hbv_seqs=hseq)


def graph_struct(d, keep):
    g = T.Graph()
    for name, dt in (("edge_off", "<u8"), ("edge_len", "<u4"), ("edge_bases", "u1"), ("fwd_xlat", "<i4"), ("rev_xlat", "<i4"),
                     ("involution", "<i4"), ("edge_vertices", "<i4")):
        keep[name] = np.ascontiguousarray(np.asarray(d[name]).reshape(-1), dtype=dt)
        setattr(g, name, keep[name].ctypes.data)
    g.n_edges, g.n_vertices, g.n_hbv_edges = d["n_edges"], d["n_vertices"], d["n_hbv_edges"]
    return g


def write_gfa(d, path, cov=None):
    keep = {}
    g = graph_struct(d, keep)
    err = C.create_string_buffer(512)
    cv = np.ascontiguousarray(cov, COV_DTYPE) if cov is not None else None
    rc = lib().w2rap_write_gfa(str(path).encode(), C.byref(g), cv.ctypes.data if cv is not None else None, err, 512)
    assert rc == 0, err.value
    return open(path).read()


# ---------------------------------------------------------------- CPU: interface

def declared_symbols():
    txt = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "w2rap_coverage.h")).read(), flags=re.S)
    return sorted(set(re.findall(r"\b(w2rap_[a-z0-9_]+)\s*\(", txt)))


def test_every_declared_symbol_is_exported():
    assert declared_symbols() == ["w2rap_counts_coverage", "w2rap_write_gfa"]
    lb = lib()
    for n in declared_symbols():
        assert hasattr(lb, n), "missing export " + n


def test_struct_sizes_match_header(tmp_path):
    src = tmp_path / "sz.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "w2rap_coverage.h"\nint main(void){printf("%zu %zu %zu %zu %zu\\n",'
                   'sizeof(w2rap_seqs),sizeof(w2rap_seq_cov),offsetof(w2rap_seqs,len),offsetof(w2rap_seq_cov,min),offsetof(w2rap_seq_cov,max));return 0;}\n')
    exe = tmp_path / "sz"
    subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), "-o", str(exe), str(src)], check=True)
    got = [int(x) for x in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()]
    assert got == [C.sizeof(Seqs), C.sizeof(SeqCov), Seqs.len.offset, SeqCov.min.offset, SeqCov.max.offset] == [32, 32, 24, 24, 28]
    assert COV_DTYPE.itemsize == 32


def test_refusals_happen_before_the_handle_is_used():
    lb, err = lib(), C.create_string_buffer(512)
    fake = C.c_void_p(16)          # never dereferenced: every call below is refused first
    ok = SeqSet([np.zeros(100, np.uint8), np.ones(70, np.uint8)])
    out = np.zeros(2, COV_DTYPE)
    assert lb.w2rap_counts_coverage(None, C.byref(ok.c()), out.ctypes.data, None, err, 512) == BAD_ARG
    assert lb.w2rap_counts_coverage(fake, None, out.ctypes.data, None, err, 512) == BAD_ARG
    assert lb.w2rap_counts_coverage(fake, C.byref(ok.c()), None, None, err, 512) == BAD_ARG
    for field in ("bases", "base_off", "len"):
        s = ok.c()
        setattr(s, field, None)
        assert lb.w2rap_counts_coverage(fake, C.byref(s), out.ctypes.data, None, err, 512) == BAD_ARG, field
    short = SeqSet([np.zeros(100, np.uint8), np.ones(70, np.uint8)])
    short.base_off[1] = 24                               # 100 bases need 25 bytes
    assert lb.w2rap_counts_coverage(fake, C.byref(short.c()), out.ctypes.data, None, err, 512) == BAD_ARG
    assert b"sequence 0" in err.value
    back = SeqSet([np.zeros(100, np.uint8), np.ones(70, np.uint8)])
    back.base_off[2] = 3                                 # offsets going backwards
    assert lb.w2rap_counts_coverage(fake, C.byref(back.c()), out.ctypes.data, None, err, 512) == BAD_ARG
    # the GFA writer: null arguments, and graphs without the arrays it reads
    d = hand_graph([np.random.default_rng(1).integers(0, 4, 80, dtype=np.uint8)])
    keep = {}
    g = graph_struct(d, keep)
    assert lb.w2rap_write_gfa(None, C.byref(g), None, err, 512) == BAD_ARG
    assert lb.w2rap_write_gfa(b"/nonexistent/x.gfa", None, None, err, 512) == BAD_ARG
    for field in ("edge_vertices", "fwd_xlat", "involution", "edge_bases"):
        g = graph_struct(d, keep)
        setattr(g, field, None)
        assert lb.w2rap_write_gfa(b"/nonexistent/x.gfa", C.byref(g), None, err, 512) == BAD_ARG, field


def hand_graphs():
    rng = np.random.default_rng(5)
    a = rng.integers(0, 4, 100, dtype=np.uint8)
    b1, b2 = rng.integers(0, 4, 30, dtype=np.uint8), rng.integers(0, 4, 45, dtype=np.uint8)
    b1[0], b2[0] = 0, 1
    linear = [a, np.concatenate([a[-59:], b1]), np.concatenate([a[-59:], b2])]     # one edge forking into two
    half = rng.integers(0, 4, 30, dtype=np.uint8)
    pal = np.concatenate([half, T.revcomp(half)])                                  # a palindromic one-k-mer edge
    into = np.concatenate([rng.integers(0, 4, 20, dtype=np.uint8), pal[:59]])      # an edge running into it
    s = rng.integers(0, 4, 90, dtype=np.uint8)
    circle = [np.concatenate([s, s[:59]])]                                         # a self-loop: start and end are one vertex
    return dict(linear=linear, palindrome=[pal, into], circle=circle, all=linear + [pal, into] + circle)


@pytest.mark.parametrize("name", ["linear", "palindrome", "circle", "all"])
def test_gfa_of_hand_built_graphs(tmp_path, name):
    d = hand_graph(hand_graphs()[name])
    got = write_gfa(d, tmp_path / "a.gfa")
    assert got == gfa_text(d)
    segs, links = parse_gfa(got)
    pairs, inv = derived_links(d["_hbv_seqs"])
    hl = gfa_links_as_hbv(links, inv)
    assert len(hl) == len(set(hl)) and set(hl) == pairs, (sorted(hl), sorted(pairs))
    assert all(min(p, (inv[p[1]], inv[p[0]])) == p for p in hl)
    for i in range(d["n_edges"]):
        assert segs[int(d["fwd_xlat"][i])]["seq"] == "".join("ACGT"[x] for x in np.frombuffer(d["_hbv_seqs"][d["fwd_xlat"][i]], np.uint8))
    if name == "palindrome":
        assert len(links) == 1 and d["n_hbv_edges"] == 3
    if name == "circle":
        assert len(links) == 1 and links[0][0] == links[0][2]
    cov = np.zeros(d["n_edges"], COV_DTYPE)
    cov["n_kmers"] = d["edge_len"] - 59
    cov["sum"] = 7 * np.arange(d["n_edges"]) + 3
    with_cov = write_gfa(d, tmp_path / "b.gfa", cov)
    assert with_cov == gfa_text(d, cov) and "\tKC:i:3\tDP:f:" in with_cov


# ---------------------------------------------------------------- CPU: the tile functions, serially

@pytest.fixture(scope="module")
def hc():
    src = os.path.join(HERE, "hostcheck", "coverage.cpp")
    deps = [src, os.path.join(ROOT, "include", "w2rap_coverage.h")]
    deps += [os.path.join(ROOT, "w2rap-contigger_b200", "csrc", f) for f in ("coverage.cuh", "kmer.cuh")]
    if not os.path.exists(HC_SO) or any(os.path.getmtime(x) > os.path.getmtime(HC_SO) for x in deps):
        os.makedirs(os.path.dirname(HC_SO), exist_ok=True)
        subprocess.run(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-x", "c++", "-o", HC_SO, src], check=True)
    lb = C.CDLL(HC_SO)
    lb.hc_coverage.argtypes = [C.c_void_p, C.c_uint64, C.c_uint32, C.POINTER(Seqs), C.c_void_p]
    return lb


@pytest.mark.parametrize("f0", [1, 3])
def test_tile_functions_against_the_oracle_counts(hc, f0):
    rs = T.rich_set(seed=9, genome=20000, cov=40, families=2, palindromes=3, plasmid=700)
    dump = T.run_oracle(rs, T.default_params(min_freq=f0, dump_kmers=2, want_paths=0))["dump"]
    rng = np.random.default_rng(f0)
    seqs = mixed_sequences(rs, rng)
    ss = SeqSet(seqs)
    got = np.zeros(len(seqs), COV_DTYPE)
    assert hc.hc_coverage(dump.ctypes.data, len(dump), f0, C.byref(ss.c()), got.ctypes.data) == 0
    want = expected_coverage(seqs, kept_dict(dump, f0))
    assert_cov_equal(want, got, "hostcheck f0=%d" % f0)
    assert want["n_absent"].sum() > 0 and (want["sum"] > 0).sum() > len(seqs) // 2 and want["n_kmers"].max() > 100 * 512


# ---------------------------------------------------------------- GPU

class Session:
    def __init__(self, rs=None):
        self.lib, self.err, self.h, self.counts = lib(), C.create_string_buffer(1024), C.c_void_p(), []
        if rs is not None:
            self.check(self.lib.w2rap_step2_upload(C.byref(rs.c()), -1, C.byref(self.h), self.err, 1024))

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

    def build(self, ch, **kw):
        g = T.Graph()
        self.check(self.lib.w2rap_step2_build(self.h, ch, C.byref(T.default_params(**kw)), C.byref(g), self.err, 1024))
        d = T.graph_to_dict(g)
        self.lib.w2rap_step2_free(C.byref(g))
        return d

    def coverage(self, ch, ss):
        """ss: anything with c() -> Seqs (it owns the arrays for the duration of the call)."""
        sv = ss.c()
        out = np.zeros(max(1, int(sv.n)), COV_DTYPE)
        ms = C.c_float(-1)
        self.check(self.lib.w2rap_counts_coverage(ch, C.byref(sv), out.ctypes.data, C.byref(ms), self.err, 1024))
        return out[:int(sv.n)], ms.value

    def close(self):
        for ch in self.counts:
            self.lib.w2rap_step2_counts_release(ch)
        self.lib.w2rap_step2_release(self.h)


def edges_of(d):
    return T.unpack_edges(d)


class GraphEdges:
    """The edge arrays of a w2rap_graph dict as a sequence set, as they are."""

    def __init__(self, d):
        self.d = d

    def c(self):
        return Seqs(self.d["n_edges"], self.d["edge_bases"].ctypes.data, self.d["edge_off"].ctypes.data, self.d["edge_len"].ctypes.data)


@pytest.mark.gpu
@pytest.mark.parametrize("f0", [1, 3])
def test_coverage_of_mixed_sequences(f0):
    rs = T.rich_set(seed=9, genome=20000, cov=40, families=2, palindromes=3, plasmid=700)
    dump = T.run_oracle(rs, T.default_params(min_freq=f0, dump_kmers=2, want_paths=0))["dump"]
    kept = kept_dict(dump, f0)
    s = Session(rs)
    try:
        ch, summ = s.count(min_freq=f0)
        assert summ["n_solid"] == len(kept)
        seqs = mixed_sequences(rs, np.random.default_rng(f0))
        got, ms = s.coverage(ch, SeqSet(seqs))
        assert_cov_equal(expected_coverage(seqs, kept), got, "f0=%d" % f0)
        assert ms > 0
        reads = seqs_of_reads(rs)                        # every read
        got, _ = s.coverage(ch, SeqSet(reads))
        assert_cov_equal(expected_coverage(reads, kept), got, "reads f0=%d" % f0)
        empty, ms0 = s.coverage(ch, SeqSet([]))           # the index build alone
        assert len(empty) == 0 and ms0 > 0
    finally:
        s.close()


@pytest.mark.gpu
def test_edges_of_builds_from_one_count():
    """f0 = 2, builds at 3, 4 and 6: every k-mer of an edge is kept and seen >= F times; the edges hold each solid k-mer once."""
    rs = T.rich_set(seed=2, genome=60000, cov=50, pq_mode=1)
    dump = T.run_oracle(rs, T.default_params(min_freq=2, dump_kmers=2, want_paths=0))["dump"]
    kept = kept_dict(dump, 2)
    s = Session(rs)
    try:
        ch, _ = s.count(min_freq=2)
        for mf in (3, 4, 6):
            d = s.build(ch, min_freq=mf)
            edges = edges_of(d)
            got, _ = s.coverage(ch, SeqSet(edges))
            assert (got["n_absent"] == 0).all() and (got["min"] >= mf).all(), mf
            assert int(got["n_kmers"].sum()) == d["n_solid"], mf
            assert np.array_equal(got["n_kmers"], d["edge_len"] - 59)
            assert_cov_equal(expected_coverage(edges, kept), got, "edges min_freq=%d" % mf)
    finally:
        s.close()


@pytest.mark.gpu
def test_every_reduce_path_gives_the_same_coverage():
    rs = T.rich_set(seed=6, genome=12000, cov=30, families=2, palindromes=1, plasmid=600)
    seqs = mixed_sequences(rs, np.random.default_rng(3))
    ss = SeqSet(seqs)
    s = Session(rs)
    try:
        ch, _ = s.count(min_freq=2)
        want, _ = s.coverage(ch, ss)
        for kw in (dict(force_passes=3), dict(table_slots=64)):
            ch2, summ = s.count(min_freq=2, **kw)
            assert summ["timings"]["count_passes"] >= 3, kw
            got, _ = s.coverage(ch2, ss)
            assert_cov_equal(want, got, str(kw))
        dump = T.run_oracle(rs, T.default_params(min_freq=2, dump_kmers=2, want_paths=0))["dump"]
        assert_cov_equal(expected_coverage(seqs, kept_dict(dump, 2)), want, "plain count vs oracle")
    finally:
        s.close()


@pytest.mark.gpu
def test_config1_scale():
    """Config 1 (4.6 Mbp, 100x, 1.84 M reads): the edges of builds at 3 and 5, and the coverage of every read."""
    lb, err = lib(), C.create_string_buffer(512)
    s = Session()
    sp = T.SynthParams(4_600_000, 250, 100, 11, 0, 0, 0, 0)
    assert lb.w2rap_step2_synth(C.byref(sp), -1, C.byref(s.h), err, 512) == 0, err.value
    hr = T.Reads()
    try:
        ch, summ = s.count(min_freq=2)
        for mf in (3, 5):
            d = s.build(ch, min_freq=mf, want_paths=0)
            got, _ = s.coverage(ch, GraphEdges(d))
            assert (got["n_absent"] == 0).all() and (got["min"] >= mf).all() and int(got["n_kmers"].sum()) == d["n_solid"], mf
        s.check(lb.w2rap_step2_download_reads(s.h, C.byref(hr), s.err, 1024))
        n = int(hr.n_reads)
        assert n == 1_840_000
        lens = T._arr(hr.len, n, "<u4")
        got, ms = s.coverage(ch, type("HostReads", (), {"c": lambda self: Seqs(n, hr.bases, hr.base_off, hr.len)})())
        assert ms > 0
        assert np.array_equal(got["n_kmers"], np.maximum(lens.astype(np.int64) - 59, 0))
        has = got["n_kmers"] > got["n_absent"]
        assert (got["min"] <= got["max"]).all() and (got["max"][has] >= 2).all() and (got["max"] <= 255).all()
        assert (got["sum"] <= 255 * (got["n_kmers"] - got["n_absent"])).all()
        assert (got["sum"] >= 2 * (got["n_kmers"] - got["n_absent"])).all()
        assert has.mean() > 0.95
    finally:
        if hr.bases:
            lb.w2rap_step2_free_host_reads(C.byref(hr))
        s.close()


@pytest.mark.gpu
def test_cli_gfa(tmp_path):
    exe = os.path.join(T.PKG_DIR, "step2")
    if not os.path.exists(exe):
        pytest.skip("step2 binary not built")
    runs = {"sweep": ("3,4", True), "sweep_plain": ("3,4", False), "one": ("4", True), "one_plain": ("4", False)}
    for k, (arg, gfa) in runs.items():
        d = tmp_path / k
        d.mkdir()
        for f in ("frag_reads_orig.fastb", "frag_reads_orig.qualp"):
            shutil.copy(os.path.join(GOLD, "circ", f), d)
        r = subprocess.run([exe, str(d), "x", "--min_freq", arg, "--quiet"] + (["--gfa"] if gfa else []), capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stdout + r.stderr
    for a, b in (("sweep", "sweep_plain"), ("one", "one_plain")):
        names = sorted(p.name for p in (tmp_path / a).iterdir() if not p.name.endswith(".gfa"))
        assert names == sorted(p.name for p in (tmp_path / b).iterdir())
        for nm in names:
            assert (tmp_path / a / nm).read_bytes() == (tmp_path / b / nm).read_bytes(), nm
    assert sorted(p.name for p in (tmp_path / "sweep").glob("*.gfa")) == ["x_mf3.small_K.gfa", "x_mf4.small_K.gfa"]
    assert sorted(p.name for p in (tmp_path / "one").glob("*.gfa")) == ["x.small_K.gfa"]
    rs = T.read_fastb_qualp(os.path.join(GOLD, "circ"))
    s = Session(rs)
    try:
        ch, _ = s.count(min_freq=3)
        for gfa, hbv, mf in (("sweep/x_mf3.small_K.gfa", "sweep/x_mf3.small_K.hbv", 3), ("sweep/x_mf4.small_K.gfa", "sweep/x_mf4.small_K.hbv", 4),
                             ("one/x.small_K.gfa", "one/x.small_K.hbv", 4)):
            segs, links = parse_gfa((tmp_path / gfa).read_text())
            hseqs = [e.tobytes() for e in T.parse_hbv(str(tmp_path / hbv))["edges"]]
            d = s.build(ch, min_freq=mf)
            assert len(segs) == d["n_edges"]
            for name, sg in segs.items():
                assert sg["seq"] == "".join("ACGT"[x] for x in np.frombuffer(hseqs[name], np.uint8)), name
            cov, _ = s.coverage(ch, SeqSet(edges_of(d)))
            for i in range(d["n_edges"]):
                sg = segs[int(d["fwd_xlat"][i])]
                assert int(sg["tags"]["KC"]) == int(cov["sum"][i]) and int(sg["tags"]["LN"]) == int(d["edge_len"][i])
            pairs, inv = derived_links(hseqs)
            hl = gfa_links_as_hbv(links, inv)
            assert len(hl) == len(set(hl)) and set(hl) == pairs, gfa
    finally:
        s.close()
