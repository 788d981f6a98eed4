"""Runs the read-batch cases of test_upload_batches.py in a fresh process: the library reads W2RAP_UPLOAD_BATCHES (and the other
diagnostic switches) once per process, so each switch setting needs a process of its own.

usage: batch_case_runner.py hook|reject

Every case runs the product through w2rap_step2_run twice, from the numpy buffers (pageable) and from buffers taken from
w2rap_step2_host_alloc (pinned: only then does the copy of batch b+1 overlap the map of batch b), and compares both with the oracle
bit for bit.  It also checks timings.count_launches: one scatter launch per non-empty read batch and counting pass, so a batch that
was not mapped, or a re-sized retry of the map, shows up.  One line per case; the exit code is the number of failed cases.
"""
import ctypes as C
import os
import sys
import traceback

import numpy as np

import w2r_testlib as T

NB = int(os.environ.get("W2RAP_UPLOAD_BATCHES", "1")) if os.environ.get("W2RAP_UPLOAD_BATCHES", "1").isdigit() else 0


def batch_of(n_reads):
    """Read batch of every read index: the upload gives batch b the reads [n*b/NB, n*(b+1)/NB)."""
    b = np.zeros(n_reads, np.int64)
    for k in range(NB):
        b[n_reads * k // NB:n_reads * (k + 1) // NB] = k
    return b


def expected_launches(rs, npass):
    if rs.n == 0 or not (rs.len > 59).any():      # no read has a k-mer: nothing is mapped
        return 0
    return len(np.unique(batch_of(rs.n))) * npass


def run_pinned(rs, params):
    """w2rap_step2_run from library-allocated pinned buffers filled from the numpy ones."""
    lib = T.product_lib()
    lib.w2rap_step2_host_alloc.restype = C.c_void_p
    lib.w2rap_step2_host_alloc.argtypes = [C.c_size_t]
    lib.w2rap_step2_host_free.restype = None
    lib.w2rap_step2_host_free.argtypes = [C.c_void_p]
    bufs = []
    try:
        ptrs = []
        for a in (rs.bases, rs.base_off, rs.len, rs.quals, rs.qual_off):
            p = lib.w2rap_step2_host_alloc(max(1, a.nbytes))
            assert p, "w2rap_step2_host_alloc(%d) failed" % a.nbytes
            bufs.append(p)
            C.memmove(p, a.ctypes.data, a.nbytes)
            ptrs.append(p)
        reads = T.Reads(rs.n, *ptrs)
        g = T.Graph()
        err = C.create_string_buffer(1024)
        rc = lib.w2rap_step2_run(C.byref(reads), C.byref(params), C.byref(g), err, len(err))
        if rc != 0:
            raise RuntimeError("w2rap_step2_run failed (%d): %s" % (rc, err.value.decode(errors="replace")))
        d = T.graph_to_dict(g)
        lib.w2rap_step2_free(C.byref(g))
        return d
    finally:
        for p in bufs:
            lib.w2rap_step2_host_free(p)


def check(name, rs, want, check_passes=None, **kw):
    """Both host memories against `want` (the oracle on the same reads); returns the pinned result."""
    npass = kw.get("force_passes", 0) or 1
    for mem in ("pageable", "pinned"):
        p = T.default_params(**kw)
        got = T.run_product(rs, p) if mem == "pageable" else run_pinned(rs, p)
        T.assert_graph_equal(want, got, "%s (%s, %d batches)" % (name, mem, NB))
        launches, exp = got["timings"]["count_launches"], expected_launches(rs, npass)
        assert launches == exp, "%s (%s): %d scatter launches, expected %d (batches x passes)" % (name, mem, launches, exp)
        if check_passes:
            assert check_passes(got["timings"]["count_passes"]), "%s (%s): %d reduce groups" % (name, mem, got["timings"]["count_passes"])
    print("  %s: %d reads, %d distinct, %d solid, %d edges, %d scatter launches, %d reduce groups" % (
        name, rs.n, got["n_distinct"], got["n_solid"], got["n_edges"], launches, got["timings"]["count_passes"]))
    return got


def oracle(rs, **kw):
    return T.run_oracle(rs, T.default_params(**{k: v for k, v in kw.items() if k not in ("table_slots", "force_passes")}))


# ---------------------------------------------------------------- (a) a rich read set, 14 k reads of 30-250 bases

def rich_cases():
    rs = T.rich_set(seed=41, genome=60000, cov=50, families=4, palindromes=3, plasmid=2000, pq_mode=1, vary_len=True)
    kw = dict(dump_kmers=2, apply_fixpaths=1)
    want = oracle(rs, **kw)
    yield "rich", lambda: check("rich", rs, want, **kw)
    yield "rich, 2 forced passes", lambda: check("rich, 2 forced passes", rs, want, force_passes=2, **kw)
    yield "rich, region fallback", lambda: check("rich, region fallback", rs, want, check_passes=lambda g: g > 3, table_slots=60000, **kw)


def tiny_region_case():
    """A 4-slot shared-memory table and a 64-slot region: the per-partition retry and the hash sub-range split with roll-back."""
    rs = T.rich_set(seed=6, genome=12000, cov=30, families=2, palindromes=1, plasmid=600)
    want = oracle(rs, dump_kmers=2)
    check("tiny region", rs, want, check_passes=lambda g: g > 1000, dump_kmers=2, table_slots=64)


# ---------------------------------------------------------------- (b) counts that only add up across batches

def spread_set(seed=43, n_reads=640, min_freq=4):
    """Singleton background reads plus planted reads whose copies sit in different read batches:
    A: min_freq copies (solid only if every batch's copy is counted), B: min_freq - 1 copies (never solid),
    C: 300 copies over all batches (saturates at 255 only summed over batches), and four 62-base reads around one 60-mer X with
    predecessor j and successor j+1 (mod 4) in different batches: X's context is complete only as the OR over batches."""
    rng = np.random.default_rng(seed)
    L = 150
    a, b, c = (rng.integers(0, 4, L, dtype=np.uint8) for _ in range(3))
    x = rng.integers(0, 4, 60, dtype=np.uint8)
    planted = []                                          # (batch, codes)
    planted += [((j * NB) // min_freq, a) for j in range(min_freq)]
    planted += [(((2 * j + 1) * NB) // (2 * (min_freq - 1)), b) for j in range(min_freq - 1)]
    planted += [(j % NB, c) for j in range(300)]
    planted += [(((2 * j + 1) * NB) // 8, np.concatenate([[j], x, [(j + 1) % 4]]).astype(np.uint8)) for j in range(4)]
    bo = batch_of(n_reads)
    free = {k: list(np.nonzero(bo == k)[0]) for k in range(NB)}
    codes = rng.integers(0, 4, (n_reads, L), dtype=np.uint8)      # background: random, so every k-mer is a singleton
    lens = np.full(n_reads, L, np.uint32)
    for k, seq in planted:
        i = free[k].pop(0)
        codes[i, :len(seq)] = seq
        lens[i] = len(seq)
    return T.flatten_reads(codes, np.full((n_reads, L), 35, np.uint8), lens)


def spread_case():
    rs = spread_set()
    want = oracle(rs, dump_kmers=2, min_freq=4)
    got = check("counts across batches", rs, want, dump_kmers=2, min_freq=4)
    d = got["dump"]
    nk = 150 - 59
    # C: 300 copies -> count 255 (saturated), histogram bin 100 holds exactly its k-mers
    assert (d["count"] == 255).sum() == nk and got["hist"][100] == nk, (int((d["count"] == 255).sum()), int(got["hist"][100]))
    # B: 3 copies, never solid; A: 4 copies, solid; X: 4 copies from four reads
    assert (d["count"] == 3).sum() == nk, int((d["count"] == 3).sum())
    assert (d["count"] == 4).sum() == nk + 1, int((d["count"] == 4).sum())
    # X: all four predecessors and all four successors, each seen in another batch
    full = d[d["ctx"] == 0xff]
    assert len(full) == 1 and full["count"][0] == 4, full
    # solid: exactly A's and C's k-mers and X
    assert got["n_solid"] == 2 * nk + 1, got["n_solid"]


# ---------------------------------------------------------------- (c) degenerate batches

def degenerate_cases():
    rng = np.random.default_rng(44)
    g = rng.integers(0, 4, 2500, dtype=np.uint8)
    L = 150

    def sample(n):
        st = rng.integers(0, len(g) - L, n)
        return np.stack([g[s:s + L] for s in st]), np.full((n, L), 30, np.uint8), np.full(n, L, np.uint32)

    # fewer reads than batches: batches without reads
    codes, quals, lens = sample(5)
    rs = T.flatten_reads(codes, quals, lens)
    for mf in (1, 6):                                      # min_freq 6: nothing solid, the empty graph
        yield "5 reads, min_freq %d" % mf, (lambda rs=rs, mf=mf: check("5 reads, min_freq %d" % mf, rs, oracle(rs, dump_kmers=2, apply_fixpaths=1, min_freq=mf),
                                                                         dump_kmers=2, apply_fixpaths=1, min_freq=mf))
    # one batch of reads shorter than 60 bases, another of reads entirely below min_qual
    n = 24 * NB
    codes, quals, lens = sample(n)
    bo = batch_of(n)
    short = bo == 0
    lens[short] = rng.integers(1, 60, int(short.sum())).astype(np.uint32)
    quals[bo == NB - 1] = 3
    rs = T.flatten_reads(codes, quals, lens)
    yield "short and low-quality batches", lambda: check("short and low-quality batches", rs, oracle(rs, dump_kmers=2, apply_fixpaths=1, min_freq=2),
                                                         dump_kmers=2, apply_fixpaths=1, min_freq=2)
    # every read of every batch shorter than 60 bases: nothing to map
    rs2 = T.flatten_reads(codes, quals, rng.integers(1, 60, n).astype(np.uint32))
    yield "all reads short", lambda: check("all reads short", rs2, oracle(rs2, dump_kmers=2, apply_fixpaths=1, min_freq=1), dump_kmers=2, apply_fixpaths=1, min_freq=1)


def main():
    mode = sys.argv[1]
    if mode == "reject":
        rs = T.smoke_set(seed=3, genome=3000, cov=10)
        try:
            T.run_product(rs)
        except RuntimeError as e:
            print("REJECTED %s" % e)
            return 0
        print("ACCEPTED")
        return 1
    T.build_oracle()
    cases = []
    if mode == "hook":
        cases += list(rich_cases())
        if NB == 8:
            cases.append(("tiny region", tiny_region_case))
        cases.append(("counts across batches", spread_case))
        cases += list(degenerate_cases())
    else:
        raise SystemExit("unknown mode " + mode)
    failed = 0
    for name, fn in cases:
        try:
            fn()
            print("OK %s" % name)
        except Exception:
            failed += 1
            print("FAIL %s\n%s" % (name, traceback.format_exc()))
        sys.stdout.flush()
    return failed


if __name__ == "__main__":
    sys.exit(main())
