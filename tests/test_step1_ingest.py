"""Step-1 producer (SURVEY §8 N2, include/w2rap_step1.h): paired FASTQ -> flattened read stores + the reference's step files.

Pinned on files written by the UNMODIFIED reference: tests/golden/step1 (its step 1 run on a FASTQ pair whose content is kept in
expected.npz) and, where oracle/_ref/w2rap-contigger is present, fresh runs of its step 1 on FASTQ pairs generated here (runs of
equal qualities longer than 255, 'N's, lower-case bases, reads of very different lengths).  Equality is byte for byte on
frag_reads_orig.fastb and frag_reads_orig.qualp."""
import ctypes as C
import gzip
import os
import subprocess

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
SO = os.path.join(ROOT, "w2rap-contigger_b200", "libw2rap_step1.so")


class S1Params(C.Structure):
    _fields_ = [("abi_version", C.c_uint32), ("threads", C.c_uint32), ("alloc", C.c_void_p), ("release", C.c_void_p)]


class S1Stats(C.Structure):
    _fields_ = [("n_pairs", C.c_uint64), ("n_bases", C.c_uint64), ("n_converted", C.c_uint64), ("qual_bytes", C.c_uint64),
                ("read_s", C.c_double), ("parse_s", C.c_double), ("merge_s", C.c_double)]


@pytest.fixture(scope="module")
def s1(T):
    if not os.path.exists(SO):
        subprocess.run(["make", "-C", os.path.join(ROOT, "w2rap-contigger_b200"), os.path.join(ROOT, "w2rap-contigger_b200", "libw2rap_step1.so")], check=True)
    lib = C.CDLL(SO)
    lib.w2rap_step1_fastq_pair.argtypes = [C.c_char_p, C.c_char_p, C.POINTER(S1Params), C.POINTER(T.Reads), C.POINTER(S1Stats), C.c_char_p, C.c_size_t]
    lib.w2rap_step1_free.argtypes = [C.POINTER(S1Params), C.POINTER(T.Reads)]
    lib.w2rap_step1_write_stores.argtypes = [C.c_char_p, C.POINTER(T.Reads), C.c_char_p, C.c_size_t]
    lib.w2rap_step1_pq_encode.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p]
    lib.w2rap_step1_pq_encode.restype = C.c_size_t
    assert lib.w2rap_step1_abi_version() == 1
    return lib


def write_fastq_pair(d, seqs, quals, gz=False):
    """seqs/quals: lists of (str, bytes-like of phred values), mates interleaved (2i, 2i+1)."""
    names = []
    for k in range(2):
        fn = os.path.join(d, "r%d.fastq%s" % (k + 1, ".gz" if gz else ""))
        with (gzip.open(fn, "wt") if gz else open(fn, "w")) as f:
            for i in range(k, len(seqs), 2):
                f.write("@r%d/%d\n%s\n+\n%s\n" % (i // 2, k + 1, seqs[i], "".join(chr(33 + int(x)) for x in quals[i])))
        names.append(fn)
    return names


def ingest(T, s1, fq1, fq2, threads=3):
    p = S1Params(1, threads, None, None)
    r, st = T.Reads(), S1Stats()
    err = C.create_string_buffer(1024)
    rc = s1.w2rap_step1_fastq_pair(fq1.encode(), fq2.encode(), C.byref(p), C.byref(r), C.byref(st), err, 1024)
    return rc, err.value.decode(), p, r, st


def golden_fastq(T, tmp_path):
    exp = np.load(os.path.join(HERE, "golden", "step1", "expected.npz"))
    seqs, quals, off = [], [], 0
    for L in exp["lens"]:
        L = int(L)
        seqs.append("".join("ACGT"[b] for b in exp["bases"][off:off + L])); quals.append(exp["quals"][off:off + L]); off += L
    return seqs, quals


@pytest.mark.parametrize("threads,gz", [(1, False), (3, False), (8, True)])
def test_golden_step1_files_byte_for_byte(T, s1, tmp_path, threads, gz):
    seqs, quals = golden_fastq(T, tmp_path)
    fq1, fq2 = write_fastq_pair(str(tmp_path), seqs, quals, gz=gz)
    rc, err, p, r, st = ingest(T, s1, fq1, fq2, threads)
    assert rc == 0, err
    assert r.n_reads == len(seqs) and st.n_pairs == len(seqs) // 2 and st.n_bases == sum(len(s) for s in seqs)
    err2 = C.create_string_buffer(512)
    assert s1.w2rap_step1_write_stores(str(tmp_path).encode(), C.byref(r), err2, 512) == 0, err2.value
    s1.w2rap_step1_free(C.byref(p), C.byref(r))
    for f in ("frag_reads_orig.fastb", "frag_reads_orig.qualp"):
        assert open(os.path.join(str(tmp_path), f), "rb").read() == open(os.path.join(HERE, "golden", "step1", f), "rb").read(), f


def test_run_length_form_equals_the_programme(s1):
    """The producer emits blocks run by run (closed form); w2rap_step1_pq_encode is the reference's dynamic programme restated
    (PQVec.cc:18-85).  Same bytes on run-heavy, random and degenerate quality vectors."""
    s1.w2rap_step1_pq_encode_fastq.argtypes = [C.c_char_p, C.c_uint32, C.c_void_p]
    s1.w2rap_step1_pq_encode_fastq.restype = C.c_size_t
    rng = np.random.default_rng(2)
    a, b = np.zeros(3 * 70000 + 8, np.uint8), np.zeros(3 * 70000 + 8, np.uint8)
    for trial in range(400):
        kind = trial % 6
        n = int(rng.choice([0, 1, 2, 254, 255, 256, 509, 510, 511, 765, 1000, 3000])) if kind < 3 else int(rng.integers(1, 1200))
        if kind == 0:
            q = np.full(n, int(rng.integers(0, 64)))
        elif kind == 1:
            q = np.repeat(rng.integers(0, 64, n // 200 + 2), rng.integers(1, 600, n // 200 + 2))[:n]
        elif kind == 2:
            q = np.repeat(rng.integers(0, 64, n // 255 + 2), 255)[:n]
        elif kind == 3:
            q = rng.integers(0, 64, n)
        elif kind == 4:
            q = np.repeat(rng.integers(30, 34, n // 3 + 1), 3)[:n]
        else:
            q = np.concatenate([np.full(n // 2, 37), rng.integers(2, 40, n - n // 2)])
        q = q.astype(np.uint8)
        n = len(q)
        na = s1.w2rap_step1_pq_encode(q.ctypes.data if n else a.ctypes.data, n, a.ctypes.data)
        nb = s1.w2rap_step1_pq_encode_fastq(bytes((q + 33).tolist()), n, b.ctypes.data)
        assert na == nb and na > 0 and np.array_equal(a[:na], b[:nb]), (trial, n)
    bad = np.array([10, 64], np.uint8)
    assert s1.w2rap_step1_pq_encode(bad.ctypes.data, 2, a.ctypes.data) == 0
    assert s1.w2rap_step1_pq_encode_fastq(bytes((bad + 33).tolist()), 2, b.ctypes.data) == 0


def tricky_reads(seed, n_pairs):
    rng = np.random.default_rng(seed)
    seqs, quals = [], []
    for i in range(2 * n_pairs):
        L = int(rng.choice([1, 2, 59, 60, 61, 100, 250, 255, 256, 257, 300, 511, 600, 1000]))
        s = rng.integers(0, 4, L)
        kind = i % 5
        if kind == 0:
            q = np.full(L, 37)                                              # one run, longer than a block when L > 255
        elif kind == 1:
            q = np.repeat(rng.integers(2, 42, L // 7 + 1), 7)[:L]           # short runs
        elif kind == 2:
            q = np.concatenate([np.full(L - L // 3, 40), rng.integers(0, 64, L // 3)])
        elif kind == 3:
            q = rng.integers(0, 64, L)
        else:
            q = np.repeat(rng.integers(30, 41, L // 300 + 2), 300)[:L]      # runs of exactly 300: 255 + 45 or 45 + 255?
        txt = "".join("ACGT"[b] for b in s)
        if i % 3 == 0 and L > 4:
            txt = txt[:2] + "N" + txt[3:L - 1] + "N"
        if i % 4 == 1:
            txt = txt.lower().replace("n", "N")
        seqs.append(txt); quals.append(q.astype(np.uint8))
    return seqs, quals


def test_against_the_reference_binary_on_fresh_fastq(T, s1, tmp_path):
    """Runs the reference's own step 1, so it needs the reference built from its sources (W2RAP_REFERENCE at build time) and skips
    without it; test_golden_step1_files_byte_for_byte (files the reference wrote) and test_stores_feed_step2_formats ('N' and lower
    case on these kinds of reads) keep running."""
    if not os.path.exists(T.REF_BIN):
        pytest.skip("oracle/_ref/w2rap-contigger not built (needs the reference's sources: W2RAP_REFERENCE=<checkout> at build time)")
    seqs, quals = tricky_reads(5, 400)
    fq1, fq2 = write_fastq_pair(str(tmp_path), seqs, quals)
    ref = tmp_path / "ref"; ref.mkdir()
    subprocess.run([T.REF_BIN, "-t", "2", "-o", str(ref), "-p", "x", "-r", fq1 + "," + fq2, "--to_step", "1"], check=True, stdout=subprocess.DEVNULL)
    rc, err, p, r, st = ingest(T, s1, fq1, fq2, threads=4)
    assert rc == 0, err
    assert st.n_converted == sum(s.count("N") for s in seqs)
    mine = tmp_path / "mine"; mine.mkdir()
    err2 = C.create_string_buffer(512)
    assert s1.w2rap_step1_write_stores(str(mine).encode(), C.byref(r), err2, 512) == 0, err2.value
    s1.w2rap_step1_free(C.byref(p), C.byref(r))
    for f in ("frag_reads_orig.fastb", "frag_reads_orig.qualp"):
        assert open(str(mine / f), "rb").read() == open(str(ref / f), "rb").read(), f


def test_stores_feed_step2_formats(T, s1, tmp_path):
    """What the producer returns is what the step-2 entry points take: same arrays as reading the files it writes back."""
    seqs, quals = tricky_reads(9, 60)
    fq1, fq2 = write_fastq_pair(str(tmp_path), seqs, quals)
    rc, err, p, r, st = ingest(T, s1, fq1, fq2, threads=2)
    assert rc == 0, err
    n = int(r.n_reads)
    lens = T._arr(r.len, n, "<u4"); boff = T._arr(r.base_off, n + 1, "<u8"); qoff = T._arr(r.qual_off, n + 1, "<u8")
    assert list(lens) == [len(s) for s in seqs]
    bases = T._arr(r.bases, int(boff[-1]), "u1"); qs = T._arr(r.quals, int(qoff[-1]), "u1")
    err2 = C.create_string_buffer(512)
    assert s1.w2rap_step1_write_stores(str(tmp_path).encode(), C.byref(r), err2, 512) == 0
    s1.w2rap_step1_free(C.byref(p), C.byref(r))
    rs = T.read_fastb_qualp(str(tmp_path))
    assert np.array_equal(rs.len, lens) and np.array_equal(rs.base_off, boff) and np.array_equal(rs.qual_off, qoff)
    assert np.array_equal(rs.bases[:int(boff[-1])], bases) and np.array_equal(rs.quals[:int(qoff[-1])], qs)
    # decoded qualities and bases are the FASTQ's ('N' -> 'A', case folded)
    buf = np.zeros(70000, np.uint8)
    lib = T.oracle_lib()
    for i in range(n):
        m = lib.oracle_pq_decode(rs.quals.ctypes.data + int(rs.qual_off[i]), buf.ctypes.data)
        assert m == len(seqs[i]) and np.array_equal(buf[:m], quals[i])
        want = np.array(["ACGT".index(c) for c in seqs[i].upper().replace("N", "A")], np.uint8)
        assert np.array_equal(rs.read_codes(i), want)


def test_errors_the_reference_scrams_on(T, s1, tmp_path):
    seqs, quals = tricky_reads(3, 6)
    d = str(tmp_path)
    fq1, fq2 = write_fastq_pair(d, seqs, quals)

    def expect(code, text, a=fq1, b=fq2):
        rc, err, p, r, st = ingest(T, s1, a, b)
        assert rc == code and text in err, (rc, err)
        assert not r.bases and r.n_reads == 0
    expect(7, "cannot open", a=os.path.join(d, "missing.fastq"))
    short = os.path.join(d, "short.fastq")
    open(short, "w").write("".join(open(fq2).read().splitlines(True)[:-4]))
    expect(1, "different numbers of records", b=short)
    open(short, "w").write("".join(open(fq2).read().splitlines(True)[:-1]))
    expect(1, "incomplete record", b=short)
    bad = os.path.join(d, "bad.fastq")
    lines = open(fq2).read().splitlines(True)
    lines[3] = lines[3][:-2] + "\n"
    open(bad, "w").write("".join(lines))
    expect(1, "inconsistent base/quality lengths", b=bad)
    lines = open(fq2).read().splitlines(True)
    lines[1] = "R" + lines[1][1:]
    open(bad, "w").write("".join(lines))
    expect(1, "character 'R'", b=bad)
    lines = open(fq2).read().splitlines(True)
    lines[3] = chr(33 + 64) + lines[3][1:]
    open(bad, "w").write("".join(lines))
    expect(1, "quality score above 63", b=bad)


def test_empty_files(T, s1, tmp_path):
    a, b = str(tmp_path / "a.fastq"), str(tmp_path / "b.fastq")
    open(a, "w").close(); open(b, "w").close()
    rc, err, p, r, st = ingest(T, s1, a, b)
    assert rc == 0 and r.n_reads == 0 and st.n_pairs == 0
    s1.w2rap_step1_free(C.byref(p), C.byref(r))


def test_fastq_to_step_files_program(T, s1, tmp_path):
    """host/step12_main.cc: FASTQ pair -> frag_reads_orig.* (step 1) -> step 2 on the B200.  Here (no device) it must write the
    step-1 files, identical to the library's, and then stop loudly at step 2: there is no CPU path."""
    exe = os.path.join(ROOT, "w2rap-contigger_b200", "step12")
    if not os.path.exists(exe):
        pytest.skip("step12 not built (run __graft_entry__.build())")
    seqs, quals = golden_fastq(T, tmp_path)
    fq1, fq2 = write_fastq_pair(str(tmp_path), seqs, quals)
    out = tmp_path / "out"; out.mkdir()
    r = subprocess.run([exe, fq1, fq2, str(out), "x", "--stores-only"], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    for f in ("frag_reads_orig.fastb", "frag_reads_orig.qualp"):
        assert open(str(out / f), "rb").read() == open(os.path.join(HERE, "golden", "step1", f), "rb").read(), f
    if T.product_lib().w2rap_step2_device_count() == 0:
        r = subprocess.run([exe, fq1, fq2, str(out), "x"], capture_output=True, text=True)
        assert r.returncode == 1 and "step 2 failed (2)" in r.stderr and "no CPU path" in r.stderr, (r.returncode, r.stderr)
        assert not os.path.exists(str(out / "x.small_K.hbv"))
