"""Independent validators of the step-2 products (SURVEY.md §8f N1/N3): the reference's own downstream reader `hbv2gfa`
(src/modules/hbv2gfa.cc: BinaryReader of the .hbv, hbv.Involution + TestInvolution, LoadReadPathVec, GFA dump with paths),
built unmodified into oracle/_ref/hbv2gfa, is run on the files this repo writes; and the involution the C ABI exports is
checked against its definition (paths/HyperBasevector.cc:648-660).

hbv2gfa is reference code run on files written during each test, so no stored output can stand in for it: the two tests skip unless
the reference was built from its sources (W2RAP_REFERENCE at build time).  The written formats are still parsed back and compared in
test_abi.py::test_host_format_writers_roundtrip and test_gpu_parity.py::test_resident_and_file_level_entry_points."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

HBV2GFA = None


def _hbv2gfa(T):
    exe = os.path.join(os.path.dirname(T.REF_BIN), "hbv2gfa")
    if not os.path.exists(exe):
        pytest.skip("oracle/_ref/hbv2gfa not built (needs the reference's sources: W2RAP_REFERENCE=<checkout> at build time)")
    return exe


def run_hbv2gfa(T, prefix_in, prefix_out, stats_only):
    r = subprocess.run([_hbv2gfa(T), "-i", prefix_in, "-o", prefix_out, "--stats_only", "1" if stats_only else "0"], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "Abort" not in r.stdout, r.stdout[-3000:] + r.stderr[-2000:]      # TestInvolution prints "Abort." and tracebacks on a bad graph
    size = [int(l.split(":")[1]) for l in r.stdout.splitlines() if l.startswith("Canonical graph sequences size")]
    assert size, r.stdout[-2000:]
    return size[0], r.stdout


def check_involution(T, d):
    """inv is an involution without fixed points other than palindromes, and edge inv[e] spells the reverse complement of edge e."""
    inv = d["involution"]
    assert len(inv) == d["n_hbv_edges"]
    assert np.array_equal(inv[inv], np.arange(len(inv)))
    seqs, _, _ = T.hbv_view(d)
    for e in range(len(inv)):
        assert T.revcomp(np.frombuffer(seqs[e], np.uint8)).tobytes() == seqs[int(inv[e])]


def test_oracle_involution_and_reference_reader_accept_written_files(T, tmp_path):
    """No GPU: the oracle's graph through the product's host-side format writers, read back and validated by the reference."""
    rs = T.rich_set(seed=4, genome=30000, cov=40, families=3, palindromes=3, plasmid=1200)
    g = T.Graph()
    p = T.default_params(apply_fixpaths=1)
    assert T.oracle_lib().oracle_step2_run(C.byref(rs.c()), C.byref(p), C.byref(g)) == 0
    d = T.graph_to_dict(g)
    check_involution(T, d)
    lib = T.product_lib()
    err = C.create_string_buffer(512)
    pre = str(tmp_path / "x.small_K")
    assert lib.w2rap_write_hbv((pre + ".hbv").encode(), C.byref(g), err, 512) == 0, err.value
    assert lib.w2rap_write_paths((pre + ".paths").encode(), C.byref(g), err, 512) == 0, err.value
    T.oracle_lib().oracle_step2_free(C.byref(g))
    size, _ = run_hbv2gfa(T, pre, str(tmp_path / "out"), stats_only=False)
    assert size == int(d["edge_len"].sum())                  # canonical (FWD or palindromic) sequences = our edge list
    assert os.path.getsize(str(tmp_path / "out") + ".gfa") > 0 if os.path.exists(str(tmp_path / "out") + ".gfa") else True


@pytest.mark.gpu
def test_reference_reader_accepts_step2_output(T, tmp_path):
    """The file-level drop-in's .hbv/.paths (w2rap_step2_run_files on the B200) through the reference's hbv2gfa."""
    lib = T.product_lib()
    rs = T.rich_set(seed=5, genome=60000, cov=40, families=4, palindromes=3, plasmid=1500)
    T.write_fastb_qualp(str(tmp_path), rs)
    err = C.create_string_buffer(512)
    g = T.Graph()
    assert lib.w2rap_step2_run_files(str(tmp_path).encode(), b"x", C.byref(T.default_params()), C.byref(g), err, 512) == 0, err.value
    d = T.graph_to_dict(g)
    lib.w2rap_step2_free(C.byref(g))
    check_involution(T, d)
    size, _ = run_hbv2gfa(T, str(tmp_path / "x.small_K"), str(tmp_path / "out"), stats_only=False)
    assert size == int(d["edge_len"].sum())
