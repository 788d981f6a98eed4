"""The host-buffer entry point with several read batches, against the oracle.

From 2^20 reads on, w2rap_step2_run uploads the reads as 8 batches and maps each batch as soon as it has landed, so every k-mer
partition is made of 8 record runs (one per batch), counted together by the multi-run branches of k_count_smem and k_count_region.
Smaller read sets are one batch.  The test hook W2RAP_UPLOAD_BATCHES=n splits any read set into n batches; the library reads it
once per process, so the hook cases run in child processes (batch_case_runner.py).  Every case compares every array with the
oracle bit for bit, from pageable and from pinned host memory, and checks that one scatter launch ran per non-empty batch and pass.
"""
import ctypes as C
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))


def run_child(mode, batches, timeout=900):
    e = dict(os.environ, W2RAP_UPLOAD_BATCHES=str(batches), PYTHONPATH=HERE)
    return subprocess.run([sys.executable, os.path.join(HERE, "batch_case_runner.py"), mode], env=e, capture_output=True, text=True, timeout=timeout)


@pytest.mark.parametrize("batches", [2, 3, 8, 16])
def test_batched_runs_match_the_oracle(batches):
    """A rich read set of 30-250-base reads (dump level 2, FixPaths) plain, in 2 forced passes and through the region fallback;
    at 8 batches also a 64-slot region (hash sub-range split with roll-back); reads whose counts and contexts only add up over
    the batches; batches without reads, of reads shorter than K and of reads below min_qual."""
    r = run_child("hook", batches)
    assert r.returncode == 0 and "FAIL" not in r.stdout, (r.stdout[-6000:], r.stderr[-3000:])
    assert r.stdout.count("OK ") == (9 if batches == 8 else 8), r.stdout


@pytest.mark.parametrize("value", ["0", "17", "eight"])
def test_out_of_range_batch_count_is_rejected(value):
    r = run_child("reject", value, timeout=300)
    assert r.returncode == 0, (r.stdout[-3000:], r.stderr[-3000:])
    assert "failed (1)" in r.stdout and "1..16" in r.stdout, r.stdout


def test_natural_batch_threshold(T):
    """No hook: 1,048,578 reads (2^20 + 2, so the 8 batches differ in size), resident (one batch) and through w2rap_step2_run from
    the pinned download and from a pageable copy (8 batches): every array equal at dump level 2; the pinned run also against the
    oracle."""
    lib = T.product_lib()
    err = C.create_string_buffer(512)
    sp = T.SynthParams(6_000_000, 150, 0, 17, 30, 0, 1_048_578, 0)
    h = C.c_void_p()
    assert lib.w2rap_step2_synth(C.byref(sp), -1, C.byref(h), err, 512) == 0, err.value
    r = T.Reads()
    assert lib.w2rap_step2_download_reads(h, C.byref(r), err, 512) == 0, err.value
    n = int(r.n_reads)
    assert n == 1_048_578
    try:
        def run(reads, resident, **kw):
            g = T.Graph()
            p = T.default_params(**kw)
            rc = lib.w2rap_step2_run_resident(h, C.byref(p), C.byref(g), err, 512) if resident else lib.w2rap_step2_run(C.byref(reads), C.byref(p), C.byref(g), err, 512)
            assert rc == 0, err.value
            d = T.graph_to_dict(g)
            lib.w2rap_step2_free(C.byref(g))
            return d
        res = run(None, True, dump_kmers=2)
        pinned = run(r, False, dump_kmers=2)
        boff, qoff = T._arr(r.base_off, n + 1, "<u8"), T._arr(r.qual_off, n + 1, "<u8")
        rs = T.ReadSet(T._arr(r.bases, int(boff[-1]), "u1"), boff, T._arr(r.len, n, "<u4"), T._arr(r.quals, int(qoff[-1]), "u1"), qoff)
        pageable = T.run_product(rs, T.default_params(dump_kmers=2))
        assert res["timings"]["count_launches"] == 1
        assert pinned["timings"]["count_launches"] == 8 and pageable["timings"]["count_launches"] == 8, (
            pinned["timings"]["count_launches"], pageable["timings"]["count_launches"])
        T.assert_graph_equal(res, pinned, "resident vs pinned host buffers")
        T.assert_graph_equal(res, pageable, "resident vs pageable host buffers")
        assert len(res["dump"]) == res["n_distinct"] > 0 and res["n_solid"] > 0
        got = run(r, False, apply_fixpaths=1, dump_kmers=1)
        want = T.run_oracle(rs, T.default_params(apply_fixpaths=1, dump_kmers=1))
        T.assert_graph_equal(want, got, "8 batches vs oracle")
        assert got["n_pathed"] > 0.9 * n
    finally:
        lib.w2rap_step2_free_host_reads(C.byref(r))
        lib.w2rap_step2_release(h)
