"""bench.py --dump-outputs: what the timed entry point returned, written as float64 .npy files that two builds can compare."""
import importlib.util
import os

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def load_bench():
    spec = importlib.util.spec_from_file_location("bench", os.path.join(ROOT, "bench.py"))
    B = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(B)
    return B


def test_dump_outputs_exact_sampled_and_bounded(T, tmp_path):
    B = load_bench()
    d = T.run_oracle(T.rich_set(seed=33, genome=60000, cov=40), T.default_params(apply_fixpaths=1, places_K2=200))
    assert d["n_places"] > 0
    B.dump_outputs(d, str(tmp_path / "a"))
    for name in B.DUMP_ARRAYS:
        a = np.load(str(tmp_path / "a" / (name + ".npy")))
        want = np.asarray(d[name]).reshape(-1)
        assert a.dtype == np.float64 and np.array_equal(a.astype(want.dtype), want), name
    c = np.load(str(tmp_path / "a" / "counts.npy"))
    assert [int(x) for x in c[:len(B.DUMP_COUNTS)]] == [d[k] for k in B.DUMP_COUNTS]
    assert (int(c[-4]) << 32 | int(c[-3]), int(c[-2]) << 32 | int(c[-1])) == (d["digest_graph"], d["digest_paths"])
    # without places the step fills no place arrays: none is written, and no file is empty
    B.dump_outputs(dict(d, place_off=d["place_off"][:0], place_edges=d["place_edges"][:0]), str(tmp_path / "n"))
    names = sorted(os.listdir(str(tmp_path / "n")))
    assert names == sorted(["counts.npy"] + [n + ".npy" for n in B.DUMP_ARRAYS if not n.startswith("place_")])
    assert all(np.load(str(tmp_path / "n" / f)).size > 0 for f in names)
    # an array longer than the cap: the same seeded positions in every run, in order
    big = dict(d, path_edges=np.arange(3 * B.DUMP_CAP, dtype=np.int32))
    for sub in ("b", "c"):
        B.dump_outputs(big, str(tmp_path / sub))
    pe = np.load(str(tmp_path / "b" / "path_edges.npy"))
    assert len(pe) == B.DUMP_CAP and (np.diff(pe) > 0).all()
    assert np.array_equal(pe, np.load(str(tmp_path / "c" / "path_edges.npy")))
    # every array at the cap, plus the counters, stays under 64 MB
    assert (len(B.DUMP_ARRAYS) * B.DUMP_CAP + len(B.DUMP_COUNTS) + 4) * 8 < 64e6


@pytest.mark.gpu
def test_bench_dumps_what_the_timed_entry_point_returns(T, tmp_path):
    """bench.py itself on a small workload: --steps sets the number of timed steps, and --dump-outputs writes what
    w2rap_step2_run_resident returns for the same seeded reads and parameters."""
    import ctypes as C
    import json
    import subprocess
    import sys
    B = load_bench()
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--genome-mbp", "2", "--coverage", "20", "--steps", "2", "--warmup", "0",
                        "--no-cpu-baseline", "--no-e2e", "--dump-outputs", str(tmp_path / "bench")], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    line = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
    assert line["steps"] == 2 and len(line["per_step"]["resident_ms"]) == 2
    lib = T.product_lib()
    err = C.create_string_buffer(512)
    sp = T.SynthParams(2_000_000, 250, 20, 1000, 0, 0, 160_000, 0)        # bench.py's read set for these arguments
    h = C.c_void_p()
    assert lib.w2rap_step2_synth(C.byref(sp), -1, C.byref(h), err, 512) == 0, err.value
    g = T.Graph()
    assert lib.w2rap_step2_run_resident(h, C.byref(T.default_params(apply_fixpaths=1)), C.byref(g), err, 512) == 0, err.value
    d = T.graph_to_dict(g)
    lib.w2rap_step2_free(C.byref(g))
    lib.w2rap_step2_release(h)
    B.dump_outputs(d, str(tmp_path / "direct"))
    names = sorted(os.listdir(str(tmp_path / "direct")))
    assert sorted(os.listdir(str(tmp_path / "bench"))) == names and "path_edges.npy" in names
    for f in names:
        assert np.array_equal(np.load(str(tmp_path / "bench" / f)), np.load(str(tmp_path / "direct" / f))), f
