"""bench.py --dump-outputs (CPU): the dumped float64 words are the output bytes exactly, at the same seeded rows on
every run, under 64 MB; and the step counts that would leave no timed step are refused before any GPU work."""
import importlib.util
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench():
    spec = importlib.util.spec_from_file_location("bench", os.path.join(ROOT, "bench.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def test_dump_outputs_round_trips_the_output_bytes(tmp_path):
    bench = _bench()
    n = bench.BATCH
    out = np.random.Generator(np.random.PCG64(7)).integers(0, 256, size=576 * n, dtype=np.uint8)
    out[::48] = 0xff                                  # top words above 2^31: no sign or rounding slip
    bench.dump_outputs(str(tmp_path / "a"), out)
    bench.dump_outputs(str(tmp_path / "b"), out)
    names = sorted(os.listdir(tmp_path / "a"))
    assert names == ["pairing_rows.npy", "pairings.npy"]
    assert sum(os.path.getsize(tmp_path / "a" / nm) for nm in names) <= 64 * 2 ** 20
    words = np.load(tmp_path / "a" / "pairings.npy")
    rows = np.load(tmp_path / "a" / "pairing_rows.npy")
    assert words.dtype == np.float64 and rows.dtype == np.float64
    assert words.shape == (bench.DUMP_ROWS, 12, 12) and rows.shape == (bench.DUMP_ROWS,)
    r = rows.astype(np.int64)
    assert np.all(np.diff(r) > 0) and r[0] >= 0 and r[-1] < n
    back = np.ascontiguousarray(words.astype(">u4")).view(np.uint8).reshape(len(r), 576)
    assert np.array_equal(back, out.reshape(n, 576)[r])
    for nm in names:
        assert np.array_equal(np.load(tmp_path / "a" / nm), np.load(tmp_path / "b" / nm))


def test_bench_refuses_an_empty_timed_window():
    for argv in (["--steps", "0"], ["--warmup", "-1"]):
        res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + argv, capture_output=True, text=True)
        assert res.returncode == 2 and "--steps must be at least 1" in res.stderr
