"""CPU: bench.py's command line and the file --dump-outputs writes."""
import os
import subprocess
import sys

import numpy as np
import pytest

import bench

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dump_outputs_writes_the_token_ids_as_float32(tmp_path):
    toks = {u: [(u * 1000 + j) * 31 % 128256 for j in range(bench.GEN_LEN)] for u in range(bench.USERS)}
    bench.dump_outputs(str(tmp_path / "out"), toks)
    got = np.load(tmp_path / "out" / "tokens.npy")
    assert got.dtype == np.float32 and got.shape == (bench.USERS, bench.GEN_LEN)
    assert got.astype(np.int64).tolist() == [toks[u] for u in range(bench.USERS)]


def test_dump_outputs_refuses_a_short_stream(tmp_path):
    toks = {u: [1] * bench.GEN_LEN for u in range(bench.USERS)}
    toks[5] = toks[5][:-1]
    with pytest.raises((RuntimeError, ValueError)):
        bench.dump_outputs(str(tmp_path), toks)
    assert not (tmp_path / "tokens.npy").exists()


@pytest.mark.parametrize("argv", [["--steps", "0"], ["--warmup", "-1"], ["--impl", "reference", "--dump-outputs", "x"]])
def test_bench_rejects_bad_arguments(argv):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + argv, capture_output=True, text=True, timeout=120)
    assert r.returncode == 2 and "error:" in r.stderr
