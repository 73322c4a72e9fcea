"""bench.py's command line and output dump, without a GPU."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import bench

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dump_outputs_writes_float32_npy_with_exact_ids(tmp_path):
    ids = torch.randint(0, 21178, (2, 5, 4), dtype=torch.int32)
    wav = torch.randn(2, 300)
    bench.dump_outputs(str(tmp_path / "out"), {"ids": ids, "wav": wav})
    a, w = np.load(tmp_path / "out" / "ids.npy"), np.load(tmp_path / "out" / "wav.npy")
    assert a.dtype == w.dtype == np.float32 and np.array_equal(a, ids.numpy()) and np.array_equal(w, wav.numpy())


def test_dump_outputs_refuses_more_than_the_limit(tmp_path):
    with pytest.raises(ValueError):
        bench.dump_outputs(str(tmp_path / "out"), {"x": torch.zeros(bench.DUMP_LIMIT_BYTES // 4 + 1)})
    assert not (tmp_path / "out").exists()


@pytest.mark.parametrize("argv", [["--steps", "0"], ["--impl", "reference", "--dump-outputs", "x"]])
def test_bad_arguments_are_rejected_before_any_work(argv):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *argv], capture_output=True, text=True, timeout=300)
    assert r.returncode == 2 and "error:" in r.stderr
