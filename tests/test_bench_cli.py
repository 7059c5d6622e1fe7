"""CPU: bench.py's command line - the step counts are validated and --dump-outputs writes float32 / float64 .npy files
within its size limit."""
import os
import sys

import numpy as np
import pytest
import torch

import bench


@pytest.mark.parametrize("argv", [["--steps", "0"], ["--warmup", "-1"], ["--steps", "1.5"],
                                  ["--impl", "reference", "--dump-outputs", "out"]])
def test_bench_rejects_bad_arguments(monkeypatch, argv):
    monkeypatch.setattr(sys, "argv", ["bench.py", *argv])
    with pytest.raises(SystemExit) as e:
        bench.parse_args()
    assert e.value.code == 2


def test_bench_steps_and_dump_dir_are_taken_as_given(monkeypatch):
    monkeypatch.setattr(sys, "argv", ["bench.py", "--gpus", "1", "--steps", "7", "--warmup", "0", "--dump-outputs", "d"])
    args = bench.parse_args()
    assert (args.steps, args.warmup, args.dump_outputs) == (7, 0, "d")


def test_dump_outputs_dtypes_names_and_limit(tmp_path, monkeypatch):
    half = torch.arange(6, dtype=torch.float16).reshape(3, 2)
    bench.dump_outputs(str(tmp_path / "d"), {"logits": half, "x": torch.full((2,), 0.1, dtype=torch.float64)}, "_rank1")
    a = np.load(tmp_path / "d" / "logits_rank1.npy")
    assert a.dtype == np.float32 and np.array_equal(a, half.float().numpy())
    b = np.load(tmp_path / "d" / "x_rank1.npy")
    assert b.dtype == np.float64 and b[0] == 0.1
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", 16)
    with pytest.raises(ValueError, match="limit"):
        bench.dump_outputs(str(tmp_path / "big"), {"logits": torch.zeros(5)})
    assert not os.path.exists(tmp_path / "big")
