"""bench.py's command line: --steps is the number of timed steps, and --dump-outputs writes what the last timed step
computed, on inputs that are the same from run to run."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BENCH = os.path.join(ROOT, "bench.py")


def _bench(*argv, env=None):
    return subprocess.run([sys.executable, BENCH, *argv], capture_output=True, text=True, timeout=600,
                          env={**os.environ, **(env or {})})


@pytest.mark.parametrize("argv", [["--steps", "0"], ["--impl", "reference", "--dump-outputs", "out"]])
def test_bench_rejects_arguments_it_cannot_honour(argv):
    out = _bench(*argv, env={"CUDA_VISIBLE_DEVICES": ""})
    assert out.returncode == 2 and "error:" in out.stderr, out.stderr[-500:]


@pytest.mark.gpu
def test_bench_dump_is_the_timed_output_and_steps_are_timed(tmp_path):
    import torch

    import bench
    import mevi_b200

    n = 100003
    lines = {}
    for steps in (1, 3):
        out = _bench("--docs", str(n), "--steps", str(steps), "--warmup", "1", "--no-extras", "--no-cpu-baseline",
                     "--dump-outputs", str(tmp_path / f"s{steps}"))
        assert out.returncode == 0, out.stderr[-2000:]
        lines[steps] = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])
        assert lines[steps]["steps"] == steps
    assert lines[1]["gpu_launches"] > 0 and lines[3]["gpu_launches"] == 3 * lines[1]["gpu_launches"]
    codes = np.load(tmp_path / "s3" / "codes.npy")
    rows = np.load(tmp_path / "s3" / "codes_rows.npy")
    assert codes.dtype == np.float32 and codes.shape == (n, bench.M_LEVELS)
    assert rows.dtype == np.float64 and np.array_equal(rows, np.arange(n))
    assert np.array_equal(np.load(tmp_path / "s1" / "codes.npy"), codes)
    # the same corpus and codebook regenerated here give the same codes
    X = bench.make_corpus(n, bench.D, torch.device("cuda", 0), 1234)
    want = mevi_b200.get_context(0).rq_encode(X, bench.load_codebook().cuda(0), mode="auto").cpu().numpy()
    assert np.array_equal(codes, want.astype(np.float32))
    assert int(want.astype(np.int64).sum()) == lines[3]["codes_checksum"]
