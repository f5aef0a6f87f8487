"""bench.py --dump-outputs: float32 arrays within the size budget, the same values at the same positions in every run."""
import os
import subprocess
import sys

import numpy as np

import bench
from conftest import ROOT


class _Calc:
    """The two calls dump_outputs makes, on fixed data.  A 1280x960 P010 output frame holds more values than one array of a
    dump may (it is sampled); the 640x480 flow does not (it is stored whole)."""
    W, H, LW, LH = 1280, 960, 640, 480
    outputFrameBytes = W * H * 3 // 2 * 2

    def __init__(self):
        self.k = 0

    def downloadFrame(self, a):
        a[:] = (np.arange(a.size, dtype=np.int64) * (2 * self.k + 1)) % 65536
        self.k += 1

    def readFlow(self, latest=False):
        assert latest, "the dump holds the flow the step computed, not the one its warps read"
        return (np.arange(2 * self.LH * self.LW) % 301 - 150).astype(np.int16).reshape(2, self.LH, self.LW)


def test_dump_outputs_are_float32_within_the_budget_and_repeatable(tmp_path):
    blends = [0.1, 0.25, 0.4, 0.55, 0.7, 0.85, 0.95]
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), _Calc(), blends, True)
    names = sorted(p.name for p in (tmp_path / "a").iterdir())
    assert names == ["flow.npy"] + [f"output{k}.npy" for k in range(len(blends))]
    assert sum(p.stat().st_size for p in (tmp_path / "a").iterdir()) <= bench.DUMP_BYTES
    for name in names:
        a, b = np.load(tmp_path / "a" / name), np.load(tmp_path / "b" / name)
        assert a.dtype == np.float32 and np.array_equal(a, b), name
    assert np.array_equal(np.load(tmp_path / "a" / "flow.npy"), _Calc().readFlow(latest=True).reshape(-1))
    out = np.load(tmp_path / "a" / "output3.npy")
    assert out.size == bench.DUMP_SAMPLES < _Calc.outputFrameBytes // 2
    assert not np.array_equal(out, np.load(tmp_path / "a" / "output2.npy")), "every output frame is its own array"


def test_dump_outputs_is_refused_outside_the_single_stream_cuda_path(tmp_path):
    for extra in (["--impl", "reference"], ["--workload", "cfg4"], ["--streams-per-gpu", "2"]):
        res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--dump-outputs", str(tmp_path)] + extra,
                             capture_output=True, text=True, timeout=120, cwd=ROOT)
        assert res.returncode == 2 and "--dump-outputs" in res.stderr, extra
    assert not any(tmp_path.iterdir())
