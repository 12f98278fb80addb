"""GPU tier: `bench.py --dump-outputs` writes the change set of the last timed step; with the same arguments the inputs are the
same, so two runs (different step counts) dump identical files, equal to the oracle's change set of that workload."""
import importlib
import json
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
REPO = Path(__file__).resolve().parent.parent
N = 20_000


def _bench(out_dir, steps):
    out = subprocess.run([sys.executable, str(REPO / "bench.py"), "--objects", str(N), "--steps", str(steps), "--warmup", "1", "--no-cpu-baseline",
                          "--dump-outputs", str(out_dir)], capture_output=True, text=True, timeout=900, cwd=str(REPO))
    assert out.returncode == 0, out.stderr[-3000:]
    line = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])
    assert line["steps"] == steps and line["parity"]["equal"] is True
    return line


def test_dump_outputs_repeat_and_equal_the_oracle(garecon, oracle, tmp_path):
    _bench(tmp_path / "a", 2)
    _bench(tmp_path / "b", 3)
    import __graft_entry__ as ge
    ge.build_synth()
    synth = importlib.import_module("aws-global-accelerator-controller_b200.synth")
    bench = importlib.import_module("bench")
    cfg = synth.preset(3, N)
    cfg.layout = 1
    snap = synth.SynthSnapshot(cfg)
    names = bench.dump_outputs(oracle.diff(snap, snap.cluster, mode=1), tmp_path / "want")
    for k in names:
        want = np.load(tmp_path / "want" / f"{k}.npy")
        for d in ("a", "b"):
            got = np.load(tmp_path / d / f"{k}.npy")
            assert got.dtype == np.float64 and np.array_equal(got, want), (d, k)
    assert sum((tmp_path / "a" / f"{k}.npy").stat().st_size for k in names) <= 64 << 20
