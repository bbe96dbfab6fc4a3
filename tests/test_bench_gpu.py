"""-m gpu: bench.py --dump-outputs.  Two runs with the same arguments must dump the same arrays (same seeded inputs,
same sample positions), so that the dumps of two builds of the project can be compared output for output; one more
timed step must change them (the dump is the LAST timed step's, and --steps sets how many there are)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LOSSES = ("d_loss", "g_loss", "cat_loss", "cont_loss", "affine_loss", "relative_cat_loss", "total")


def _bench(out_dir, steps):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--config", "dsprites", "--steps", str(steps),
                        "--warmup", "3", "--no-parity", "--no-cpu-baseline", "--dump-outputs", str(out_dir)],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-3000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, r.stdout
    return json.loads(lines[0])


def test_dump_outputs_is_reproducible_and_follows_the_timed_steps(cuda, tmp_path):
    _bench(tmp_path / "a", 2)
    _bench(tmp_path / "b", 2)
    _bench(tmp_path / "c", 3)
    names = sorted(os.listdir(tmp_path / "a"))
    assert names == sorted(os.listdir(tmp_path / "b")) == sorted(os.listdir(tmp_path / "c"))
    assert {n + ".npy" for n in LOSSES} | {"G.conv_block.0.weight.npy", "D.conv_block.0.weight_orig.npy"} <= set(names)
    load = lambda run, n: np.load(tmp_path / run / n).astype(np.float64)
    total, rerun, one_more = 0, 0.0, 0.0
    for n in names:
        a, b, c = load("a", n), load("b", n), load("c", n)
        assert np.load(tmp_path / "a" / n).dtype in (np.float32, np.float64) and a.shape == b.shape == c.shape, n
        assert np.isfinite(a).all(), n
        total += np.load(tmp_path / "a" / n).nbytes
        if n[:-4] in LOSSES:
            assert abs(a - b).max() <= 1e-4 * max(1.0, abs(b).max()), n     # same arguments: same step
        else:
            rerun += np.abs(a - b).mean()
            one_more += np.abs(a - c).mean()
    for n in ("d_loss.npy", "g_loss.npy", "G.conv_block.0.weight.npy", "D.conv_block.0.weight_orig.npy"):
        assert (load("a", n) != load("c", n)).any(), n    # the third timed step's losses / Adam updates are in the dump
    # run to run the step differs only by the order of the fp64 atomics of the BatchNorm sums (and the bf16 roundings
    # that can flip); one Adam step moves the state by ~lr per element
    assert one_more > 0 and rerun <= 1e-2 * one_more, (rerun, one_more)
    assert total <= 64 << 20
