"""bench.py --dump-outputs: what the last timed training step computed, written as float32 .npy files, is the same on
every run with the same arguments (seeded inputs and initialisation, fixed-order reductions), so that two builds of the
project can be compared output for output."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench(out_dir, steps):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup", "3",
                        "--batch", "4", "--no-cpu-baseline", "--no-profile", "--no-predict", "--no-extra",
                        "--dump-outputs", str(out_dir)], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-3000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    arrays = {f[:-4]: np.load(out_dir / f) for f in sorted(os.listdir(out_dir))}
    return line, arrays


def test_dump_outputs_is_reproducible(tmp_path):
    line, a = _bench(tmp_path / "a", 2)
    assert line["steps"] == 2
    assert sorted(a) == ["grads_sample", "logits", "loss", "params_sample"]
    assert all(v.dtype == np.float32 and np.isfinite(v).all() for v in a.values())
    assert sum(v.nbytes for v in a.values()) <= 64 << 20
    assert a["logits"].shape == (4, 2, 256, 256)
    assert a["loss"][0] == np.float32(line["final_loss"])
    _, b = _bench(tmp_path / "b", 2)
    for k in a:
        assert np.array_equal(a[k], b[k]), k
    # one more timed step is one more update: the dumped step is the last timed one
    _, c = _bench(tmp_path / "c", 3)
    assert not np.array_equal(a["params_sample"], c["params_sample"])
