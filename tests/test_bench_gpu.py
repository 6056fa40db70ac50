"""GPU: `bench.py --dump-outputs DIR` writes what the last timed step computed (loss, grad norm, a seeded sample of the
updated trainable parameters and of AdamW's first moment) as float32 / float64 .npy files of bounded size; the dumped
loss is the step's loss the JSON line reports, and two runs with the same arguments write the same bits.  A batch of 2
keeps it short."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FILES = ["adam_exp_avg.npy", "grad_norm.npy", "loss.npy", "sample_index.npy", "trainable_params.npy"]


def _bench_dump(out):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "3", "--batch", "2",
                        "--no-cpu-baseline", "--dump-outputs", out], cwd=ROOT, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-3000:]
    line = json.loads([l for l in r.stdout.splitlines() if l.lstrip().startswith("{")][-1])
    assert sorted(os.listdir(out)) == FILES, os.listdir(out)
    assert sum(os.path.getsize(os.path.join(out, f)) for f in FILES) <= 64 << 20
    return line, {f[:-4]: np.load(os.path.join(out, f)) for f in FILES}


def test_dump_outputs_writes_the_last_timed_step(cuda, tmp_path):
    line, a = _bench_dump(str(tmp_path / "run1"))
    assert line["steps"] == 2
    assert all(v.dtype in (np.float32, np.float64) for v in a.values())
    assert np.isfinite(a["loss"]).all() and a["loss"][0] == np.float32(line["final_loss"])
    assert a["grad_norm"][0] > 0
    idx = a["sample_index"]
    assert idx.shape == a["trainable_params"].shape == a["adam_exp_avg"].shape and (np.diff(idx) >= 0).all()
    assert np.isfinite(a["trainable_params"]).all() and np.abs(a["adam_exp_avg"]).max() > 0
    # a second run with the same arguments: same inputs, fixed-order reductions -> the same bits
    _, b = _bench_dump(str(tmp_path / "run2"))
    for k in a:
        assert np.array_equal(a[k], b[k]), (k, np.abs(a[k].astype(np.float64) - b[k]).max())
