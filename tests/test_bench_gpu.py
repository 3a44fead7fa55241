"""bench.py's GPU arm with --dump-outputs: what the last timed step returned is written as .npy files, and the same
arguments give the same outputs whatever the number of timed steps."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from bitswap_b200 import synthetic
from bitswap_b200.config import preset

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NAMES = ("base", "heads", "lengths", "pixels", "streams", "words")


def _bench(out, steps):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup", "1",
                        "--batch", "48", "--lanes", "2", "--no-cpu-baseline", "--dump-outputs", str(out)],
                       stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["steps"] == steps and line["roundtrip_ok"]
    return {n: np.load(os.path.join(out, n + ".npy")) for n in NAMES}


def test_dump_outputs_are_the_coded_batch_and_do_not_depend_on_steps(tmp_path):
    a = _bench(tmp_path / "a", 1)
    b = _bench(tmp_path / "b", 3)
    assert sorted(os.listdir(tmp_path / "a")) == sorted(n + ".npy" for n in NAMES)
    for n in NAMES:
        assert a[n].dtype in (np.float32, np.float64), n
        assert np.array_equal(a[n], b[n]), n
    assert sum(os.path.getsize(tmp_path / "a" / (n + ".npy")) for n in NAMES) <= 64 << 20
    cfg = preset("cifar8")
    assert np.array_equal(a["streams"], np.arange(48))
    assert np.array_equal(a["pixels"], synthetic.synthetic_images(cfg, 48, seed=7).astype(np.float32))
    assert a["lengths"].sum() == a["words"].size and (a["lengths"] > 0).all()
    assert (a["words"] == np.floor(a["words"])).all() and a["words"].min() >= 0 and a["words"].max() < 2 ** 32
    assert a["heads"].shape == (48, 2) and (a["heads"][:, 1] >= 1).all() and a["heads"].max() < 2 ** 32   # 2^32 <= head < 2^64
