"""GPU: `bench.py --dump-outputs` writes what the LAST timed step computed (every view's image, the loss, the parameter
gradients) as float32 .npy files.  The dump of a bench process is compared with a replay in this process: the same
workload, the same seed and noise-call counter, `--steps` steps.  Images and loss agree within 1e-6, gradients within
1e-4 of their largest entry (the backward's atomic additions land in any order); the step before the last renders
different images (the plane-feature noise changes every step), so a dump of any other step would not match."""
import json
import os
import subprocess
import sys
from types import SimpleNamespace

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
STEPS = 3


def _bench_dump(d):
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "c1", "--steps", str(STEPS), "--warmup", "1",
                        "--no-cpu", "--no-gpu-baseline", "--dump-outputs", d], capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [l for l in p.stdout.strip().splitlines() if l.startswith("{")]
    assert len(lines) == 1 and json.loads(lines[0])["steps"] == STEPS
    return {f[:-len(".npy")]: np.load(os.path.join(d, f)) for f in os.listdir(d)}


def _replay():
    """Outputs after STEPS - 1 and after STEPS timed steps, started the way bench.run_ours starts its timed loop."""
    import bench
    from splatco_b200 import decode
    w = bench.Workload(SimpleNamespace(torch_scaling_reg=False), "c1", torch.device("cuda", 0), 0, 1)
    w.keep_outputs = True
    prev_calls = decode._noise_calls
    try:
        with torch.random.fork_rng(devices=[0]):
            torch.manual_seed(0)
            decode._noise_calls = 0
            outs = []
            for _ in range(STEPS):
                w.step(False)
                outs.append(w.outputs())
    finally:
        decode._noise_calls = prev_calls
    return outs[-2], outs[-1]


def test_dump_outputs_are_the_last_timed_step(tmp_path):
    got = _bench_dump(str(tmp_path / "dump"))
    before_last, want = _replay()
    assert sorted(got) == sorted(want)
    assert {"loss", "render_view0", "grad._anchor", "grad.mlp_opacity.0.weight"} <= set(got)
    assert sum(v.nbytes for v in got.values()) <= 64 << 20
    assert got["render_view0"].shape == (3, 256, 256) and got["loss"].shape == () and float(got["loss"]) > 0
    for k in got:
        a, b = got[k], want[k]
        assert a.dtype == np.float32 and a.shape == b.shape and np.isfinite(a).all(), k
        if k.startswith("grad."):
            assert np.abs(a - b).max() <= 1e-4 * np.abs(b).max() + 1e-12, k
        else:
            assert np.abs(a - b).max() <= 1e-6 * max(np.abs(b).max(), 1.0), k
    assert np.abs(before_last["render_view0"] - want["render_view0"]).max() > 1e-5
