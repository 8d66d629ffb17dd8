"""CPU: the reference arm of bench.py (`--impl reference`: the oracle port on the host cores) prints one JSON line with
the keys the measurement contract names, on the reference's own CPU-runnable configuration (BASELINE configs[0])."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_json_line():
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "c1", "--steps", "1",
                        "--warmup", "0"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [l for l in p.stdout.strip().splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "fwd_bwd_ms_per_view" and d["unit"] == "ms/view"
    assert d["higher_is_better"] is False and d["vs_baseline"] is None and d["value"] > 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "ms/view", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and "model" not in d["config"]


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2")
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "c1", "--steps", "1",
                        "--warmup", "0", "--gpus", "2"], capture_output=True, text=True, timeout=600, cwd=ROOT, env=env)
    assert p.returncode == 0 and p.stdout.strip() == ""


def test_dump_outputs_samples_large_arrays_at_fixed_positions(tmp_path):
    """--dump-outputs: small arrays are written whole, a large one as the same seeded sample in every call, all float32;
    a dump over the size limit writes no file."""
    import numpy as np
    import pytest
    sys.path.insert(0, ROOT)
    import bench
    big = np.arange(3 * bench.DUMP_MAX_ELEMS, dtype=np.float32).reshape(3, -1)
    arrays = {"loss": np.array(2.5, np.float32), "grad.small": np.ones((4, 3), np.float64), "render_view0": big}
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), {k: bench.dump_sample(v) for k, v in arrays.items()})
    too_big = {f"render_view{v}": big for v in range(bench.DUMP_MAX_BYTES // big.nbytes + 1)}
    with pytest.raises(RuntimeError):
        bench.dump_outputs(str(tmp_path / "c"), too_big)
    assert not (tmp_path / "c").exists()
    a = {f: np.load(str(tmp_path / "a" / f)) for f in os.listdir(str(tmp_path / "a"))}
    assert sorted(a) == ["grad.small.npy", "loss.npy", "render_view0.npy"]
    assert all(v.dtype == np.float32 for v in a.values())
    assert a["loss.npy"].shape == () and a["grad.small.npy"].shape == (4, 3)
    s = a["render_view0.npy"]
    assert s.shape == (bench.DUMP_MAX_ELEMS,) and np.all(np.diff(s) > 0) and np.isin(s, big).all()
    assert np.array_equal(s, np.load(str(tmp_path / "b" / "render_view0.npy")))


def test_committed_evidence_is_readable_by_the_bench():
    """The roofline object takes `traffic` and the issue-slot numbers from the newest committed ncu capture and `peak` from
    MEASURED_PEAKS.json: both helpers must parse what is in the tree (a malformed file would only show up on the GPU box)."""
    sys.path.insert(0, ROOT)
    import bench
    ev = bench.ncu_evidence()
    assert ev["_file"].startswith("profiles/r2") and ev["_file"].endswith("_traffic.json")
    tags = sorted((f for f in os.listdir(os.path.join(ROOT, "profiles")) if f.endswith("_traffic.json")), key=lambda f: (len(f), f))
    assert ev["_file"] == "profiles/" + tags[-1]
    kernels = {k: v for k, v in ev.items() if isinstance(v, dict)}
    for name in ("blend_bwd", "blend_fwd"):          # names as tools/collect_profiles.py normalises them
        hit = [v for k, v in kernels.items() if name in k]
        assert hit, f"{name} missing from {ev['_file']}"
        assert hit[0]["dram_bytes"] > 0 and 0 < hit[0]["issue_active_pct"] <= 100
    peak, src = bench.peaks()
    assert src in ("measured", "fallback") and 3000 < peak < 9000
