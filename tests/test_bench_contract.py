"""bench.py's reference arm runs on the CPU, so its half of the driver contract can be checked without a GPU: exactly one
JSON line on stdout, the keys the driver reads, and the synthetic image generators."""
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--batch", "4096", "--steps", "1",
                          "--warmup", "3"], cwd=ROOT, capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, out.stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["higher_is_better"] is True and d["unit"] == "images/s" and d["value"] > 0
    assert d["metric"].startswith("MNIST-16x16 images/sec") and d["config"]["workload"].startswith("fc:")
    assert d["e2e"] == {"value": d["value"], "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["cpu_baseline"]["kind"] in ("reference", "port") and d["cpu_baseline"]["cores"] >= 1 and d["gpu_launches"] == 0


def test_reference_arm_dumps_the_last_step(tmp_path):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--batch", "4096", "--steps", "2",
                          "--warmup", "3", "--dump-outputs", str(tmp_path)], cwd=ROOT, capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr[-2000:]
    n = json.loads(out.stdout)["config"]["sample_per_step"]
    sys.path.insert(0, ROOT)
    import bench
    from oracle.oracle import Oracle
    want_logits, want_labels = Oracle().infer(bench.load_model("fc"), bench.synth_images(4096, 256, 1234)[:n])
    logits, labels = np.load(tmp_path / "logits.npy"), np.load(tmp_path / "labels.npy")
    assert logits.dtype == labels.dtype == np.float32 and sorted(os.listdir(tmp_path)) == ["labels.npy", "logits.npy"]
    assert np.array_equal(logits, want_logits) and np.array_equal(labels, want_labels)


def test_dump_outputs_samples_rows_above_the_limit(tmp_path, monkeypatch):
    sys.path.insert(0, ROOT)
    import bench
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", 1000)
    logits = np.arange(4000, dtype=np.int32).reshape(400, 10) * 5000        # beyond 2**24: float64
    labels = np.arange(400, dtype=np.uint32)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), {"logits": logits, "labels": labels})
    got = {f: np.load(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a")}
    assert sorted(got) == ["labels.npy", "logits.npy", "rows.npy"] and sum(a.nbytes for a in got.values()) <= 1000
    rows = got["rows.npy"].astype(np.int64)
    assert got["logits.npy"].dtype == np.float64 and np.array_equal(got["logits.npy"], logits[rows])
    assert got["labels.npy"].dtype == np.float32 and np.array_equal(got["labels.npy"], labels[rows])
    assert np.array_equal(np.load(tmp_path / "b" / "rows.npy"), got["rows.npy"])   # the same sample every time


def test_reference_arm_other_ranks_stay_silent():
    env = dict(os.environ, RANK="1", LOCAL_RANK="1", WORLD_SIZE="2")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--batch", "4096",
                          "--steps", "1"], cwd=ROOT, env=env, capture_output=True, text=True, timeout=120)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_synthetic_image_generators():
    sys.path.insert(0, ROOT)
    import bench
    u = bench.synth_images(1000, 256, 7, "uniform")
    m = bench.synth_images(1000, 256, 7, "mnist")
    assert u.shape == m.shape == (1000, 256) and u.dtype == m.dtype == np.int8
    assert np.array_equal(u, bench.synth_images(1000, 256, 7, "uniform"))           # seeded
    assert abs(int(np.median(m)) + 20) <= 2 and m.max() == 127 and u.min() == -128   # background near -20, strokes to 127


def test_clock_sampler_selector_never_raises(monkeypatch):
    """ADVICE r1: CUDA_VISIBLE_DEVICES may hold UUIDs or be narrowed to one device per rank; the auxiliary clock sampler must cope."""
    sys.path.insert(0, ROOT)
    import bench
    monkeypatch.setenv("CUDA_VISIBLE_DEVICES", "GPU-3a4b5c6d-0000-1111-2222-333344445555,GPU-deadbeef-0000-1111-2222-333344445555")
    assert bench.ClockSampler.device_selector(1).startswith("GPU-deadbeef")
    monkeypatch.setenv("CUDA_VISIBLE_DEVICES", "5")
    assert bench.ClockSampler.device_selector(3) == "5"            # narrowed list: fall back to its only entry
    monkeypatch.setenv("CUDA_VISIBLE_DEVICES", "2,3")
    assert bench.ClockSampler.device_selector(1) == "3"
    s = bench.ClockSampler("GPU-not-a-real-uuid")
    s.start()
    out = s.stop(0.0, 1.0, "test")                                  # no nvidia-smi / bad selector: a dict, not an exception
    assert isinstance(out, dict) and "reasons" in out


def test_epilogue_alu_bound_and_int_alu_peak():
    sys.path.insert(0, ROOT)
    import bench
    from bitnetmcu_b200.model import Model
    fc = Model.load(os.path.join(ROOT, "tests", "golden", "models", "fc.bnm"))
    b160 = Model.load(os.path.join(ROOT, "tests", "golden", "models", "binary160.bnm"))
    a, b = bench.epilogue_alu_bound(fc, 1965.0), bench.epilogue_alu_bound(b160, 1965.0)
    assert a["hidden_accumulators_per_image"] == 192 and b["hidden_accumulators_per_image"] == 480
    assert abs(a["images_per_s"] / b["images_per_s"] - 480 / 192) < 1e-9 and 3.5e10 < a["images_per_s"] < 4.5e10
    assert abs(bench.int_alu_peak_ops(1965.0) - 148 * 64 * 8 * 1965e6) < 1
