"""The bench.py contract: the reference arm's JSON line and the refusal without a GPU on the CPU; the b200 arm's
--dump-outputs on the GPU."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_json_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1",
                          "--ref-blocks", "16"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1, "exactly one JSON line"
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "encode+decode Mpixel/s" and d["unit"] == "Mpixel/s"
    assert d["n_gpus"] == 1 and d["steps"] == 1 and d["warmup"] == 1 and d["higher_is_better"] is True
    assert d["value"] > 0 and d["ms_per_step"] > 0 and d["vs_baseline"] is None and d["scaling"] == "weak"
    assert d["e2e"] == {"value": d["value"], "unit": "Mpixel/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and "blocks" in cb["sample"]
    assert "workload" in d["config"] and "model" not in d["config"]


def test_b200_arm_fails_loudly_without_gpu():
    # the child sees no GPU, so this also runs on a machine that has one
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "1"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT,
                         env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))
    assert out.returncode != 0, "the product arm must not fall back to the CPU"
    assert not [l for l in out.stdout.splitlines() if l.startswith('{"metric"')]


def test_dump_outputs_sample_is_fixed_and_within_budget(tmp_path):
    """bench.dump_outputs on host tensors larger than its sample: float32 / float64 arrays, 64 MB at most, the same
    positions in every run, stream bytes taken from inside each stream."""
    import torch
    import bench
    g = torch.Generator().manual_seed(0)
    zhat = torch.rand(3, 192, 90, 96, generator=g)                   # 5 M values > bench.DUMP_ELEMENTS
    lens = torch.tensor([8, 4096, 1000], dtype=torch.int32)
    streams = torch.randint(0, 256, (3, 4096), dtype=torch.uint8, generator=g)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), zhat, lens, streams, zhat.clone())
    names = sorted(os.listdir(tmp_path / "a"))
    assert names == ["lens.npy", "streams.npy", "zdec.npy", "zhat.npy"]
    got = {n[:-4]: np.load(tmp_path / "a" / n) for n in names}
    for n, a in got.items():
        assert a.dtype in (np.float32, np.float64) and np.array_equal(a, np.load(tmp_path / "b" / f"{n}.npy"))
    assert sum(a.nbytes for a in got.values()) <= 64 << 20
    assert got["zhat"].size == bench.DUMP_ELEMENTS
    assert np.array_equal(got["zhat"], got["zdec"]) and np.isin(got["zhat"], zhat.numpy()).all()
    assert np.array_equal(got["lens"], [8, 4096, 1000])
    s = got["streams"]
    assert s.shape == (3, 2048)
    for i, n in enumerate((8, 4096, 1000)):
        assert np.isin(s[i], streams[i, :n].numpy()).all()
    assert set(s[0]) == set(streams[0, :8].tolist())                 # every byte of a short stream


@pytest.mark.gpu
def test_dump_outputs_of_the_b200_arm(tmp_path):
    """--dump-outputs: the last timed step's reconstructions and streams, identical in two runs with the same arguments;
    --warmup 0 is allowed and --steps is what the JSON line reports."""
    args = [sys.executable, os.path.join(ROOT, "bench.py"), "--images", "3", "--height", "64", "--width", "96",
            "--warmup", "0", "--no-cpu-baseline", "--no-e2e", "--no-reference-container", "--no-single-image"]
    got = []
    for run, steps in (("a", 2), ("b", 1)):
        out = subprocess.run(args + ["--steps", str(steps), "--dump-outputs", str(tmp_path / run)],
                             capture_output=True, text=True, timeout=900, cwd=ROOT)
        assert out.returncode == 0, out.stderr[-3000:]
        line = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])
        assert line["steps"] == steps and line["enc_dec_identical"] is True
        got.append({n[:-4]: np.load(tmp_path / run / n) for n in os.listdir(tmp_path / run)})
    a, b = got
    assert sorted(a) == ["lens", "streams", "zdec", "zhat"]
    assert a["zhat"].size == 3 * 192 * 8 * 12 and np.array_equal(a["zhat"], a["zdec"])
    assert a["lens"].shape == (3,) and (a["lens"] > 8).all()
    for n in a:
        assert a[n].dtype in (np.float32, np.float64) and np.array_equal(a[n], b[n]), n
