"""Checks of the bench.py contract.  Without a GPU: the reference arm (the oracle timed on the host cores) prints one
well-formed JSON line, non-zero ranks of a torchrun launch stay silent and exit 0, and the product arm refuses to run without
a CUDA device instead of falling back to anything.  On the GPU: --dump-outputs writes reproducible outputs."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(args, env=None, timeout=600):
    e = dict(os.environ)
    e.update(env or {})
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True, env=e,
                          timeout=timeout, cwd=ROOT)


def test_reference_arm_prints_contract_line():
    r = _run(["--impl", "reference", "--size", "64", "--steps", "1", "--warmup", "1"])
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "512x512 images/sec" and d["unit"] == "images/s"
    assert d["value"] > 0 and d["ms_per_step"] > 0 and d["higher_is_better"] is True and d["n_gpus"] == 1
    assert d["e2e"] == {"value": d["value"], "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and "sample" in cb
    assert "workload" in d["config"] and "model" not in d["config"]


def test_reference_arm_other_ranks_are_silent():
    r = _run(["--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "1"], env={"RANK": "1", "WORLD_SIZE": "2",
                                                                                            "LOCAL_RANK": "1"})
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_product_arm_needs_a_gpu():
    import torch
    if torch.cuda.is_available():
        return
    r = _run(["--steps", "1", "--warmup", "1"], timeout=300)
    assert r.returncode != 0 and "{" not in r.stdout          # no number is printed, nothing falls back to the CPU


def test_dump_outputs_over_budget_keep_one_seeded_sample(tmp_path, monkeypatch):
    """Outputs larger than the dump budget are cut to the same seeded sample of their elements on every call, within budget."""
    import torch
    sys.path.insert(0, ROOT)
    import bench
    monkeypatch.setattr(bench, "DUMP_BYTES", 4096)
    outs = {"image": torch.randn(2, 3, 32, 32, dtype=torch.bfloat16), "latent": torch.randn(2, 4, 4, 4, dtype=torch.bfloat16)}
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), outs)
    got = {n: np.load(tmp_path / "a" / f"{n}.npy") for n in outs}
    assert sum(a.nbytes for a in got.values()) <= 4096
    for n, t in outs.items():
        assert got[n].dtype == np.float32 and got[n].size > 0
        assert np.array_equal(got[n], np.load(tmp_path / "b" / f"{n}.npy"))
        assert np.isin(got[n], t.float().numpy().ravel()).all()


@pytest.mark.gpu
def test_dump_outputs_repeat_bit_for_bit(tmp_path):
    """--dump-outputs writes the last timed step's image and latent as float32 .npy; --steps sets the timed step count; two runs
    with the same arguments get the same seeded inputs, so the dumps of one build agree bit for bit."""
    dumps = []
    for i in range(2):
        d = tmp_path / f"run{i}"
        r = _run(["--steps", "2", "--warmup", "1", "--batch", "1", "--configs", "none", "--no-cpu-baseline",
                  "--dump-outputs", str(d)], timeout=900)
        assert r.returncode == 0, r.stderr[-3000:]
        line = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
        assert line["steps"] == 2 and line["finite"]
        assert sorted(os.listdir(d)) == ["image.npy", "latent.npy"]
        a = {n: np.load(d / f"{n}.npy") for n in ("image", "latent")}
        assert a["image"].shape == (1, 3, 512, 512) and a["latent"].shape == (1, 4, 64, 64)
        assert all(v.dtype == np.float32 and np.isfinite(v).all() for v in a.values())
        dumps.append(a)
    for n in dumps[0]:
        assert np.array_equal(dumps[0][n], dumps[1][n]), n
