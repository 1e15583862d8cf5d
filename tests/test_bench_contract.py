"""bench.py's contract, as far as it can be checked without a GPU: the reference arm prints one JSON line with the
keys the driver reads, and the product arm refuses to run on a CPU (no fallback path exists)."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(*args):
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True,
                          cwd=ROOT, env=env, timeout=600)


def test_reference_arm_prints_one_json_line_with_the_contract_keys():
    res = _run("--impl", "reference", "--steps", "1", "--warmup", "1")
    assert res.returncode == 0, res.stderr
    lines = [ln for ln in res.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["n_gpus"] == 1 and d["steps"] == 1 and d["warmup"] == 1
    assert d["unit"] == "images/s" and d["higher_is_better"] is True and d["scaling"] == "weak"
    assert d["vs_baseline"] is None and d["dtype"] == "f32" and d["data"] == "synthetic"
    assert d["value"] > 0 and d["ms_per_step"] > 0
    assert "workload" in d["config"] and "model" not in d["config"]
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("port", "reference") and cb["cores"] >= 1 and cb["sample"] and cb["value"] == d["value"]
    e2e = d["e2e"]
    assert e2e["value"] == d["value"] and e2e["unit"] == d["unit"]
    assert e2e["h2d_bytes_per_step"] == 0 and e2e["d2h_bytes_per_step"] == 0
    # the same metric and workload as the product arm reports (BASELINE.json's north star)
    with open(os.path.join(ROOT, "BASELINE.json")) as f:
        base = json.load(f)
    assert "metric" in base and d["metric"]


def test_steps_below_one_and_dumps_of_the_cpu_arm_are_rejected():
    res = _run("--impl", "reference", "--steps", "0")
    assert res.returncode != 0 and "--steps must be at least 1" in res.stderr
    res = _run("--impl", "reference", "--steps", "1", "--dump-outputs", os.devnull)
    assert res.returncode != 0 and "--dump-outputs writes the outputs of --impl ours" in res.stderr


def test_explicit_steps_are_the_timed_steps():
    """The CPU arm used to cap --steps at 5 (and the stress workload replaced an explicit 2000 by 200)."""
    res = _run("--impl", "reference", "--batch", "8", "--steps", "7", "--warmup", "0")
    assert res.returncode == 0, res.stderr
    assert json.loads(res.stdout.strip().splitlines()[-1])["steps"] == 7


def test_dump_sample_keeps_the_budget_with_one_fixed_subset_of_images(monkeypatch):
    import numpy as np
    import torch
    import bench
    monkeypatch.setattr(bench, "DUMP_BYTES", 10_000)
    loc = torch.arange(8 * 100 * 4, dtype=torch.float32).reshape(8, 100, 4)
    cls = torch.arange(8 * 100, dtype=torch.int32).reshape(8, 100)
    a = bench.dump_sample({"losses": torch.ones(2)}, {"loc": loc, "cls": cls})
    b = bench.dump_sample({"losses": torch.ones(2)}, {"loc": loc, "cls": cls})
    assert a["loc"].dtype == np.float32 and a["cls"].dtype == np.float64 and a["losses"].dtype == np.float32
    assert sum(x.nbytes for x in a.values()) <= 10_000 and a["loc"].shape == (4, 100, 4)      # 2400 B per image
    imgs = a["loc"][:, 0, 0].astype(np.int64) // 400
    assert list(imgs) == sorted(imgs) and np.array_equal(a["cls"][:, 0].astype(np.int64) // 100, imgs)
    assert all(np.array_equal(a[k], b[k]) for k in a)
    whole = bench.dump_sample({}, {"loc": loc[:2], "cls": cls[:2]})
    assert np.array_equal(whole["loc"], loc[:2].numpy())


def test_product_arm_refuses_to_run_without_a_gpu():
    res = _run("--steps", "1", "--warmup", "1")
    assert res.returncode != 0
    assert "no CPU fallback" in (res.stdout + res.stderr)
    assert not [ln for ln in res.stdout.splitlines() if ln.strip().startswith("{")], "no result line may be printed"


@pytest.mark.gpu
def test_dump_outputs_of_the_timed_step(tmp_path):
    """--dump-outputs on the GPU: the training step's losses and a seeded image subset of its gradients within 64 MB,
    the same files from two runs with the same arguments; the detections with the slots past each count zeroed."""
    import numpy as np

    def dump(name, *args):
        res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "3", "--warmup", "3",
                              "--no-others", "--dump-outputs", str(tmp_path / name), *args],
                             capture_output=True, text=True, cwd=ROOT, timeout=900)
        assert res.returncode == 0, res.stderr
        assert len([ln for ln in res.stdout.splitlines() if ln.strip()]) == 1
        files = sorted(os.listdir(tmp_path / name))
        assert sum(os.path.getsize(tmp_path / name / f) for f in files) <= 64_000_000
        return {f[:-4]: np.load(tmp_path / name / f) for f in files}

    a, b = dump("train_a"), dump("train_b")
    assert sorted(a) == ["grad_conf", "grad_loc", "loss_sums", "losses"]
    assert a["losses"].dtype == np.float32 and a["loss_sums"].dtype == np.float64
    k = a["grad_loc"].shape[0]
    assert 0 < k < 256 and a["grad_loc"].shape == (k, 8732, 4) and a["grad_conf"].shape == (k, 8732, 21)
    assert (a["grad_conf"] != 0).any() and np.isfinite(a["losses"]).all()
    assert all(np.array_equal(a[n], b[n]) for n in a)
    d = dump("detect", "--workload", "detect")
    assert sorted(d) == ["boxes", "cls", "cnt", "prior", "prob"] and d["cnt"].dtype == np.float64
    assert d["boxes"].shape == (64, 200, 4) and d["prob"].shape == d["cls"].shape == d["prior"].shape == (64, 200)
    past = np.arange(200)[None, :] >= d["cnt"][:, None]
    assert (d["prob"][past] == 0).all() and (d["boxes"][past] == 0).all() and (d["prob"][~past] > 0).all()
