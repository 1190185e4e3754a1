"""bench.py --dump-outputs: what the last timed step returned, as float .npy files under a size cap."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import bench
from conftest import ROOT

BIAS = torch.full((15,), -6.21875, dtype=torch.bfloat16)


def load(d):
    return {n[:-4]: np.load(os.path.join(d, n)) for n in os.listdir(d)}


def test_dump_zeroes_rows_past_each_count(tmp_path):
    g = torch.Generator().manual_seed(0)
    dets = torch.randn(3, 5, 6, generator=g) + 10.0
    labels = torch.randint(0, 15, (3, 5), generator=g).float() + 1.0
    counts = torch.tensor([2, 0, 5], dtype=torch.int32)
    bench.dump_outputs(str(tmp_path), dets, labels, counts, BIAS)
    out = load(str(tmp_path))
    assert sorted(out) == ["counts", "dets", "image_index", "labels", "odm_cls_bias"]
    assert all(a.dtype in (np.float32, np.float64) for a in out.values())
    np.testing.assert_array_equal(out["counts"], [2, 0, 5])
    np.testing.assert_array_equal(out["image_index"], [0, 1, 2])
    np.testing.assert_array_equal(out["odm_cls_bias"], np.full(15, -6.21875))
    for i, k in enumerate((2, 0, 5)):
        np.testing.assert_array_equal(out["dets"][i, :k], dets[i, :k].numpy())
        np.testing.assert_array_equal(out["labels"][i, :k], labels[i, :k].numpy())
        assert not out["dets"][i, k:].any() and not out["labels"][i, k:].any()


def test_dump_samples_images_under_the_cap(tmp_path, monkeypatch):
    n, K = 50, 4
    per_image = K * 6 * 4 + K * 4 + 16
    cap = 10 * per_image + 15 * 8
    monkeypatch.setattr(bench, "DUMP_MAX_BYTES", cap)
    dets = torch.arange(n, dtype=torch.float32)[:, None, None].expand(n, K, 6).contiguous()
    counts = torch.full((n,), K, dtype=torch.int32)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), dets, torch.ones(n, K), counts, BIAS)
    a, b = load(str(tmp_path / "a")), load(str(tmp_path / "b"))
    assert a["dets"].shape == (10, K, 6) and sum(v.nbytes for v in a.values()) <= cap
    np.testing.assert_array_equal(a["dets"][:, 0, 0], a["image_index"])      # the rows of the images it names
    for k in a:                                                               # the same sample every run
        np.testing.assert_array_equal(a[k], b[k])


@pytest.mark.gpu
def test_bench_dumps_the_last_timed_step_identically(tmp_path):
    """The wiring in bench.main(): two runs with the same arguments write identical files, and they are the step whose
    detection count the JSON line reports."""
    lines = []
    for d in ("a", "b"):
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "3", "--warmup", "3",
                            "--batch", "2", "--no-extra", "--no-cpu-baseline", "--dump-outputs", str(tmp_path / d)],
                           cwd=str(tmp_path), stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=600)
        assert r.returncode == 0, r.stderr[-2000:]
        lines.append(json.loads(r.stdout.strip().splitlines()[-1]))
    a, b = load(str(tmp_path / "a")), load(str(tmp_path / "b"))
    for k in ("dets", "labels", "counts", "image_index", "odm_cls_bias"):
        np.testing.assert_array_equal(a[k], b[k])
    assert a["dets"].shape == (2, 2000, 6) and a["labels"].shape == (2, 2000)
    np.testing.assert_array_equal(a["image_index"], [0, 1])
    assert int(a["counts"].mean()) == lines[0]["config"]["detections_per_image"] > 0
    assert float(a["odm_cls_bias"].mean()) == pytest.approx(lines[0]["config"]["odm_cls_bias"], abs=1e-5)
    for i, k in enumerate(a["counts"].astype(int)):
        s = a["dets"][i, :k, 5]
        assert np.all((s > 0.05) & (s <= 1.0)) and np.all((a["labels"][i, :k] >= 0) & (a["labels"][i, :k] < 15))
