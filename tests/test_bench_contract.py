"""bench.py contract checks: the product arm refuses to run without a CUDA device (no CPU
fallback), the reference arm prints one JSON line with the agreed keys and times --steps steps,
--dump-outputs writes the task's outputs within its size budget, and (GPU) the dumped outputs of
the last timed step repeat exactly from run to run and agree with the oracle."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import bench
from helpers import assert_close

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(*args, timeout=600):
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], cwd=ROOT,
                          capture_output=True, text=True, timeout=timeout)


@pytest.mark.skipif(torch.cuda.is_available(), reason="only meaningful on a machine without a GPU")
def test_product_arm_fails_loudly_without_a_gpu():
    r = _run("--steps", "1", "--warmup", "1")
    assert r.returncode != 0
    assert "no CPU fallback" in (r.stderr + r.stdout)
    assert not r.stdout.strip().startswith("{")       # no bench line was produced


def test_reference_arm_json_contract():
    r = _run("--impl", "reference", "--steps", "1", "--warmup", "1")
    assert r.returncode == 0, r.stderr[-2000:]
    line = [ln for ln in r.stdout.strip().splitlines() if ln.startswith("{")][-1]
    d = json.loads(line)
    assert d["impl"] == "reference" and d["higher_is_better"] is True and d["unit"] == "clouds/s"
    for key in ("metric", "value", "n_gpus", "steps", "warmup", "ms_per_step", "scaling", "dtype",
                "data", "config", "cpu_baseline", "e2e"):
        assert key in d, key
    assert d["value"] > 0 and d["steps"] == 1
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("port", "reference") and cb["cores"] >= 1 and "sample" in cb
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert abs(d["e2e"]["value"] - d["value"]) < 1e-9 * max(1.0, d["value"])
    assert "workload" in d["config"] and "model" not in d["config"]


def test_reference_arm_times_every_requested_step():
    r = _run("--impl", "reference", "--config", "cfg1", "--steps", "6", "--warmup", "1")
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads([ln for ln in r.stdout.strip().splitlines() if ln.startswith("{")][-1])
    assert d["steps"] == 6 and d["cpu_baseline"]["sample"].startswith("6 steps ")


@pytest.mark.parametrize("args,flag", [(("--steps", "0"), "--steps"),
                                       (("--impl", "reference", "--dump-outputs", "unused"),
                                        "--dump-outputs")])
def test_arguments_the_run_would_not_honour_are_refused(args, flag):
    r = _run(*args)
    assert r.returncode != 0 and flag in r.stderr
    assert not os.path.exists(os.path.join(ROOT, "unused"))


class _Crit:
    forward_loss_array = torch.tensor([1.0, 2.0])
    backward_loss_array = torch.tensor([3.0, 4.0])


@pytest.mark.parametrize("task,names", [
    ("classifier", ["feature", "loss", "score"]),
    ("segmenter", ["feature", "loss", "score_segmenter"]),
    ("autoencoder", ["chamfer_loss_arrays", "feature", "loss", "loss_chamfer",
                     "loss_chamfer_conv4", "predicted_pc"])])
def test_step_outputs_names_and_types(task, names):
    m = type("M", (), {})()
    for n in names:
        setattr(m, n, torch.arange(6, dtype=torch.float64).view(2, 3))
    m.loss_chamfer_conv5 = None                  # not computed for 1024 conv points: left out
    m.chamfer_criteria = _Crit()
    out = bench.step_outputs(task, m)
    assert sorted(out) == names
    assert all(t.dtype == torch.float32 and t.device.type == "cpu" for t in out.values())
    if task == "autoencoder":
        assert out["chamfer_loss_arrays"].tolist() == [[1.0, 3.0], [2.0, 4.0]]


def test_dump_outputs_samples_over_budget_at_fixed_positions(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_BUDGET", 1000)        # 125 float32 elements per array
    arrays = {"big": torch.arange(600, dtype=torch.float32).view(20, 30),
              "small": torch.arange(7, dtype=torch.float32)}
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), arrays)
    assert sorted(os.listdir(tmp_path / "a")) == ["big.npy", "small.npy"]
    big = np.load(tmp_path / "a" / "big.npy")
    assert big.dtype == np.float32 and big.shape == (125,)
    # values equal their flat positions: distinct, ascending, in range
    assert (np.diff(big) > 0).all() and big[0] >= 0 and big[-1] < 600
    assert np.array_equal(big, np.load(tmp_path / "b" / "big.npy"))
    assert np.array_equal(np.load(tmp_path / "a" / "small.npy"), arrays["small"].numpy())
    total = sum(np.load(tmp_path / "a" / n).nbytes for n in ("big.npy", "small.npy"))
    assert total <= 1000


def _dump(d, *args):
    r = _run(*args, "--steps", "3", "--warmup", "1", "--dump-outputs", str(d))
    assert r.returncode == 0, r.stderr[-3000:]
    line = json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("{")][-1])
    assert line["steps"] == 3
    out = {n[:-len(".npy")]: np.load(d / n) for n in os.listdir(d)}
    assert all(a.dtype == np.float32 and np.isfinite(a).all() for a in out.values())
    assert sum(a.nbytes for a in out.values()) <= bench.DUMP_BUDGET
    return out


@pytest.mark.gpu
def test_dump_outputs_repeat_exactly(tmp_path):
    """Two runs with the same arguments dump the same arrays; the first run also checks the timed
    rows (the dumped score) against the CPU arm (bench.py exits non-zero on a parity failure), and
    feature -> score and score -> loss are recomputed independently."""
    from oracle import oracle
    from sonet_b200 import synth
    a = _dump(tmp_path / "a", "--config", "cfg1")
    b = _dump(tmp_path / "b", "--config", "cfg1", "--no-cpu-baseline")
    assert sorted(a) == ["feature", "loss", "score"] == sorted(b)
    for n in a:
        assert np.array_equal(a[n], b[n]), n
    assert a["score"].shape == (8, 40)
    _, st_h = bench.make_states("classifier", 8, 1024)
    assert_close(a["score"], oracle.classifier_forward(st_h, torch.from_numpy(a["feature"])),
                 "score from the dumped feature")
    label = synth.synth_inputs(8, 1024, seed=0)["label"]
    assert_close(a["loss"], F.cross_entropy(torch.from_numpy(a["score"]), label), "loss")


@pytest.mark.gpu
def test_dump_outputs_segmenter(tmp_path):
    o = _dump(tmp_path, "--config", "cfg3", "--no-cpu-baseline")
    assert sorted(o) == ["feature", "loss", "score_segmenter"]
    assert o["score_segmenter"].shape == (32, 50, 1024)
    seg = bench.input_list("segmenter", dict.fromkeys(("pc", "sn", "label", "node", "node_knn_I")),
                           32, 1024)[3]
    assert_close(o["loss"], F.cross_entropy(torch.from_numpy(o["score_segmenter"]), seg), "loss")


@pytest.mark.gpu
def test_dump_outputs_autoencoder(tmp_path):
    from oracle import oracle
    from sonet_b200 import synth
    o = _dump(tmp_path, "--config", "cfg4", "--no-cpu-baseline")
    assert sorted(o) == ["chamfer_loss_arrays", "feature", "loss", "loss_chamfer",
                         "loss_chamfer_conv4", "predicted_pc"]
    assert o["predicted_pc"].shape == (32, 3, 1280) and o["chamfer_loss_arrays"].shape == (32, 2)
    ch = oracle.chamfer(torch.from_numpy(o["predicted_pc"]), synth.synth_inputs(32, 5000, seed=0)["pc"])
    assert_close(o["chamfer_loss_arrays"],
                 torch.stack((ch["forward_loss_array"], ch["backward_loss_array"]), dim=1),
                 "Chamfer terms of the dumped prediction")
    assert_close(o["loss_chamfer"], ch["loss"], "loss_chamfer")
    assert_close(o["loss"], o["loss_chamfer"] + o["loss_chamfer_conv4"], "loss", 1e-6)
