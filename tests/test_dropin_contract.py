"""INTEGRATION.md section 2, executed: our model classes under the package's restatement of the reference's Config /
RecDataset / dataloaders / Trainer, kernels replaced by oracle-backed CPU stand-ins, against what the reference's own
harness and model classes produced (tests/golden, recorded by tests/golden/make_golden.py).  No GPU needed."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_our_model_class_under_the_reference_trainer():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "dropin_contract_worker.py")], capture_output=True, text=True,
                         timeout=600)
    lines = [l for l in out.stdout.splitlines() if l.startswith("CONTRACT ")]
    assert out.returncode == 0 and lines, out.stdout[-3000:] + out.stderr[-3000:]
    r = json.loads(lines[-1][len("CONTRACT "):])
    assert r["init_identical"], "init_seed(999) must reproduce the reference's initial weights under the reference's harness"
    assert r["valid"].keys() == r["want_valid"].keys()
    for k, v in r["want_valid"].items():
        assert abs(r["valid"][k] - v) < 1e-9, (k, r["valid"][k], v)
    for k, v in r["want_test"].items():
        assert abs(r["test"][k] - v) < 1e-9, (k, r["test"][k], v)
    assert abs(r["loss"] - r["want_loss"]) <= 1e-5 * abs(r["want_loss"])
    assert r["has_grads"]


def test_our_mmgcn_class_against_the_reference_model_code():
    """MMGCN (torch_geometric absent): our PyG-free class under the package's harness reproduces what the reference's own
    model code produced under the PyG shim -- initial weights bit for bit, forward / loss / gradients / scores to fp32 rounding,
    and the metrics of the reference's `Trainer.evaluate`."""
    out = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "dropin_contract_worker.py"), "mmgcn"], capture_output=True,
                         text=True, timeout=600)
    lines = [l for l in out.stdout.splitlines() if l.startswith("CONTRACT ")]
    assert out.returncode == 0 and lines, out.stdout[-3000:] + out.stderr[-3000:]
    r = json.loads(lines[-1][len("CONTRACT "):])
    assert r["init_identical"]
    assert r["fwd_rel"] < 1e-6 and r["grad_rel"] < 1e-4 and r["score_err"] < 1e-6
    assert abs(r["loss"] - r["want_loss"]) <= 1e-6 * abs(r["want_loss"])
    for k, v in r["want_valid"].items():
        assert abs(r["valid"][k] - v) < 1e-9, (k, r["valid"][k], v)


@pytest.mark.parametrize("name", ["BM3", "MGCN", "LightGCN", "LayerGCN"])
def test_our_model_classes_under_the_reference_harness(name):
    """The other north-star classes as drop-ins under the package's Config / RecDataset / loaders / Trainer (kernels replaced by
    torch-CPU stand-ins): initial weights bit for bit, `forward` (MGCN: the no-autograd gate / fuse / stacked-table route),
    the loss on the recorded batch under the reference's RNG stream -- BM3's always-on `F.dropout` branch (`bm3.py:110-119`)
    included, which the device tests can only check with dropout switched off --, gradients, first-batch scores and the
    reference Trainer's valid / test metrics."""
    out = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "dropin_contract_worker.py"), name], capture_output=True, text=True,
                         timeout=600)
    lines = [l for l in out.stdout.splitlines() if l.startswith("CONTRACT ")]
    assert out.returncode == 0 and lines, out.stdout[-3000:] + out.stderr[-3000:]
    r = json.loads(lines[-1][len("CONTRACT "):])
    assert r["init_identical"] and r["grad_ok"]
    assert r["fwd_rel"] < 1e-6 and r["score_err"] < 1e-6
    assert abs(r["loss"] - r["want_loss"]) <= 1e-6 * abs(r["want_loss"])
    for k, v in r["want_valid"].items():
        assert abs(r["valid"][k] - v) < 1e-9, (k, r["valid"][k], v)
    for k, v in r["want_test"].items():
        assert abs(r["test"][k] - v) < 1e-9, (k, r["test"][k], v)


@pytest.mark.parametrize("name", ["LightGCN", "FREEDOM"])
def test_reference_training_loop_drives_our_class(name):
    """Two epochs of `Trainer._train_epoch` (torch's Adam, the scheduler, the reference loader's recorded batches) on OUR class:
    the same batches, every batch loss and the per-epoch valid / test metrics of the trajectory the reference's class recorded."""
    out = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "dropin_contract_worker.py"), "traj:" + name], capture_output=True,
                         text=True, timeout=900)
    lines = [l for l in out.stdout.splitlines() if l.startswith("CONTRACT ")]
    assert out.returncode == 0 and lines, out.stdout[-3000:] + out.stderr[-3000:]
    r = json.loads(lines[-1][len("CONTRACT "):])
    assert r["same_batches"] and r["n_batches"] == 8
    assert r["loss_max_rel"] < 1e-6 and r["metric_max_abs"] < 1e-9


@pytest.mark.parametrize("key", ["FREEDOM-prune", "LayerGCN", "BM3", "MGCN"])
def test_reference_training_loop_with_pruning_and_dropout(key):
    """The same two-epoch replay where the model draws random numbers inside the loop: FREEDOM's and LayerGCN's per-epoch
    degree-sensitive pruning (`freedom.py:128-162`: the `torch.multinomial` stream and the graph rebuilt from it), BM3's dropout,
    and MGCN (whose evaluations go through the fused inference route).  Same batches, every loss and metric exactly."""
    out = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "dropin_contract_worker.py"), "traj:" + key], capture_output=True,
                         text=True, timeout=900)
    lines = [l for l in out.stdout.splitlines() if l.startswith("CONTRACT ")]
    assert out.returncode == 0 and lines, out.stdout[-3000:] + out.stderr[-3000:]
    r = json.loads(lines[-1][len("CONTRACT "):])
    assert r["same_batches"] and r["n_batches"] == 8
    assert r["loss_max_rel"] < 1e-6 and r["metric_max_abs"] < 1e-9
