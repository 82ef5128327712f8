"""The reference's own example scripts, BYTE-IDENTICAL, run against this package through the `normflow`
alias (north_star: "existing scripts run unchanged"; SURVEY 8b).

The scripts are not committed here: oracle/stage_ref.py stages /root/reference/examples/*.py next to the
staged reference package in the git-ignored oracle/_ref/ (which travels to the GPU box with the snapshot).
The tests execute those files as they are -- `from normflow import ...` resolves to normflow__b200 -- for
a few epochs, and check what the scripts themselves print / return."""

import importlib.util
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EXAMPLES = os.path.join(ROOT, "oracle", "_ref", "examples")


def _load(name):
    path = os.path.join(EXAMPLES, name + ".py")
    if not os.path.exists(path):
        pytest.skip("oracle/_ref/examples is not staged (run `python -m oracle.stage_ref` in the build container)")
    spec = importlib.util.spec_from_file_location("ref_example_" + name, path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod, path


def test_alias_package_is_the_same_modules():
    """`normflow.X` IS `normflow__b200.X` (CPU-side check: no kernels run)."""
    import normflow
    import normflow__b200
    import normflow.nn.scalar.couplings_ as a
    import normflow__b200.nn.scalar.couplings_ as b
    assert a is b and normflow.Model is normflow__b200.Model
    for sub in ("action", "mask", "nn", "prior", "mcmc"):           # src/__init__.py:9-13
        assert getattr(normflow, sub) is getattr(normflow__b200, sub)
    from normflow import np as np_, torch as torch_, backward_sanitychecker  # noqa: F401  (src/__init__.py:5-6)
    assert np_ is np


def test_staged_examples_are_the_reference_files():
    """Where the reference tree is present (the build container) the staged scripts are byte-identical."""
    ref = "/root/reference/examples"
    if not os.path.isdir(ref) or not os.path.isdir(EXAMPLES):
        pytest.skip("needs both /root/reference and the staged copy")
    for name in ("scalar_zerodim.py", "scalar_affine.py"):
        with open(os.path.join(ref, name), "rb") as f, open(os.path.join(EXAMPLES, name), "rb") as g:
            assert f.read() == g.read()


@pytest.mark.gpu
def test_reference_scalar_zerodim_runs_unchanged(tmp_path, capsys, monkeypatch):
    """examples/scalar_zerodim.py: main() as written, 300 epochs: the loss heads for -log Z = -1.112773 and
    the script's own backward_sanitychecker prints round-off-sized numbers.  The script's snapshot path
    points into its author's home directory; the snapshot it saves is written to tmp_path instead."""
    mod, path = _load("scalar_zerodim")
    import torch
    from normflow__b200._normflowcore import Fitter
    save = Fitter._save_snapshot

    def save_into_tmp_path(fitter, epoch):
        snapshot_path = fitter.checkpoint_dict['snapshot_path']
        fitter.checkpoint_dict['snapshot_path'] = str(tmp_path / os.path.basename(snapshot_path))
        try:
            save(fitter, epoch)
        finally:
            fitter.checkpoint_dict['snapshot_path'] = snapshot_path
    monkeypatch.setattr(Fitter, "_save_snapshot", save_into_tmp_path)
    torch.manual_seed(0)
    np.random.seed(0)
    model = mod.main(n_epochs=300, batch_size=1024)
    out = capsys.readouterr().out
    assert "number of model parameters =" in out
    loss = model.fit.train_history['loss']
    assert len(loss) == 300 and np.isfinite(loss).all()
    assert abs(np.mean(loss[-20:]) + 1.112773) < 0.02
    nums = [float(v) for v in out.strip().splitlines()[-1].split()]
    assert len(nums) == 2 and max(nums) < 1e-3


@pytest.mark.gpu
def test_reference_scalar_affine_runs_unchanged(tmp_path, capsys, monkeypatch):
    """examples/scalar_affine.py: main() as written (PSD block, DistConvertor_, 4 affine ConvAct couplings,
    parameter groups, snapshots under ../torch-snapshots relative to the working directory)."""
    mod, path = _load("scalar_affine")
    import torch
    torch.manual_seed(0)
    np.random.seed(0)
    work = tmp_path / "run"
    work.mkdir()
    (tmp_path / "torch-snapshots").mkdir()
    monkeypatch.chdir(work)
    model = mod.main(n_epochs=40, batch_size=128)
    out = capsys.readouterr().out
    assert "number of model parameters =" in out and "nranks is 1" in out
    loss = model.fit.train_history['loss']
    assert len(loss) == 40 and np.isfinite(loss).all()
    assert np.mean(loss[-5:]) < np.mean(loss[:5])
    # (save_every=200 in the script: no snapshot is due within 40 epochs)
    nums = [float(v) for v in out.strip().splitlines()[-1].split()]
    assert len(nums) == 2 and max(nums) < 1e-2
