"""Boundary by execution: the reference's UNMODIFIED ``Main.py`` (Main.py:11-15 star-imports ``util_functions``,
``models``, ``train_eval``) runs on the drop-in modules under ``shims/`` - dataset construction through
``eval(dataset_class)(...)``, ``IGMC(...)``, ``train_multiple_epochs`` with its ``logger`` (log.txt + checkpoints) and
the checkpoint ensemble of ``test_once`` - with the data loaders stubbed by a synthetic split (tests/main_stubs).

Main.py is read from oracle/_ref/, the git-ignored copy that build() places through oracle/make_ref.py when it finds a
checkout of the reference; without it the test is skipped (the reference's source is not part of this repository)."""
import os
import re
import subprocess
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pytestmark = pytest.mark.gpu


def _main_py():
    p = os.path.join(ROOT, "oracle", "_ref", "Main.py")
    return p if os.path.isfile(p) else None


@pytest.mark.skipif(_main_py() is None, reason="reference Main.py not available (run oracle/make_ref.py)")
@pytest.mark.parametrize("extra", [["--dynamic-train", "--dynamic-test"], ["--dynamic-train"], []],
                         ids=["dynamic", "static-test", "static"])
def test_reference_main_runs_on_the_drop_in_modules(tmp_path, extra):
    env = dict(os.environ)
    env["PYTHONPATH"] = os.pathsep.join([os.path.join(ROOT, "tests", "main_stubs"), os.path.join(ROOT, "shims"), ROOT,
                                         env.get("PYTHONPATH", "")])
    env["MPLBACKEND"] = "Agg"
    # the script's own directory leads sys.path: run a copy from the (otherwise empty) working directory so that
    # `from util_functions import *` resolves to shims/, not to the reference file that sits next to Main.py
    import shutil
    shutil.copyfile(_main_py(), str(tmp_path / "Main.py"))
    cmd = [sys.executable, "Main.py", "--data-name", "ml_1m", "--testing", "--epochs", "20", "--save-interval", "5",
           "--ensemble", "--keep-old", "--max-nodes-per-hop", "10", "--batch-size", "50", "--lr-decay-step-size", "8",
           "--save-appendix", "_t"] + extra
    r = subprocess.run(cmd, cwd=str(tmp_path), env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-3000:] + "\n" + r.stderr[-3000:]
    res = tmp_path / "results" / "ml_1m_t_testmode"
    log = (res / "log.txt").read_text().strip().splitlines()
    ep = [l for l in log if re.match(r"Epoch \d+, train loss [\d.]+, test rmse [\d.]+$", l)]
    assert len(ep) == 20, log
    losses = [float(l.split("train loss ")[1].split(",")[0]) for l in ep]
    assert losses[-1] < losses[0]                                   # it trains
    assert log[-1].startswith("Epoch ensemble of range(5, 20, 5)")  # Main.py:437-466 -> logger(eval_info, None, None)
    assert "Ensemble test rmse is:" in r.stdout and "Total number of parameters is 49233" in r.stdout
    for e in (5, 10, 15, 20):
        sd = torch.load(res / ("model_checkpoint%d.pth" % e))
        assert "convs.0.basis" in sd and "lin2.bias" in sd         # reference state_dict names
        od = torch.load(res / ("optimizer_checkpoint%d.pth" % e))
        assert len(od["state"]) == 20 and od["param_groups"][0]["lr"] <= 1e-3
