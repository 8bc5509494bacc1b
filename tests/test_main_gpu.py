"""Drop-in boundary on hardware (SURVEY.md 8b): the reference's UNMODIFIED main.py (shipped to git-ignored
oracle/_ref by oracle/ship_reference.py during build()) trains, checkpoints, reloads and evaluates THIS repository's
`disvae` package on the B200, then the reference's own visualiser decodes traversals through it
(reference main.py:165-247, utils/visualize.py:121-123,217-222).  Runs in a child process so that the
reference's `main`/`utils` modules and the synthetic loader never leak into the other tests."""
import json
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.path.join(ROOT, "oracle", "_ref")


@pytest.mark.parametrize("loss", ["btcvae", "factor"])
def test_unmodified_main_drives_this_package(loss, tmp_path):
    if not os.path.isfile(os.path.join(REF, "main.py")):
        pytest.skip("oracle/_ref not shipped: build() found no checkout of the reference")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "run_reference_main.py"), loss, str(tmp_path)],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-3000:] + "\n" + r.stderr[-6000:]
    out = json.loads(r.stdout.strip().splitlines()[-1])
    # trained by main.py: checkpoints of training.py:92-94, final model + metadata of main.py:220, logs of both phases
    assert {"model.pt", "specs.json", "train_losses.log", "test_losses.log", "model-0.pt", "model-1.pt"} <= set(out["files"]) \
        or {"model.pt", "specs.json", "train_losses.log", "test_losses.log", "model-0.pt"} <= set(out["files"])
    assert out["log_head"] == "Epoch,Loss,Value"
    assert {"recon_loss", "kl_loss", "loss", "kl_loss_0"} <= set(out["logged"])
    if loss == "btcvae":
        assert {"mi_loss", "tc_loss", "dw_kl_loss"} <= set(out["logged"])
        assert out["img_size"] == [1, 64, 64]
    else:
        assert {"tc_loss", "discrim_loss"} <= set(out["logged"])
        assert out["img_size"] == [3, 64, 64]
    assert {"recon_loss", "kl_loss", "loss"} <= set(out["test_losses"])
    assert all(v == v and abs(v) < 1e9 for v in out["test_losses"].values())          # finite
    assert out["param_device"].startswith("cuda") and out["meta_loss"] == loss
    assert out["native_launches"] > 100                                               # the .so did the work
    assert len(out["traversal_shape"]) == 3 and len(out["reconstruct_shape"]) == 3
