"""SURVEY §8(b) "what scripts call must keep working unchanged", on the REAL scripts: ref:ssp_vit2spn_tiny.py and
ref:octmnist_ft_vit2spn.py from a checkout of the original ViT-2SPN at $V2S_REFERENCE_DIR (not part of this
repository) run UNMODIFIED under ``python -m vit2spn.run``.  Skipped when they are absent.  (File name: runs last — it
takes ~2.5 minutes: 100 epochs of the reference's own loop.)"""
import os
import subprocess

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF_DIR = os.environ.get("V2S_REFERENCE_DIR", "")
SCRIPTS = ("ssp_vit2spn_tiny.py", "octmnist_ft_vit2spn.py")
pytestmark = pytest.mark.gpu


@pytest.mark.skipif(not (REF_DIR and all(os.path.isfile(os.path.join(REF_DIR, s)) for s in SCRIPTS)),
                    reason="V2S_REFERENCE_DIR does not name a checkout of the original ViT-2SPN")
def test_unmodified_reference_scripts_run_under_the_launcher(tmp_path):
    out, work = tmp_path / "logs", tmp_path / "work"
    env = dict(os.environ, V2S_WORKDIR=str(work))
    r = subprocess.run(["bash", os.path.join(ROOT, "tools", "run_reference_scripts.sh"), str(out)], env=env,
                       capture_output=True, text=True, timeout=1500)
    ssp = (out / "ssp_vit2spn_tiny.log").read_text()
    ft = (out / "octmnist_ft_vit2spn.log").read_text()
    assert r.returncode == 0, r.stdout[-2000:] + (out / "ssp_vit2spn_tiny.err").read_text()[-3000:] + \
        (out / "octmnist_ft_vit2spn.err").read_text()[-3000:]
    # pretraining: the reference's own loop ran all 100 epochs through autocast + GradScaler + its .data EMA loop
    assert "SYNTHETIC DATA" in ssp and "Total parameters: 11681408" in ssp          # ref:235-239, README "11.68 M"
    assert "Epoch 100/100, Loss: " in ssp and "Checkpoint saved at epoch 100" in ssp and "Pretrained model saved" in ssp
    losses = [float(l.split("Loss: ")[1]) for l in ssp.splitlines() if l.startswith("Epoch ") and "Loss: " in l]
    assert len(losses) == 100 and losses[-1] < losses[0] - 0.3, (losses[0], losses[-1])   # it learns (cosine -> -1)
    # the hand-off of ref:ssp_vit2spn_tiny.py:246 -> ref:octmnist_ft_vit2spn.py:190: HF key names, strict load
    sd = torch.load(work / "ssp_retinaloct_tbme" / "vit2spn_tiny" / "octmnist_vit2spn_tiny_model.pth", map_location="cpu")
    assert len(sd) == 200 and all(k.startswith("vit.") for k in sd)
    import vit2spn
    vit2spn.ViTBackbone().load_state_dict(sd, strict=True)
    ck = torch.load(work / "ssp_retinaloct_tbme" / "vit2spn_tiny" / "octmnist_vit2spn_tiny_checkpoint.pth", map_location="cpu")
    assert set(ck) == {"epoch", "model_state_dict", "optimizer_state_dict", "loss"} and ck["epoch"] == 100
    assert len(ck["model_state_dict"]) == 808 and len(ck["optimizer_state_dict"]["state"]) == 400
    # fine-tuning: 10 folds, evaluation on the test subset, AUC summary (on fabricated data: only the plumbing counts)
    assert "SYNTHETIC DATA" in ft and "Fold 10/10" in ft and "Evaluating on test data with the best model" in ft
    assert "Mean AUC across folds:" in ft
