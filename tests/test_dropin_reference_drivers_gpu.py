"""The drop-in proof (SURVEY section 4 item 4, section 8b): the reference's UNMODIFIED main.py / train_model.py / dataset.py /
utils.py, byte-compiled into oracle/_ref by __graft_entry__.build() where the original project is present
(oracle/stage_reference.py), import `module` from dropin/ and train on a synthetic (datetime, instrument) pickle:
`from module import ...` (main.py:12, utils.py:6) resolves to the B200-native classes, main.main runs its epochs with Adam +
CosineAnnealingLR on OUR parameters, writes its best-validation checkpoint, utils.load_model + load_state_dict reload it,
train_model.validate and utils.generate_prediction_scores run on it.  The same harness is then run with the reference's own
module.py (PyTorch eager on the same GPU): both trajectories must agree up to the noise they draw differently."""
import json
import os
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.path.join(ROOT, "oracle", "_ref")


def _drive(module_dir, work, env_extra=None):
    env = dict(os.environ, WANDB_MODE="disabled", **(env_extra or {}))
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "_dropin_driver.py"), module_dir, REF, str(work)],
                       capture_output=True, text=True, timeout=900, cwd=ROOT, env=env)
    if r.returncode != 0:
        sys.stdout.write("---- driver stdout ----\n" + r.stdout[-3000:] + "\n---- driver stderr ----\n" + r.stderr[-6000:])
    assert r.returncode == 0, r.stderr[-1500:]
    return json.loads(r.stdout.strip().splitlines()[-1])


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_unmodified_reference_drivers_train_on_the_dropin(precision, tmp_path, cuda_device):
    if not os.path.exists(os.path.join(REF, "main.pyc")):
        pytest.skip("oracle/_ref is absent (made by __graft_entry__.build() where the original project is present)")
    ours = _drive(os.path.join(ROOT, "dropin"), tmp_path / "ours", {"FVAE_PRECISION": precision})
    print("drop-in driver result:", ours)
    assert ours["module_file"].startswith(os.path.join(ROOT, "dropin")), ours["module_file"]
    assert ours["device"].startswith("cuda")
    ep = ours["epochs"]
    assert len(ep) == 3 and all(torch.isfinite(torch.tensor(e)).all() for e in ep), ep
    assert ep[-1][0] < ep[0][0] and ep[-1][1] < ep[0][1], ep                       # train and validation loss decrease
    assert ours["checkpoint"] and ours["state_keys"] == 28 + 5 * 8
    assert ours["load_state_dict"] == "<All keys matched successfully>"
    assert ours["score_frame_shape"][1] == 1 and ours["scores_finite"]
    theirs = _drive(REF, tmp_path / "theirs")                                       # the reference's own module.py, eager
    assert theirs["module_file"].startswith(REF)
    print("drop-in  :", ep, ours["reloaded_val_loss"])
    print("reference:", theirs["epochs"], theirs["reloaded_val_loss"])
    assert ours["score_frame_shape"] == theirs["score_frame_shape"]
    for (a_tr, a_va), (b_tr, b_va) in zip(ep, theirs["epochs"]):
        assert abs(a_tr - b_tr) <= 0.25 * abs(b_tr), (ep, theirs["epochs"])
        assert abs(a_va - b_va) <= 0.25 * abs(b_va), (ep, theirs["epochs"])
