"""-m gpu: the reference's own train.py / evaluate.py / predict.py, UNMODIFIED (baseline/_ref, staged by
__graft_entry__.build()), run on the drop-in modules and -- same files, same seeds, same data -- on stock PyTorch.
See tests/callers_ref_worker.py.  Those scripts are not part of this repository: the test skips unless build() ran with
UNETB200_REFERENCE_DIR naming a checkout of the reference, which stages them under baseline/_ref."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
REF = os.path.join(ROOT, "baseline", "_ref")


def _run(mode, tmp):
    out = os.path.join(tmp, f"{mode}.json")
    p = subprocess.run([sys.executable, os.path.join(HERE, "callers_ref_worker.py"), "--mode", mode, "--work",
                        os.path.join(tmp, mode), "--out", out], capture_output=True, text=True, timeout=900)
    sys.stdout.write(p.stdout[-3000:])
    sys.stderr.write(p.stderr[-3000:])
    assert p.returncode == 0, f"{mode} run failed"
    with open(out) as f:
        return json.load(f), np.load(out + ".mask.npy")


@pytest.mark.skipif(not os.path.isfile(os.path.join(REF, "train.py")),
                    reason="needs the reference's own scripts in baseline/_ref (build() with UNETB200_REFERENCE_DIR set)")
def test_reference_callers_run_unchanged_on_the_dropin(tmp_path):
    ours, mask_o = _run("dropin", str(tmp_path))
    ref, mask_r = _run("stock", str(tmp_path))
    # the loop ran: 3 ids x 4 rotations / batch 2 = 6 optimisation steps, one evaluate() with PNGs, a checkpoint
    for r in (ours, ref):
        assert len(r["losses"]) == 6 and all(v == v for v in r["losses"])
        assert r["num_batches_tracked"] == 6 and r["weights_moved"] > 0 and r["saved_model"] and r["pngs"] >= 4
        assert r["state_keys"] == 118
    assert ours["unet_from"].endswith(os.path.join("unet-medical-image-contour-segmentation_b200", "unet"))
    # same trajectory as the stock fp16-autocast run, at reduced-precision tolerance
    lo, lr_ = np.array(ours["losses"]), np.array(ref["losses"])
    assert np.abs(lo - lr_).max() / np.abs(lr_).max() < 2e-2, (lo, lr_)
    for k in ("running_mean_inc", "running_var_up4"):
        a, b = np.array(ours[k]), np.array(ref[k])
        assert np.abs(a - b).max() / np.abs(b).max() < 5e-2, k
    # (original, post-processed, minimum) dice of evaluate(): the post-processed score passes through OpenCV's
    # connected-component filter, which can drop a whole blob on a one-pixel difference -- compare the other two
    vo, vr = np.array(ours["val_scores"]), np.array(ref["val_scores"])
    assert abs(vo[0] - vr[0]) < 5e-2 and abs(vo[2] - vr[2]) < 5e-2 and 0.0 <= vo[1] <= 1.0
    assert (mask_o == mask_r).mean() > 0.9
