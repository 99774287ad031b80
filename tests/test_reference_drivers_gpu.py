"""The acceptance test the north star names, against stored numbers: this repository's trainer
(r2_gaussian_b200.trainer, the flow and defaults of the reference's train.py) on the synthetic case of
scripts/make_synthetic_case.py reaches the 3-D PSNR that the reference's own train.py and test.py reached on the
reference's own CUDA kernels with the same case and schedule (scripts/run_reference_drivers.py, recorded in
tests/golden/reference_drivers_psnr.json)."""
import json
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden", "reference_drivers_psnr.json")


def test_trainer_reaches_the_psnr_of_the_reference_drivers(tmp_path):
    with open(GOLDEN) as f:
        G = json.load(f)
    c, it = G["case"], G["iterations"]
    case = str(tmp_path / "case_phantom")
    subprocess.check_call([sys.executable, os.path.join(ROOT, "scripts", "make_synthetic_case.py"), case,
                           "--det", str(c["detector"]), "--vox", str(c["volume"]), "--train", str(c["train_views"]),
                           "--test", str(c["test_views"]), "--init", str(c["init_points"])])
    model = str(tmp_path / "model")
    r = subprocess.run([sys.executable, "-m", "r2_gaussian_b200.trainer", "-s", case, "-m", model,
                        "--iterations", str(it), "--densify_from_iter", str(G["densify_from"]),
                        "--densify_until_iter", str(G["densify_until"]), "--test_iterations", str(it)],
                       cwd=ROOT, capture_output=True, text=True, timeout=1500)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    res = json.loads(r.stdout.strip().splitlines()[-1])
    assert os.path.exists(os.path.join(model, "point_cloud", f"iteration_{it}", "point_cloud.pickle"))
    ref = G["arms"]["refkernels"]["test_eval"]["psnr_3d"]
    assert res["psnr_3d"] > 20.0, res
    assert abs(res["psnr_3d"] - ref) <= 0.2, (res["psnr_3d"], ref)
