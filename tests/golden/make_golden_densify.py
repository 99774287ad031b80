"""Writes tests/golden/densify_prune_reference.json: the reference's own GaussianModel.densify_and_prune
(r2_gaussian/gaussian/gaussian_model.py of the original R2-Gaussian code), run on a GPU from the state
tests/test_train_gpu.py::densify_case builds, recorded as SHA-256 digests of every tensor it leaves behind.

    python tests/golden/make_golden_densify.py --reference <dir holding the reference's r2_gaussian/> [--out FILE]

The reference's module imports plyfile at load time; scripts/ref_shims stands in for it, and simple_knn is this
repository's.  Run it with the same torch as the tests: the starting state is drawn from torch's CUDA generator, and
the test checks that it starts from the recorded state before it compares the result.
"""
import argparse
import importlib
import json
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reference", required=True)
    ap.add_argument("--out", default=os.path.join(HERE, "densify_prune_reference.json"))
    a = ap.parse_args()
    for p in (ROOT, os.path.join(ROOT, "tests"), os.path.join(ROOT, "scripts", "ref_shims"), os.path.abspath(a.reference)):
        sys.path.insert(0, p)
    import test_train_gpu as T

    RefModel = importlib.import_module("r2_gaussian.gaussian.gaussian_model").GaussianModel
    golden = {}
    for max_num in (None, 10):
        gm, xyz, dens, args = T.densify_case(max_num)
        ref = RefModel(np.array(gm.scale_bound))
        ref.create_from_pcd(xyz, dens, 1.0)
        ref.training_setup(T._opt_args())
        with torch.no_grad():
            for name, attr in T.DENSIFY_GROUPS:
                getattr(ref, attr).copy_(getattr(gm, attr))
        for g_ref, (name, attr) in zip(ref.optimizer.param_groups, T.DENSIFY_GROUPS):
            assert g_ref["name"] == name
            src = gm.optimizer.state[getattr(gm, attr)]
            ref.optimizer.state[g_ref["params"][0]] = {"step": src["step"].clone(), "exp_avg": src["exp_avg"].clone(),
                                                       "exp_avg_sq": src["exp_avg_sq"].clone()}
        ref.max_radii2D = gm.max_radii2D.clone()
        ref.xyz_gradient_accum = gm.xyz_gradient_accum.clone()
        ref.denom = gm.denom.clone()
        before = T.densify_state_digests(ref)
        assert before == T.densify_state_digests(gm)
        torch.manual_seed(123)
        with torch.no_grad():
            returned = ref.densify_and_prune(*args)
        golden[str(max_num)] = {
            "before": before,
            "returned": T.tensor_digest(returned),
            "cuda_rng_state_after": torch.cuda.get_rng_state().numpy().tobytes().hex(),
            "after": T.densify_state_digests(ref),
        }
    golden["recorded_with"] = {"torch": torch.__version__, "device": torch.cuda.get_device_name(0)}
    with open(a.out, "w") as f:
        json.dump(golden, f, indent=1)
    print(f"wrote {a.out}")


if __name__ == "__main__":
    main()
