"""Golden data for the tests that compare with the REFERENCE's own modules, so that they run without the reference tree.

TEST INFRASTRUCTURE ONLY.  Run where the reference tree is present (``G4D_REFERENCE_ROOT``):
    python oracle/make_golden_reference.py
Writes
  * tests/golden/ref_state_dicts.json: for the dnerf / hypernerf / dynerf configs, the reference ``deform_network``'s
    state_dict (key order, shape, dtype) and the shapes of its ``get_mlp_parameters()`` / ``get_grid_parameters()`` groups;
  * tests/golden/ref_outputs.npz: the reference module's fp64 forward (seed-11 weights, 129 seed-7 points, t = 0.73) for
    the tiny and dynerf configs, and its l1_loss / ssim / regulariser on the seed-5 inputs of make_golden_loss.py.
"""
from __future__ import annotations

import json
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))

from oracle import deform_ref as dr  # noqa: E402
from oracle.make_golden_deform import param_checksum, synth_inputs  # noqa: E402
from oracle.make_golden_loss import inputs, load_reference_loss_modules, reference_compute_regulation  # noqa: E402
from oracle.ref_loader import load_reference_deform_network  # noqa: E402

GOLD = os.path.join(os.path.dirname(HERE), "tests", "golden")
AABB = torch.tensor([[1.31, 1.27, 1.3], [-1.29, -1.3, -1.22]])
DEFORM_OUTPUTS = ("pts", "scales", "rot", "opacity", "shs")
FP64_SEED, FP64_POINTS, FP64_POINT_SEED, FP64_TIME = 11, 129, 7, 0.73
LOSS_SEED, LOSS_WEIGHTS = 5, (0.01, 0.0001, 0.0001)


def state_dict_layouts():
    out = {}
    for name in ("dnerf", "hypernerf", "dynerf"):
        net = load_reference_deform_network(dr.CONFIGS[name])
        out[name] = {"state_dict": [[k, list(v.shape), str(v.dtype)] for k, v in net.state_dict().items()],
                     "mlp_parameters": [list(p.shape) for p in net.get_mlp_parameters()],
                     "grid_parameters": [list(p.shape) for p in net.get_grid_parameters()]}
    return out


def reference_outputs():
    out = {}
    for name in ("tiny", "dynerf"):
        cfg = dr.CONFIGS[name]
        prm = dr.random_params(cfg, seed=FP64_SEED, aabb=AABB, dtype=torch.float64)
        net = load_reference_deform_network(cfg).double()
        sd = net.state_dict()
        sd.update(dr.params_to_state_dict(prm))
        net.load_state_dict(sd)
        (xyz, sc, rot, op, shs), _ = synth_inputs(FP64_POINTS, FP64_POINT_SEED, dtype=torch.float64)
        with torch.no_grad():
            ref = net(xyz, sc, rot, op, shs, torch.tensor(FP64_TIME, dtype=torch.float64).repeat(FP64_POINTS, 1))
        out["deform_%s_param_checksum" % name] = np.float64(param_checksum(prm))
        for nm, o in zip(DEFORM_OUTPUTS, ref):
            out["deform_%s_%s" % (name, nm)] = o.numpy()
    lu, reg = load_reference_loss_modules()
    img1, img2, grids = inputs(seed=LOSS_SEED)
    out["loss_l1"] = lu.l1_loss(img1, img2).numpy()
    out["loss_ssim"] = lu.ssim(img1.float(), img2.float()).numpy()
    out["loss_reg"] = reference_compute_regulation(reg, grids, *LOSS_WEIGHTS).numpy()
    out["loss_reg_weights"] = np.array(LOSS_WEIGHTS)
    return out


def main():
    path = os.path.join(GOLD, "ref_state_dicts.json")
    with open(path, "w") as f:
        json.dump(state_dict_layouts(), f, indent=1)
        f.write("\n")
    print("wrote", path)
    path = os.path.join(GOLD, "ref_outputs.npz")
    np.savez_compressed(path, **reference_outputs())
    print("wrote", path, os.path.getsize(path) // 1024, "KiB")


if __name__ == "__main__":
    main()
