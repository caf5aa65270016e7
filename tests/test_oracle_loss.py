"""Pins oracle/loss_ref.py (CPU restatement of l1_loss / ssim / compute_regulation) to the reference:
golden vectors produced by the reference's own functions (tests/golden/loss_ref.npz), and the values those functions
give on a second set of inputs (tests/golden/ref_outputs.npz, oracle/make_golden_reference.py)."""
import os

import numpy as np
import torch

from oracle import loss_ref as lr
from oracle.make_golden_loss import inputs

GOLD = os.path.join(os.path.dirname(__file__), "golden", "loss_ref.npz")
REF_OUTPUTS = os.path.join(os.path.dirname(__file__), "golden", "ref_outputs.npz")


def test_loss_oracle_matches_reference_goldens():
    z = np.load(GOLD)
    img1, img2, grids = inputs()
    a = img1.clone().requires_grad_(True)
    l = lr.l1_loss(a, img2); l.backward()
    assert abs(float(l) - float(z["l1"])) <= 1e-14 and np.abs(a.grad.numpy() - z["l1_grad"]).max() <= 1e-16
    a = img1.float().clone().requires_grad_(True)
    s = lr.ssim(a, img2.float()); s.backward()
    assert abs(float(s) - float(z["ssim"])) <= 1e-6 and np.abs(a.grad.numpy() - z["ssim_grad"]).max() <= 1e-8
    leaves = [[p.clone().requires_grad_(True) for p in lvl] for lvl in grids]
    w = tuple(float(x) for x in z["reg_weights"])
    r = lr.compute_regulation(leaves, *w); r.backward()
    assert abs(float(r) - float(z["reg"])) <= 1e-15
    for l_, lvl in enumerate(leaves):
        for k, p in enumerate(lvl):
            assert np.abs(p.grad.numpy() - z["reg_grad_%d_%d" % (l_, k)]).max() <= 1e-15, (l_, k)


def test_loss_oracle_matches_reference_live():
    z = np.load(REF_OUTPUTS)
    img1, img2, grids = inputs(seed=5)
    assert abs(float(lr.l1_loss(img1, img2)) - float(z["loss_l1"])) <= 1e-15
    assert abs(float(lr.ssim(img1.float(), img2.float())) - float(z["loss_ssim"])) <= 1e-6
    w = tuple(float(x) for x in z["loss_reg_weights"])
    assert abs(float(lr.compute_regulation(grids, *w)) - float(z["loss_reg"])) <= 1e-15
