"""Pins oracle/deform_ref.py against golden vectors produced by the REFERENCE's own
scene.deformation.deform_network (oracle/make_golden_deform.py, and its fp64 forward from
oracle/make_golden_reference.py)."""
import os

import numpy as np
import pytest
import torch

from oracle import deform_ref as dr
from oracle.make_golden_deform import param_checksum, synth_inputs

GOLD = os.path.join(os.path.dirname(__file__), "golden")
AABB = torch.tensor([[1.31, 1.27, 1.3], [-1.29, -1.3, -1.22]])
NAMES = ("pts", "scales", "rot", "opacity", "shs")


def _load(name):
    z = np.load(os.path.join(GOLD, f"deform_{name}.npz"))
    cfg = dr.CONFIGS[name]
    prm = dr.random_params(cfg, seed=int(z["seed"]), aabb=AABB)
    assert abs(param_checksum(prm) - float(z["param_checksum"])) <= 1e-6 * float(z["param_checksum"]), \
        "CPU RNG drift: regenerate goldens"
    return z, cfg, prm


@pytest.mark.parametrize("name", ["tiny", "dnerf", "hypernerf", "dynerf"])
def test_forward_matches_reference_golden(name):
    z, cfg, prm = _load(name)
    (xyz, sc, rot, op, shs), _ = synth_inputs(int(z["n"]), int(z["seed"]))
    for ti, t in enumerate(z["times"]):
        outs = dr.deform_forward(cfg, prm, xyz, sc, rot, op, shs, float(t))
        for nm, o in zip(NAMES, outs):
            ref = torch.from_numpy(z[f"t{ti}_{nm}"])
            assert o.shape == ref.shape
            # fp32 vs fp32: summation order differs (ATen GEMM vs matmul here) -> a few ulp
            assert (o - ref).abs().max().item() <= 2e-5, (name, nm)


@pytest.mark.parametrize("name", ["tiny", "dynerf"])
def test_forward_fp64_restatement_close_to_fp32_golden(name):
    z, cfg, prm = _load(name)
    (xyz, sc, rot, op, shs), _ = synth_inputs(int(z["n"]), int(z["seed"]))
    p64 = prm.to(torch.float64)
    outs = dr.deform_forward(cfg, p64, xyz.double(), sc.double(), rot.double(), op.double(), shs.double(),
                             float(z["times"][0]))
    for nm, o in zip(NAMES, outs):
        assert (o - torch.from_numpy(z[f"t0_{nm}"]).double()).abs().max().item() <= 2e-5


@pytest.mark.parametrize("name", ["tiny", "dnerf", "dynerf"])
def test_backward_matches_reference_golden(name):
    z, cfg, prm = _load(name)
    (xyz, sc, rot, op, shs), probes = synth_inputs(int(z["n"]), int(z["seed"]))
    for ti, t in enumerate(z["times"]):
        xyz_r = xyz.clone().requires_grad_(True)
        w0 = prm.w0.clone().requires_grad_(True)
        p02 = prm.planes[0][2].clone().requires_grad_(True)
        p10 = prm.planes[1][0].clone().requires_grad_(True)
        planes = [list(l) for l in prm.planes]
        planes[0][2] = p02
        planes[1][0] = p10
        q = dr.DeformParams(aabb=prm.aabb, planes=planes, w0=w0, b0=prm.b0, heads=prm.heads)
        outs = dr.deform_forward(cfg, q, xyz_r, sc, rot, op, shs, float(t))
        loss = sum((o * p).sum() for o, p in zip(outs, probes))
        loss.backward()
        for got, key in ((xyz_r.grad, "g_xyz"), (w0.grad, "g_w0"), (p02.grad, "g_plane02"), (p10.grad, "g_plane10")):
            ref = torch.from_numpy(z[f"t{ti}_{key}"])
            scale = max(1.0, ref.abs().max().item())
            assert (got - ref).abs().max().item() <= 5e-5 * scale, (name, key)


def test_tiny_golden_stores_weights_explicitly():
    z, cfg, prm = _load("tiny")
    for k, v in dr.params_to_state_dict(prm).items():
        assert np.array_equal(z["w_" + k], v.numpy())


def test_state_dict_round_trip():
    cfg = dr.CONFIGS["tiny"]
    prm = dr.random_params(cfg, seed=5)
    back = dr.params_from_state_dict(dr.params_to_state_dict(prm), cfg.levels)
    for a, b in zip(prm.leaves(), back.leaves()):
        assert torch.equal(a, b)


def test_time_axis_and_flipped_aabb_quirks():
    """SURVEY §8a3: xyz_max maps to -1 (first texel), t=0 maps to the CENTRE row of the time axis."""
    cfg = dr.DeformConfig(channels=1, resolution=(3, 3, 3, 5), multires=(1,), net_width=4)
    prm = dr.random_params(cfg, seed=0, dtype=torch.float64)
    for k in range(6):
        prm.planes[0][k].fill_(1.0)
    ramp = torch.arange(5, dtype=torch.float64).reshape(1, 1, 5, 1).expand(1, 1, 5, 3).clone()
    prm.planes[0][2] = ramp                     # plane (x,t): H axis is t
    xyz = prm.aabb[0:1].clone()                 # the max corner
    f0 = dr.hexplane_features(prm.planes, xyz, prm.aabb, torch.tensor([0.0], dtype=torch.float64))
    f1 = dr.hexplane_features(prm.planes, xyz, prm.aabb, torch.tensor([1.0], dtype=torch.float64))
    assert abs(f0.item() - 2.0) < 1e-12 and abs(f1.item() - 4.0) < 1e-12
    assert torch.allclose(dr.normalize(xyz, prm.aabb), -torch.ones(1, 3, dtype=torch.float64))


@pytest.mark.parametrize("name", ["tiny", "dynerf"])
def test_live_reference_module_fp64(name):
    """The reference module run in fp64 on the same weights and points (tests/golden/ref_outputs.npz)."""
    z = np.load(os.path.join(GOLD, "ref_outputs.npz"))
    cfg = dr.CONFIGS[name]
    prm = dr.random_params(cfg, seed=11, aabb=AABB, dtype=torch.float64)
    want = float(z[f"deform_{name}_param_checksum"])
    assert abs(param_checksum(prm) - want) <= 1e-12 * want, "CPU RNG drift: regenerate goldens"
    (xyz, sc, rot, op, shs), _ = synth_inputs(129, 7, dtype=torch.float64)
    got = dr.deform_forward(cfg, prm, xyz, sc, rot, op, shs, 0.73)
    for nm, a in zip(NAMES, got):
        b = torch.from_numpy(z[f"deform_{name}_{nm}"])
        assert a.shape == b.shape and (a - b).abs().max().item() < 1e-12, nm
