"""Host-side logic of the drop-in modules that needs no GPU: state_dict compatibility with the reference module,
parameter grouping, time-scalar quirks, settings tuple, oracle-side composition helpers used by the GPU tests."""
import importlib
import json
import os

import numpy as np
import pytest
import torch

from util_scene import g4d, make_module, oracle_params_from_module, oracle_render, synth

# the reference deform_network's state_dict layout and parameter groups (oracle/make_golden_reference.py)
REF_LAYOUT = os.path.join(os.path.dirname(__file__), "golden", "ref_state_dicts.json")


def test_state_dict_keys_shapes_and_layout():
    mod = g4d.deform_network(synth.hidden_args("dynerf"))
    sd = mod.state_dict()
    assert len(sd) == 43
    assert sd["deformation_net.grid.grids.0.2"].shape == (1, 16, 150, 64)     # (x,t) plane: H = T, W = 64
    assert sd["deformation_net.grid.grids.1.0"].shape == (1, 16, 128, 128)
    assert sd["deformation_net.shs_deform.3.weight"].shape == (48, 128)
    assert sd["deformation_net.grid.aabb"].shape == (2, 3)
    p = mod.deformation_net.grid.grids[0][2]
    assert p.is_contiguous(memory_format=torch.channels_last) and p.stride() == (150 * 64 * 16, 1, 64 * 16, 16)
    assert float(p.min()) == 1.0 and float(p.max()) == 1.0                      # time planes start at one
    s = mod.deformation_net.grid.grids[0][0]
    assert 0.1 <= float(s.min()) and float(s.max()) <= 0.5
    assert len(mod.get_mlp_parameters()) == 26 and len(mod.get_grid_parameters()) == 13
    mod.deformation_net.set_aabb([1.0, 2.0, 3.0], [-1.0, -2.0, -3.0])
    amax, amin = mod.get_aabb
    assert amax.tolist() == [1.0, 2.0, 3.0] and amin.tolist() == [-1.0, -2.0, -3.0]
    assert mod.head_mask() == 31
    assert g4d.deform_network(synth.hidden_args("dnerf")).head_mask() == 7


@pytest.mark.parametrize("name", ["dnerf", "hypernerf", "dynerf"])
def test_state_dict_round_trips_with_reference_module(name):
    with open(REF_LAYOUT) as f:
        ref = json.load(f)[name]
    mine = g4d.deform_network(synth.hidden_args(name))
    sd = mine.state_dict()
    # same keys in the same order, same shapes and dtypes: the reference's strict load_state_dict accepts ours
    assert list(sd.keys()) == [k for k, _, _ in ref["state_dict"]]
    for k, shape, dtype in ref["state_dict"]:
        assert list(sd[k].shape) == shape and str(sd[k].dtype) == dtype, k
    # and ours loads what the reference's state_dict() holds: plain contiguous tensors of its layout
    g = torch.Generator().manual_seed(0)
    theirs = {k: torch.rand(shape, generator=g).to(getattr(torch, dtype.split(".")[1])) for k, shape, dtype in ref["state_dict"]}
    mine.load_state_dict(theirs)
    assert all(torch.equal(v, theirs[k]) for k, v in mine.state_dict().items())
    assert mine.deformation_net.grid.grids[0][0].is_contiguous(memory_format=torch.channels_last)
    assert [list(p.shape) for p in mine.get_mlp_parameters()] == ref["mlp_parameters"]
    assert [list(p.shape) for p in mine.get_grid_parameters()] == ref["grid_parameters"]


def test_flat_parameter_cache_follows_the_module():
    """flat_parameters() caches the Parameter OBJECTS in C-ABI order (nn.Module container indexing costs ~0.1 ms per render): the
    cache must survive in-place updates (load_state_dict, optimizer steps) and be dropped by .to()/.float() and invalidate_cache()."""
    mod = g4d.deform_network(synth.hidden_args("dynerf"))
    a = mod.flat_parameters()
    assert len(a) == 12 + 2 + 4 * 5
    assert a[12] is mod.deformation_net.feature_out[0].weight and a[-1] is mod.deformation_net.shs_deform[3].bias
    b = mod.flat_parameters()
    assert all(x is y for x, y in zip(a, b)) and a is not b                 # same objects, a fresh list each call
    mod.load_state_dict({k: v.clone() for k, v in mod.state_dict().items()})
    assert all(x is y for x, y in zip(a, mod.flat_parameters()))
    mod.double(); mod.float()                                                # _apply: the cache is rebuilt
    c = mod.flat_parameters()
    assert all(x is y for x, y in zip(c, [p for lvl in mod.deformation_net.grid.grids for p in lvl]))
    mod.invalidate_cache()
    assert mod._flat_cache is None and len(mod.flat_parameters()) == len(a)


def test_scalar_time_quirks():
    d = importlib.import_module("4dgaussians_b200.deformation")
    assert d.scalar_time(0) == 0.0 and d.scalar_time(0.25) == 0.25
    assert d.scalar_time(torch.tensor(0.5)) == 0.5
    assert d.scalar_time(torch.tensor(0.75).repeat(7, 1)) == 0.75
    assert d.scalar_time(torch.zeros(3, 1, dtype=torch.int64)) == 0.0
    with pytest.raises(RuntimeError):
        d.scalar_time(None)


def test_dead_options_are_rejected():
    a = synth.hidden_args("dnerf")
    a.static_mlp = True
    with pytest.raises(NotImplementedError):
        g4d.deform_network(a)


def test_settings_namedtuple_and_dropin_install():
    rs = g4d.GaussianRasterizationSettings(image_height=4, image_width=5, tanfovx=0.5, tanfovy=0.4, bg=torch.zeros(3),
                                           scale_modifier=1.0, viewmatrix=torch.eye(4), projmatrix=torch.eye(4), sh_degree=3,
                                           campos=torch.zeros(3), prefiltered=False, debug=False)
    assert rs._fields == ("image_height", "image_width", "tanfovx", "tanfovy", "bg", "scale_modifier", "viewmatrix",
                          "projmatrix", "sh_degree", "campos", "prefiltered", "debug")
    importlib.import_module("4dgaussians_b200.dropin").install()
    from diff_gaussian_rasterization import GaussianRasterizationSettings, GaussianRasterizer  # noqa: F401
    assert GaussianRasterizer is g4d.GaussianRasterizer
    rz = importlib.import_module("4dgaussians_b200.rasterizer")
    cam = rz.camera_from_settings(rs, time=0.3)
    assert cam.image_width == 5 and abs(cam.time - 0.3) < 1e-7 and cam.viewmatrix[5] == 1.0 and not cam.d_viewmatrix
    r = GaussianRasterizer(rs)
    with pytest.raises(Exception, match="excatly one"):
        r(means3D=None, means2D=None, opacities=None, shs=None, colors_precomp=None, scales=1, rotations=1)


def test_oracle_composition_helpers_run_on_cpu():
    """The oracle-side render composition used by the GPU tests (deform oracle -> activations -> C rasterizer oracle,
    with autograd through all of it)."""
    scene = synth.make_scene(300, seed=1, scale_mean=0.1)
    mod = make_module("small64", seed=1, device="cpu", aabb=scene["aabb"])
    cfg, prm = oracle_params_from_module(mod)
    cam = synth.make_camera(10.0, 48, 32, time=0.4)
    leaves = {k: v.clone().requires_grad_(True) for k, v in scene.items() if k != "aabb"}
    color, depth, radii, rc, _ = oracle_render(cfg, prm, leaves, cam, 0.4, (1, 1, 1), sh_degree=2)
    assert color.shape == (3, 32, 48) and int((radii > 0).sum()) > 10
    color.sum().backward()
    assert float(leaves["xyz"].grad.abs().max()) > 0 and float(prm.w0.grad.abs().max()) > 0
    assert float(prm.planes[0][2].grad.abs().max()) > 0
