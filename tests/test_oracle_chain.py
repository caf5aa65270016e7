"""The backward-parity harness itself (util_scene), on the CPU: the fp64 chain oracle against autograd through the whole
oracle composition, the kink-free scene, and kink_rows at the last frame (t = 1)."""
import numpy as np
import torch

from oracle import deform_ref as dr
from oracle import raster_ref as rr
from util_scene import (SCENE_LEAVES, kink_free_scene, kink_rows, make_module, oracle_chain_grads,
                        oracle_params_from_module, oracle_render, rel_err, synth)

T = 0.35


def _small(net="small128", n=1500, seed=3):
    scene = synth.make_scene(n, seed=seed, scale_mean=0.05)
    mod = make_module(net, seed=seed, device="cpu", aabb=scene["aabb"])
    cfg, prm = oracle_params_from_module(mod)
    return scene, cfg, prm


def test_chain_oracle_matches_autograd_through_oracle_render():
    scene, cfg, prm = _small()
    scene = kink_free_scene(scene, cfg, prm, [T])
    cam = synth.make_camera(25.0, 96, 72, radius=3.0, time=T)
    bg = (0.1, 0.2, 0.3)
    leaves = {k: scene[k].clone().requires_grad_(True) for k in SCENE_LEAVES}
    color, _, radii, rc, (pts, s, r, o, sh) = oracle_render(cfg, prm, leaves, cam, T, bg, sh_degree=3)
    dL = torch.randn(color.shape, generator=torch.Generator().manual_seed(1))
    (color * dL).sum().backward()
    assert int((radii > 0).sum()) > 100
    ins = [x.detach().numpy().astype(np.float32) for x in (pts, s, r, o, sh)]
    g_r = rr.rasterize_backward(rc, *ins, rr.rasterize_forward(rc, *ins), dL.numpy())
    per, params = oracle_chain_grads(cfg, prm, scene, T, g_r, chunk=400)      # several chunks: parameter grads accumulate
    for k in SCENE_LEAVES:
        assert float(leaves[k].grad.abs().max()) > 0, k
        assert rel_err(per[k].numpy(), leaves[k].grad.numpy()) <= 1e-4, k
    assert np.array_equal(per["means2D"].numpy(), g_r["means2D"])
    ref = dr.params_to_state_dict(prm)
    assert set(params) == set(ref) - {"deformation_net.grid.aabb"}
    for k, g in params.items():
        if ref[k].grad is None:
            assert g is None, k
        else:
            assert float(ref[k].grad.abs().max()) > 0, k
            assert rel_err(g.numpy(), ref[k].grad.numpy()) <= 1e-4, k


def test_kink_free_scene_has_no_kink_rows():
    scene, cfg, prm = _small("dynerf", n=20000)
    times = [0.0, T, 1.0]
    before = sum(int(kink_rows(cfg, prm, scene["xyz"], t).sum()) for t in times)
    assert before > 0                                   # something had to be re-drawn
    free = kink_free_scene(scene, cfg, prm, times)
    for t in times:
        assert not bool(kink_rows(cfg, prm, free["xyz"], t).any()), t
    moved = (free["xyz"] != scene["xyz"]).any(dim=1)
    assert 0 < int(moved.sum()) <= before
    lo, hi = scene["aabb"][1], scene["aabb"][0]
    assert bool(((free["xyz"] >= lo) & (free["xyz"] <= hi)).all())
    for k in SCENE_LEAVES[1:]:
        assert free[k] is scene[k]


def test_kink_rows_at_the_last_frame_flags_only_spatial_kinks():
    """t = 1 lies on the last grid line of every time plane: that must not flag every row (no gradient is taken with
    respect to t).  A row put on a spatial grid line is still flagged, at t = 1 as at any other time."""
    scene, cfg, prm = _small("dnerf", n=5000)
    xyz = scene["xyz"].clone()
    hi, lo = prm.aabb[0].detach(), prm.aabb[1].detach()
    W = prm.planes[0][0].shape[3]                       # plane (x, y): W follows x
    xyz[0, 0] = float(hi[0] + (lo[0] - hi[0]) * 17 / (W - 1))    # normalised x on grid line 17
    for t in (1.0, 0.0, T):
        m = kink_rows(cfg, prm, xyz, t)
        assert bool(m[0]), t
        assert float(m.float().mean()) <= 0.05, (t, float(m.float().mean()))
