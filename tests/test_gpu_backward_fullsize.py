"""Full-size backward parity: render() gradients at the BASELINE sizes C1 (70k, dnerf net -> FFMA backward), C2 (200k,
hypernerf net, L=3) and C3 (300k, dynerf net, 5 heads) against an fp64 oracle -- the sizes at which the persistent dgrad
loop, the FFMA backward's per-CTA accumulators and the split-K tensor-core weight-gradient kernel own many tiles per CTA.

Two discrete effects would make the GPU and the oracle take different branches; both are removed instead of tolerated:
  (i)  rasterizer decisions: the oracle rasterizer is fed the GPU's own deformed tensors (index data asserted bit-exact) and
       the same dL/dcolor (util_scene.same_inputs_raster_grads);
  (ii) deformation kinks: every row near a ReLU kink or a spatial HexPlane grid line at any of the test's times is re-drawn
       (util_scene.kink_free_scene), then the rasterizer's gradients are pushed through activations and deformation in
       fp64 autograd (util_scene.oracle_chain_grads).
Every gradient -- the six per-Gaussian tensors, the screen-space points, every plane, w0 / b0 and every head's weights --
is then held to GRAD_TOL relative to the tensor's max, with no percentile.  The measured errors go to the same statistics
file as the forward's (test_gpu_fullsize._record).
"""
import importlib

import numpy as np
import pytest
import torch

from test_gpu_fullsize import _record
from util_scene import (SCENE_LEAVES, cam_tuple, g4d, kink_free_scene, make_module, oracle_chain_grads,
                        oracle_params_from_module, rel_err, same_inputs_raster_grads, synth)

pytestmark = pytest.mark.gpu
GRAD_TOL = 2e-3
td = importlib.import_module("4dgaussians_b200.train_dp")


class _Pipe:
    convert_SHs_python = False
    compute_cov3D_python = False
    debug = False


def _setup(wl, times, aabb_scale=1.0, seed=0):
    w = synth.WORKLOADS[wl]
    scene = synth.make_scene(w["n"], seed=seed, scale_mean=w["scale_mean"])
    mod = make_module(w["net"], seed=seed, aabb=scene["aabb"] * aabb_scale)
    cfg, prm = oracle_params_from_module(mod)
    scene = kink_free_scene(scene, cfg, prm, times, seed=seed)
    return w, scene, mod, cfg, prm


def _view(w, theta, t, seed):
    cam = synth.make_camera(theta, w["width"], w["height"], radius=w["radius"], focal=w["focal"], time=t)
    rc, _ = cam_tuple(cam, w["bg"], sh_degree=3)
    dL = torch.randn(3, w["height"], w["width"], generator=torch.Generator().manual_seed(seed))
    return cam, rc, dL


def _oracle_view(out, mod, cfg, prm, scene, rc, t, dL):
    """Oracle gradients of one rendered view; `out` is the render() result, whose context still holds the forward."""
    ctx = out["render"].grad_fn.lease.ctx
    g_r, R, n_clamp = same_inputs_raster_grads(ctx, out["radii"].cpu().numpy(), rc, scene, not mod.args.no_dshs, dL)
    per, params = oracle_chain_grads(cfg, prm, scene, t, g_r)
    return per, params, {"R": int(R), "clamp_bit_mismatch": n_clamp}


def _compare(gpu_per, mod, per, params):
    """rel. errors of every gradient; asserts the vacuity guards (enabled heads non-zero, disabled heads no gradient)"""
    stats = {}
    for k, g in gpu_per.items():
        assert float(per[k].abs().max()) > 0, k
        stats[k] = rel_err(g.detach().cpu().numpy().reshape(per[k].shape), per[k].numpy())
    for k, p in mod.named_parameters():
        if k not in params:
            continue
        ref = params[k]
        if ref is None:                      # a head the config disables
            assert p.grad is None or float(p.grad.abs().max()) == 0.0, k
            continue
        assert float(ref.abs().max()) > 0, k
        assert p.grad is not None, k
        stats[k] = rel_err(p.grad.cpu().numpy(), ref.numpy())
    return stats


def _assert_within(stats):
    bad = {k: e for k, e in stats.items() if isinstance(e, float) and e > GRAD_TOL}
    assert not bad, bad


def _render_backward_case(wl, t, theta, aabb_scale=1.0, key=None):
    w, scene, mod, cfg, prm = _setup(wl, [t], aabb_scale=aabb_scale)
    pc = synth.SyntheticGaussianModel(scene, mod, sh_degree=3, requires_grad=True)
    cam, rc, dL = _view(w, theta, t, seed=7)
    out = g4d.render(cam, pc, _Pipe(), torch.tensor(w["bg"], dtype=torch.float32, device="cuda"))
    per, params, info = _oracle_view(out, mod, cfg, prm, scene, rc, t, dL)
    out["render"].backward(dL.cuda())
    gpu = dict(zip(SCENE_LEAVES, pc.gaussian_parameters()))
    gpu = {k: p.grad for k, p in gpu.items()}
    gpu["means2D"] = out["viewspace_points"].grad
    stats = _compare(gpu, mod, per, params)
    info["max_rel_err"] = max(stats.values())
    _record(key or "render_bwd_%s" % wl, dict(stats, **info))
    _assert_within(stats)
    return scene, mod


@pytest.mark.parametrize("wl,t,theta", [("C1", 0.0, 30.0), ("C2", 0.55, -20.0), ("C3", 0.8, 30.0)])
def test_full_size_render_backward_vs_fp64_oracle(wl, t, theta):
    _render_backward_case(wl, t, theta)


def test_full_size_render_backward_points_outside_aabb():
    """C2 size with the aabb shrunk to 0.8: about a third of the points sample the planes through the border clamp, where
    the xyz gradient of the clamped coordinates is zero."""
    scene, mod = _render_backward_case("C2", 1.0, 60.0, aabb_scale=0.8, key="render_bwd_C2_outside_aabb")
    aabb = mod.deformation_net.grid.aabb.detach().cpu()
    inside = ((scene["xyz"] <= aabb[0]) & (scene["xyz"] >= aabb[1])).all(dim=1)
    assert 0.2 < float((~inside).float().mean()) < 0.8


def test_train_step_fused_accumulation_C3_vs_fp64_oracle():
    """The training path: DPTrainer's FlatState (network gradients accumulated by the kernels straight into the flat
    buffer, deform_network.fused_grad_accumulation) over two views with different cameras at t = 0 and t = 1 (the first
    and last frame of the reference loaders' time / max_time).  First forward -> backward per view, as DPTrainer.step
    does; then both forwards before both backwards (the reference's batch_size > 1 pattern).  Both times every slice of
    the flat gradient buffer must equal the sum of the two views' oracle gradients."""
    views = [(30.0, 0.0, 11), (-75.0, 1.0, 12)]
    w, scene, mod, cfg, prm = _setup("C3", [t for _, t, _ in views])
    gs = td.GaussianSet(scene, mod)
    tr = td.DPTrainer(gs)
    assert mod.fused_grad_accumulation
    bg = torch.tensor(w["bg"], dtype=torch.float32, device="cuda")
    cams = [_view(w, th, t, s) for th, t, s in views]
    per_sum, par_sum, m2d_ref, deformed, infos = None, None, [], [], {}
    for order in ("per_view", "batched"):
        tr.state.zero_grad()
        outs = []
        for i, (cam, rc, dL) in enumerate(cams):
            out = g4d.render(cam, gs, _Pipe, bg)
            ctx = out["render"].grad_fn.lease.ctx
            if order == "per_view":
                deformed.append(ctx.read("deformed"))
                per, params, infos["view%d" % i] = _oracle_view(out, mod, cfg, prm, scene, rc, views[i][1], dL)
                m2d_ref.append(per.pop("means2D"))
                per_sum = per if per_sum is None else {k: per_sum[k] + per[k] for k in per}
                par_sum = params if par_sum is None else {k: None if v is None else par_sum[k] + v for k, v in params.items()}
                out["render"].backward(dL.cuda())
            else:                                # the same forward as in the first pass: the oracle above applies
                assert np.array_equal(ctx.read("deformed"), deformed[i])
            outs.append(out)
        if order == "batched":
            torch.autograd.backward([o["render"] for o in outs], [dL.cuda() for _, _, dL in cams])
        assert tr.state.attached()               # every .grad below is a view of its flat-buffer slice
        gpu = dict(zip(SCENE_LEAVES, (gs._xyz, gs._scaling, gs._rotation, gs._opacity, gs._features_dc, gs._features_rest)))
        stats = _compare({k: p.grad for k, p in gpu.items()}, mod, per_sum, par_sum)
        for i, out in enumerate(outs):           # the screen-space points are per view, not accumulated
            stats["means2D_view%d" % i] = rel_err(out["viewspace_points"].grad.cpu().numpy(), m2d_ref[i].numpy())
        _record("train_step_C3_%s" % order, dict(stats, **infos, max_rel_err=max(stats.values())))
        _assert_within(stats)
