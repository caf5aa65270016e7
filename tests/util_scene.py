"""Shared helpers for tests: small synthetic scenes in the rasterizer's post-activation input space."""
import math
from importlib import import_module

import numpy as np
import torch

synth = import_module("4dgaussians_b200.synth")


def raster_inputs(n, seed, scale_mean=0.08, sh_scale=0.3):
    """(means3D, scales, rots[normalised], opac, shs) as fp64 torch tensors that are exactly fp32-representable."""
    sc = synth.make_scene(n, seed=seed, scale_mean=scale_mean)
    g = torch.Generator().manual_seed(seed + 77)
    means3D = sc["xyz"].double()
    scales = torch.exp(sc["scaling"]).float().double()
    rots = torch.nn.functional.normalize(sc["rotation"], dim=-1).float().double()
    opac = torch.sigmoid(sc["opacity"]).float().double()
    shs = torch.cat([sc["features_dc"], torch.randn(n, 15, 3, generator=g) * sh_scale], dim=1).float().double()
    return means3D, scales, rots, opac, shs


def cam_tuple(camera, bg, sh_degree=3, scale_modifier=1.0):
    from oracle import raster_ref as rr
    from oracle.dense_ref import cam_dict_from
    cd = cam_dict_from(camera, bg, sh_degree, scale_modifier)
    rc = rr.make_cam(cd["H"], cd["W"], cd["tanfovx"], cd["tanfovy"], cd["view"], cd["proj"], cd["campos"], cd["bg"],
                     sh_degree, scale_modifier)
    # use the fp32-rounded tangents in the dense path too
    cd["tanfovx"] = float(np.float32(cd["tanfovx"])); cd["tanfovy"] = float(np.float32(cd["tanfovy"]))
    return rc, cd


# ---------------------------------------------------------------------------------------------------
# helpers for the GPU parity tests: oracle-side composition of the whole render() path
# ---------------------------------------------------------------------------------------------------
import importlib

g4d = importlib.import_module("4dgaussians_b200")


class OracleRaster(torch.autograd.Function):
    """CPU autograd wrapper around the C rasterizer oracle (forward + hand-derived backward)."""

    @staticmethod
    def forward(ctx, means3D, shs, opac, scales, rots, rc):
        from oracle import raster_ref as rr
        arrs = [t.detach().numpy().astype(np.float32) for t in (means3D, scales, rots, opac, shs)]
        f = rr.rasterize_forward(rc, *arrs)
        ctx.rc, ctx.f, ctx.arrs = rc, f, arrs
        return torch.from_numpy(f["color"].copy()), torch.from_numpy(f["depth"].copy()), torch.from_numpy(f["radii"].copy())

    @staticmethod
    def backward(ctx, g_color, _gd, _gr):
        from oracle import raster_ref as rr
        g = rr.rasterize_backward(ctx.rc, *ctx.arrs, ctx.f, g_color.numpy().astype(np.float32))
        ctx.means2D_grad = g["means2D"]
        OracleRaster.last_means2D_grad = g["means2D"]
        return (torch.from_numpy(g["means3D"]), torch.from_numpy(g["shs"]), torch.from_numpy(g["opacities"]),
                torch.from_numpy(g["scales"]), torch.from_numpy(g["rots"]), None)


def oracle_params_from_module(module):
    """DeformConfig + DeformParams (CPU fp32 leaves with requires_grad) mirroring a g4d deform_network."""
    from oracle import deform_ref as dr
    a = module.args
    kc = a.kplanes_config
    cfg = dr.DeformConfig(channels=kc["output_coordinate_dim"], resolution=tuple(kc["resolution"]), multires=tuple(a.multires),
                          net_width=a.net_width, no_dx=a.no_dx, no_ds=a.no_ds, no_dr=a.no_dr, no_do=a.no_do, no_dshs=a.no_dshs)
    sd = {k: v.detach().cpu().contiguous().clone() for k, v in module.state_dict().items()}
    prm = dr.params_from_state_dict(sd, cfg.levels)
    for t in prm.leaves():
        t.requires_grad_(True)
    return cfg, prm


def oracle_render(cfg, prm, scene_cpu, camera, t, bg, sh_degree=3, stage="fine", scale_modifier=1.0):
    """Reference composition (gaussian_renderer/__init__.py:80-128) on the oracle: deform -> activations -> rasterize.
    scene_cpu: dict of CPU tensors (leaves may require grad).  Returns (color, depth, radii, rc)."""
    from oracle import deform_ref as dr
    shs = torch.cat([scene_cpu["features_dc"], scene_cpu["features_rest"]], dim=1)
    if stage == "fine":
        pts, sc, rot, op, sh = dr.deform_forward(cfg, prm, scene_cpu["xyz"], scene_cpu["scaling"], scene_cpu["rotation"],
                                                 scene_cpu["opacity"], shs, float(t))
    else:
        pts, sc, rot, op, sh = scene_cpu["xyz"], scene_cpu["scaling"], scene_cpu["rotation"], scene_cpu["opacity"], shs
    s, r, o = dr.activate(sc, rot, op)
    rc, _ = cam_tuple(camera, bg, sh_degree=sh_degree, scale_modifier=scale_modifier)
    color, depth, radii = OracleRaster.apply(pts, sh, o, s, r, rc)
    return color, depth, radii, rc, (pts, s, r, o, sh)


def make_module(net: str, seed: int = 0, device="cuda", aabb=None):
    torch.manual_seed(1234 + seed)          # nn.Linear / plane initialisation draws from the global generator
    m = g4d.deform_network(synth.hidden_args(net))
    synth.perturb_deformation(m, seed)
    if aabb is not None:
        m.deformation_net.set_aabb(aabb[0].tolist(), aabb[1].tolist())
    return m.to(device)


def rel_err(got, ref, floor=1e-3):
    got = np.asarray(got, dtype=np.float64); ref = np.asarray(ref, dtype=np.float64)
    return float(np.abs(got - ref).max() / max(floor, np.abs(ref).max()))


def rel_err_bulk(got, ref, floor=1e-3, q=99.9):
    """(q-th percentile, max) of |got - ref| relative to max|ref|.  For gradients that pass through ReLU / floor()
    decisions: an input sitting within fp32 rounding of a kink may legitimately land on the other side on the GPU."""
    got = np.asarray(got, dtype=np.float64); ref = np.asarray(ref, dtype=np.float64)
    e = np.abs(got - ref).reshape(-1) / max(floor, np.abs(ref).max())
    return float(np.percentile(e, q)), float(e.max())


def kink_rows(cfg, prm, xyz, t, delta_act=2e-6, delta_grid=2e-4):
    """[N] bool: Gaussians sitting within rounding distance of a NON-DIFFERENTIABLE point of the deformation network,
    evaluated in fp64 on the oracle: a pre-activation of an active ReLU within delta_act of 0, or a spatial HexPlane sample
    coordinate within delta_grid (in texels) of a grid line, where floor() picks the bilinear cell.  On such rows an fp32
    implementation may legitimately take the other branch, and the gradient is then the (equally valid) one-sided
    derivative of the neighbouring piece.  Everywhere else gradients must agree to the stated tolerance.

    The time coordinate is never a kink: no gradient is taken with respect to t, and with t on a time grid line the
    bilinear weights put 1 on the same texel row whichever cell floor() picks, so the sample and its derivative along the
    spatial axis of an (a, t) plane are the same on both sides.  (t = 0 and t = 1, the first and last frame, are on grid
    lines of every time plane.)"""
    from oracle import deform_ref as dr
    with torch.no_grad():
        x64 = xyz.detach().double().cpu()
        n = x64.shape[0]
        planes = [[p.detach().double() for p in lvl] for lvl in prm.planes]
        aabb = prm.aabb.detach().double()
        tt = torch.full((n,), float(t), dtype=torch.float64)
        p = dr.normalize(x64, aabb)
        mask = torch.zeros(n, dtype=torch.bool)
        for l, lvl in enumerate(planes):
            for k, (c0, c1) in enumerate(dr.PLANE_AXES):
                _, _, H, W = lvl[k].shape
                for axis, size in ((c0, W), (c1, H)):
                    if axis == 3:
                        continue
                    g = (p[:, axis] + 1.0) / 2.0 * (size - 1)     # unclamped: far outside the aabb the border rule is smooth
                    mask |= ((g - torch.round(g)).abs() < delta_grid) & (g > -delta_grid) & (g < size - 1 + delta_grid)
        feat = dr.hexplane_features(planes, x64, aabb, tt)
        hidden = feat @ prm.w0.detach().double().t() + prm.b0.detach().double()
        mask |= (hidden.abs() < delta_act).any(dim=1)
        active = {"pos": not cfg.no_dx, "scales": not cfg.no_ds, "rotations": not cfg.no_dr, "opacity": not cfg.no_do,
                  "shs": not cfg.no_dshs}
        a = torch.relu(hidden)
        for name, on in active.items():
            if not on:
                continue
            w1, b1, _, _ = prm.heads[name]
            z = a @ w1.detach().double().t() + b1.detach().double()
            mask |= (z.abs() < delta_act).any(dim=1)
    return mask


def kink_free_scene(scene, cfg, prm, times, seed=0, max_initial_frac=0.05, rounds=8):
    """A copy of ``scene`` in which every row that ``kink_rows`` flags at any of ``times`` has been given a fresh ``xyz``,
    drawn uniformly from the scene's box (``scene["aabb"]`` when present, else the module's aabb), until no row is flagged.
    With no row at a kink, the fp32 GPU and the fp64 oracle take the same branch of every ReLU and floor(), and gradients
    can be held to the strict tolerance without a percentile.  At most ``max_initial_frac`` of the rows may be flagged to
    begin with, so the statement stays about the scene that was asked for."""
    box = scene["aabb"] if "aabb" in scene else prm.aabb.detach()
    hi, lo = box[0].float(), box[1].float()
    xyz = scene["xyz"].detach().clone()
    g = torch.Generator().manual_seed(4242 + seed)
    rows = torch.arange(xyz.shape[0])
    for r in range(rounds):
        flagged = torch.zeros(rows.shape[0], dtype=torch.bool)
        for t in times:
            flagged |= kink_rows(cfg, prm, xyz[rows], t)
        if r == 0:
            frac = float(flagged.float().mean()) if rows.numel() else 0.0
            assert frac <= max_initial_frac, ("kink rows", frac)
        rows = rows[flagged]
        if rows.numel() == 0:
            return dict(scene, xyz=xyz)
        xyz[rows] = lo + torch.rand(rows.shape[0], 3, generator=g) * (hi - lo)
    raise AssertionError("%d rows still at a kink after %d rounds" % (rows.numel(), rounds))


def params64(prm):
    """fp64 leaf copies (requires_grad) of oracle DeformParams; the aabb stays a constant."""
    from oracle import deform_ref as dr
    c = lambda x: x.detach().double().clone().requires_grad_(True)
    p64 = dr.DeformParams(aabb=prm.aabb.detach().double(), planes=[[c(p) for p in lvl] for lvl in prm.planes],
                          w0=c(prm.w0), b0=c(prm.b0), heads={k: tuple(c(x) for x in v) for k, v in prm.heads.items()})
    return p64


SCENE_LEAVES = ("xyz", "scaling", "rotation", "opacity", "features_dc", "features_rest")


def oracle_chain_grads(cfg, prm, scene, t, g_raster, stage="fine", chunk=65536):
    """fp64 backward of deform -> activations, fed with the rasterizer's gradients ``g_raster`` (what
    ``rr.rasterize_backward`` returns: dL/d means3D, activated scales, normalised rotations, activated opacities, SH).
    Runs in chunks of at most ``chunk`` rows to bound host memory; the parameter gradients accumulate across chunks.
    Returns ({scene leaf -> [N,...] fp64 gradient, "means2D" -> the rasterizer's}, {state_dict key -> fp64 gradient, or None
    for a head the config disables})."""
    from oracle import deform_ref as dr
    p64 = params64(prm)
    n = scene["xyz"].shape[0]
    gr = {k: torch.as_tensor(np.asarray(g_raster[k])).double() for k in ("means3D", "scales", "rots", "opacities", "shs")}
    out = {k: torch.zeros(scene[k].shape, dtype=torch.float64) for k in SCENE_LEAVES}
    for a in range(0, n, chunk):
        sl = slice(a, min(n, a + chunk))
        x = {k: scene[k][sl].detach().double().requires_grad_(True) for k in SCENE_LEAVES}
        shs = torch.cat([x["features_dc"], x["features_rest"]], dim=1)
        if stage == "fine":
            pts, sc, rot, op, sh = dr.deform_forward(cfg, p64, x["xyz"], x["scaling"], x["rotation"], x["opacity"], shs, float(t))
        else:
            pts, sc, rot, op, sh = x["xyz"], x["scaling"], x["rotation"], x["opacity"], shs
        s, r, o = dr.activate(sc, rot, op)
        loss = ((pts * gr["means3D"][sl]).sum() + (s * gr["scales"][sl]).sum() + (r * gr["rots"][sl]).sum()
                + (o * gr["opacities"][sl].reshape(o.shape)).sum() + (sh * gr["shs"][sl].reshape(sh.shape)).sum())
        loss.backward()
        for k in SCENE_LEAVES:
            out[k][sl] = x[k].grad
    out["means2D"] = torch.as_tensor(np.asarray(g_raster["means2D"])).double()
    params = {k: (v.grad if v.requires_grad else None) for k, v in dr.params_to_state_dict(p64).items()
              if k != "deformation_net.grid.aabb"}
    return out, params


def _assert_index_data_bit_exact(ctx, radii_gpu, ref, colour_exact=True):
    pr, bn = ref["proj"], ref["bin"]
    assert np.array_equal(radii_gpu, ref["radii"])
    for name, want in (("depth", pr.depth), ("rect", pr.rect), ("tiles_touched", pr.tiles_touched), ("xy", pr.xy),
                       ("conic_opacity", pr.conic_op), ("rgb", pr.rgb), ("clamped", pr.clamped)):
        got = ctx.read(name)
        assert got.shape == want.shape, name
        if name in ("rgb", "clamped") and not colour_exact:
            # the fused tensor-core kernel evaluates the SH polynomial with all 16 basis values in registers (a different
            # association order from the standalone preprocess kernel) and also for culled Gaussians (whose colour nobody
            # reads): colours of the VISIBLE Gaussians agree to fp32 rounding, not bit for bit
            vis = ref["radii"] > 0
            if name == "rgb":
                assert float(np.abs(got[vis] - want[vis]).max()) <= 2e-6, name
            else:
                assert float((got[vis] != want[vis]).mean()) <= 1e-4, name
            continue
        assert np.array_equal(got.view(np.uint8), want.view(np.uint8)), name
    st = ctx.stats()
    assert st.num_rendered == bn.R and st.num_visible == int((ref["radii"] > 0).sum())
    assert np.array_equal(ctx.read("sorted_ids"), bn.ids)
    assert np.array_equal(ctx.read("ranges"), bn.ranges)
    assert np.array_equal(ctx.read("sorted_keys"), bn.keys)
    return bn.R


def same_inputs_raster_grads(ctx, radii_gpu, rc, scene, has_sh_head, dL):
    """Oracle rasterizer forward + backward fed with EXACTLY the deformed, activated tensors the fused kernel handed to its
    projection stage (read from the render context ``ctx``, which must have kept them).  Asserts that the index data are
    bit-exact, so that both sides composite the same instances in the same order.  The SH colour clamp (rgb < 0) is
    a discrete decision taken on values that agree only to fp32 rounding; the oracle's backward takes the GPU's clamp bits.
    Returns (rasterizer gradients as rr.rasterize_backward gives them, number of instances R, visible clamp-bit mismatches)."""
    from oracle import raster_ref as rr
    dfm = ctx.read("deformed")
    if has_sh_head:
        shs = ctx.read("deformed_shs").reshape(-1, 16, 3)
    else:
        shs = torch.cat([scene["features_dc"], scene["features_rest"]], dim=1).numpy()
    ins = [np.ascontiguousarray(a, dtype=np.float32) for a in (dfm[:, 0:3], dfm[:, 3:6], dfm[:, 6:10], dfm[:, 10:11], shs)]
    ref = rr.rasterize_forward(rc, *ins)
    R = _assert_index_data_bit_exact(ctx, radii_gpu, ref, colour_exact=False)
    clamped = ctx.read("clamped")
    vis = ref["radii"] > 0
    n_clamp = int((clamped[vis] != ref["proj"].clamped[vis]).any(axis=-1).sum())
    ref["proj"].clamped = np.ascontiguousarray(clamped)
    g = rr.rasterize_backward(rc, *ins, ref, np.asarray(dL, dtype=np.float32))
    return g, R, n_clamp
