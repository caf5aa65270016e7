"""Import the REFERENCE's own ``scene.deformation.deform_network`` on CPU (this container only).

TEST / BASELINE INFRASTRUCTURE ONLY.  /root/reference does not exist on the GPU box: there the unmodified copies that
``oracle/make_ref.py`` put into ``oracle/_ref/`` at build() time are imported instead; callers must check
``reference_available()`` first.  Used by the ``oracle/make_golden_*.py`` scripts (the golden vectors the tests
compare against) and by ``bench.py --impl reference`` when present.

Two shims make the module importable without the reference's heavy dependencies (SURVEY §8c):
  * an empty package object ``scene`` whose ``__path__`` points at /root/reference/scene, so
    ``scene/__init__.py`` (plyfile / open3d / simple_knn imports) never runs;
  * a stub ``tkinter`` exposing ``W`` (``scene/deformation.py:5`` does ``from tkinter import W``).
Nothing is copied: the reference sources are imported from where they lie.
"""
from __future__ import annotations

import os
import sys
import types
from argparse import Namespace

_HERE = os.path.dirname(os.path.abspath(__file__))
REF_ROOT = os.environ.get("G4D_REFERENCE_ROOT", "/root/reference")
if not os.path.isfile(os.path.join(REF_ROOT, "scene", "deformation.py")):
    # GPU box: the unmodified copies made by oracle/make_ref.py at build() time (git-ignored, shipped with the snapshot)
    REF_ROOT = os.path.join(_HERE, "_ref")


def reference_available() -> bool:
    return os.path.isfile(os.path.join(REF_ROOT, "scene", "deformation.py"))


def reference_origin() -> str:
    return "oracle/_ref (copied from /root/reference at build time)" if REF_ROOT.endswith("_ref") else REF_ROOT


def _install_shims():
    if "tkinter" not in sys.modules:
        try:
            import tkinter  # noqa: F401
        except Exception:
            tk = types.ModuleType("tkinter")
            tk.W = "w"
            sys.modules["tkinter"] = tk
    if "scene" not in sys.modules or not hasattr(sys.modules["scene"], "__path__") or \
            os.path.join(REF_ROOT, "scene") not in list(sys.modules["scene"].__path__):
        pkg = types.ModuleType("scene")
        pkg.__path__ = [os.path.join(REF_ROOT, "scene")]
        sys.modules["scene"] = pkg
    if REF_ROOT not in sys.path:
        sys.path.append(REF_ROOT)      # for ``utils.graphics_utils``


def hidden_args(cfg) -> Namespace:
    """ModelHiddenParams (arguments/__init__.py:74-107) with the path-shaping fields taken from cfg."""
    return Namespace(
        net_width=cfg.net_width, timebase_pe=4, defor_depth=1, posebase_pe=10, scale_rotation_pe=2,
        opacity_pe=2, timenet_width=64, timenet_output=32, bounds=1.6, grid_pe=0,
        kplanes_config={"grid_dimensions": 2, "input_coordinate_dim": 4,
                        "output_coordinate_dim": cfg.channels, "resolution": list(cfg.resolution)},
        multires=list(cfg.multires), no_dx=cfg.no_dx, no_grid=False, no_ds=cfg.no_ds, no_dr=cfg.no_dr,
        no_do=cfg.no_do, no_dshs=cfg.no_dshs, empty_voxel=False, static_mlp=False, apply_rotation=False)


def load_reference_deform_network(cfg):
    """Returns an instance of the reference's ``deform_network`` built for ``cfg`` (CPU, fp32)."""
    if not reference_available():
        raise RuntimeError("reference tree not present at %s" % REF_ROOT)
    _install_shims()
    import contextlib
    import io
    from scene.deformation import deform_network  # type: ignore
    with contextlib.redirect_stdout(io.StringIO()):
        net = deform_network(hidden_args(cfg))
    return net
