"""CPU: PLY / .pth IO (street_gaussians_b200/io.py) — layout of the reference's files (attribute order, channel-major SH, element
names), round trips, and an independent byte-level parse of the written file."""
import os
import struct

import numpy as np
import torch

import compose_case as CC
from street_gaussians_b200 import io as sio


def models(sem=0):
    ms = CC.make_case(3, 50, [20, 7], 16, 5)
    for m in ms:
        m["semantic"] = torch.randn(m["xyz"].shape[0], sem)
    return {"background": ms[0], "obj_000": ms[1], "obj_001": ms[2]}


def test_multi_element_ply_layout_and_round_trip(tmp_path):
    ms = models(sem=2)
    path = str(tmp_path / "point_cloud" / "iteration_7" / "point_cloud.ply")
    sio.save_ply(path, ms)
    raw = open(path, "rb").read()
    head = raw[: raw.index(b"end_header\n")].decode().splitlines()
    assert head[:2] == ["ply", "format binary_little_endian 1.0"]
    assert [ln for ln in head if ln.startswith("element")] == ["element vertex_background 50", "element vertex_obj_000 20", "element vertex_obj_001 7"]
    props_bk = head[3: 3 + 6 + 3 + 45 + 1 + 3 + 4 + 2]
    assert props_bk[:7] == [f"property float {a}" for a in ("x", "y", "z", "nx", "ny", "nz", "f_dc_0")]
    assert props_bk[9] == "property float f_rest_0" and props_bk[-3:] == ["property float rot_3", "property float semantic_0", "property float semantic_1"]
    # independent parse of the first background row: x y z | normals = 0 | f_dc channel-major
    body = raw[raw.index(b"end_header\n") + 11:]
    row0 = struct.unpack("<64f", body[: 64 * 4])
    bk = ms["background"]
    assert np.allclose(row0[:3], bk["xyz"][0].numpy()) and row0[3:6] == (0.0, 0.0, 0.0)
    assert np.allclose(row0[6:9], bk["features_dc"][0, 0].numpy())                  # C = 1: (r, g, b)
    assert np.allclose(row0[9:9 + 15], bk["features_rest"][0, :, 0].numpy())        # channel-major: all 15 red coefficients first
    back = sio.load_ply(path)
    assert list(back) == ["background", "obj_000", "obj_001"]
    for name, m in ms.items():
        for k in ("xyz", "features_dc", "features_rest", "opacity", "scaling", "rotation", "semantic"):
            assert back[name][k].shape == m[k].shape and torch.equal(back[name][k], m[k].float()), (name, k)
    # actors keep their fourier_dim = 5 DC rows through the channel-major flattening
    assert back["obj_000"]["features_dc"].shape == (20, 5, 3)


def test_single_element_and_ascii(tmp_path):
    m = models()["background"]
    p = str(tmp_path / "one.ply")
    sio.save_ply(p, {"background": m}, single_element=True)
    back = sio.load_ply(p)
    assert list(back) == [""] and torch.equal(back[""]["rotation"], m["rotation"])
    # an ascii file with the same header conventions (what a text export of the reference's file looks like)
    q = str(tmp_path / "ascii.ply")
    rows = sio.make_ply(m)[:3]
    with open(q, "w") as f:
        f.write("ply\nformat ascii 1.0\ncomment made by hand\nelement vertex 3\n" + "".join(f"property float {a}\n" for a in sio.attribute_names(m)) + "end_header\n")
        for r in rows:
            f.write(" ".join(repr(float(v)) for v in r) + "\n")
    b2 = sio.load_ply(q)[""]
    assert torch.allclose(b2["xyz"], m["xyz"][:3]) and torch.allclose(b2["features_rest"], m["features_rest"][:3])


def test_checkpoint_keys_match_reference(tmp_path):
    ms = models()
    p = str(tmp_path / "trained_model" / "iteration_30000.pth")
    sio.save_checkpoint(p, ms, 30000, extras={"background": dict(spatial_lr_scale=3.5, active_sh_degree=3)})
    sd = torch.load(p, weights_only=False)
    assert sd["iter"] == 30000 and set(sd["background"]) >= {"xyz", "feature_dc", "feature_rest", "scaling", "rotation", "opacity", "semantic",
                                                            "spatial_lr_scale", "active_sh_degree"}
    back = sio.load_checkpoint(p)
    assert torch.equal(back["obj_001"]["features_dc"], ms["obj_001"]["features_dc"]) and back["background"]["spatial_lr_scale"] == 3.5


def test_attribute_order_and_rows_equal_the_reference_model():
    """The reference's own GaussianModel.construct_list_of_attributes / make_ply / state_dict(is_final=True) on the same parameters,
    as recorded from the unmodified reference (tests/golden/callsite/ply_attributes.npz, tests/golden/make_io_golden.py)."""
    z = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "callsite", "ply_attributes.npz"))
    for name in ("background", "obj"):
        sub = {"_" + k: torch.from_numpy(z[f"{name}_{k}"]) for k in sio.RAW}
        assert sio.attribute_names(sub) == list(z[name + "_attributes"])
        ref_rows = z[name + "_ply"]  # structured array built by the reference
        mine = sio.make_ply(sub)
        assert mine.shape == (len(ref_rows), len(ref_rows.dtype.names))
        for j, n in enumerate(ref_rows.dtype.names):
            assert np.array_equal(mine[:, j], ref_rows[n]), n
        sd = sio.model_state_dict(sub)
        ref_sd = dict(e.split(":") for e in z[name + "_state_dict"])  # state_dict key -> the raw parameter it holds
        assert set(sd) == set(ref_sd) and all(sd[k] is sub["_" + r] for k, r in ref_sd.items())
