"""Generates tests/golden/callsite/ply_attributes.npz: what the reference's own GaussianModel.construct_list_of_attributes,
make_ply and state_dict(is_final=True) (lib/models/gaussian_model.py) return for the background and the first actor of a
seeded StreetGaussianModel, with those sub-models' parameters.  Recorded through tests/refharness.py on a box that has the
reference's sources; tests/test_io_cpu.py::test_attribute_order_and_rows_equal_the_reference_model holds street_gaussians_b200.io
against it.  Run from the repo root:  python tests/golden/make_io_golden.py
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
import refharness as H  # noqa: E402
from street_gaussians_b200 import io as sio  # noqa: E402


def main():
    ns = H.load()
    model = H.make_street_model(ns, n_bkgd=11, n_obj=1, per_obj=5)
    out = {}
    for name, sub in (("background", model.background), ("obj", getattr(model, model.obj_list[0]))):
        for k in sio.RAW:
            out[f"{name}_{k}"] = getattr(sub, "_" + k).detach().numpy()
        out[name + "_attributes"] = np.array(sub.construct_list_of_attributes())
        out[name + "_ply"] = sub.make_ply()
        # which raw parameter each state_dict entry is (the entries are the parameters themselves, not copies)
        sd = sub.state_dict(is_final=True)
        out[name + "_state_dict"] = np.array([f"{k}:{next(r for r in sio.RAW if v is getattr(sub, '_' + r))}" for k, v in sd.items()])
    path = os.path.join(HERE, "callsite", "ply_attributes.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
