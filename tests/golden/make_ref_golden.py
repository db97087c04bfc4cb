"""Generates tests/golden/reference/*.npz: what the UNMODIFIED reference CUDA code (oracle/_ref, built by oracle/build_ref.sh)
computes for the scenes of the reference-parity tests of tests/test_parity_gpu.py and of __graft_entry__.smoke(), so that
those comparisons run wherever this repository is checked out.  The full outputs at these sizes are far too large to
commit: each file holds a fingerprint (tests/util.py fingerprint: seeded samples, whole-tensor hashes and sums).  Needs a
GPU and oracle/_ref:

    python tests/golden/make_ref_golden.py [OUT_DIR]      (default: tests/golden/reference)
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import __graft_entry__ as entry  # noqa: E402
import test_parity_gpu as T  # noqa: E402
import util  # noqa: E402
from street_gaussians_b200 import synthetic  # noqa: E402


def main():
    out = sys.argv[1] if len(sys.argv) > 1 else util.REF_GOLDEN
    os.makedirs(out, exist_ok=True)
    assert util.ref_available(), "oracle/_ref is missing: build it with oracle/build_ref.sh"
    ref = util.load_ref()

    def save(name, fp):
        path = os.path.join(out, name + ".npz")
        np.savez_compressed(path, **fp)
        print(f"{name}: {os.path.getsize(path)} bytes", flush=True)

    scenes = [("smoke", lambda: synthetic.make_scene(**entry.SMOKE_SCENE)), ("callsite_render_kernel", T.callsite_scene)]
    scenes += [("medium_" + name, lambda kw=kw: synthetic.make_scene(**kw)) for name, kw in T.MEDIUM]
    scenes += [("config_C", lambda: synthetic.make_config("C", seed=0))]
    for name, make in scenes:
        scene = make()
        save(name, util.fingerprint(util.run_api(ref, scene), scene))
        del scene
        torch.cuda.empty_cache()
    save("geometry_100k", T.reference_geometry_fingerprint(ref, synthetic.make_scene(**T.GEOM_KW)))
    save("knn_visible_filter", T.reference_knn_visible(ref, util.load_ref_knn(), synthetic.make_scene(**T.VIS_KW)))


if __name__ == "__main__":
    main()
