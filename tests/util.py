"""Shared helpers for the parity tests: run the candidate (libsgr.so through the reference-compatible API), the compiled
reference (oracle/_ref, GPU) and the CPU oracle (oracle/sgr_oracle.c) on the same seeded scene, and compare the candidate
with the reference outputs recorded under tests/golden/reference/ (tests/golden/make_ref_golden.py)."""
from __future__ import annotations

import hashlib
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GRAD_KEYS = ["means3D", "means2D", "shs", "opacities", "scales", "rotations"]
REF_GOLDEN = os.path.join(ROOT, "tests", "golden", "reference")
IMAGE_KEYS = ("color", "depth", "alpha", "semantic")
INPUT_KEYS = ("means3D", "shs", "opacities", "scales", "rotations", "semantics", "colors_precomp", "grad_color", "grad_depth",
              "grad_alpha", "grad_semantic")


def sha256(a) -> str:
    if torch.is_tensor(a):
        a = a.detach().cpu().numpy()
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def fingerprint(res, scene, n_pix=1024, n_rows=96, seed=0):
    """A small record of one forward+backward result (run_api's dict) that check_fingerprint can hold a full result against:
    radii as a hash (they must match exactly); per image a seeded pixel sample, the per-channel sums and max|.|; per gradient
    a seeded sample of visible rows, max|.| and sum|.|; the float64 sum of every input, so that a change of the seeded
    generators shows up as such rather than as a parity failure."""
    rng = np.random.default_rng(seed)
    radii = np.asarray(res["radii"], np.int32)
    fp = dict(radii_sha256=np.array(sha256(radii)), radii_visible=np.int64((radii > 0).sum()))
    npx = scene["cam"]["image_height"] * scene["cam"]["image_width"]
    fp["pix"] = np.sort(rng.choice(npx, min(n_pix, npx), replace=False)).astype(np.int32)
    for k in IMAGE_KEYS:
        if res.get(k) is not None and np.asarray(res[k]).size:
            a = np.asarray(res[k], np.float32).reshape(np.asarray(res[k]).shape[0], -1)
            fp[k + "_val"], fp[k + "_sum"], fp[k + "_maxabs"] = a[:, fp["pix"]], a.sum(1, dtype=np.float64), np.float32(np.abs(a).max())
    vis = np.flatnonzero(radii > 0)
    fp["rows"] = np.sort(rng.choice(vis, min(n_rows, vis.size), replace=False)).astype(np.int32)
    for k, g in res.items():
        if k.startswith("g_") and g is not None and np.asarray(g).size:
            g = np.asarray(g, np.float32)
            fp[k + "_val"], fp[k + "_maxabs"], fp[k + "_l1"] = g[fp["rows"]], np.float32(np.abs(g).max()), np.abs(g).sum(dtype=np.float64)
    for k in INPUT_KEYS:
        if k in scene:
            fp["in_sum_" + k] = np.float64(scene[k].double().sum())
    return fp


def load_ref_golden(name):
    with np.load(os.path.join(REF_GOLDEN, name + ".npz")) as z:
        return {k: z[k] for k in z.files}


def check_fingerprint(res, fp, scene, fwd_tol=1e-4, grad_tol=1e-3):
    """Holds a full result against a recorded fingerprint with the bars of a full comparison (no pixel above fwd_tol, every
    gradient within grad_tol * max|ref|) on the sampled entries, and with the consequences of those bars that the whole tensors
    must meet: bit-equal radii, per-channel image sums within npx * fwd_tol, max|.| and sum|.| of every gradient within
    grad_tol * max|ref| and numel * grad_tol * max|ref|."""
    for k in INPUT_KEYS:
        if "in_sum_" + k in fp:
            got = float(scene[k].double().sum())
            assert abs(got - float(fp["in_sum_" + k])) <= 1e-9 * max(1.0, abs(got)), f"input {k} differs from the recorded one: regenerate"
    radii = np.asarray(res["radii"], np.int32)
    assert sha256(radii) == str(fp["radii_sha256"]), f"radii differ ({int((radii > 0).sum())} visible, reference {int(fp['radii_visible'])})"
    pix = fp["pix"]
    for k in IMAGE_KEYS:
        if k + "_val" not in fp:
            continue
        a = np.asarray(res[k], np.float64).reshape(fp[k + "_val"].shape[0], -1)
        npx = a.shape[1]
        scale = max(1.0, float(fp[k + "_maxabs"])) if k == "depth" else 1.0  # depth is un-normalised metres
        d = np.abs(a[:, pix] - fp[k + "_val"])
        assert d.max() <= fwd_tol * scale, (k, float(d.max()))
        assert (np.abs(a.sum(1) - fp[k + "_sum"]) <= fwd_tol * scale * npx).all(), (k, a.sum(1), fp[k + "_sum"])
    rows, n = fp["rows"], 0
    for key in fp:
        if not (key.startswith("g_") and key.endswith("_val")):
            continue
        k = key[:-4]
        g = np.asarray(res[k], np.float64)
        ref_max = float(fp[k + "_maxabs"]) + 1e-12
        e = float(np.abs(g[rows] - fp[key]).max()) / ref_max
        assert e <= grad_tol, (k, e)
        assert abs(float(np.abs(g).max()) - ref_max) <= grad_tol * ref_max, (k, float(np.abs(g).max()), ref_max)
        assert abs(float(np.abs(g).sum()) - float(fp[k + "_l1"])) <= grad_tol * ref_max * g.size, (k, float(np.abs(g).sum()), float(fp[k + "_l1"]))
        n += 1
    return n


def ref_available() -> bool:
    return os.path.exists(os.path.join(ROOT, "oracle", "_ref", "ref_dgr", "_C.so"))


def load_ref():
    """The unmodified reference rasterizer built by oracle/build_ref.sh (test infrastructure)."""
    p = os.path.join(ROOT, "oracle", "_ref")
    if p not in sys.path:
        sys.path.insert(0, p)
    import ref_dgr  # noqa
    return ref_dgr


def load_ref_knn():
    p = os.path.join(ROOT, "oracle", "_ref")
    if p not in sys.path:
        sys.path.insert(0, p)
    from ref_knn import _C  # noqa
    return _C


def settings_from(mod, cam, device, debug=False):
    return mod.GaussianRasterizationSettings(
        image_height=cam["image_height"], image_width=cam["image_width"], tanfovx=cam["tanfovx"], tanfovy=cam["tanfovy"],
        bg=cam["bg"].to(device), scale_modifier=cam["scale_modifier"], viewmatrix=cam["viewmatrix"].to(device),
        projmatrix=cam["projmatrix"].to(device), sh_degree=cam["sh_degree"], campos=cam["campos"].to(device),
        prefiltered=False, debug=debug)


def run_api(mod, scene, device="cuda", backward=True, use_colors_precomp=False, use_cov3d=None, rasterizer_kwargs=None):
    """Run forward(+backward) through a module exposing the reference API.  Returns dict of numpy arrays."""
    cam = scene["cam"]
    st = settings_from(mod, cam, device)
    rast = mod.GaussianRasterizer(st, **(rasterizer_kwargs or {}))
    leaf = lambda t: t.to(device).clone().requires_grad_(backward)
    means3D = leaf(scene["means3D"])
    means2D = torch.zeros_like(means3D, requires_grad=backward)
    opac = leaf(scene["opacities"])
    kw = {}
    inputs = dict(means3D=means3D, means2D=means2D, opacities=opac)
    if use_colors_precomp:
        inputs["colors_precomp"] = leaf(scene["colors_precomp"]); kw["colors_precomp"] = inputs["colors_precomp"]
    else:
        inputs["shs"] = leaf(scene["shs"]); kw["shs"] = inputs["shs"]
    if use_cov3d is not None:
        inputs["cov3D_precomp"] = leaf(use_cov3d); kw["cov3D_precomp"] = inputs["cov3D_precomp"]
    else:
        inputs["scales"] = leaf(scene["scales"]); inputs["rotations"] = leaf(scene["rotations"])
        kw["scales"] = inputs["scales"]; kw["rotations"] = inputs["rotations"]
    if "semantics" in scene:
        inputs["semantics"] = leaf(scene["semantics"]); kw["semantics"] = inputs["semantics"]
    color, radii, depth, alpha, sem = rast(means3D=means3D, means2D=means2D, opacities=opac, **kw)
    out = dict(color=color, radii=radii, depth=depth, alpha=alpha, semantic=sem)
    res = {k: v.detach().cpu().numpy() for k, v in out.items()}
    if backward:
        loss = (color * scene["grad_color"].to(device)).sum() + (depth * scene["grad_depth"].to(device)).sum() + \
               (alpha * scene["grad_alpha"].to(device)).sum()
        if "semantics" in scene:
            loss = loss + (sem * scene["grad_semantic"].to(device)).sum()
        loss.backward()
        for k, v in inputs.items():
            res["g_" + k] = v.grad.detach().cpu().numpy() if v.grad is not None else None
    torch.cuda.synchronize()
    return res


def run_oracle(scene, backward=True, use_colors_precomp=False, use_cov3d=None):
    from oracle import oracle as O
    cam = scene["cam"]
    c = O.Camera(cam["image_height"], cam["image_width"], cam["tanfovx"], cam["tanfovy"], cam["bg"].numpy(), cam["scale_modifier"],
                 cam["viewmatrix"].numpy(), cam["projmatrix"].numpy(), cam["sh_degree"], cam["campos"].numpy())
    fw = O.Forward(c, scene["means3D"], scene["opacities"], shs=None if use_colors_precomp else scene["shs"],
                   colors_precomp=scene.get("colors_precomp") if use_colors_precomp else None,
                   scales=None if use_cov3d is not None else scene["scales"],
                   rotations=None if use_cov3d is not None else scene["rotations"], cov3D_precomp=use_cov3d,
                   semantics=scene.get("semantics"))
    res = dict(color=fw.color, radii=fw.radii, depth=fw.depth, alpha=fw.alpha, semantic=fw.semantic, num_rendered=fw.num_rendered,
               pairs_evaluated=fw.pairs_evaluated, pairs_blended=fw.pairs_blended)
    if backward:
        g = fw.backward(scene["grad_color"], scene["grad_depth"], scene["grad_alpha"], scene.get("grad_semantic"))
        res.update(g_means3D=g["means3D"], g_means2D=g["means2D"], g_opacities=g["opacities"], g_semantics=g["semantics"])
        if use_colors_precomp:
            res["g_colors_precomp"] = g["colors_precomp"]
        else:
            res["g_shs"] = g["sh"]
        if use_cov3d is not None:
            res["g_cov3D_precomp"] = g["cov3D_precomp"]
        else:
            res["g_scales"] = g["scales"]; res["g_rotations"] = g["rotations"]
    res["_fw"] = fw
    return res


def rel_err(a, b):
    """max|a-b| / (max|b| + 1e-12): the per-tensor gradient metric of SURVEY.md §8d."""
    a = np.asarray(a, np.float64); b = np.asarray(b, np.float64)
    if a.size == 0 and b.size == 0:
        return 0.0
    return float(np.max(np.abs(a - b)) / (np.max(np.abs(b)) + 1e-12))


def compare(res, ref, keys=None, verbose=True, tag=""):
    """Returns dict of error metrics: forward max-abs errors and gradient relative errors."""
    out = {}
    for k in ("color", "depth", "alpha", "semantic"):
        if res.get(k) is None or ref.get(k) is None or np.asarray(ref[k]).size == 0:
            continue
        d = np.abs(np.asarray(res[k], np.float64) - np.asarray(ref[k], np.float64))
        out[k + "_maxabs"] = float(d.max())
        out[k + "_n_gt_1e-4"] = int((d > 1e-4).sum())
    out["radii_mismatch"] = int((np.asarray(res["radii"]) != np.asarray(ref["radii"])).sum())
    for k in res:
        if k.startswith("g_") and res[k] is not None and ref.get(k) is not None:
            out[k + "_rel"] = rel_err(res[k], ref[k])
    if verbose:
        print(tag, {k: (f"{v:.3e}" if isinstance(v, float) else v) for k, v in out.items()})
    return out


def flip_bound(scene_or_maxc, bg=None):
    """SURVEY.md §7 'Discontinuities' (ii)/(iv): ONE flipped hard threshold changes a pixel by at most
         alpha<1/255 skip   : (1/255) * T * |c_i - C_behind|   <= (1/255) * (max|c| + max|bg|)
         T(1-alpha)<1e-4 stop: 1e-4 * (max|c| + max|bg|)
    where max|c| is the largest per-Gaussian colour (or depth / feature) value that can be blended."""
    return (1.0 / 255.0 + 1e-4) * float(scene_or_maxc + (0.0 if bg is None else bg))


def check_forward_flip_protocol(res, ref, max_value, tol=1e-4, max_flips_per_pixel=2, max_pixels=None, names=("color",)):
    """The parity protocol of SURVEY.md §7: enumerate EVERY pixel whose difference exceeds `tol` and require each to be explained
    by at most `max_flips_per_pixel` threshold flips (flip_bound); all other pixels are within `tol`.  Returns the offender list
    [(name, channel, y, x, diff)] so callers can print / count it.  `max_value[name]` = largest blendable value of that image."""
    offenders = []
    for name in names:
        a, b = np.asarray(res[name], np.float64), np.asarray(ref[name], np.float64)
        if b.size == 0:
            continue
        d = np.abs(a - b)
        scale = max(1.0, float(np.abs(b).max())) if name == "depth" else 1.0
        idx = np.argwhere(d > tol * scale)
        bound = max_flips_per_pixel * flip_bound(max_value[name]) * 1.05
        for c, y, x in idx:
            assert d[c, y, x] <= bound, f"{name}[{c},{y},{x}] differs by {d[c, y, x]:.3e} > {max_flips_per_pixel} threshold flips ({bound:.3e})"
            offenders.append((name, int(c), int(y), int(x), float(d[c, y, x])))
        assert np.median(d) <= 1e-6 * scale, (name, float(np.median(d)))
    if max_pixels is not None:
        px = {(o[2], o[3]) for o in offenders}
        assert len(px) <= max_pixels, f"{len(px)} pixels above {tol}: {offenders[:10]}"
    return offenders
