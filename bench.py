#!/usr/bin/env python
"""bench.py — rasterizer fwd+bwd frames/s on the BASELINE.json workload, one process per GPU.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl sgr|reference] [--workload C|B|E|A] [--dump-outputs DIR]

A "step" = one forward + backward pass of the rasterizer over one synthetic frame (config C of BASELINE.md by default:
1.5M background + 8x50k vehicle Gaussians, 1920x1280, SH degree 3).  Prints ONE JSON line (rank 0).

  value      : frames/s with the Gaussian parameters already resident in HBM (device-timed, CUDA events, max over ranks)
  e2e        : same metric through the public API starting from PINNED HOST buffers: every step copies that step's inputs
               host->device (double-buffered on a copy stream) and reads the scalar loss back device->host
  roofline   : dominant kernel (blend_bwd), algorithmic bytes / CUDA-event time / measured HBM peak (MEASURED_PEAKS.json)
  cpu_baseline: the CPU oracle port (oracle/sgr_oracle.c, OpenMP) on a bounded sample of the same frame
  --impl reference : the UNMODIFIED reference CUDA rasterizer built from the reference's sources into oracle/_ref
               (stock code path through its own Python API), same workload/metric/timing; the reference has no CPU
               implementation of this path, so the CPU port is reported beside it in cpu_baseline.  If oracle/_ref is
               absent the arm times the CPU oracle port instead.
  --dump-outputs DIR : after the timed steps, what the last of them returned to the caller (images, radii, the gradient of
               every input) as DIR/<name>.npy, float32 (indices float64); larger outputs as a fixed seeded sample.  The inputs
               are seeded, so two builds (or the two --impl arms) can be compared output for output.
N > 1: strong scaling — the SAME frame is tile-row sharded across ranks (street_gaussians_b200.sharded), one NCCL
all-reduce of the per-Gaussian screen-space gradient sums per step.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

from street_gaussians_b200 import synthetic  # noqa: E402

PARAM_KEYS = ("means3D", "shs", "opacities", "scales", "rotations")


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="sgr", choices=["sgr", "reference"])
    ap.add_argument("--workload", default="C", choices=list(synthetic.CONFIGS.keys()))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true", help="skip the end-to-end (host buffer) leg")
    ap.add_argument("--sync-free", dest="sync_free", action="store_true", default=None,
                    help="InstanceCapacity mode of the public API (sgr_forward_bounded: no host read-back inside forward); "
                         "this is the default for the timed region; the exact drop-in mode is timed beside it "
                         "(config.exact_mode_ms_per_step)")
    ap.add_argument("--exact", dest="sync_free", action="store_false", help="force the exact (read-back) mode")
    ap.add_argument("--mp-mode", choices=["gaussian", "gaussian-p2p", "gaussian-p2p-staged", "gaussian-p2p-allgather", "replicated"], default="gaussian-p2p",
                    help="N > 1 only. gaussian: every rank owns P/N Gaussians and a tile-row band (NCCL all-gather of records, "
                         "reduce-scatter of grad2d; GaussianShardedRasterizer).  gaussian-p2p: same partition, but records / grad2d rows "
                         "move by direct NVLink stores / loads to exactly the ranks that need them (exchange='p2p'), one C-ABI call per "
                         "forward / backward (sgr_sharded_forward / sgr_sharded_backward).  gaussian-p2p-staged: the same exchange driven "
                         "stage by stage from Python (round-1 path).  gaussian-p2p-allgather: gaussian-p2p followed by an NCCL all-gather of "
                         "every parameter gradient, so that EVERY rank ends with all gradients (the north-star's literal contract).  "
                         "replicated: parameters replicated, tile rows sharded, one all-reduce (ShardedGaussianRasterizer)")
    ap.add_argument("--graph", choices=["auto", "on", "off"], default="auto",
                    help="timed region: capture ONE fwd+bwd step (through the public API, autograd included) in a CUDA graph after the warm-up "
                         "and replay it K times — no per-kernel launch latency, no Python between kernels.  Needs the sync-free mode (nothing "
                         "in the step may talk to the host); the Gaussian-sharded peer-memory step is graph-safe because its barrier epochs "
                         "live on the device.  auto = on where supported, falling back to the eager loop if capture fails")
    ap.add_argument("--no-clock-sampler", action="store_true")
    ap.add_argument("--diag", action="store_true", help="per-rank host/all-reduce timing breakdown on stderr")
    ap.add_argument("--cpu-sample-stride", type=int, default=0, help="CPU baseline uses every k-th Gaussian (0 = auto)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step to DIR/<name>.npy (single GPU; at most 64 MB, larger outputs sampled)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


DUMP_PIXELS, DUMP_GAUSSIANS = 1 << 20, 1 << 16  # sample sizes: 5 image channels + 63 floats per Gaussian + indices stay under 64 MB


def dump_outputs(out_dir, color, radii, depth, alpha, params, means2D):
    """The outputs of one step as out_dir/<name>.npy: images, radii and the gradients of every input.  Images with more than
    DUMP_PIXELS pixels are sampled at a fixed seeded set of pixels (pixel_index.npy), per-Gaussian arrays with more than
    DUMP_GAUSSIANS rows at a fixed seeded set of Gaussians (gaussian_index.npy), so that the files stay under 64 MB."""
    os.makedirs(out_dir, exist_ok=True)
    dev = color.device
    H, W = color.shape[1:]
    P = radii.shape[0]
    rng = np.random.default_rng(0)
    pix = np.sort(rng.choice(H * W, DUMP_PIXELS, replace=False)) if H * W > DUMP_PIXELS else np.arange(H * W)
    rows = np.sort(rng.choice(P, DUMP_GAUSSIANS, replace=False)) if P > DUMP_GAUSSIANS else np.arange(P)
    pix_t, rows_t = torch.from_numpy(pix).to(dev), torch.from_numpy(rows).to(dev)
    out = {name: img.detach().reshape(img.shape[0], -1).index_select(1, pix_t) for name, img in (("color", color), ("depth", depth), ("alpha", alpha))}
    out["radii"] = radii.index_select(0, rows_t)
    out.update({"grad_" + k: p.grad.index_select(0, rows_t) for k, p in params.items()})
    out["grad_means2D"] = means2D.grad.index_select(0, rows_t)
    arrays = {k: v.float().cpu().numpy() for k, v in out.items()}
    arrays.update(pixel_index=pix.astype(np.float64), gaussian_index=rows.astype(np.float64))
    total = sum(a.nbytes for a in arrays.values())
    assert total <= 64_000_000, f"outputs of {total} bytes exceed 64 MB"
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), a)


class ClockSampler:
    """SM clock / throttle-reason sampler running DURING the timed region (B200_PROFILING.md 'clocks' line).

    In-process NVML polling from a background thread (pynvml).  An external `nvidia-smi -lms 100` loop was measured to
    perturb this host-synchronising workload badly (4.0 ms/step with it vs 2.2 ms without: every query takes driver
    locks that the mid-forward cudaStreamSynchronize then waits on); if NVML is unavailable the record says so."""
    REASONS = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40}

    def __init__(self, gpu_index: int, period_s: float = 0.05):
        import threading
        self.samples, self.marks, self._stop = [], [None, None], threading.Event()
        self.h = None
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[gpu_index]) if vis and vis.split(",")[gpu_index].strip().isdigit() else gpu_index
            self.nv, self.h = pynvml, pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.sm_max = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.h = None
        self.period = period_s
        self.t = threading.Thread(target=self._run, daemon=True)
        self.t.start()

    def _run(self):
        while not self._stop.is_set():
            if self.h is not None:
                try:
                    sm = float(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM))
                    try:
                        rs = int(self.nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
                    except Exception:
                        rs = int(self.nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
                    self.samples.append((time.perf_counter(), sm, rs))
                except Exception:
                    pass
            self._stop.wait(self.period)

    def mark(self, which: int):
        self.marks[which] = time.perf_counter()

    def stop(self):
        self._stop.set()
        self.t.join(timeout=2)
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0, "source": "nvml" if self.h is not None else "unavailable"}
        t0, t1 = self.marks
        sel = [s for s in self.samples if (t0 is None or s[0] >= t0) and (t1 is None or s[0] <= t1)] or self.samples[-3:]
        if sel:
            reasons = set()
            for _, _, rs in sel:
                for nm, bit in self.REASONS.items():
                    if rs & bit:
                        reasons.add(nm)
            out.update(sm_mhz=float(np.median([s[1] for s in sel])), sm_max_mhz=self.sm_max, reasons=sorted(reasons), samples=len(sel))
        return out


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            j = json.load(open(p))
            return float(j["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_traffic(kernel: str, source: str, workload):
    """(dram bytes per launch, issue-active %, stale) of `kernel` from profiles/ncu_traffic.json.  The first two are None when the
    committed capture is for another workload or for another version of the kernel's source file (sha256 of the .cu as of the
    capture's commit); `stale` then describes that earlier capture so the line can still point at it without claiming it."""
    import hashlib
    if workload is None:  # (multi-GPU runs: the per-rank kernel is a different launch than the captured single-GPU one)
        return None, None, None
    try:
        j = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))[kernel]
        sha = hashlib.sha256(open(os.path.join(ROOT, "street_gaussians_b200", "csrc", source), "rb").read()).hexdigest()[:16]
        if workload is not None and j.get("workload") == workload and j.get("source_sha16") == sha:
            return float(j["dram_bytes"]), j.get("issue_active_pct"), None
        return None, None, dict(dram_bytes=float(j["dram_bytes"]), issue_active_pct=j.get("issue_active_pct"), kernel_us=j.get("time_us"),
                                commit=j.get("commit"), workload=j.get("workload"),
                                note="ncu capture of an EARLIER build of this kernel (source changed since); not a measurement of this build")
    except Exception:
        pass
    return None, None, None


def make_settings(mod, cam, dev):
    return mod.GaussianRasterizationSettings(
        image_height=cam["image_height"], image_width=cam["image_width"], tanfovx=cam["tanfovx"], tanfovy=cam["tanfovy"],
        bg=cam["bg"].to(dev), scale_modifier=cam["scale_modifier"], viewmatrix=cam["viewmatrix"].to(dev),
        projmatrix=cam["projmatrix"].to(dev), sh_degree=cam["sh_degree"], campos=cam["campos"].to(dev), prefiltered=False,
        debug=False)


def cpu_baseline(scene, stride: int, budget_pairs: float = 6e8):
    """CPU oracle port on every `stride`-th Gaussian of the same frame at full resolution; linear extrapolation in P."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from oracle import oracle as O
    P = scene["means3D"].shape[0]
    H, W = scene["cam"]["image_height"], scene["cam"]["image_width"]
    if stride <= 0:  # auto: aim for a few 1e8 (pixel, splat) evaluations ~ 10-30 s on 8 cores
        stride = max(1, int(P * 12 * 256 / budget_pairs))
    sub = {k: (v[::stride].contiguous() if (torch.is_tensor(v) and v.dim() >= 1 and v.shape[0] == P) else v) for k, v in scene.items()}
    cam = scene["cam"]
    c = O.Camera(H, W, cam["tanfovx"], cam["tanfovy"], cam["bg"].numpy(), cam["scale_modifier"], cam["viewmatrix"].numpy(),
                 cam["projmatrix"].numpy(), cam["sh_degree"], cam["campos"].numpy())
    cores = O.num_threads()
    try:  # honour a cgroup CPU quota (this pool: 16 cores visible as 64): oversubscribing it makes the port SLOWER
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            cores = max(1, min(cores, int(int(q) / int(per))))
            O.set_num_threads(cores)
    except Exception:
        pass
    t0 = time.perf_counter()
    fw = O.Forward(c, sub["means3D"], sub["opacities"], shs=sub["shs"], scales=sub["scales"], rotations=sub["rotations"])
    fw.backward(scene["grad_color"], scene["grad_depth"], scene["grad_alpha"])
    dt = time.perf_counter() - t0
    n_sub = sub["means3D"].shape[0]
    fps_full = 1.0 / (dt * (P / n_sub))
    info = dict(value=fps_full, unit="frames/s", cores=cores, kind="port",
                sample=f"every {stride}th Gaussian ({n_sub} of {P}) of the same frame at full {W}x{H}, fwd+bwd, {dt:.2f} s measured, "
                       f"extrapolated x{P / n_sub:.1f} in Gaussian count; R_sample={fw.num_rendered}, pairs={fw.pairs_evaluated}")
    fw.close()
    return info


def check_parity_n(mod, rast, scene, cam, dev, rank, world, H, lo, hi, params, means2D, upstream):
    """Before timing at N > 1: this rank's band of colour / depth / alpha must be BIT-equal to a single-GPU render of the same
    tensors, and the gradients this rank ends up with — of the Gaussians it owns (Gaussian-sharded) or of all of them (replicated
    parameters) — within 1e-3 of the single-GPU gradients of the FULL loss (max|d| / max|ref| per tensor, BASELINE.json's bar; the
    exchange sums the bands, so float summation order is the only expected difference, ~2.5e-5)."""
    from street_gaussians_b200.sharded import band_of_rows
    full = {k: scene[k].to(dev).requires_grad_(True) for k in PARAM_KEYS}
    m2 = torch.zeros((full["means3D"].shape[0], 3), device=dev, requires_grad=True)
    one = mod.GaussianRasterizer(make_settings(mod, cam, dev))
    c1, r1, d1, a1, _ = one(means3D=full["means3D"], means2D=m2, opacities=full["opacities"], shs=full["shs"], scales=full["scales"],
                            rotations=full["rotations"])
    torch.autograd.backward([c1, d1, a1], [scene[k].to(dev) for k in ("grad_color", "grad_depth", "grad_alpha")])
    for v in list(params.values()) + [means2D]:
        v.grad = None
    color, radii, depth, alpha, _ = rast(means3D=params["means3D"], means2D=means2D, opacities=params["opacities"], shs=params["shs"],
                                         scales=params["scales"], rotations=params["rotations"])
    torch.autograd.backward([color, depth, alpha], list(upstream))
    rows = band_of_rows(H, rank, world).to(dev)
    ok = all(bool(torch.equal(a.detach()[:, rows], b.detach()[:, rows])) for a, b in ((color, c1), (depth, d1), (alpha, a1)))
    ok = ok and bool(torch.equal(radii, r1[lo:hi]))
    worst = 0.0
    for got, ref in [(params[k].grad, full[k].grad[lo:hi]) for k in PARAM_KEYS] + [(means2D.grad, m2.grad[lo:hi])]:
        worst = max(worst, float((got.double() - ref.double()).abs().max() / (ref.double().abs().max() + 1e-12)))
    del full, m2, one, c1, d1, a1
    torch.cuda.empty_cache()
    return dict(ok=ok and worst <= 1e-3, grad_rel_max=worst)


def rank_models(raw, lo, hi, dev):
    """The slice [lo, hi) of the composed index space as a list of raw sub-models (background first, possibly empty; then the actors
    that intersect the slice) — leaf tensors on `dev` — plus the indices of those actors."""
    models, actors, at = [], [], 0
    for k, m in enumerate(raw["models"]):
        n = m["xyz"].shape[0]
        a, b = max(lo, at) - at, min(hi, at + n) - at
        at += n
        if k > 0 and b <= a:
            continue
        a, b = (a, b) if b > a else (0, 0)
        models.append({key: v[a:b].to(dev).contiguous().requires_grad_(True) for key, v in m.items()})
        if k > 0:
            actors.append(k - 1)
    return models, actors


def composed_e2e(args, mod, rast, scene, cam, dev, lo, hi, means2D, upstream, ref_cuda, barrier, use_dist, n_e2e, capacity=None):
    """frames/s of  compose -> rasterize -> backward  with the raw parameters resident on the device and the per-frame inputs
    (view / projection matrix, camera centre, actor poses) copied from PINNED HOST memory inside the timed region; the scalar loss is
    read back.  Reference arm: the reference's own compose math as the PyTorch ops it is (oracle/compose_oracle.py restates
    lib/models/street_gaussian_model.py:287-449 line by line) in front of the unmodified reference rasterizer."""
    raw = scene["raw"]
    models, actors = rank_models(raw, lo, hi, dev)
    n_act = len(actors)
    poses_host = raw["poses"][actors].contiguous().pin_memory() if n_act else None
    idft_dev = raw["idft"][actors].to(dev) if n_act else None
    cam_host = torch.cat([cam["viewmatrix"].reshape(-1), cam["projmatrix"].reshape(-1), cam["campos"].reshape(-1)]).float().pin_memory()
    cam_dev = [torch.empty_like(cam_host, device=dev) for _ in range(2)]
    poses_dev = [torch.empty((n_act, 7), device=dev) for _ in range(2)] if n_act else [None, None]
    loss_host = torch.zeros(1).pin_memory()
    gc, gd, ga = upstream
    h2d = cam_host.numel() * 4 + (poses_host.numel() * 4 if n_act else 0)
    if ref_cuda:
        from oracle import compose_oracle as CO  # the reference's compose math as torch ops (bench.py may run oracle/ for this arm)

    def frame(i):
        cam_dev[i].copy_(cam_host, non_blocking=True)
        pd = None
        if n_act:
            poses_dev[i].copy_(poses_host, non_blocking=True)
            pd = poses_dev[i].detach().requires_grad_(True)
        st = mod.GaussianRasterizationSettings(
            image_height=cam["image_height"], image_width=cam["image_width"], tanfovx=cam["tanfovx"], tanfovy=cam["tanfovy"],
            bg=rast.raster_settings.bg, scale_modifier=cam["scale_modifier"], viewmatrix=cam_dev[i][:16].view(4, 4),
            projmatrix=cam_dev[i][16:32].view(4, 4), sh_degree=cam["sh_degree"], campos=cam_dev[i][32:35], prefiltered=False, debug=False)
        for m in models:
            for v in m.values():
                v.grad = None
        means2D.grad = None
        if ref_cuda:
            o = CO.compose(models, pd if n_act else torch.zeros(0, 7, device=dev), idft_dev if n_act else torch.zeros(0, 1, device=dev), None, None)
            xyz, rot, scale, opac, sh = o["xyz"], o["rotation"], o["scaling"], o["opacity"], o["features"]
            r = mod.GaussianRasterizer(st)
        else:
            xyz, rot, scale, opac, sh = mod.compose(models, pd, idft_dev)
            rast.raster_settings = st
            r = rast
        color, radii, depth, alpha, sem = r(means3D=xyz, means2D=means2D, opacities=opac, shs=sh, scales=scale, rotations=rot)
        loss = (color * gc).sum() + (depth * gd).sum() + (alpha * ga).sum()
        loss.backward()
        loss_host.copy_(loss.detach().view(1), non_blocking=True)

    old_settings = getattr(rast, "raster_settings", None)
    for i in range(3):
        frame(i % 2)
    barrier()
    # The whole frame — pinned-host -> device copies of the camera and poses, compose, rasterize, loss, backward through both, loss ->
    # pinned host — as ONE CUDA graph (the copies are graph nodes: every replay re-reads the pinned buffers, which is where a trainer
    # writes the next frame's camera / poses).  Falls back to the eager loop when capture is impossible, like the main timed region.
    graph, graph_note = None, None
    if (not ref_cuda and args.graph != "off" and capacity is not None and capacity.capacity is not None
            and (not use_dist or args.mp_mode == "gaussian-p2p")):
        try:
            capacity.freeze()
            side = torch.cuda.Stream(device=dev)
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                for _ in range(2):
                    frame(0)
            torch.cuda.current_stream().wait_stream(side)
            barrier()
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                frame(0)
            for _ in range(2):
                graph.replay()
            torch.cuda.synchronize()
        except Exception as e:  # noqa: BLE001
            graph, graph_note = None, f"capture failed, eager loop timed instead: {e!r}"[:300]
            try:
                torch.cuda.synchronize()
            except Exception:  # noqa: BLE001
                pass
        if use_dist:
            flag = torch.tensor([1 if graph is not None else 0], device=dev)
            dist.all_reduce(flag, op=dist.ReduceOp.MIN)
            if int(flag.item()) == 0:
                graph, graph_note = None, graph_note or "capture failed on another rank; eager loop timed instead"
        if graph is None:
            capacity.freeze(False)
            frame(0)
        barrier()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for i in range(n_e2e):
        if graph is not None:
            graph.replay()
        else:
            frame(i % 2)
    b.record()
    barrier()
    _ = float(loss_host.item())
    timed_graph = graph is not None
    ms = a.elapsed_time(b) / n_e2e
    if use_dist:
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
        t = torch.tensor([float(h2d)], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        h2d = int(t.item())
    if old_settings is not None and not ref_cuda:
        rast.raster_settings = old_settings
    if graph is not None:
        capacity.freeze(False)
        del graph
    return dict(value=1000.0 / ms, unit="frames/s", ms_per_step=ms, h2d_bytes_per_step=int(h2d), d2h_bytes_per_step=4,
                timed_region=("CUDA graph of the whole frame (H2D copies, compose, rasterize, loss, backward, D2H loss), replayed %d times" % n_e2e)
                if timed_graph else ("eager Python loop" + (" (%s)" % graph_note if graph_note else "")),
                note=("compose (sgr_compose_*) -> rasterize -> backward through both; raw per-model parameters resident in HBM; camera matrices + "
                      "%d actor poses copied from pinned host memory every step; scalar loss read back" % n_act) if not ref_cuda else
                     ("reference compose math as PyTorch ops -> unmodified reference rasterizer -> autograd backward; same residency and "
                      "per-step copies"))


def main():
    args = parse()
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference" and rank != 0:
        if world > 1:  # the reference is single-GPU: rank 0 alone runs it
            pass
        return 0
    if not torch.cuda.is_available():
        print(json.dumps({"error": "no CUDA device", "impl": args.impl}))
        return 1
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    use_dist = world > 1 and args.impl == "sgr"
    if use_dist and args.dump_outputs:
        print(json.dumps({"error": "--dump-outputs writes the outputs of one process: run it with --gpus 1"}))
        return 1
    if use_dist:
        dist.init_process_group("nccl", device_id=dev)

    ref_so = os.path.join(ROOT, "oracle", "_ref", "ref_dgr", "_C.so")
    ref_cuda = args.impl == "reference" and os.path.exists(ref_so)
    cpu_only_reference = args.impl == "reference" and not ref_cuda

    scene = synthetic.make_config(args.workload, seed=0, **({} if synthetic.CONFIGS[args.workload]["kind"] == "smoke" else {"with_raw": True}))
    cam = scene["cam"]
    P = scene["means3D"].shape[0]
    H, W = cam["image_height"], cam["image_width"]
    wl_desc = {"C": "config C: 1.5M background + 8x50k vehicle Gaussians composed, 1920x1280, SH deg 3, fwd+bwd",
               "B": "config B: 500k Gaussians static scene, 1920x1280, SH deg 3, fwd+bwd",
               "E": "config E: 8M Gaussians, 3840x2160, SH deg 3", "A": "config A: smoke-script replay 10k, 256x256",
               "A_native": "config A native: smoke-script replay 10k, 1242x375"}[args.workload]

    if cpu_only_reference:
        cb = cpu_baseline(scene, args.cpu_sample_stride)
        line = dict(metric="rasterizer_fwd_bwd_fps", value=cb["value"], unit="frames/s", n_gpus=args.gpus, steps=args.steps,
                    warmup=args.warmup, ms_per_step=1000.0 / cb["value"], higher_is_better=True, scaling="strong", vs_baseline=None,
                    dtype="f32", data="synthetic", impl="reference", config=dict(workload=wl_desc, P=P, width=W, height=H),
                    cpu_baseline=cb, e2e=dict(value=cb["value"], unit="frames/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0),
                    gpu_launches=0, note="oracle/_ref (reference CUDA build) absent: CPU oracle port timed instead")
        print(json.dumps(line))
        return 0

    if ref_cuda:
        sys.path.insert(0, os.path.join(ROOT, "oracle", "_ref"))
        import ref_dgr as mod
        rast = mod.GaussianRasterizer(make_settings(mod, cam, dev))
    else:
        import street_gaussians_b200 as mod
        from street_gaussians_b200.sharded import ShardedGaussianRasterizer
        if args.sync_free is None:
            # The timed region uses the sync-free mode of the public API (GaussianRasterizer(capacity=InstanceCapacity())):
            # with no host wait inside the step the measurement does not depend on host scheduling noise (one run on a
            # busy box measured 4.9 ms/step in the exact mode while every kernel ran at its usual speed), and it is what
            # lets 8 ranks share this pool's 16-core container quota (1.64 ms exact vs 1.28 ms sync-free at N = 8).  On a
            # quiet box the two modes agree within 3 % on one GPU (1.91-1.95 exact vs 1.96 ms); the exact drop-in mode —
            # what the UNCHANGED reference call site gets — is timed right after and reported as exact_mode_ms_per_step.
            args.sync_free = True
        capacity = mod.InstanceCapacity() if args.sync_free else None
        if use_dist and args.mp_mode.startswith("gaussian"):
            from street_gaussians_b200.sharded import GaussianShardedRasterizer
            chunk = (P + world - 1) // world
            rast = GaussianShardedRasterizer(make_settings(mod, cam, dev), capacity=capacity, chunk=chunk,
                                             exchange="p2p" if args.mp_mode.startswith("gaussian-p2p") else "nccl",
                                             fused=args.mp_mode != "gaussian-p2p-staged")
            if args.mp_mode.startswith("gaussian-p2p"):
                # the peer-memory exchange needs torch symmetric memory (CUDA VMM handles shared between the ranks); if any
                # rank cannot set it up, ALL ranks fall back to the NCCL exchange (measured 2.5 % slower at N = 8)
                ok = 1
                try:
                    rast.workspace(dev)
                except Exception as e:  # noqa: BLE001
                    ok = 0
                    print(f"[rank {rank}] peer workspace unavailable ({e!r}); falling back to the NCCL exchange", file=sys.stderr, flush=True)
                flag = torch.tensor([ok], device=dev)
                dist.all_reduce(flag, op=dist.ReduceOp.MIN)
                if int(flag.item()) == 0:
                    args.mp_mode = "gaussian"
                    rast = GaussianShardedRasterizer(make_settings(mod, cam, dev), capacity=capacity, chunk=chunk, exchange="nccl")
        else:
            rast = ShardedGaussianRasterizer(make_settings(mod, cam, dev), capacity=capacity)

    gauss_sharded = use_dist and args.mp_mode.startswith("gaussian") and not ref_cuda
    p2p = gauss_sharded and args.mp_mode.startswith("gaussian-p2p")
    literal = gauss_sharded and args.mp_mode == "gaussian-p2p-allgather"
    lo, hi = (min(P, rank * chunk), min(P, (rank + 1) * chunk)) if gauss_sharded else (0, P)
    local_scene = {k: scene[k][lo:hi].contiguous() for k in PARAM_KEYS}  # this rank's Gaussians (all of them unless Gaussian-sharded)
    params = {k: local_scene[k].to(dev).requires_grad_(True) for k in PARAM_KEYS}
    means2D = torch.zeros((hi - lo, 3), device=dev, requires_grad=True)
    gc, gd, ga = (scene[k].to(dev) for k in ("grad_color", "grad_depth", "grad_alpha"))
    if use_dist:  # band-local loss: upstream grads are only defined on this rank's rows
        from street_gaussians_b200.sharded import band_of_rows
        m = band_of_rows(H, rank, world).to(dev).view(1, H, 1).float()
        gc, gd, ga = gc * m, gd * m, ga * m

    def step(p=params):
        for v in p.values():
            v.grad = None
        means2D.grad = None
        color, radii, depth, alpha, sem = rast(means3D=p["means3D"], means2D=means2D, opacities=p["opacities"], shs=p["shs"],
                                               scales=p["scales"], rotations=p["rotations"])
        torch.autograd.backward([color, depth, alpha], [gc, gd, ga])
        if literal:  # north-star literal contract: every rank ends the step holding ALL per-Gaussian gradients
            for k in PARAM_KEYS:
                gl = p[k].grad
                if gl.shape[0] < chunk:
                    gl = torch.cat([gl, gl.new_zeros((chunk - gl.shape[0],) + tuple(gl.shape[1:]))])
                dist.all_gather_into_tensor(full_grads[k].view(-1), gl.contiguous().view(-1))
        return color, radii, depth, alpha

    full_grads = {k: torch.empty((chunk * world,) + tuple(params[k].shape[1:]), device=dev) for k in PARAM_KEYS} if literal else None

    # ---- N > 1: verify THIS run against a single-GPU render of the same tensors before anything is timed ----
    parity_n = None
    if use_dist and not ref_cuda:
        for _ in range(3):  # exact frame (learns the capacities), first fused frame, steady-state fused frame
            step()
        parity_n = check_parity_n(mod, rast, scene, cam, dev, rank, world, H, lo, hi, params, means2D, (gc, gd, ga))
        ok = torch.tensor([1 if parity_n["ok"] else 0], device=dev)
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        worst = torch.tensor([parity_n["grad_rel_max"]], device=dev)
        dist.all_reduce(worst, op=dist.ReduceOp.MAX)
        parity_n = dict(ok=bool(int(ok.item())), images="band rows bit-equal to the single-GPU render on every rank" if int(ok.item()) else "MISMATCH",
                        grad_rel_max=float(worst.item()), grad_tol=1e-3)
        if not parity_n["ok"]:
            if rank == 0:
                print(json.dumps(dict(error="multi-GPU result differs from the single-GPU render", parity_n=parity_n)))
            dist.destroy_process_group()
            return 2

    def barrier():
        if use_dist:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident throughput ----
    sampler = ClockSampler(local_rank) if (rank == 0 and not args.no_clock_sampler) else None
    diag = {"ar": [], "host": []}
    if args.diag and use_dist and getattr(rast, "grad_reduce", None) is not None:
        inner = rast.grad_reduce

        def timed_reduce(g2d, gsem):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            out = inner(g2d, gsem)
            b.record()
            diag["ar"].append((a, b))
            return out

        rast.grad_reduce = timed_reduce
    for _ in range(max(args.warmup, 3)):
        step()
    diag["ar"].clear()
    barrier()
    if not ref_cuda:
        from street_gaussians_b200 import _capi as _sgr_capi

    # ---- optional: the step as a CUDA graph ----
    graph, graph_note, launches_per_replay = None, None, 0
    graph_ok = (not ref_cuda and args.graph != "off" and args.sync_free and capacity is not None and capacity.capacity is not None
                and not args.diag and (not use_dist or args.mp_mode == "gaussian-p2p"))
    if graph_ok:
        try:
            capacity.freeze()
            side = torch.cuda.Stream(device=dev)
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):  # warm-up on a side stream, as torch.cuda.graph requires
                for _ in range(3):
                    step()
            torch.cuda.current_stream().wait_stream(side)
            barrier()
            l0 = int(_sgr_capi.lib().sgr_launch_count())
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                outputs = step()
            launches_per_replay = int(_sgr_capi.lib().sgr_launch_count()) - l0
            for _ in range(3):
                graph.replay()
            torch.cuda.synchronize()
        except Exception as e:  # noqa: BLE001
            graph, graph_note = None, f"capture failed, eager loop timed instead: {e!r}"[:300]
            try:
                torch.cuda.synchronize()
            except Exception:  # noqa: BLE001
                pass
        if use_dist:  # every rank must take the same path (the device barriers pair replays with replays)
            flag = torch.tensor([1 if graph is not None else 0], device=dev)
            dist.all_reduce(flag, op=dist.ReduceOp.MIN)
            if int(flag.item()) == 0:
                graph = None
                graph_note = graph_note or "capture failed on another rank; eager loop timed instead"
        if graph is None:
            capacity.freeze(False)
            for _ in range(3):
                step()
        barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    if sampler:
        sampler.mark(0)
    launches0 = int(_sgr_capi.lib().sgr_launch_count()) if not ref_cuda else 0
    e0.record()
    for _ in range(args.steps):
        t_h = time.perf_counter()
        if graph is not None:
            graph.replay()
        else:
            outputs = step()
        diag["host"].append((time.perf_counter() - t_h) * 1e3)
    e1.record()
    barrier()
    ms_total = e0.elapsed_time(e1)
    color, radii = outputs[:2]
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, *outputs, params, means2D)
    # kernels of libsgr.so enqueued by THIS rank inside the timed region (counted in the library at launch / capture time; cub's sort
    # and scan kernels excluded)
    if ref_cuda:
        gpu_launches = 0
    elif graph is not None:
        gpu_launches = launches_per_replay * args.steps
    else:
        gpu_launches = int(_sgr_capi.lib().sgr_launch_count()) - launches0
    host_ms = float(np.median(diag["host"]))
    if graph is not None:
        capacity.freeze(False)  # the legs below (stage table, exact mode, e2e) run eagerly with tracking on
    if args.diag:
        ar = [a.elapsed_time(b) for a, b in diag["ar"]]
        print(f"[diag rank {rank}] step {ms_total / args.steps:.3f} ms | host loop per step: median {np.median(diag['host']):.3f} max {max(diag['host']):.3f} ms"
              + (f" | all-reduce (device, incl. waiting for peers): median {np.median(ar):.3f} min {min(ar):.3f} max {max(ar):.3f} ms" if ar else ""),
              file=sys.stderr, flush=True)
    if use_dist:
        t = torch.tensor([ms_total], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_total = float(t.item())
    ms_step = ms_total / args.steps
    vis_t = (radii > 0).sum()
    if gauss_sharded:
        dist.all_reduce(vis_t, op=dist.ReduceOp.SUM)
    visible = int(vis_t.item())
    exact_ms = None
    if not ref_cuda and args.sync_free and not use_dist:
        rast_exact = mod.GaussianRasterizer(make_settings(mod, cam, dev))

        def step_exact():
            for v in params.values():
                v.grad = None
            color, radii_, depth, alpha, sem = rast_exact(means3D=params["means3D"], means2D=means2D, opacities=params["opacities"],
                                                           shs=params["shs"], scales=params["scales"], rotations=params["rotations"])
            torch.autograd.backward([color, depth, alpha], [gc, gd, ga])

        for _ in range(3):
            step_exact()
        torch.cuda.synchronize()
        x0, x1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        x0.record()
        for _ in range(args.steps):
            step_exact()
        x1.record()
        torch.cuda.synchronize()
        exact_ms = x0.elapsed_time(x1) / args.steps

    # ---- per-stage device times (CUDA events around the staged C-ABI calls) + roofline of the dominant kernel ----
    roofline, stages, n_inst = None, {}, None
    if gauss_sharded:
        from street_gaussians_b200 import sharded as SH
        st_obj = make_settings(mod, cam, dev)
        band = rast.band
        with torch.no_grad():
            lt = SH._local_tensors(params["means3D"], params["shs"], None, None, params["opacities"], params["scales"], params["rotations"], None)
            names = ("project", "scatter+barrier" if p2p else "all_gather", "forward_records", "blend_bwd",
                     "barrier+gather" if p2p else "reduce_scatter", "preprocess_bwd")
            acc = {k: [] for k in names}
            ws = rast.workspace(dev) if p2p else None
            for it in range(3 + 5):
                evs = [torch.cuda.Event(enable_timing=True) for _ in range(7)]
                evs[0].record()
                rec, radii_l = SH.project_records(lt, st_obj, chunk)
                evs[1].record()
                if p2p:
                    SH.scatter_records(st_obj, ws, rec, radii_l, hi - lo)
                    ws.barrier()
                    fs, radii_all, gb, ib = SH.peer_forward_state(ws), ws.radii_all, ws.geom_bytes, ws.img_bytes
                else:
                    fs, rec_all, gb, ib = SH.alloc_gathered(st_obj, chunk * world, 0, dev)
                    radii_all = torch.empty((chunk * world,), device=dev, dtype=torch.int32)
                    dist.all_gather_into_tensor(rec_all.view(-1), rec.view(-1))
                    dist.all_gather_into_tensor(radii_all, radii_l)
                evs[2].record()
                col, dep, alp, sem = SH.forward_records(st_obj, band, fs, (gb, ib), radii_all, None)
                evs[3].record()
                g2d, gsem = SH.backward_blend_records(st_obj, band, fs, chunk * world, None, alp, gc, gd, ga, None,
                                                      grad2d_out=ws.grad2d if p2p else None)
                evs[4].record()
                if p2p:
                    ws.barrier()
                    g2l = SH.gather_grad2d(st_obj, ws, rec, radii_l, hi - lo)
                else:
                    g2l = torch.empty((chunk, 12), device=dev)
                    dist.reduce_scatter_tensor(g2l.view(-1), g2d.view(-1))
                evs[5].record()
                SH.backward_geom_local(st_obj, lt, rec, radii_l, g2l)
                evs[6].record()
                torch.cuda.synchronize()
                if it >= 3:
                    for i, k in enumerate(names):
                        acc[k].append(evs[i].elapsed_time(evs[i + 1]))
            stages = {k: float(np.median(v)) for k, v in acc.items()}
            n_inst = int(fs.num_instances)
    elif not ref_cuda:
        from street_gaussians_b200 import rasterizer as R
        st_obj = make_settings(mod, cam, dev)
        band = rast.band
        with torch.no_grad():
            def ev():
                return torch.cuda.Event(enable_timing=True)
            acc = {"forward": [], "blend_bwd": [], "preprocess_bwd": []}
            for it in range(3 + 5):
                a, b, c, d = ev(), ev(), ev(), ev()
                a.record()
                col, rad, dep, alp, sem, fst, tens = R._forward_impl(params["means3D"], params["shs"], None, None, params["opacities"],
                                                                      params["scales"], params["rotations"], None, st_obj, band)
                b.record()
                g2d, gsem = R._backward_blend_impl(st_obj, band, fst, tens, alp, gc, gd, ga, None)
                c.record()
                R._backward_geom_impl(st_obj, band, fst, tens, rad, g2d)
                d.record()
                torch.cuda.synchronize()
                if it >= 3:
                    acc["forward"].append(a.elapsed_time(b)); acc["blend_bwd"].append(b.elapsed_time(c)); acc["preprocess_bwd"].append(c.elapsed_time(d))
            stages = {k: float(np.median(v)) for k, v in acc.items()}
            n_inst = int(fst.num_instances)
    if not ref_cuda:
        npx = W * H
        # SURVEY.md §8(d): blend_bwd = R*44 + Npx*28 + V*44 bytes (R = this library's instance count, this rank's band)
        rows_frac = 1.0 / world if use_dist else 1.0
        alg_bytes = n_inst * 44 + npx * rows_frac * 28 + visible * 44
        peak, peak_src = measured_peaks()
        achieved = alg_bytes / (stages["blend_bwd"] * 1e-3) / 1e9
        # dram__bytes_read.sum + dram__bytes_write.sum of the kernel from the committed `ncu --set full` capture: only reported when
        # profiles/ncu_traffic.json holds a capture of THIS workload taken from THIS version of the kernel source (sha256 of the .cu)
        traffic, issue_pct, traffic_stale = ncu_traffic("blend_bwd2_kernel", "blend_bwd2.cu", args.workload if not use_dist else None)
        roofline = dict(bound="hbm", kernel="blend_bwd2_kernel", achieved=achieved, peak=peak, unit="GB/s", frac=achieved / peak,
                        traffic=traffic, issue_active_pct=issue_pct, peak_source=peak_src, algorithmic_bytes=alg_bytes, kernel_ms=stages["blend_bwd"],
                        note="blend kernels are FP32/SFU-issue bound, not HBM bound (SURVEY.md §8d; ncu of the round-1 build: 76 % issue-active, "
                             "1.4 % DRAM): real DRAM traffic is ~8x BELOW the algorithmic bytes because the tile lists and records are L2 hits; "
                             "the HBM fraction is reported as the contract asks; kernel_ms includes the cudaMemsetAsync of the accumulators")
        if traffic is None and traffic_stale is not None:
            roofline["traffic_earlier_build"] = traffic_stale

    # ---- end to end from pinned host memory ----
    if args.no_e2e:
        if sampler:
            sampler.mark(1)
        clocks = sampler.stop() if sampler else None
        if rank == 0:
            fps = 1000.0 / ms_step
            print(json.dumps(dict(metric="rasterizer_fwd_bwd_fps", value=fps, unit="frames/s", n_gpus=world if use_dist else 1, steps=args.steps,
                                  warmup=max(args.warmup, 3), ms_per_step=ms_step, higher_is_better=True, scaling="strong", dtype="f32",
                                  config=dict(workload=wl_desc, stage_ms=stages), clocks=clocks, note="--no-e2e diagnostic line")))
        if use_dist:
            dist.destroy_process_group()
        return 0
    host = {k: local_scene[k].pin_memory() for k in PARAM_KEYS}
    h2d_bytes = sum(v.numel() * 4 for v in host.values())  # this rank's share; summed over ranks below when Gaussian-sharded
    copy_stream = torch.cuda.Stream(device=dev)
    bufs = [{k: torch.empty_like(v, device=dev) for k, v in host.items()} for _ in range(2)]
    ready = [torch.cuda.Event(), torch.cuda.Event()]
    consumed = [torch.cuda.Event(), torch.cuda.Event()]
    loss_host = torch.zeros(1).pin_memory()

    def upload(i):
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(consumed[i])
            for k in PARAM_KEYS:
                bufs[i][k].copy_(host[k], non_blocking=True)
            ready[i].record(copy_stream)

    def e2e_step(i):
        torch.cuda.current_stream().wait_event(ready[i])
        p = {k: bufs[i][k].detach().requires_grad_(True) for k in PARAM_KEYS}
        color, radii, depth, alpha, sem = rast(means3D=p["means3D"], means2D=means2D, opacities=p["opacities"], shs=p["shs"],
                                               scales=p["scales"], rotations=p["rotations"])
        loss = (color * gc).sum() + (depth * gd).sum() + (alpha * ga).sum()
        loss.backward()
        consumed[i].record()
        loss_host.copy_(loss.detach().view(1), non_blocking=True)

    for ev_ in consumed:
        ev_.record()
    n_e2e = max(3, min(args.steps, 10))
    upload(0)
    for i in range(3):  # warm-up
        upload((i + 1) % 2)
        e2e_step(i % 2)
    barrier()
    upload(0)
    e0.record()
    for i in range(n_e2e):
        upload((i + 1) % 2)
        e2e_step(i % 2)
    e1.record()
    barrier()
    _ = float(loss_host.item())
    e2e_ms = e0.elapsed_time(e1) / n_e2e
    if use_dist:
        t = torch.tensor([e2e_ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_ms = float(t.item())
    if gauss_sharded:
        t = torch.tensor([float(h2d_bytes)], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        h2d_bytes = int(t.item())
    # ---- end to end through the COMPOSER (SURVEY.md §8 f1): the raw per-model parameters stay resident in HBM like the nn.Parameters of
    # a training run; what a frame brings from the host is the camera and the tracked actor poses ----
    e2e_comp = None
    if "raw" in scene:
        e2e_comp = composed_e2e(args, mod, rast, scene, cam, dev, lo, hi, means2D, (gc, gd, ga), ref_cuda, barrier, use_dist, n_e2e,
                                capacity=None if ref_cuda else capacity)
    if sampler:
        sampler.mark(1)
    clocks = sampler.stop() if sampler else None

    if rank == 0:
        cb = None if args.no_cpu_baseline else cpu_baseline(scene, args.cpu_sample_stride)
        fps = 1000.0 / ms_step
        line = dict(metric="rasterizer_fwd_bwd_fps", value=fps, unit="frames/s", n_gpus=world if use_dist else 1, steps=args.steps,
                    warmup=max(args.warmup, 3), ms_per_step=ms_step, higher_is_better=True, scaling="strong", vs_baseline=None,
                    dtype="f32", data="synthetic (seeded; street_gaussians_b200/synthetic.py)",
                    config=dict(workload=wl_desc, P=P, visible=visible, width=W, height=H, sh_degree=cam["sh_degree"],
                                l2="inputs (%.0f MB of Gaussian parameters) exceed the 126 MB L2; no explicit flush" % (h2d_bytes / 1e6),
                                parallelism=(("Gaussian-sharded x%d (P/N Gaussians + cyclic tile rows per rank): %s; parameters and gradients stay sharded"
                                              % (world, ("48-B records stored / grad2d rows loaded over NVLink peer memory to/from only the ranks whose band "
                                                         "a Gaussian touches (stores fused into the projection kernel, loads into the chain-rule kernel), 2 device-side "
                                                         "barriers per step, no NCCL on the data path" + ("; PLUS an NCCL all-gather of all parameter gradients so every "
                                                         "rank holds all of them (north-star literal contract)" if literal else "")) if p2p else
                                                 "NCCL all-gather of 48-B records, reduce-scatter of grad2d[P,12]")) if gauss_sharded else
                                             ("tile-row sharded x%d (cyclic rows), parameters replicated, 1 NCCL all-reduce of grad2d[P,12]/step" % world))
                                if use_dist else "single GPU",
                                mp_mode=(args.mp_mode if use_dist else None),
                                num_instances=n_inst, gaussians_pixels_per_s=P * W * H * fps, stage_ms=stages,
                                stage_ms_note=("per-stage CUDA events of the STAGED calls (one C-ABI call per stage, run after the timed region); "
                                               "the timed region itself issues each forward / backward as one fused call") if p2p else None,
                                binning_mode="sync-free (InstanceCapacity)" if args.sync_free else "exact (drop-in default: one 4-byte read-back per forward)",
                                exact_mode_ms_per_step=exact_ms),
                    e2e=dict(value=1000.0 / e2e_ms, unit="frames/s", ms_per_step=e2e_ms, h2d_bytes_per_step=h2d_bytes, d2h_bytes_per_step=4,
                             note="pinned host -> device copy of all 59 floats/Gaussian every step (each rank uploads the Gaussians it owns), double-buffered on a copy stream; scalar loss read back"),
                    gpu_launches=gpu_launches, clocks=clocks)
        line["config"]["host_ms_per_step"] = host_ms
        line["config"]["timed_region"] = ("CUDA graph: one fwd+bwd step through the public API (autograd included) captured after the warm-up, "
                                          "replayed %d times" % args.steps) if graph is not None else "eager Python loop"
        if graph_note:
            line["config"]["graph_note"] = graph_note
        if parity_n is not None:
            line["parity_n"] = parity_n
        if e2e_comp is not None:
            # headline end-to-end number: the call a user of the framework makes per training frame (compose -> rasterize -> backward
            # through both), per-frame inputs (camera + actor poses) copied from pinned host memory; the full-parameter upload variant
            # of round 1 is kept beside it
            line["e2e_full_upload"] = line["e2e"]
            line["e2e"] = e2e_comp
        if roofline:
            line["roofline"] = roofline
        if cb:
            line["cpu_baseline"] = cb
        if ref_cuda:
            line["impl"] = "reference"
            line["config"]["reference"] = "unmodified DGR sources compiled for sm_100 into oracle/_ref (stock CUDA rasterizer, on the GPU)"
            line["gpu_launches"] = 0
        print(json.dumps(line))
    if use_dist:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
