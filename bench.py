#!/usr/bin/env python
"""bench.py -- train-step images/sec (fwd+bwd) @1080p, 3M Gaussians, SH-3 (BASELINE.json).

  python bench.py --gpus N --steps K --warmup W            our sm_100a path
  python bench.py --impl reference --gpus N ...            the CPU restatement of the same path, WHOLE frames on the
                                                           host cores (the reference's own source for it is absent)
  python bench.py --impl reference-cuda ...                the reference's own CUDA build, if baseline/refprobe.py finds
                                                           one on this machine (else one line saying it is unavailable)

A "step" (SURVEY.md 8d) = LOD cut (expand_to_size + get_interpolation_weights) -> cut gather / parent lerp ->
rasterizer forward -> L1 loss gradient -> rasterizer backward -> gradient scatter to the full parameter arrays.
Three host forms of that step are timed (same kernels, same results -- tests/test_gpu_graphstep.py, test_gpu_pipeline.py):

  value         --mode graph (default on hierarchy workloads): the sync-free step of h3dgs.graphstep -- device-side LOD
                cut, capacity-sized binning, the whole step replayed from two CUDA graphs, nothing returns to the host;
  value_api     --mode api: call by call through the drop-in packages (gaussian_hierarchy._C + GaussianRasterizer) with the
                cut gather / lerp fused into K1/K9 (settings.render_indices / parent_indices -- an opt-in: the reference's
                call sites leave those fields empty);
  value_dropin  what the reference's unmodified render_post() flow costs on top of the packages: its ~25 PyTorch gather /
                lerp kernels around the rasterizer, index_add in backward (h3dgs.pipeline.render_hier).

N > 1: one process per GPU, the frame is screen-tile-sharded (h3dgs.dist), strong scaling.  Prints ONE JSON line on rank 0.
The stage profiler (cudaEvents around every library launch) is OFF in every timed region; per-stage times come from a
separate pass."""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "hierarchical-3d-gaussians_b200")
for p in (ROOT, PKG, os.path.join(ROOT, "baseline")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402

METRIC = "train-step images/sec (fwd+bwd) @1080p, 3M Gaussians, SH-3"
UNIT = "images/s"
W, H = 1920, 1080                # overridden by the 4K workload (main)
RESOLUTION = {"hier20m4k": (3840, 2160)}
TAU = 6.0
N_VIEWS = 8
WORKLOADS = {"hier3m": "config #3: N_all=3M (1.5M leaves + 1,499,999 interior nodes), 1920x1080, SH-3, LOD cut tau=6px, "
                       "fwd+bwd, 8 synthetic views (cloud v2: BASELINE.md section 2a)",
             "flat1m": "config #2: 1M flat Gaussians (cloud v1), 1920x1080, SH-3, fwd+bwd",
             "tiny": "smoke-size hierarchy",
             "hier20m4k": "config #5: N_all=20M (10M leaves + 9,999,999 interior nodes), 3840x2160, SH-3, LOD cut tau=6px, "
                          "fwd+bwd, 8 synthetic views"}


# ----------------------------------------------------------------------------- workload
def build_workload(name, cache_dir="/tmp/h3dgs_cache", device=None):
    """Synthetic scene + cameras.  hier3m: 1.5M leaves + 1,499,999 interior nodes (config #3); flat1m: 1M flat
    Gaussians (config #2), both numpy, cached under /tmp.  hier20m4k: 10M leaves + 9,999,999 interior nodes at
    3840x2160 (config #5), generated with torch ops directly on `device` (h3dgs.synth_torch; seconds on a GPU
    where the numpy builder needs minutes) -- tensors, not cached."""
    from h3dgs import synth
    os.makedirs(cache_dir, exist_ok=True)
    path = os.path.join(cache_dir, f"{name}_v3.npz")
    cams = [synth.make_camera(W, H)]
    rs = np.random.default_rng(2)
    for i in range(1, N_VIEWS):
        cams.append(synth.yaw_camera(W, H, float(rs.uniform(-15, 15)), rs.uniform(-0.5, 0.5, 3)))
    if name == "hier20m4k":
        from h3dgs import synth_torch
        leaves = synth_torch.cloud(10_000_000, cams[0].tanfovx, cams[0].tanfovy, sh_degree=3, zmin=2.0, zmax=60.0, seed=0,
                                   device=device or "cpu")
        return synth_torch.build_hierarchy(leaves), cams
    if os.path.exists(path):
        z = np.load(path)
        return {k: z[k] for k in z.files}, cams
    cam = cams[0]
    if name == "hier3m":
        # Cloud v2 (a documented deviation from SURVEY.md 8d's cloud v1, BASELINE.md section 2a): like cloud v1 but the
        # world-space size grows as sqrt(z) (screen size shrinks with distance), so the tau=6px cut really merges far
        # leaves instead of returning all 1.5M of them; z ~ U[2,60]
        leaves = synth.cloud_v1(1_500_000, cam, sh_degree=3, zmin=2.0, zmax=60.0, seed=0, scale_k=1.0)
        z = leaves["means3D"][:, 2:3]
        g = np.random.default_rng(7)
        leaves["scales"] = (2.4e-3 * np.sqrt(2.0 * z) * np.exp(0.5 * g.standard_normal((z.shape[0], 3)))).astype(np.float32)
        arrays = synth.build_hierarchy(leaves)
    elif name == "flat1m":
        arrays = synth.cloud_v1(1_000_000, cam, sh_degree=3, seed=0)
    elif name == "tiny":
        leaves = synth.cloud_v1(20_000, cam, sh_degree=3, zmin=2.0, zmax=60.0, seed=0, scale_k=8e-3)
        arrays = synth.build_hierarchy(leaves)
    else:
        raise ValueError(name)
    tmp = path + f".{os.getpid()}.tmp.npz"
    np.savez(tmp, **arrays)
    os.replace(tmp, path)
    return arrays, cams


def alg_bytes(P, V, D, hier, N_nodes=0, fused=False):
    """ALGORITHMIC bytes per image, per stage (SURVEY.md 8d derivation: every array once per stage that must produce /
    consume it, fp32/i32, sort idealised as one read + one write).  `total` is the section's base formula
    60 P + 792 V + 160 D + 52 Px + 8 T; the section's add-ons for what this step also does are listed separately:
    hierarchy (t, k) + 8 P, LOD cut + 60 per node visited, cut gather / lerp fused into ours + 3*236 P each way."""
    Px, T = W * H, ((W + 15) // 16) * ((H + 15) // 16)
    b = {
        "preprocess": 44 * P + 8 * P + 40 * V,
        "preprocess_color": 192 * V,
        "scan": 8 * P,                             # per-tile path: 8 T (tile histogram scan)
        "key_emission": 12 * D,
        "sort": 24 * D,                            # per-tile path: fused with the record gather (tile_sort_gather)
        "identify_tile_ranges": 8 * D + 8 * T,     # fallback path only
        "gather_records": 0,                       # fallback path only; implementation choice (TMA staging)
        "render_forward": 40 * D + 20 * Px,
        "render_backward": 40 * D + 36 * D + 32 * Px,
        "preprocess_backward": (36 + 44 + 40) * V + 56 * V,
        "sh_backward": 192 * V + 192 * V,
    }
    b["total"] = sum(b.values())
    addons = {"hierarchy_t_k": 8 * P if hier else 0, "lod_cut": 60 * N_nodes if hier else 0,
              "gather_lerp_fused_fwd": 3 * 236 * P if fused else 0, "gather_lerp_fused_bwd": 3 * 236 * P if fused else 0}
    b["addons"] = addons
    b["total_with_addons"] = b["total"] + sum(addons.values())
    b["lod_cut"] = addons["lod_cut"]
    return b


# ----------------------------------------------------------------------------- clocks
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx, self.rows, self.proc = gpu_index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.idx)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm = [float(r[1]) for r in self.rows if len(r) >= 9 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 9 and r[2].replace(".", "").isdigit()]
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            if len(r) >= 9:
                for n, v in zip(names, r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ----------------------------------------------------------------------------- CPU arms
def cpu_step_fn(arrays, cams, frac=1):
    """Returns a callable running ONE step of the path on the host cores with the oracle (kind "port"): LOD cut +
    weights + gather/lerp + forward + L1 grad + backward at full resolution; frac > 1 keeps every frac-th Gaussian of
    the cut (only used when a whole frame does not fit the time budget, e.g. on a laptop)."""
    from oracle import oracle
    from h3dgs import synth
    hier = "nodes" in arrays

    def step(i):
        cam = cams[i % len(cams)]
        if hier:
            thr = synth.tau_threshold(TAU, cam)
            n, ri, pi, ni = oracle.expand_to_size(arrays["nodes"], arrays["boxes"], thr, cam.camera_center)
            ts, kids = oracle.get_interpolation_weights(ni, thr, arrays["nodes"], arrays["boxes"], cam.camera_center)
            sel = slice(0, n, frac)
            (means, shs, opac, scales, rots), _ = oracle.lerp_cut(arrays["means3D"], arrays["shs"], arrays["opacities"],
                                                                  arrays["scales"], arrays["rotations"], ri[sel], pi[sel], ts[sel])
            ts, kids = ts[sel], kids[sel]
        else:
            sel = slice(0, None, frac)
            means, scales, shs, opac, rots = (arrays[k][sel] for k in ("means3D", "scales", "shs", "opacities", "rotations"))
            ts = kids = None
        f = oracle.rasterize_forward(means, shs, None, opac, scales, rots, None, cam.world_view_transform,
                                     cam.full_proj_transform, cam.camera_center, np.zeros(3, np.float32), W, H,
                                     cam.tanfovx, cam.tanfovy, ts=ts, kids=kids)
        g = synth.l1_grad(f["color"], seed=3 + i)
        oracle.rasterize_backward(f, g)
        return f["num_rendered"]
    return step


def run_cpu_arm(arrays, cams, steps, warmup, budget_s=25.0, frac=0):
    """Times whole frames (frac = 1).  frac = 0: one probe frame decides -- if it alone exceeds the budget the arm falls
    back to every 16th Gaussian of the cut and SAYS so (value then is an extrapolation, reported as such)."""
    arrays = {k: (v.detach().cpu().numpy() if hasattr(v, "detach") else v) for k, v in arrays.items()}
    from oracle import oracle
    oracle.set_threads(os.cpu_count() or 1)          # torchrun exports OMP_NUM_THREADS=1
    t0 = time.perf_counter()
    probe_s = None
    if frac == 0:
        cpu_step_fn(arrays, cams, 1)(0)
        probe_s = time.perf_counter() - t0
        frac = 1 if probe_s <= budget_s else 16
    step = cpu_step_fn(arrays, cams, frac)
    w_done = 1 if (probe_s is not None and frac == 1) else 0          # the probe frame was a warm-up frame
    while w_done < warmup and time.perf_counter() - t0 < 0.3 * budget_s:
        step(w_done); w_done += 1
    t1 = time.perf_counter()
    done = 0
    for i in range(steps):
        step(warmup + i)
        done += 1
        if time.perf_counter() - t0 > budget_s:
            break
    dt = (time.perf_counter() - t1) / done
    return dict(ms_per_step=dt * 1e3, value=1.0 / (dt * frac), steps_run=done, warmup_run=w_done, frac=frac,
                cores=oracle.num_threads())


def run_pytorch_config1():
    """BASELINE.json configs[0] in full: 1k random Gaussians, 128x128, SH-0, 1 view -- the naive pure-PyTorch CPU
    point-splat (oracle/torch_splat.py, dense [pixels x Gaussians], autograd backward) on all host cores."""
    import torch
    from h3dgs import synth
    from oracle import torch_splat
    n = os.cpu_count() or 1
    torch.set_num_threads(n)
    cam = synth.make_camera(128, 128)
    sc = synth.cloud_v1(1000, cam, sh_degree=0, seed=0, scale_k=2e-2)
    t = lambda a: torch.tensor(a, dtype=torch.float32, requires_grad=True)
    p = {k: t(sc[k]) for k in ("means3D", "shs", "opacities", "scales", "rotations")}
    c = lambda a: torch.tensor(a, dtype=torch.float32)
    times = []
    for _ in range(4):
        for v in p.values():
            v.grad = None
        t0 = time.perf_counter()
        img, radii, _ = torch_splat.splat(p["means3D"], p["shs"], None, p["opacities"], p["scales"], p["rotations"], None,
                                          c(cam.world_view_transform), c(cam.full_proj_transform), c(cam.camera_center),
                                          torch.zeros(3), 128, 128, cam.tanfovx, cam.tanfovy, sh_degree=0)
        (img - 0.5).abs().mean().backward()
        times.append(time.perf_counter() - t0)
    dt = float(np.median(times[1:]))
    return {"value": 1.0 / dt, "unit": UNIT, "cores": n, "kind": "pytorch", "ms_per_step": dt * 1e3,
            "sample": "config #1 in full: 1k Gaussians, 128x128, SH-0, 1 view, fwd+bwd (autograd), median of 3 after 1 warm-up; "
                      "oracle/torch_splat.py, torch.set_num_threads(%d)" % n}


def time_classic(scene, cam, bg, thr, hier, stage_ms, iters=10):
    """Times baseline/classic/libclassic.so (one index gather per thread per round, one pixel per
    thread, one global atomic per pixel per gradient value -- the formulation of the 3DGS paper; the
    reference's own kernels are absent) on the SAME binned state as our blend kernels."""
    import ctypes as C
    import torch
    from h3dgs import pipeline
    from diff_gaussian_rasterization import _C as rc
    lib = C.CDLL(os.path.join(ROOT, "baseline", "classic", "libclassic.so"))
    with torch.no_grad():
        if hier:
            n = pipeline.lod_cut(scene, cam, thr)
            m, s, r, o, sh = pipeline.interpolate_cut(scene, n)
        else:
            m, s, r, o, sh = scene.means3D, scene.scales, scene.rotations, scene.opacities, scene.shs
            n = m.shape[0]
        D, color, radii, gb, bb, ib, _ = rc.rasterize_gaussians(bg, m, None, o, s, r, 1.0, None, cam.viewmatrix,
                                                                cam.projmatrix, cam.tanfovx, cam.tanfovy, cam.H, cam.W,
                                                                sh, 3, cam.campos, False, False)
        sv = rc.state_view(n, cam.W, cam.H, D, gb, bb, ib)
        ptr = lambda t: C.c_void_p(t.data_ptr())
        out = torch.empty_like(color); fT = torch.empty((cam.H, cam.W), device=color.device)
        nc = torch.empty((cam.H, cam.W), dtype=torch.int32, device=color.device)
        g = torch.sign(color - torch.rand_like(color)) / color.numel()
        accum = torch.zeros((n, 10), device=color.device)
        st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
        fwd = lambda: lib.classic_render_forward(cam.W, cam.H, ptr(sv["ranges"]), ptr(sv["point_list"]), ptr(sv["records"]),
                                                 ptr(bg), ptr(out), ptr(fT), ptr(nc), st)
        bwd = lambda: lib.classic_render_backward(cam.W, cam.H, ptr(sv["ranges"]), ptr(sv["point_list"]), ptr(sv["records"]),
                                                  ptr(bg), ptr(fT), ptr(nc), ptr(g), ptr(accum), st)
        res = {}
        for name, fn in (("render_forward", fwd), ("render_backward", bwd)):
            for _ in range(3):
                fn()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(iters):
                fn()
            e1.record(); torch.cuda.synchronize()
            res[name + "_ms"] = e0.elapsed_time(e1) / iters
        res["image_max_abs_diff_vs_ours"] = float((out - color).abs().max().item())
        res["ours_ms"] = {k: stage_ms.get(k) for k in ("render_forward", "render_backward", "gather_records", "sort")}
        res["note"] = ("classic = stand-in for the absent reference kernels (paper formulation, flat alpha, no "
                       "hierarchy weight); ours includes the record materialisation (sort / gather_records) it relies on")
    return res


# ----------------------------------------------------------------------------- reference arms
def reference_arm(args, config, rank):
    """--impl reference: rank 0 alone, the CPU restatement of the path on the box's host cores, whole frames."""
    if rank != 0:
        return
    arrays, cams = build_workload(args.workload)
    r = run_cpu_arm(arrays, cams, args.steps, args.warmup, budget_s=150.0)
    whole = r["frac"] == 1
    sample = (f"{r['steps_run']} whole frame(s) at {W}x{H} after {r['warmup_run']} warm-up frame(s), no extrapolation" if whole else
              f"every {r['frac']}th Gaussian of the cut at {W}x{H} (a whole frame exceeds the time budget on this host), "
              f"{r['steps_run']} step(s), images/s extrapolated linearly (x1/{r['frac']})") + "; oracle/oracle.c with OpenMP"
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": r["value"], "unit": UNIT, "n_gpus": args.gpus,
        "steps": r["steps_run"], "warmup": r["warmup_run"], "ms_per_step": r["ms_per_step"] if whole else r["ms_per_step"] * r["frac"],
        "ms_per_sample_step": r["ms_per_step"], "extrapolated": not whole,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": config,
        "cpu_baseline": {"value": r["value"], "unit": UNIT, "cores": r["cores"], "kind": "port", "sample": sample},
        "e2e": {"value": r["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": "the reference's own implementation of this path (hierarchy-rasterizer, gaussian-hierarchy) is "
                "absent from /root/reference and is CUDA-only; this arm times the CPU restatement (oracle port). "
                "steps/warmup are what fitted the 150 s budget of this arm"}))


def reference_cuda_arm(args, config, rank, local_rank):
    """--impl reference-cuda: the reference's own CUDA packages on the same inputs, when baseline/refprobe.py finds a
    build (flat workloads through GaussianRasterizer; hierarchy workloads through the reference's render_post flow:
    PyTorch gather/lerp + its rasterizer with interpolation_weights / num_node_kids)."""
    if rank != 0:
        return
    import refprobe
    pr = refprobe.probe()
    if not pr["available"]:
        print(json.dumps({"impl": "reference-cuda", "unavailable": pr["note"], "probe": pr}))
        return
    import torch
    from h3dgs import pipeline, synth
    ref = refprobe.load("diff_gaussian_rasterization")
    refh = refprobe.load("gaussian_hierarchy")
    dev = f"cuda:{local_rank}"
    torch.cuda.set_device(local_rank)
    arrays, cams = build_workload(args.workload, device=dev)
    scene = pipeline.Scene(arrays, device=dev)
    dcams = [pipeline.DeviceCamera(c, device=dev) for c in cams]
    thr = [synth.tau_threshold(TAU, c) for c in cams]
    bg = torch.zeros(3, device=dev)
    gts = [torch.rand((3, H, W), generator=torch.Generator().manual_seed(5 + v)).to(dev) for v in range(N_VIEWS)]
    # swap the package handles h3dgs.pipeline drives for the reference's
    pipeline.GaussianRasterizationSettings, pipeline.GaussianRasterizer = ref.GaussianRasterizationSettings, ref.GaussianRasterizer
    if refh is not None:
        pipeline.expand_to_size, pipeline.get_interpolation_weights = refh._C.expand_to_size, refh._C.get_interpolation_weights
    step = lambda i: pipeline.l1_step(scene, dcams[i % N_VIEWS], bg, gts[i % N_VIEWS], thr[i % N_VIEWS] if scene.hier else None, fused=False)
    for i in range(max(args.warmup, 20)):
        step(i)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(args.steps):
        step(i)
    e1.record(); torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / args.steps
    print(json.dumps({"impl": "reference-cuda", "metric": METRIC, "value": 1000.0 / ms, "unit": UNIT, "n_gpus": 1, "steps": args.steps,
                      "warmup": max(args.warmup, 20), "ms_per_step": ms, "higher_is_better": True, "scaling": "strong",
                      "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config, "probe": pr,
                      "note": "the reference's unmodified packages driven through its own render_post-style flow "
                              "(PyTorch gather/lerp around its rasterizer); compare with value_dropin of the default arm"}))


# ----------------------------------------------------------------------------- outputs
DUMP_MAX_ELEMENTS = 1 << 20       # per array: at most 8 MB each, so the seven arrays of a step stay under 64 MB


def dump_outputs(out_dir, arrays):
    """Writes each tensor as out_dir/<name>.npy (integers and float64 as float64, everything else as float32), so that
    two builds run with the same arguments can be compared output for output.  An array of more than DUMP_MAX_ELEMENTS
    elements is written as the flat sample of that many elements at positions drawn with a fixed seed (sorted), the
    same positions for every array of that size."""
    import torch
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        t = t.detach()
        if t.numel() > DUMP_MAX_ELEMENTS:
            idx = np.sort(np.random.default_rng(0).choice(t.numel(), DUMP_MAX_ELEMENTS, replace=False))
            t = t.reshape(-1)[torch.from_numpy(idx).to(t.device)]
        dtype = torch.float32 if t.dtype in (torch.float32, torch.float16, torch.bfloat16) else torch.float64
        np.save(os.path.join(out_dir, name + ".npy"), t.to(dtype).cpu().numpy())


# ----------------------------------------------------------------------------- GPU arm
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "reference-cuda"])
    ap.add_argument("--workload", default="hier3m", choices=list(WORKLOADS))
    ap.add_argument("--mode", default=None, choices=["graph", "api"],
                    help="host form of the headline `value` (default: graph on hierarchy workloads, api on flat ones)")
    ap.add_argument("--graph", action="store_true", help="same as --mode graph")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the value_api / value_dropin / N-rank check passes")
    ap.add_argument("--no-peer", action="store_true",
                    help="N > 1, graph mode: NCCL all-gather + reduce-scatter instead of the collectives fused into the blend "
                         "kernels over peer memory (the default on 2, 4 or 8 GPUs)")
    ap.add_argument("--classic", action="store_true",
                    help="also time the classic-formulation blend kernels (baseline/classic) on the same binned state")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last of them computed as DIR/<name>.npy (see dump_outputs)")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    hier = args.workload != "flat1m"
    mode = args.mode or ("graph" if (args.graph or hier) else "api")
    # N > 1 without an explicit --mode: the graphed step with the collectives fused over peer memory when the ranks can map
    # each other's memory (validated on 2 GPUs incl. the N-rank equality check: profiles/r02_m2b_*); otherwise the call-by-call
    # NCCL form (--mode graph --no-peer selects the graphed NCCL form explicitly)
    auto_mode = world > 1 and not args.mode and not args.graph
    if mode == "graph" and not hier:
        raise SystemExit("--mode graph drives the hierarchy step (LOD cut + fused gather/lerp)")
    global W, H
    W, H = RESOLUTION.get(args.workload, (W, H))
    config = {"workload": WORKLOADS[args.workload],
              "l2": "inputs larger than L2 (parameter arrays 0.7 GB, per-step state > 1 GB); no explicit flush",
              "parallelism": f"screen-tile-sharded x{world}" if world > 1 else "single GPU",
              "mode": {"graph": "sync-free step replayed from CUDA graphs (h3dgs.graphstep)",
                       "api": "call by call through the drop-in packages, cut gather/lerp fused into K1/K9"}[mode]}

    if args.impl == "reference":
        return reference_arm(args, config, rank)
    if args.impl == "reference-cuda":
        return reference_cuda_arm(args, config, rank, local_rank)

    # ---------------- our arm ----------------
    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py (impl ours) needs a CUDA device: there is no CPU fallback for this path")
    if args.dump_outputs and world > 1:
        raise SystemExit("--dump-outputs writes one process's outputs: run it on one GPU")
    torch.cuda.set_device(local_rank)
    dev = f"cuda:{local_rank}"
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device(dev))
    if rank == 0 or args.workload == "hier20m4k":        # the 4K workload is generated on every rank's own GPU
        arrays, cams = build_workload(args.workload, device=dev)
    if world > 1:
        dist.barrier()
    if rank != 0 and args.workload != "hier20m4k":
        arrays, cams = build_workload(args.workload)

    from h3dgs import _lib, pipeline, synth
    from h3dgs import dist as hdist
    from diff_gaussian_rasterization import _C as rc
    scene = pipeline.Scene(arrays, device=dev)
    dcams = [pipeline.DeviceCamera(c, device=dev) for c in cams]
    thr = [synth.tau_threshold(TAU, c) for c in cams]
    bg = torch.zeros(3, device=dev)
    g = torch.Generator(device="cpu").manual_seed(5)
    gts_host = [torch.rand((3, H, W), generator=g).pin_memory() for _ in range(N_VIEWS)]
    gts_dev = [t.to(dev) for t in gts_host]
    sharder = hdist.TileSharder(world, rank, dev) if world > 1 else None
    copy_stream = torch.cuda.Stream(device=dev)
    host_cams = [(torch.tensor(c.world_view_transform).pin_memory(), torch.tensor(c.full_proj_transform).pin_memory(),
                  torch.tensor(c.camera_center).pin_memory()) for c in cams]
    thr_host = [torch.tensor([t], dtype=torch.float32).pin_memory() for t in thr]

    gs = None
    if mode == "graph":
        from h3dgs.graphstep import GraphedStep
        c0 = cams[0]
        use_peer, peer_note = world in (2, 4, 8) and not args.no_peer, ""
        if use_peer:
            from h3dgs import peer as hpeer
            use_peer, peer_note = hpeer.probe(world, rank, dev)           # same answer on every rank
            if not use_peer:
                config["peer_probe"] = (f"peer memory unavailable on this box ({peer_note}): " +
                                        ("call-by-call NCCL form of the sharded step" if auto_mode else "graphed NCCL form of the sharded step"))
        if auto_mode and not use_peer:
            mode = "api"
            config["mode"] = "call by call through the drop-in packages, cut gather/lerp fused into K1/K9"
    if mode == "graph":
        config["collectives"] = ("fused into the kernels over NVLink peer memory (image: the L1 kernel forwards a rank's rendered tile rows to "
                                 "every rank with coalesced stores; gradients: a push of the partial [P,10] rows into the owners' staging areas, "
                                 "summed by the owner's chain-rule kernels) + 2 device-side barrier kernels per step" if use_peer else
                                 ("NCCL all-gather (image slabs) + reduce-scatter ([P,10] sums)" if world > 1 else "none"))
        mk = lambda **kw: GraphedStep(scene, W, H, c0.tanfovx, c0.tanfovy, bg, thr[0], world=world, rank=rank, peer=use_peer, **kw)
        # capacities: one eager sync-free pass over the views with generous sizes, then +15 % head room
        # (rows and entries) and the next power of two (longest tile list)
        probe = mk(bin_capacity=(1 << 23) if W <= 1920 else (1 << 27), sort_capacity=8192, capture=False)
        need = {"rows": 0, "D": 0, "longest_list": 0}
        for v in range(N_VIEWS):
            probe.set_threshold(thr[v])
            probe.step(dcams[v], gts_dev[v])
            st = probe.status()
            if st["overflow"]:
                raise SystemExit(f"--mode graph: view {v} does not fit the probe capacities: {st}")
            need = {k: max(need[k], st[k]) for k in need}
        if probe.arena is not None:
            probe.arena.close()
        del probe
        torch.cuda.empty_cache()
        rows_cap = min(int(need["rows"] * 1.15) + 1, scene.means3D.shape[0])
        if world > 1:       # the row blocks of the reduce-scatter must agree on every rank
            t = torch.tensor([rows_cap], device=dev); dist.all_reduce(t, op=dist.ReduceOp.MAX); rows_cap = int(t.item())
        sort_cap = 32
        while sort_cap < min(int(need["longest_list"] * 1.25), 8192):
            sort_cap *= 2
        gs = mk(row_capacity=rows_cap, bin_capacity=int(need["D"] * 1.15) + 1, sort_capacity=sort_cap, capture=False)
        gs.set_camera(dcams[0]); gs.gt.copy_(gts_dev[0])
        gs.capture()
        config["graph"] = {"row_capacity": rows_cap, "bin_capacity": gs.bin_capacity, "sort_capacity": sort_cap,
                           "library_launches_per_step": int(gs.launches_per_step)}

    def step_graph(i, resident=True):
        v = i % N_VIEWS
        ready = gs.upload_target(gts_dev[v] if resident else gts_host[v], copy_stream)
        gs.threshold_dev.copy_(thr_host[v], non_blocking=True)      # this view's LOD threshold: a device scalar the graph reads
        if resident:
            gs.set_camera(dcams[v])
        else:
            gs.view.copy_(host_cams[v][0].reshape(16), non_blocking=True)
            gs.proj.copy_(host_cams[v][1].reshape(16), non_blocking=True)
            gs.campos.copy_(host_cams[v][2], non_blocking=True)
        gs.step(gt_ready=ready)
        return gs.status_dev[0], gs.radii, -1

    def step_api(i, resident=True, fused=True):
        v = i % N_VIEWS
        ready = None
        if resident:
            cam, gt = dcams[v], gts_dev[v]
        else:       # e2e: this step's camera and target come from pinned host memory
            cam = pipeline.DeviceCamera.__new__(pipeline.DeviceCamera)
            c = cams[v]
            cam.W, cam.H, cam.tanfovx, cam.tanfovy = c.W, c.H, c.tanfovx, c.tanfovy
            cam.viewmatrix = host_cams[v][0].to(dev, non_blocking=True)
            cam.projmatrix = host_cams[v][1].to(dev, non_blocking=True)
            cam.campos = host_cams[v][2].to(dev, non_blocking=True)
            cam.campos_cpu = host_cams[v][2]
            # the 25 MB target is only needed at the loss: upload it on a copy stream, overlapped with
            # this step's LOD cut and forward pass
            with torch.cuda.stream(copy_stream):
                gt = gts_host[v].to(dev, non_blocking=True)
                ready = torch.cuda.Event(); ready.record(copy_stream)
            gt.record_stream(torch.cuda.current_stream())
        if sharder is None:
            return pipeline.l1_step(scene, cam, bg, gt, thr[v] if hier else None, gt_ready=ready, fused=fused)
        return sharder.l1_step(scene, cam, bg, gt, thr[v] if hier else None, gt_ready=ready)

    step = step_graph if gs is not None else step_api
    read_stream = torch.cuda.Stream(device=dev)
    loss_pinned = torch.zeros(2, dtype=torch.float64).pin_memory()

    def timed(fn, nsteps, resident, collect=None, graph_mode=False):
        """W/K contract: barrier + synchronize on both sides, CUDA events on the launching stream, max over ranks."""
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        # e2e: the D2H read of every step's result happens one step behind, on a side stream into pinned memory --
        # the host looks at loss i-1 while the device works on step i (what a training loop's logging does), so the
        # read never drains the launch queue; all of it, including the last read, is inside the timed region
        main_s, prev_done = torch.cuda.current_stream(), None
        for i in range(nsteps):
            if prev_done is not None and graph_mode:
                main_s.wait_event(prev_done)         # graph mode: the static result buffer is not overwritten before it was read
            loss, radii, n = fn(i, resident)
            if not resident:
                ev = torch.cuda.Event(); ev.record(main_s)
                with torch.cuda.stream(read_stream):
                    read_stream.wait_event(ev)
                    loss.record_stream(read_stream)
                    loss_pinned[i % 2].copy_(loss.detach(), non_blocking=True)
                    done = torch.cuda.Event(); done.record(read_stream)
                if prev_done is not None:
                    prev_done.synchronize()
                    _ = float(loss_pinned[(i - 1) % 2])
                prev_done = done
            if collect is not None:
                collect.append(n)            # ints only: holding tensors here would defeat the caching allocator
        if prev_done is not None:
            prev_done.synchronize()
            _ = float(loss_pinned[(nsteps - 1) % 2])
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dist.barrier()
            ms = float(t.item())
        return ms

    # the clock sampler (nvidia-smi) starts BEFORE the warm-up: its NVML start-up stalls the GPU for
    # milliseconds and must not land inside the timed region
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        time.sleep(1.0)
    # set-up (untimed, not counted as warm-up): one pass over the views so that the caching allocator
    # has seen every buffer size (the cut size differs per view; a first-time size means a cudaMalloc)
    _lib.profile_enable(False)
    for i in range(N_VIEWS):
        step(i, False)
        step(i, True)
    for i in range(args.warmup):
        step(i, True)
    torch.cuda.synchronize()
    l0 = _lib.launch_count()
    stats = []
    headline, last = step, []
    if args.dump_outputs:
        def headline(i, resident):
            last[:] = [step(i, resident)]
            return last[0]
    ms_total = timed(headline, args.steps, True, stats, graph_mode=gs is not None)     # <- `value`: profiler off
    launches = _lib.launch_count() - l0
    if args.dump_outputs:
        loss, radii, _ = last[0]
        if gs is not None:
            rows = int(gs.status_dev[1].item())
            outs = {"loss": loss, "image": gs.image, "radii": radii[:rows]}
            outs.update({"grad_" + k: v for k, v in gs.grads.items()})
        else:
            outs = {"loss": loss, "radii": radii}
            outs.update({"grad_" + k: getattr(scene, k).grad for k in ("means3D", "shs", "opacities", "scales", "rotations")})
        dump_outputs(args.dump_outputs, outs)
    ms_e2e = timed(step, args.steps, False, graph_mode=gs is not None)
    clocks = sampler.stop() if rank == 0 else None
    if gs is not None:
        launches = gs.launches_per_step * args.steps            # replays bypass the library's launch counter

    # ---- the other host forms of the same step (untimed for the headline; each with its own warm-up) ----
    extras = {}
    if not args.no_extras and hier:
        if gs is not None:
            for i in range(N_VIEWS + 3):
                step_api(i, True)
            ms = timed(step_api, args.steps, True)
            extras["value_api"] = {"value": 1000.0 * args.steps / ms, "ms_per_step": ms / args.steps,
                                   "what": "call by call through the drop-in packages, fused cut gather/lerp (render_indices), "
                                           "two host synchronisations per step (expand_to_size returns an int; num_rendered)"}
        if world == 1:
            fn = lambda i, resident: step_api(i, resident, fused=False)
            k = max(3, min(args.steps, 10))
            for i in range(N_VIEWS + 2):
                fn(i, True)
            ms = timed(fn, k, True)
            extras["value_dropin"] = {"value": 1000.0 * k / ms, "ms_per_step": ms / k, "steps": k,
                                      "what": "the reference's render_post flow on the packages: PyTorch gather / parent lerp "
                                              "(~25 kernels, full-size temporaries, index_add backward) around the rasterizer -- "
                                              "what train_post.py:119-129 sees without opting in to anything"}
            scene.zero_grad()
            torch.cuda.empty_cache()

    # ---- bookkeeping + per-stage device times: a separate, profiled pass over the views ----
    Vs, Ds, Ps, NCs = [], [], [], []
    _lib.profile_reset(); _lib.profile_enable(True)
    if gs is None:
        for i in range(N_VIEWS):
            loss, radii, n = step(i, True)
            Ps.append(int(n)); Vs.append(int((radii > 0).sum().item())); Ds.append(rc.last_num_rendered())
    else:
        # graph replays bypass the library's stage events: the same sync-free step, run eagerly once per view
        graphs, gs.graph_a, gs.graph_b = (gs.graph_a, gs.graph_b), None, None
        for i in range(N_VIEWS):
            step(i, True)
            st = gs.status()
            if st["overflow"]:
                raise SystemExit(f"--mode graph: view {i} overflowed the capacities {config['graph']}: {st}; timed result invalid")
            Ps.append(st["rows"]); Ds.append(st["D"]); Vs.append(int((gs.radii > 0).sum().item()))
            NCs.append(int(gs.n_contrib_view().long().sum().item()))
        gs.graph_a, gs.graph_b = graphs
    prof = _lib.profile_read(); _lib.profile_enable(False)
    Pm, Vm, Dm = float(np.mean(Ps)), float(np.mean(Vs)), float(np.mean(Ds))
    stage_ms = {k: (v[0] / max(v[1], 1)) for k, v in prof.items() if v[1] > 0}

    # ---- N > 1: the sharded step equals the single-GPU step (gradients to fp32 sum order, same loss), and what the two
    # collectives cost on their own ----
    nrank = None
    if world > 1 and not args.no_extras and args.workload != "hier20m4k":
        v = 0
        loss1, radii1, n1 = pipeline.l1_step(scene, dcams[v], bg, gts_dev[v], thr[v] if hier else None)
        g1 = [p.grad.clone() for p in scene.params()]
        if gs is not None:
            step_graph(v, True)
            st = gs.status()
            g2 = [gs.grads[k].clone() for k in ("means3D", "scales", "rotations", "opacities", "shs")]
            same = st["rows"] == n1            # image equality of the graphed step: tests/test_gpu_dist.py
            loss2 = st["loss"]
        else:
            loss2t, radii2, n2 = sharder.l1_step(scene, dcams[v], bg, gts_dev[v], thr[v] if hier else None)
            g2 = [p.grad.clone() for p in scene.params()]
            loss2, same = float(loss2t.item()), bool(torch.equal(radii1, radii2))
        for t_ in g2:
            dist.all_reduce(t_, op=dist.ReduceOp.SUM)           # sharded by rendered row: the sum is the full gradient
        errs = [float((a - b.reshape(a.shape)).abs().max() / a.abs().max().clamp_min(1e-30)) for a, b in zip(g1, g2)]
        ok = torch.tensor([1.0 if (max(errs) < 1e-5 and abs(float(loss1.item()) - loss2) < 1e-6 and same) else 0.0], device=dev)
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        # collectives alone (same buffers / sizes as the step), CUDA events, max over ranks
        rpr = hdist.rows_per_rank(H, world)
        slab = torch.zeros((rpr, 3, 16, W), device=dev); slabs = torch.zeros((world * rpr, 3, 16, W), device=dev)
        acc = hdist.accum_scratch(int(max(Ps)), world, dev)
        comm = {}
        for name, fn in (("all_gather_image", lambda: dist.all_gather_into_tensor(slabs, slab)),
                         ("reduce_scatter_accum", lambda: hdist.reduce_accum(acc, int(max(Ps)), world, rank))):
            for _ in range(5):
                fn()
            dist.barrier(); torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(20):
                fn()
            e1.record(); torch.cuda.synchronize()
            t = torch.tensor([e0.elapsed_time(e1) / 20], device=dev); dist.all_reduce(t, op=dist.ReduceOp.MAX)
            comm[name] = round(float(t.item()), 4)
        if gs is not None and gs.peer:
            for _ in range(5):
                gs.arena.barrier()
            dist.barrier(); torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(50):
                gs.arena.barrier()
            e1.record(); torch.cuda.synchronize()
            t = torch.tensor([e0.elapsed_time(e1) / 50], device=dev); dist.all_reduce(t, op=dist.ReduceOp.MAX)
            comm = {"peer_barrier_kernel": round(float(t.item()), 4), "barrier_timed_out": gs.arena.timed_out(),
                    "nccl_for_comparison": comm}
        nrank = {"equals_single_gpu": bool(ok.item() == 1.0), "grad_rel_err_max": max(errs), "comm_ms": comm,
                 "comm_bytes": {"all_gather_image": int(slabs.numel() * 4), "reduce_scatter_accum": int(acc.numel())}}

    if rank == 0:
        ms_step = ms_total / args.steps
        value = 1000.0 / ms_step
        N_nodes = int(scene.nodes.shape[0]) if hier else 0
        out = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
               "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong",
               "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config,
               "clocks": clocks, "gpu_launches": int(launches),
               "e2e": {"value": 1000.0 / (ms_e2e / args.steps), "unit": UNIT,
                       "h2d_bytes_per_step": 3 * H * W * 4 + 16 * 4 * 2 + 3 * 4 + (4 if gs is not None else 0),
                       "d2h_bytes_per_step": 8 if gs is not None else 4},
               "stage_ms": {k: round(v, 4) for k, v in stage_ms.items()},
               "stage_ms_note": "separate profiled pass (cudaEvents around every library launch); the timed regions run with the profiler off",
               "counts": {"P_cut": Pm, "V": Vm, "D_rank0": Dm, "N_all": int(scene.means3D.shape[0]),
                          "sum_n_contrib": float(np.mean(NCs)) if NCs else None}}
        out.update(extras)
        dev_ms = sum(v for k, v in stage_ms.items() if k not in ("preprocess_color", "sh_backward"))
        out["host_gap_ms"] = round(ms_step - dev_ms, 4)
        out["host_gap_note"] = ("step time minus the summed library-kernel times on the critical stream (preprocess_color and "
                                "sh_backward overlap on the side stream): loss kernels, memsets, collectives and any launch gaps")
        if nrank is not None:
            out["nrank_check"] = nrank
        try:
            import refprobe
            out["reference_cuda"] = refprobe.probe()
        except Exception as e:        # pragma: no cover
            out["reference_cuda"] = {"available": False, "note": f"probe failed: {e}"}
        # roofline of the dominant kernel
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s"
        ncu = {}
        try:   # per-kernel figures of the committed `ncu --set full` capture (per launch)
            ncu = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
            if ncu.get("workload") != args.workload or world != 1:
                ncu = {}
        except Exception:
            pass
        if stage_ms and Dm:
            dom = max((k for k in stage_ms if k not in ("lod_cut", "lod_weights")), key=lambda k: stage_ms[k])
            # Dm is THIS rank's num_rendered: with tile sharding every rank bins ~D/world entries
            ab = alg_bytes(Pm, Vm, Dm, hier, N_nodes, fused=True)
            achieved = ab[dom] / (stage_ms[dom] * 1e-3) / 1e9
            kn = ncu.get("kernels", {}).get(dom, {})
            out["roofline"] = {"bound": "hbm", "kernel": dom, "achieved": achieved, "peak": peak, "unit": "GB/s",
                               "frac": achieved / peak, "traffic": kn.get("dram_bytes"), "peak_source": peak_src,
                               "alg_bytes_per_launch": ab[dom], "kernel_ms": stage_ms[dom],
                               "note": "the blend kernels are FP32-issue-bound, not HBM-bound (SURVEY.md 8d): see roofline_fp32"}
            # every HBM-stream stage against the same peak
            out["stage_hbm_frac"] = {k: round(ab[k] / (stage_ms[k] * 1e-3) / 1e9 / peak, 4) for k in stage_ms
                                     if k in ab and ab[k] and k not in ("render_forward", "render_backward")}
            if kn:
                out["roofline_fp32"] = {k: kn.get(k) for k in ("issue_slot_util", "ipc", "fma_pipe_pct", "alu_pipe_pct", "xu_pipe_pct",
                                                               "warp_inst", "lanes_per_inst", "source") if k in kn}
                out["roofline_fp32"]["kernel"] = dom
                out["roofline_fp32"]["note"] = ("from the committed ncu capture of this kernel (profiles/): issue_slot_util = warp "
                                                "instructions / (SMs x 4 schedulers x cycles); useful-lane fraction: DESIGN.md 3.1")
            ab = alg_bytes(Pm, Vm, Dm * world, hier, N_nodes, fused=True)       # whole frame
            out["step_roofline"] = {"alg_bytes_per_image": ab["total"], "achieved_gbs": ab["total"] / (ms_step * 1e-3) / 1e9,
                                    "frac_of_hbm_peak": ab["total"] / (ms_step * 1e-3) / 1e9 / peak,
                                    "alg_bytes_with_8d_addons": ab["total_with_addons"], "addons": ab["addons"],
                                    "frac_of_hbm_peak_with_addons": ab["total_with_addons"] / (ms_step * 1e-3) / 1e9 / peak}
        if world == 1 and args.classic:
            out["classic_blend"] = time_classic(scene, dcams[0], bg, thr[0] if hier else None, hier, stage_ms)
        if world == 1 and not args.no_cpu_baseline:
            r = run_cpu_arm(arrays, cams, 3, 1, budget_s=25.0)
            whole = r["frac"] == 1
            out["cpu_baseline"] = {"value": r["value"], "unit": UNIT, "cores": r["cores"], "kind": "port",
                                   "sample": (f"{r['steps_run']} whole frame(s) of this workload at {W}x{H}, {r['ms_per_step']:.0f} ms each, "
                                              "no extrapolation" if whole else
                                              f"every {r['frac']}th Gaussian of the cut at {W}x{H}, {r['steps_run']} step(s), "
                                              f"{r['ms_per_step']:.0f} ms each, images/s extrapolated linearly (x1/{r['frac']})")
                                             + "; oracle/oracle.c, OpenMP"}
            try:
                out["cpu_baseline_pytorch"] = run_pytorch_config1()
            except Exception as e:    # pragma: no cover
                out["cpu_baseline_pytorch"] = {"unavailable": str(e)}
        print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
