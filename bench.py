#!/usr/bin/env python
"""bench.py -- frames/sec (fwd+bwd) of the mesh-Gaussian hot path at 1080p / 1M mesh-Gaussians (BASELINE.json).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path (one process per GPU under torchrun)
    python bench.py --impl reference --gpus N --steps K ...  # the reference algorithm on the host cores (CPU oracle port)

A "step" is one training frame of gs_mesh (train.py:89-157 of the reference): fused mesh->Gaussian expansion,
rasterizer forward, L1+SSIM loss, full backward down to vertices/_alpha/_scale/features/opacity, gradient exchange
(N>1) and the Adam step.  Default workload = BASELINE config 3: synthetic closed object, F=200,000 faces x K=5 =
1,000,000 mesh-Gaussians, 1920x1080, SH degree 3, 16 cameras on two rings.  `--workload` selects the other BASELINE
configs (1: gs_flat_10k_256, 2: gs_mesh_100k_800, 4: gs_multi_mesh_2M_1080p, 5: gs_mesh_500k_1080p [--mode render_animated]).
Prints ONE JSON line (rank 0).
"""
import argparse
import json
import math
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "gaussian-mesh-splatting_b200"), os.path.join(ROOT, "tests"), os.path.join(ROOT, "baseline", "refstyle")):
    if p not in sys.path:
        sys.path.insert(0, p)

TORCH_CPU_THREADS = 8
CPU_ARM_MAX_THREADS = 32      # the oracle's composite loops stop scaling beyond this; a FIXED count keeps the arm reproducible


def _host_threads() -> int:
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    return max(1, min(n, CPU_ARM_MAX_THREADS))


HOST_THREADS = _host_threads()      # read BEFORE an OpenMP runtime binds the main thread to one core (OMP_PROC_BIND)
os.environ.setdefault("OMP_WAIT_POLICY", "passive")
if ("reference" in sys.argv and "--impl" in sys.argv) or int(os.environ.get("WORLD_SIZE", "1")) == 1:
    # The CPU arm runs two OpenMP runtimes (the oracle's libgomp, PyTorch's own): one team at a time must own the cores.
    # Passive waiting keeps an idle team from spinning against the working one (round 1: 128 + 128 spinning threads made
    # the same frame take 3 s or 25 s); thread counts are FIXED (oracle <= 32, PyTorch <= 8: its elementwise expansion ops
    # are bandwidth-trivial and only lose to fork/join overhead beyond that).
    # (Set before libgomp is loaded; overrides torchrun's OMP_NUM_THREADS=1 default.)
    os.environ["OMP_NUM_THREADS"] = str(HOST_THREADS)
    os.environ["OMP_WAIT_POLICY"] = "passive"
    os.environ["OMP_DYNAMIC"] = "false"

# The driver expects ONE JSON line on stdout.  NCCL prints its version banner with printf to fd 1 (NCCL_DEBUG_FILE does
# not cover it): keep the real stdout aside for the result line and point fd 1 at stderr for everything else.
os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
sys.stdout.flush()
_RESULT_FD = os.dup(1)
os.dup2(2, 1)


def emit_result(line: dict) -> None:
    os.write(_RESULT_FD, (json.dumps(line) + "\n").encode())


import numpy as np  # noqa: E402
import torch  # noqa: E402

WORKLOADS = {
    # name: (faces, K, W, H, n_cameras)
    "gs_mesh_1M_1080p": (200_000, 5, 1920, 1080, 16),       # BASELINE configs[2] -- the headline
    "gs_mesh_100k_800": (33_334, 3, 800, 800, 8),           # BASELINE configs[1]
    "gs_mesh_500k_1080p": (100_000, 5, 1920, 1080, 16),     # BASELINE configs[4] sizes (training step; --mode render_animated = the sweep)
    "gs_multi_mesh_2M_1080p": (400_000, 5, 1920, 1080, 16), # BASELINE configs[3]: 4 meshes x 100k faces x K=5 (merged launch)
    "gs_flat_10k_256": (10_000, 1, 256, 256, 1),            # BASELINE configs[0]: 10k free flat Gaussians (no mesh), one camera
    "tiny": (2_000, 3, 320, 240, 4),                        # CI-sized
}
METRIC = {
    "gs_mesh_1M_1080p": "frames/sec (fwd+bwd) @1080p, 1M mesh-Gaussians",
    "gs_mesh_100k_800": "frames/sec (fwd+bwd) @800x800, 100k mesh-Gaussians (num_splats=3)",
    "gs_mesh_500k_1080p": "frames/sec (fwd+bwd) @1080p, 500k mesh-Gaussians",
    "gs_multi_mesh_2M_1080p": "frames/sec (fwd+bwd) @1080p, 4 meshes / 2M mesh-Gaussians",
    "gs_flat_10k_256": "frames/sec (fwd+bwd) @256x256, 10k flat Gaussians",
    "tiny": "frames/sec (fwd+bwd) @320x240, 6k mesh-Gaussians (CI)",
}
# CPU arm: compositing fwd+bwd runs on every CPU_TILE_STRIDE-th tile (FIXED per workload, so the work is identical run to
# run) and is extrapolated; everything per-Gaussian runs in full.
CPU_TILE_STRIDE = {"gs_mesh_1M_1080p": 8, "gs_multi_mesh_2M_1080p": 16, "gs_mesh_500k_1080p": 8, "gs_mesh_100k_800": 2}
ALGO_BYTES = {  # algorithmic bytes per unit, SURVEY.md section 8(d) / DESIGN.md "Roofline accounting"
    "composite_bwd": dict(N=84, px=24), "composite_fwd": dict(N=44, px=24),
    "preprocess_fwd": dict(P=311 + 8), "preprocess_bwd": dict(P=563 - 192 + 12),     # factored SH gradient: 12 B colour gradient instead of 192 B of rows
    "expand_fwd": dict(P=56, F=60), "expand_bwd": dict(P=56, F=36),
    "emit_dups": dict(P=16, N=6), "cub_sort_tiles": dict(N=12), "cub_sort_depth": dict(P=16), "tile_ranges": dict(N=2),     # 16-bit tile keys + 32-bit Gaussian ids
    "cub_scan_tiles": dict(P=12), "ssim_stats": dict(px=3 * (8 + 12)), "ssim_grad": dict(px=3 * (12 + 8 + 4)),
    "adam": dict(P=5 * 28 + 48 * 24 + 12 + 12),   # 5 non-SH parameters/Gaussian at 28 B (p, g, m, v read; p, m, v written) + 48 SH parameters at
                                                  # 24 B (no gradient read: rebuilt from 12 B of colour gradient per rank and the 12 B centre)
}


def base_config(workload):
    """The keys BOTH arms print under `config` (identical, so the driver's same_config check holds)."""
    F, K, W, H, ncam = WORKLOADS[workload]
    return {"workload": workload, "P": F * K if workload != "gs_flat_10k_256" else F, "faces": F if workload != "gs_flat_10k_256" else 0,
            "K": K, "width": W, "height": H, "sh_degree": 3, "cameras": ncam}


def build_scene(name, seed=0):
    from gms_b200 import scenes
    F, K, W, H, ncam = WORKLOADS[name]
    if name.startswith("gs_multi_mesh"):
        # 4 disjoint objects, concatenated exactly as gaussian_multi_mesh_model.py:99-119 does (same K => merged once)
        vs, fs, off = [], [], 0
        for k, c in enumerate([(-0.75, -0.75, 0.0), (0.75, -0.75, 0.0), (-0.75, 0.75, 0.0), (0.75, 0.75, 0.0)]):
            v, f = scenes.object_mesh(F // 4)
            vs.append(v * 0.55 + np.float32(c)); fs.append(f + off); off += v.shape[0]
        verts, faces = np.concatenate(vs), np.concatenate(fs)
    else:
        verts, faces = scenes.object_mesh(F)
    params = scenes.init_mesh_gaussians(verts, faces, K, seed=seed, trained_like=True)
    cams = scenes.ring_cameras(ncam // 2, 3.4, W, H, elevation_deg=15.0) + \
        scenes.ring_cameras(ncam - ncam // 2, 4.4, W, H, elevation_deg=38.0, phase=0.3)
    return params, cams, (faces.shape[0], K, W, H)


def flat_scene(seed=0):
    """BASELINE config 1 (SURVEY.md 8d): 10k free flat Gaussians, 256x256, one camera at radius 4.03 looking at the origin."""
    from gms_b200 import scenes
    P, _, W, H, _ = WORKLOADS["gs_flat_10k_256"]
    g = scenes.flat_gaussians(P, seed=seed)
    cam = scenes.look_at_camera((4.03 * math.cos(0.5), 4.03 * math.sin(0.5), 1.2), (0, 0, 0), W, H)
    return g, cam


DUMP_MAX_ROWS = 65536            # larger outputs are dumped as a fixed, seeded sample of their rows
DUMP_MAX_BYTES = 64 << 20


def dump_outputs(out_dir, arrays):
    """--dump-outputs: write each output of the last timed step as <out_dir>/<name>.npy (float32, or float64 for float64
    tensors), so that two builds run with the same arguments can be compared array by array.  An array with more than
    DUMP_MAX_ROWS rows is reduced to the same rows every run: a sorted sample drawn with a fixed seed from its row count."""
    os.makedirs(out_dir, exist_ok=True)
    total = 0
    for name, t in arrays.items():
        a = t.detach().cpu().numpy() if isinstance(t, torch.Tensor) else np.asarray(t)
        a = a.astype(np.float64 if a.dtype == np.float64 else np.float32).reshape(a.shape or (1,))
        if a.shape[0] > DUMP_MAX_ROWS:
            a = a[np.sort(np.random.RandomState(0).choice(a.shape[0], DUMP_MAX_ROWS, replace=False))]
        total += a.nbytes
        assert total <= DUMP_MAX_BYTES, f"--dump-outputs: more than {DUMP_MAX_BYTES} bytes"
        np.save(os.path.join(out_dir, f"{name}.npy"), np.ascontiguousarray(a))


class ClockSampler(threading.Thread):
    """SM clock and throttle reasons DURING the timed region (B200_PROFILING.md 'clocks line'), sampled through NVML
    every 50 ms from a side thread (same counters nvidia-smi prints; no subprocess start-up hiccup inside the timing)."""

    def __init__(self, gpu_index=0, period_s=0.05):
        super().__init__(daemon=True)
        self.gpu_index, self.period, self.rows, self._stop_evt = gpu_index, period_s, [], threading.Event()
        self.active = False     # only samples taken while `active` count
        self.err = None

    def run(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            phys = self.gpu_index
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            if vis:
                try:
                    phys = int(vis.split(",")[self.gpu_index])
                except Exception:
                    pass
            h = nv.nvmlDeviceGetHandleByIndex(phys)
            mx = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
            R = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40}
            while not self._stop_evt.is_set():
                if self.active:
                    sm = nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)
                    try:
                        bits = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
                    except Exception:
                        bits = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                    self.rows.append((sm, mx, [k for k, b in R.items() if bits & b]))
                time.sleep(self.period)
        except Exception as e:  # pragma: no cover
            self.err = repr(e)

    def stop(self):
        self._stop_evt.set()

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable: " + str(self.err)]}
        sm = [r[0] for r in self.rows]
        reasons = sorted({x for r in self.rows for x in r[2]})
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(self.rows[0][1]), "reasons": reasons, "samples": len(sm)}


def measured_peak_gbs():
    try:
        d = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, STREAM-style copy)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_traffic_bytes(workload, kernel):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed `ncu --set full` capture of the SHIPPED
    kernel (profiles/ncu_traffic.json names the capture each figure was read from); None when there is no capture."""
    try:
        d = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
        e = d.get(workload, {}).get(kernel)
        return (float(e["dram_bytes_read"]) + float(e["dram_bytes_write"])) if e else None
    except Exception:
        return None


# ----------------------------------------------------------------------------------------------- CPU arm / baseline
def cpu_reference_frame(params, cam, dims, stride, threads):
    """One fwd+bwd frame of the SAME workload with the CPU oracle: expansion (PyTorch CPU + autograd), preprocess, binning
    and preprocess-backward on all P Gaussians, compositing fwd+bwd on every `stride`-th tile (extrapolated x stride;
    stride is a per-workload constant).  Returns (estimated seconds per full frame, description, threads)."""
    from oracle import expansion as oexp
    from oracle import raster
    from helpers import settings_from_camera
    F, K, W, H = dims
    raster.set_num_threads(threads)
    torch.set_num_threads(min(threads, TORCH_CPU_THREADS))
    S = settings_from_camera(cam, bg=(1, 1, 1))
    t0 = time.perf_counter()
    tv, ta, ts = (x.clone().requires_grad_(True) for x in (params.vertices, params._alpha, params._scale))
    xyz, sl, rr, _, _ = oexp.expand(tv, params.faces, ta, ts)
    sc, rot, op, fe = oexp.activate(sl, rr, params._opacity, params._features_dc, params._features_rest)
    t_exp_f = time.perf_counter() - t0
    t0 = time.perf_counter()
    st = raster.preprocess(S, xyz, op, shs=fe.contiguous(), scales=sc, rotations=rot)
    raster.bin_tiles(st)
    t_pre = time.perf_counter() - t0
    T = st.ranges.shape[0]
    raster.set_tile_stride(stride)
    rs = np.random.RandomState(0)
    dC = (rs.randn(3, H, W) / (W * H)).astype(np.float32)
    t0 = time.perf_counter(); raster.composite(st); t_cf = time.perf_counter() - t0
    t0 = time.perf_counter(); g = raster.composite_backward(st, dC, None); t_cb = time.perf_counter() - t0
    raster.set_tile_stride(1)
    t0 = time.perf_counter(); out = raster.preprocess_backward(st, g); t_pb = time.perf_counter() - t0
    t0 = time.perf_counter()
    torch.autograd.backward([xyz, sc, rot], [torch.tensor(out["dL_dmeans3D"]), torch.tensor(out["dL_dscales"]),
                                              torch.tensor(out["dL_drotations"])])
    t_exp_b = time.perf_counter() - t0
    frame_s = t_exp_f + t_pre + (t_cf + t_cb) * stride + t_pb + t_exp_b
    desc = (f"1 frame of the same workload (P={F * K}, {W}x{H}, N={st.N}), {threads} threads: expansion+preprocess+binning+"
            f"preprocess-bwd on all Gaussians, compositing fwd+bwd on every {stride}-th of {T} tiles (fixed stride), "
            f"extrapolated x{stride}; measured {t_exp_f + t_pre + t_cf + t_cb + t_pb + t_exp_b:.1f}s")
    return frame_s, desc, threads


def cpu_reference_flat(g, cam, threads):
    from oracle import raster
    from helpers import settings_from_camera
    raster.set_num_threads(threads); torch.set_num_threads(min(threads, TORCH_CPU_THREADS))
    S = settings_from_camera(cam, bg=(1, 1, 1))
    rs = np.random.RandomState(0)
    dC = (rs.randn(3, cam.image_height, cam.image_width) / (cam.image_width * cam.image_height)).astype(np.float32)
    t0 = time.perf_counter()
    st = raster.forward(S, g["means3D"], g["opacities"], shs=g["shs"], scales=g["scales"], rotations=g["rotations"])
    raster.backward(st, dC)
    dt = time.perf_counter() - t0
    return dt, f"full rasterizer fwd+bwd of the workload (P={g['means3D'].shape[0]}, N={st.N}), every tile, {threads} threads", threads


def run_reference_arm(args):
    """--impl reference: the reference's algorithm on the host cores (oracle port; the stock CUDA extension is an
    empty un-vendored submodule and cannot be installed)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = HOST_THREADS
    stride = CPU_TILE_STRIDE.get(args.workload, 1)
    times = []
    if args.workload == "gs_flat_10k_256":
        g, cam = flat_scene()
        for s in range(args.warmup + args.steps):
            fs, desc, cores = cpu_reference_flat(g, cam, threads)
            if s >= args.warmup:
                times.append(fs)
    else:
        params, cams, dims = build_scene(args.workload)
        for s in range(args.warmup + args.steps):
            fs, desc, cores = cpu_reference_frame(params, cams[s % len(cams)], dims, stride, threads)
            if s >= args.warmup:
                times.append(fs)
    sec = float(np.mean(times))
    line = {"impl": "reference", "metric": METRIC[args.workload], "value": 1.0 / sec,
            "unit": "frames/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": sec * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": base_config(args.workload),
            "cpu_baseline": {"value": 1.0 / sec, "unit": "frames/s", "cores": cores, "kind": "port", "sample": desc,
                             "tile_stride": stride, "threads": threads,
                             "per_step_s": {"min": float(np.min(times)), "max": float(np.max(times))}},
            "e2e": {"value": 1.0 / sec, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0,
            "note": "reference arm = CPU oracle port of the reference algorithm (stock diff-gaussian-rasterization source is "
                    "absent from the reference checkout: empty submodule); the GPU stand-in comparators are in the product "
                    "arm's `comparators` object"}
    emit_result(line)


# ----------------------------------------------------------------------------------------------- animated render
def run_render_animated(args, params, cams, dims, dev, world, rank, local):
    """scripts/render_time_animated.py:68-87: per frame t, new_vertices = transform_hotdog_fly(v, t), re-expansion from the
    moved vertices (gaussian_animated_renderer:61-73) and a rasterizer forward, under no_grad.  n_frames = 800,
    t = linspace(0, 10*pi) (:74), contiguous frame ranges per rank, no collective.  --save-images adds the image sink
    (the reference writes a PNG per frame, :86-87) inside the timed region."""
    import torch.distributed as dist
    from gms_b200 import _lib, rasterizer, scenes
    from gms_b200.model import MeshGaussianModel
    from gms_b200.trainer import render_frame
    F, K, W, H = dims
    model = MeshGaussianModel.from_params(params, dev, packed_features=True)
    bg = torch.ones(3, device=dev)
    cams_dev = [c.to(dev) for c in cams]
    n_frames = 800
    ts = torch.linspace(0, 10 * math.pi, n_frames)
    per = n_frames // world
    lo = rank * per
    v0 = model.vertices.detach().clone()
    sink = None
    if args.save_images:
        from gms_b200 import io_image
        os.makedirs(args.save_images, exist_ok=True)
        sink = io_image.ImageSink(H, W, fmt=args.image_format, device=dev,
                                  raw_path=os.path.join(args.save_images, f"rank{rank}.rgb") if args.image_format == "raw" else None)

    def frame(i):
        with torch.no_grad():
            model.vertices.data.copy_(scenes.transform_hotdog_fly(v0, float(ts[lo + (i % per)])))
            img = render_frame(model, cams_dev[i % len(cams_dev)], bg)[0]
            if sink is not None:
                sink.write(img, os.path.join(args.save_images, f"{lo + (i % per):05d}.{args.image_format}"))
            return img

    K_, W_ = args.steps, max(args.warmup, 3)
    for i in range(max(W_, 2 * len(cams_dev))):
        frame(i)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    _lib.launch_count(reset=True)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_wall = time.perf_counter()
    e0.record()
    for i in range(K_):
        img = frame(W_ + i)
    e1.record()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    if sink is not None:
        sink.close()
    t_wall = time.perf_counter() - t_wall
    ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    launches = _lib.launch_count(reset=True)
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, {"image": img})
    if rank == 0:
        ms_step = float(ms.item()) / K_
        cfg = base_config(args.workload)
        cfg.update({"mode": "render_animated", "n_frames": n_frames})
        emit_result({"metric": "frames/sec (forward only, animated-vertex sweep) @1080p", "value": world * 1000.0 / ms_step,
                     "unit": "frames/s", "n_gpus": world, "steps": K_, "warmup": W_, "ms_per_step": ms_step,
                     "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                     "config": cfg, "details": {"N_last": rasterizer.last_num_rendered,
                                                "image_sink": None if sink is None else {"format": args.image_format, "frames": sink.frames,
                                                                                        "wall_frames_per_s_incl_files": world * K_ / t_wall}},
                     "gpu_launches": int(launches)})
    if world > 1:
        dist.destroy_process_group()


# ----------------------------------------------------------------------------------------------- config 1 on the GPU
def run_flat(args, dev):
    """BASELINE config 1 on the product path: rasterizer forward + fused loss + backward of 10k free flat Gaussians."""
    import diff_gaussian_rasterization as dgr
    from gms_b200 import _lib, losses
    from helpers import settings_from_camera
    from gpu_helpers import gpu_settings
    g, cam = flat_scene()
    S = settings_from_camera(cam, bg=(1, 1, 1))
    rs = gpu_settings(S, dev)
    t = {k: v.to(dev).float().contiguous().requires_grad_(True) for k, v in g.items()}
    gt_in = flat_scene(seed=123)[0]
    with torch.no_grad():
        r = dgr.GaussianRasterizer(raster_settings=rs)
        gt = r(means3D=gt_in["means3D"].to(dev), means2D=torch.zeros(10000, 3, device=dev), opacities=gt_in["opacities"].to(dev),
               shs=gt_in["shs"].to(dev), scales=gt_in["scales"].to(dev), rotations=gt_in["rotations"].to(dev))[0].clamp(0, 1).contiguous()
    P = t["means3D"].shape[0]

    def step(_):
        for v in t.values():
            v.grad = None
        m2d = torch.zeros(P, 3, device=dev, requires_grad=True)
        img = dgr.GaussianRasterizer(raster_settings=rs)(means3D=t["means3D"], means2D=m2d, opacities=t["opacities"], shs=t["shs"],
                                                         scales=t["scales"], rotations=t["rotations"])[0]
        loss = losses.fused_training_loss(img, gt, 0.2)
        loss.backward()
        return loss

    K_, W_ = args.steps, max(args.warmup, 3)
    for s in range(W_):
        step(s)
    torch.cuda.synchronize()
    _lib.launch_count(reset=True)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for s in range(K_):
        loss = step(s)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / K_
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, dict(loss=loss, **{f"grad_{k}": v.grad for k, v in t.items()}))
    line = {"metric": METRIC[args.workload], "value": 1000.0 / ms, "unit": "frames/s", "n_gpus": 1, "steps": K_, "warmup": W_,
            "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": base_config(args.workload), "gpu_launches": int(_lib.launch_count(reset=True)),
            "details": {"path": "diff_gaussian_rasterization shim (autograd) + fused L1+SSIM; no mesh, no optimizer",
                        "l2": "working set fits in L2 (BASELINE config 1 is the reference's CPU-runnable case, not a bandwidth test)"}}
    if not args.no_cpu_baseline:
        fs, desc, cores = cpu_reference_flat(g, cam, HOST_THREADS)
        line["cpu_baseline"] = {"value": 1.0 / fs, "unit": "frames/s", "cores": cores, "kind": "port", "sample": desc}
    emit_result(line)


# ----------------------------------------------------------------------------------------------- GPU comparators
def run_comparators(model, cams_dev, gts, bg, dims, dev, n_frames=12):
    """SURVEY.md 8(d) 'how the reference's paths are timed beside it', on the same GPU, same process, same tensors:
    (1) rasterizer-only (R2-R9) fwd+bwd: product vs the ref-style stand-in (baseline/refstyle: Appendix A with the stock
        work decomposition -- NOT the stock binary, whose source is absent);
    (2) the image sink vs torchvision.utils.save_image."""
    out = {"label": "ref-style = labelled stand-in for the absent stock diff-gaussian-rasterization (SURVEY Appendix A, stock "
                    "decomposition: CTA/tile, thread/pixel, per-pixel atomics, 64-bit cub sort, host sync); not the stock binary"}
    F, K, W, H = dims

    def timeit(fn, n=n_frames, warm=3):
        for i in range(warm):
            fn(i)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(n):
            fn(warm + i)
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / n

    try:
        import diff_gaussian_rasterization as ours
        import refstyle
        with torch.no_grad():
            xyz, sc, rot = model.expand_fused(activated=True)
            op, shs = model.get_opacity.detach().clone(), model.get_features.detach().clone()
        leaves = [t.detach().clone().requires_grad_(True) for t in (xyz, sc, rot, op, shs)]
        gen = torch.Generator(device=dev).manual_seed(0)
        dC = torch.randn(3, H, W, device=dev, generator=gen) / (W * H)

        def raster_step(mod):
            def fn(i):
                cam = cams_dev[i % len(cams_dev)]
                rs = mod.GaussianRasterizationSettings(
                    image_height=H, image_width=W, tanfovx=cam.tanfovx, tanfovy=cam.tanfovy, bg=bg, scale_modifier=1.0,
                    viewmatrix=cam.world_view_transform, projmatrix=cam.full_proj_transform, sh_degree=3, campos=cam.camera_center,
                    prefiltered=False, debug=False, antialiasing=False)
                for t in leaves:
                    t.grad = None
                m2d = torch.zeros_like(leaves[0], requires_grad=True)
                img = mod.GaussianRasterizer(raster_settings=rs)(means3D=leaves[0], means2D=m2d, opacities=leaves[3], shs=leaves[4],
                                                                 scales=leaves[1], rotations=leaves[2])[0]
                img.backward(dC)
            return fn

        refstyle.GaussianRasterizationSettings = ours.GaussianRasterizationSettings
        ms_ours, ms_ref = timeit(raster_step(ours)), timeit(raster_step(refstyle))
        out["rasterizer_fwd_bwd_ms"] = {"ours": ms_ours, "refstyle": ms_ref, "through": "the diff_gaussian_rasterization autograd API, "
                                        f"{n_frames} frames cycling the cameras, CUDA events"}
        out["vs_refstyle"] = ms_ref / ms_ours
    except Exception as e:  # pragma: no cover
        out["rasterizer_error"] = repr(e)

    # (2) image sink vs torchvision.utils.save_image (scripts/render_time_animated.py:86-87), frames per second incl. the files
    try:
        import shutil
        import tempfile
        import torchvision.utils as tvu
        from gms_b200 import io_image
        frames = [g.clamp(0, 1) for g in gts[:8]]
        tmp = tempfile.mkdtemp(prefix="gms_sink_")
        res = {}
        t0 = time.perf_counter()
        for k in range(8):
            tvu.save_image(frames[k % len(frames)], os.path.join(tmp, f"ref_{k}.png"))
        torch.cuda.synchronize()
        res["torchvision_save_image_png_ms"] = (time.perf_counter() - t0) / 8 * 1e3
        for fmt in ("png", "ppm", "raw"):
            n = 48
            t0 = time.perf_counter()
            with io_image.ImageSink(H, W, fmt=fmt, device=dev, raw_path=os.path.join(tmp, "frames.rgb") if fmt == "raw" else None) as sink:
                for k in range(n):
                    sink.write(frames[k % len(frames)], os.path.join(tmp, f"ours_{k}.{fmt}"))
            res[f"image_sink_{fmt}_ms"] = (time.perf_counter() - t0) / n * 1e3
        shutil.rmtree(tmp, ignore_errors=True)
        res["what"] = "host wall-clock per 1080p frame incl. the file write (tmp dir); the sink overlaps it with rendering, save_image blocks the loop"
        out["image_sink"] = res
    except Exception as e:  # pragma: no cover
        out["image_sink_error"] = repr(e)
    return out


# ----------------------------------------------------------------------------------------------- GPU arm
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="gs_mesh_1M_1080p", choices=sorted(WORKLOADS))
    ap.add_argument("--no-optimizer", action="store_true", help="exclude the Adam step from the step")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-comparators", action="store_true", help="skip the GPU comparators (ref-style rasterizer, reference PyTorch expansion)")
    ap.add_argument("--mode", default="train", choices=["train", "render_animated"],
                    help="train: fwd+bwd step (headline). render_animated: scripts/render_time_animated.py path, forward only, "
                         "vertex animation + re-expansion every frame (BASELINE configs[4])")
    ap.add_argument("--save-images", default=None, help="render_animated: write every frame through the GPU image sink into this directory")
    ap.add_argument("--image-format", default="png", choices=["png", "ppm", "raw"])
    ap.add_argument("--opt", action="append", default=[], help="library tuning knob key=value (gms_set_option), repeatable")
    ap.add_argument("--no-native", action="store_true", help="drive the frame through PyTorch autograd instead of the one-call gms_train_frame")
    ap.add_argument("--sync-frame", action="store_true", help="stock-style frame with the 4-byte read-back of N (default: sync-free)")
    ap.add_argument("--reference-ops", action="store_true",
                    help="glue ops as the reference orders them (two-step expansion, ATen loss, torch Adam) around our rasterizer")
    ap.add_argument("--cpu-budget", type=float, default=15.0, help="(kept for compatibility; the CPU sample is now a fixed tile stride)")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="after the timed steps, write what the last one computed as DIR/<name>.npy (float32; rows of a large "
                         "array sampled with a fixed seed; at most 64 MB in all)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl ours)")
    if args.impl == "reference":
        return run_reference_arm(args)

    import torch.distributed as dist
    from gms_b200 import _lib, io_image, rasterizer
    from gms_b200.model import MeshGaussianModel
    from gms_b200.trainer import MeshTrainer, render_frame, shard_cameras

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py (impl ours) needs a GPU: the product has no CPU path"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    for kv in args.opt:
        k, v = kv.split("=")
        assert _lib.set_option(k, int(v)) >= 0, f"unknown option {k}"
    if args.workload == "gs_flat_10k_256":
        if rank == 0:
            run_flat(args, dev)
        return
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    K_, W_ = args.steps, max(args.warmup, 3)

    params, cams, dims = build_scene(args.workload)
    F, K, W, H = dims
    P = F * K
    if args.mode == "render_animated":
        return run_render_animated(args, params, cams, dims, dev, world, rank, local)
    model = MeshGaussianModel.from_params(params, dev, packed_features=not args.reference_ops)
    bg = torch.ones(3, device=dev)
    cams_dev = [c.to(dev) for c in cams]
    # Ground truth: the same object with different appearance, rendered once per camera (synthetic data) and stored the way
    # dataset images are -- 8 bits per channel.  The resident copy is the reference's (scene/cameras.py:39-46 keeps
    # original_image on the device); the e2e arm ships the uint8 image from pinned host memory every step.
    gt_params = build_scene(args.workload, seed=123)[0]
    gt_model = MeshGaussianModel.from_params(gt_params, dev)
    with torch.no_grad():
        gts_u8 = [io_image.quantize(render_frame(gt_model, c, bg)[0].clamp(0, 1).contiguous()) for c in cams_dev]      # [H, W*3] uint8
        gts = [io_image.to_device_float(g.view(H, W, 3), hwc=True) for g in gts_u8]
    del gt_model
    gts_host_u8 = [g.cpu().pin_memory() for g in gts_u8]
    gts_host_f32 = [g.cpu().pin_memory() for g in gts]
    cam_host = [torch.cat([c.world_view_transform.reshape(-1), c.full_proj_transform.reshape(-1), c.camera_center.reshape(-1)]).pin_memory()
                for c in cams]
    loss_fn = None
    if args.reference_ops:
        import aten_reference           # tests/: the ATen restatement of utils/loss_utils.py
        loss_fn = aten_reference.training_loss
    trainer = MeshTrainer(model, bg, world=world, rank=rank, optimizer_step=not args.no_optimizer, fast=not args.reference_ops,
                          native=not (args.no_native or args.reference_ops), sync_free=not args.sync_frame, loss_fn=loss_fn)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, first_step):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for s in range(steps):
            fn(first_step + s)
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    n_frames = []

    last = {}

    def step_resident(s):
        ci = shard_cameras(len(cams), s, rank, world)
        last["loss"] = trainer.step(cams_dev[ci], gts[ci])
        n_frames.append(rasterizer.last_num_rendered)

    # e2e: every step's inputs (ground-truth image + 35 camera floats) come from PINNED HOST memory; the copy of step s+1
    # runs on a side stream while step s computes (a data-loader prefetch), and the step's loss is read back to the host.
    # Both copies are inside the timed region.  Primary variant: 8-bit image (3*H*W bytes) + one dequantise kernel;
    # second figure: the fp32 image (12*H*W bytes) as in round 1.
    from gms_b200.scenes import Camera
    copy_stream = torch.cuda.Stream(dev)
    cam_bufs = [torch.empty(35, device=dev) for _ in range(2)]
    gt_u8_bufs = [torch.empty((H, W * 3), dtype=torch.uint8, device=dev) for _ in range(2)]
    gt_bufs = [torch.empty(3, H, W, device=dev) for _ in range(2)]
    ready = [torch.cuda.Event() for _ in range(2)]
    consumed = [torch.cuda.Event() for _ in range(2)]
    e2e_mode = {"u8": True}

    def prefetch(s):
        ci = shard_cameras(len(cams), s, rank, world)
        b = s & 1
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(consumed[b])
            if e2e_mode["u8"]:
                gt_u8_bufs[b].copy_(gts_host_u8[ci], non_blocking=True)
            else:
                gt_bufs[b].copy_(gts_host_f32[ci], non_blocking=True)
            cam_bufs[b].copy_(cam_host[ci], non_blocking=True)
            ready[b].record(copy_stream)

    for b in range(2):
        consumed[b].record(torch.cuda.current_stream(dev))

    loss_host = torch.zeros(1).pin_memory()
    loss_ready = torch.cuda.Event()

    def step_e2e(s):
        ci = shard_cameras(len(cams), s, rank, world)
        b = s & 1
        prefetch(s + 1)
        torch.cuda.current_stream(dev).wait_event(ready[b])
        c = cams[ci]
        cb = cam_bufs[b]
        cam = Camera(c.image_width, c.image_height, c.FoVx, c.FoVy, cb[:16].view(4, 4), cb[16:32].view(4, 4), cb[32:35], uid=("view", ci))
        if e2e_mode["u8"]:
            io_image.to_device_float(gt_u8_bufs[b].view(H, W, 3), out=gt_bufs[b], hwc=True)
        trainer.step(cam, gt_bufs[b], loss_host=loss_host, loss_ready=loss_ready)
        consumed[b].record(torch.cuda.current_stream(dev))
        loss_ready.synchronize()          # device -> host read of THIS step's loss (4 bytes into pinned memory), every step;
        return float(loss_host[0])        # the copy is queued ahead of the optimizer kernels, so Adam overlaps the next launch

    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    for s in range(max(W_, len(cams))):      # warm-up covers one sweep of the cameras (allocator sees every scratch size)
        step_resident(s)
    _lib.launch_count(reset=True)
    n_frames.clear()
    if sampler:
        sampler.active = True
    ms_total = timed(step_resident, K_, W_)
    if sampler:
        sampler.active = False
    launches = _lib.launch_count(reset=True)
    if rank == 0 and args.dump_outputs:
        # what the caller of a training step receives: the loss and the updated parameters (Adam consumes the gradients)
        dump_outputs(args.dump_outputs, {"loss": last["loss"], "vertices": model.vertices, "_alpha": model._alpha, "_scale": model._scale,
                                         "_opacity": model._opacity, "features": model.get_features})

    def run_e2e(u8):
        e2e_mode["u8"] = u8
        torch.cuda.synchronize()
        prefetch(0)
        for s in range(2):
            step_e2e(s)
        return timed(step_e2e, K_, 2)

    if sampler:
        sampler.active = True
    ms_e2e = run_e2e(True)
    if sampler:
        sampler.active = False
        sampler.stop()
    ms_e2e_f32 = run_e2e(False)
    h2d_u8 = gts_host_u8[0].numel() + 35 * 4
    h2d_f32 = gts_host_f32[0].numel() * 4 + 35 * 4
    # SURVEY 8(d)'s frame (fwd + loss + bwd, optimizer excluded) as a second figure
    frame_only = None
    if not args.no_optimizer:
        try:
            trainer.optimizer_step = False
            for s in range(3):
                step_resident(s)
            frame_only = timed(step_resident, K_, 3) / K_
        finally:
            trainer.optimizer_step = True
    # per-kernel device time (CUDA events on the launching stream, inside the library), separate pass
    _lib.set_option("time_kernels", 1)
    _lib.kernel_times(reset=True)
    barrier()
    for s in range(min(K_, 10)):
        step_resident(W_ + 2 * K_ + s)
    torch.cuda.synchronize()
    kt = _lib.kernel_times(reset=True)
    _lib.set_option("time_kernels", 0)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    ms_step = ms_total / K_
    value = world * 1000.0 / ms_step
    N_mean = float(np.mean([n for n in n_frames if n > 0])) if any(n > 0 for n in n_frames) else 0.0
    units = {"P": P, "F": F, "N": N_mean, "px": W * H}
    per_kernel = {}
    for name, (ms, cnt) in kt.items():
        if cnt:
            ab = sum(ALGO_BYTES.get(name, {}).get(u, 0) * units[u] for u in units)
            if name == "adam":
                ab += 12 * (world - 1) * P          # replicated factored optimizer: one more 12 B colour gradient per extra rank
            per_kernel[name] = {"ms": ms / cnt, "launches_per_step": cnt / min(K_, 10), "algo_bytes": ab,
                                "gbs": (ab / (ms / cnt * 1e-3) / 1e9) if ms > 0 else None}
    if "cub_sort_tiles" in per_kernel and any(o.startswith("bin_impl=1") for o in args.opt):
        per_kernel["bin_tiles"] = per_kernel.pop("cub_sort_tiles")      # --opt bin_impl=1: the cooperative counting kernel runs in that slot
    dom = max(per_kernel, key=lambda k: per_kernel[k]["ms"] * per_kernel[k]["launches_per_step"]) if per_kernel else None
    peak, peak_src = measured_peak_gbs()
    roof = None
    if dom:
        a = per_kernel[dom]["gbs"]
        roof = {"bound": "hbm", "kernel": dom, "achieved": a, "peak": peak, "unit": "GB/s", "frac": a / peak,
                "traffic": ncu_traffic_bytes(args.workload, dom), "peak_source": peak_src, "kernel_ms": per_kernel[dom]["ms"],
                "algo_bytes_per_launch": per_kernel[dom]["algo_bytes"],
                "note": "composite kernels are FP32-issue bound (exp + ~50 flops per pixel x splat), not HBM bound; see DESIGN.md"}
    frame_bytes = 1014 * P + 96 * F + 172 * N_mean + 48 * W * H
    raster_names = ("preprocess_fwd", "cub_sort_depth", "cub_scan_tiles", "emit_dups", "cub_sort_tiles", "bin_tiles", "tile_ranges",
                    "composite_fwd", "composite_bwd", "preprocess_bwd")
    raster_ms = sum(per_kernel[k]["ms"] * per_kernel[k]["launches_per_step"] for k in raster_names if k in per_kernel)
    line = {"metric": METRIC[args.workload], "value": value, "unit": "frames/s", "n_gpus": world,
            "steps": K_, "warmup": W_, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": base_config(args.workload),
            "details": {"N_mean": N_mean, "optimizer_step": not args.no_optimizer,
                        "glue": "reference-ops" if args.reference_ops else ("fused, one C call per frame (gms_train_frame)" if not args.no_native else "fused, autograd-driven"),
                        "sync_free_frame": (not args.sync_frame) and not (args.no_native or args.reference_ops),
                        "options": args.opt, "parallelism": f"frame-sharded dp{world}",
                        "l2": "inputs_exceed_l2 (per-step working set > 126 MB)",
                        "frame_algo_bytes": frame_bytes, "frame_hbm_frac": frame_bytes / (ms_step * 1e-3) / 1e9 / peak,
                        "rasterizer_only_ms": raster_ms,
                        "frame_without_optimizer": None if frame_only is None else {"ms_per_step": frame_only, "value": world * 1000.0 / frame_only,
                                                                                    "what": "SURVEY 8(d) frame: expansion + render + loss + backward (+ gradient all-reduce), no Adam"},
                        "binning_overflows": getattr(getattr(trainer, "_frame", None), "overflows", None),
                        "ground_truth": "8-bit (quantised once at set-up; resident copy dequantised to fp32, e2e ships uint8 from pinned host memory)"},
            "e2e": {"value": world * 1000.0 / (ms_e2e / K_), "unit": "frames/s", "h2d_bytes_per_step": h2d_u8, "d2h_bytes_per_step": 4,
                    "ms_per_step": ms_e2e / K_,
                    "fp32_ground_truth": {"value": world * 1000.0 / (ms_e2e_f32 / K_), "ms_per_step": ms_e2e_f32 / K_, "h2d_bytes_per_step": h2d_f32}},
            "gpu_launches": int(launches), "roofline": roof, "kernels": per_kernel,
            "clocks": sampler.summary() if sampler else None}
    if world == 1 and not args.no_comparators:
        line["comparators"] = run_comparators(model, cams_dev, gts, bg, dims, dev)
        if "rasterizer_fwd_bwd_ms" in line["comparators"]:
            line["vs_refstyle"] = line["comparators"]["vs_refstyle"]
    if world == 1 and not args.no_cpu_baseline:
        try:
            stride = CPU_TILE_STRIDE.get(args.workload, 1)
            fs, desc, cores = cpu_reference_frame(params, cams[0], dims, stride, HOST_THREADS)
            line["cpu_baseline"] = {"value": 1.0 / fs, "unit": "frames/s", "cores": cores, "kind": "port", "sample": desc, "tile_stride": stride}
        except Exception as e:  # pragma: no cover
            line["cpu_baseline"] = {"value": None, "unit": "frames/s", "cores": 0, "kind": "port", "sample": f"failed: {e}"}
    emit_result(line)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
