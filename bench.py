#!/usr/bin/env python
"""bench.py -- fwd+bwd Mpix/s of the differentiable gaussian rasterizer (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            (N>1: launched by torch.distributed.run)
    python bench.py --impl reference ...                     (the path's CPU implementation, timed alone)
    python bench.py ... --dump-outputs DIR                   (also writes the last timed step's outputs: dump_outputs())

A *step* is one pass of the hot path over one batch of synthetic input: every rank renders its
`--views-per-rank` camera views of the SAME replicated gaussians forward + backward (L1 loss against a
synthetic target image), gradients accumulate in one flat bucket, and ONE NCCL all-reduce sums the bucket
over ranks (view-parallel, weak scaling: views per rank fixed).  Workload = BASELINE.json configs[2]
(1 M random gaussians, 1920x1080, SH degree 3); with 8 views per rank, N=8 is configs[4] (64 views).

`value`   : inputs (cameras, target images) resident in HBM; device-timed (CUDA events), max over ranks.
`e2e`     : same step through the public API with HOST inputs: each view's camera matrices and target
            image are copied from pinned host memory inside the timed region (side stream, overlapping the
            view's forward kernels) and the step's loss is copied back to pinned host memory every step
            (the host<->device crossings of the reference's loop: train.py:119,148).
            The gaussians are the model state and stay resident, as they do in the reference.
`roofline`: dominant kernel (render_bwd) -- algorithmic bytes / CUDA-event time on its launch stream.
`cpu_baseline` / `--impl reference`: the CPU restatement of the path (oracle/gs_oracle.c, OpenMP over all
            host cores).  The reference's own rasterizer sources are absent from /root/reference
            (SURVEY.md section 0), so there is no oracle/_ref and kind is "port".  If a stock install of
            the reference rasterizer ever appears under baseline/_ref (diff_gaussian_rasterization built
            from the submodule the operator vendors), `--impl reference` times THAT on the GPU instead
            (kind "reference-cuda").
`single_view`: the drop-in path a user of the reference gets: one camera per iteration through
            GaussianRasterizer.forward + loss.backward() (train.py:111-142), same workload.
"""
import argparse
import gc
import importlib.util
import json
import math
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "gaussian-splatting_b200")
for _p in (ROOT, PKG):
    if _p not in sys.path:
        sys.path.insert(0, _p)

METRIC = "fwd+bwd Mpix/s @1M gaussians 1080p"
UNIT = "Mpix/s"
LOG_SCALE_MEAN = -5.3   # mean reference tiles-touched per visible gaussian ~= 7 (SURVEY.md 8d asks 4-8)
DUMP_ROWS = 65536       # gaussians sampled by --dump-outputs: 119 floats each at most (59 gradients, 59 parameters, radius) = 31 MB


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--views-per-rank", type=int, default=8)
    ap.add_argument("--gaussians", type=int, default=1_000_000)
    ap.add_argument("--width", type=int, default=1920)
    ap.add_argument("--height", type=int, default=1080)
    ap.add_argument("--sh-degree", type=int, default=3)
    ap.add_argument("--api", default="views", choices=["views", "render"],
                    help="views: fused view-batch path render_views_backward(); render: per-view render() + autograd")
    ap.add_argument("--loss", default="l1", choices=["l1", "l1_ssim"],
                    help="l1: mean |clamp(image) - target| (default, comparable across rounds); l1_ssim: the reference step's "
                         "0.8 L1 + 0.2 (1 - SSIM) (train.py:120-126), fused kernel")
    ap.add_argument("--optimizer", action="store_true",
                    help="whole training iteration: the gaussians live in gaussian_store.GaussianModel (raw parameters) and "
                         "every step ends with its fused activation-backward + Adam step (outside the BASELINE metric)")
    ap.add_argument("--no-batch", action="store_true", help="views API view by view instead of gsb_forward_batch")
    ap.add_argument("--sync", action="store_true",
                    help="A/B: the synchronous view-batch call (one instance-count read-back per step) instead of the sync-free one")
    ap.add_argument("--grad-chunks", type=int, default=1,
                    help="gaussian-range chunks of the gradient-writing kernel, each chunk's SH rows all-reduced while the next "
                         "computes.  Default 1 = one all-reduce after the last kernel: on 8 B200s the chunked variant measured "
                         "SLOWER (9.75 vs 9.47 ms/step, profiles/r2_scaling.md) -- the concurrent NCCL kernels cost the compute "
                         "kernel more than the overlap hides")
    ap.add_argument("--reduce", default="allreduce", choices=["allreduce", "peer"],
                    help="allreduce: one NCCL all-reduce of the gradient bucket after the last kernel.  peer: the FUSED reduce-"
                         "scatter -- the gradient kernel adds every row into its owner rank's peer-mapped buffer over NVLink while "
                         "it computes (gsb_backward_batch_peer), then a barrier and an in-place all-gather of the owned rows")
    ap.add_argument("--no-pin", action="store_true", help="do not pin the process to its GPU's NUMA-local cores")
    ap.add_argument("--no-single-view", action="store_true", help="skip the drop-in single-view leg (render() + autograd)")
    ap.add_argument("--workload", default="raster", choices=["raster", "train6m"],
                    help="raster: the BASELINE metric (default).  train6m: BASELINE configs[3], the 6 M-gaussian training loop "
                         "with densify/prune (tools/train_bench.py), reported as iterations/s")
    ap.add_argument("--iterations", type=int, default=1000, help="train6m: iterations")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-baseline-seconds", type=float, default=20.0)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the device-resident timed steps, write what the last of them returned to its caller as DIR/<name>.npy "
                         "(see dump_outputs), so that two builds can be compared on identical inputs")
    a = ap.parse_args()
    if a.dump_outputs and (a.impl != "ours" or a.workload != "raster"):
        ap.error("--dump-outputs applies to the rasterizer workload of this implementation (--impl ours --workload raster)")
    return a


def dump_outputs(directory, last, pc, with_params):
    """Writes what the caller of the last timed step received: the per-view losses (losses.npy, [V]) and, per gaussian, the
    largest screen radius over the step's views (radii_max.npy) and the gradient of each rasterizer input (grad_means3D.npy,
    grad_shs.npy, grad_opacities.npy, grad_scales.npy, grad_rotations.npy); with --optimizer also the inputs as the optimizer
    step left them (means3D.npy, ...).  Per-gaussian arrays hold a sample of DUMP_ROWS gaussians drawn with a fixed seed, so
    the same --gaussians gives the same rows; gaussian_index.npy lists them (float64), every other array is float32."""
    import numpy as np
    import torch
    inputs = {"means3D": pc.get_xyz, "shs": pc.get_features, "opacities": pc.get_opacity, "scales": pc.get_scaling,
              "rotations": pc.get_rotation}
    P = int(pc.get_xyz.shape[0])
    rows = torch.arange(P) if P <= DUMP_ROWS else \
        torch.randperm(P, generator=torch.Generator().manual_seed(0))[:DUMP_ROWS].sort().values
    idx = rows.to(pc.get_xyz.device)
    arrays = {"gaussian_index": rows.double(), "losses": torch.stack(list(last["losses"])),
              "radii_max": torch.stack(last["radii"]).amax(dim=0)[idx]}
    for name, t in inputs.items():
        arrays["grad_" + name] = t.grad[idx]
        if with_params:
            arrays[name] = t.detach()[idx]
    os.makedirs(directory, exist_ok=True)
    for name, t in arrays.items():
        t = t.detach().cpu()
        np.save(os.path.join(directory, name + ".npy"), t.numpy() if t.dtype == torch.float64 else t.float().numpy())


class BenchCamera:
    """The attributes render() reads from scene.cameras.Camera (/root/reference/scene/cameras.py:19-89)."""

    def __init__(self, width, height, fovx, R, T, device, camera_matrices=None):
        if camera_matrices is None:
            from gaussian_renderer.synthetic import camera_matrices
        self.image_width, self.image_height = width, height
        self.FoVx = fovx
        self.FoVy = 2.0 * math.atan(math.tan(fovx / 2) * height / width)
        wvt, full, center = camera_matrices(R, T, self.FoVx, self.FoVy)
        self.host = dict(wvt=wvt.contiguous().pin_memory() if device != "cpu" else wvt,
                         full=full.contiguous().pin_memory() if device != "cpu" else full,
                         center=center.contiguous().pin_memory() if device != "cpu" else center)
        self.world_view_transform = wvt.to(device)
        self.full_proj_transform = full.to(device)
        self.camera_center = center.to(device)
        self.image_name = "synthetic"

    def upload(self, device):
        """e2e leg: per-view camera tensors come from pinned host memory."""
        self.world_view_transform = self.host["wvt"].to(device, non_blocking=True)
        self.full_proj_transform = self.host["full"].to(device, non_blocking=True)
        self.camera_center = self.host["center"].to(device, non_blocking=True)
        return 4 * (16 + 16 + 3)


def view_pose(global_index: int, radius: float):
    """Cameras on a sphere of radius 3R looking at the origin (SURVEY.md 8d); golden-angle spiral."""
    from gaussian_renderer.synthetic import sphere_pose
    return sphere_pose(global_index, radius)


class BenchGaussians:
    """Duck-typed stand-in for scene.GaussianModel: activated tensors as leaves (the rasterizer's inputs)."""

    def __init__(self, scene, sh_degree, device):
        import torch
        self.active_sh_degree = sh_degree
        self.max_sh_degree = int(round(math.sqrt(scene["shs"].shape[1]))) - 1
        mk = lambda t: t.to(device).contiguous().requires_grad_(True)
        self._xyz, self._shs, self._opacity = mk(scene["means3D"]), mk(scene["shs"]), mk(scene["opacities"])
        self._scaling, self._rotation = mk(scene["scales"]), mk(scene["rotations"])

    def parameters(self):
        return [self._xyz, self._shs, self._opacity, self._scaling, self._rotation]

    get_xyz = property(lambda s: s._xyz)
    get_features = property(lambda s: s._shs)
    get_opacity = property(lambda s: s._opacity)
    get_scaling = property(lambda s: s._scaling)
    get_rotation = property(lambda s: s._rotation)


class Pipe:
    debug = False
    antialiasing = False
    compute_cov3D_python = False
    convert_SHs_python = False


class ClockSampler:
    """SM clock / throttle reasons sampled DURING the timed region.  In-process NVML (nvidia_ml_py) every 100 ms:
    an external `nvidia-smi -lms` loop was measured to stall kernel launches (the device-resident leg ran 2-3x
    slower than the end-to-end leg whenever it was polling), so it is only the fallback, at 500 ms."""

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.samples = []          # (wall time, sm_mhz, sm_max_mhz, reasons bitmask or list)
        self.thread = None
        self.proc = None
        self.stop_flag = False
        self.t_start, self.t_end = 0.0, float("inf")
        # NVML calls share driver locks with kernel launches and occasionally take tens of ms: a launch thread that has no lead over
        # the device yet (every timed region starts from a synchronize) passes such a stall on to the device, and through the
        # collective to every rank.  Inside a timed region the sampler therefore waits until the launch thread has enqueued the
        # region's work (timed() calls hold() / release()); the samples are still taken under load, while the device drains.
        self.clear = threading.Event()
        self.clear.set()

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            idx = int(vis.split(",")[self.gpu]) if vis and all(x.strip().isdigit() for x in vis.split(",")) else self.gpu
            h = pynvml.nvmlDeviceGetHandleByIndex(idx)
            mx = pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM)

            def loop():
                while not self.stop_flag:
                    if not self.clear.wait(0.05):
                        continue
                    try:
                        sm = pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)
                        try:
                            r = pynvml.nvmlDeviceGetCurrentClocksEventReasons(h)
                        except Exception:
                            r = pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                        self.samples.append((time.time(), float(sm), float(mx), int(r)))
                    except Exception:
                        pass
                    time.sleep(0.02 if self.draining else 0.1)
            self.thread = threading.Thread(target=loop, daemon=True)
            self.thread.start()
            self.kind = "nvml"
        except Exception:
            self._start_smi()

    def _start_smi(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "500",
                                          "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)

            def read():
                for line in self.proc.stdout:
                    f = [x.strip() for x in line.split(",")]
                    try:
                        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
                        rs = [n for n, v in zip(names, f[2:6]) if v.lower().startswith("active")]
                        self.samples.append((time.time(), float(f[0]), float(f[1]), rs))
                    except Exception:
                        pass
            self.thread = threading.Thread(target=read, daemon=True)
            self.thread.start()
            self.kind = "nvidia-smi"
        except Exception:
            self.kind = "unavailable"

    draining = False

    def hold(self):
        """the launch thread is about to enqueue a timed region: no NVML calls until release()"""
        self.draining = False
        self.clear.clear()

    def release(self):
        """the region's work is enqueued (the device is still executing it): sample now, every 20 ms"""
        self.draining = True
        self.clear.set()

    def mark(self, which):
        """start / end of the timed region (wall clock): only samples taken inside it are reported."""
        setattr(self, "t_" + which, time.time())

    def stop(self):
        self.stop_flag = True
        if self.proc:
            self.proc.terminate()
        inside = [s for s in self.samples if self.t_start <= s[0] <= self.t_end + 0.05] or self.samples[-2:]
        if not inside:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no sample"], "source": getattr(self, "kind", "?")}
        reasons = set()
        # NVML bit masks (nvml.h): 0x8 hw_slowdown, 0x40 hw_thermal, 0x20 sw_thermal, 0x4 sw_power_cap
        bits = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}
        for s in inside:
            if isinstance(s[3], int):
                reasons |= {n for b, n in bits.items() if s[3] & b}
            else:
                reasons |= set(s[3])
        return {"sm_mhz": statistics.median(s[1] for s in inside), "sm_max_mhz": max(s[2] for s in inside),
                "reasons": sorted(reasons), "samples": len(inside), "source": getattr(self, "kind", "?")}


def cpu_reference_pass(scene, cam_settings, repeats):
    """One full-frame forward+backward of the CPU oracle per repeat; returns (seconds per pass, threads)."""
    import numpy as np
    from oracle.c_oracle import COracle, threads
    H, W = cam_settings.image_height, cam_settings.image_width
    rng = np.random.default_rng(0)
    dL = rng.standard_normal((3, H, W)).astype(np.float32)
    times = []
    for _ in range(repeats):
        t0 = time.perf_counter()
        co = COracle(scene["means3D"], scene["shs"], None, scene["opacities"], scene["scales"], scene["rotations"],
                     None, cam_settings)
        co.backward(dL, None)
        co.close()
        times.append(time.perf_counter() - t0)
    return times, threads()


def oracle_settings(cam: BenchCamera, sh_degree: int):
    """Settings record for the CPU oracle (cpu_baseline / --impl reference legs only)."""
    import torch
    from oracle import torch_oracle as TO
    return TO.OracleSettings(image_height=cam.image_height, image_width=cam.image_width,
                             tanfovx=math.tan(cam.FoVx * 0.5), tanfovy=math.tan(cam.FoVy * 0.5),
                             bg=torch.zeros(3), scale_modifier=1.0, viewmatrix=cam.world_view_transform.cpu(),
                             projmatrix=cam.full_proj_transform.cpu(), sh_degree=sh_degree,
                             campos=cam.camera_center.cpu(), prefiltered=False, debug=False, antialiasing=False)


def workload_config(a, world):
    return {"workload": f"{a.gaussians} random gaussians, {a.width}x{a.height}, SH degree {a.sh_degree}, fwd+bwd "
                        f"(BASELINE.json configs[2]); {a.views_per_rank} views per rank",
            "gaussians": a.gaussians, "image": [a.width, a.height], "sh_degree": a.sh_degree,
            "views_per_rank": a.views_per_rank, "views_total": a.views_per_rank * world,
            "parallelism": f"view-parallel x{world}, gaussians replicated, one all-reduce of 59 floats/gaussian",
            "api": a.api, "loss": a.loss, "optimizer": "fused_adam_store" if a.optimizer else "none",
            "l2": "inputs_exceed_l2 (236 MB parameters + 8 distinct views per step; no explicit flush)",
            "scene": f"xyz~U([-1,1]^3), log-scale~N({LOG_SCALE_MEAN},0.5), opacity=sigmoid(U(-2,4)), cameras on sphere r=3, seed 0"}


def _load_synthetic():
    """gaussian_renderer/synthetic.py by FILE PATH: importing the package would map libgs_b200.so into the reference arm."""
    spec = importlib.util.spec_from_file_location("gsb_synthetic", os.path.join(PKG, "gaussian_renderer", "synthetic.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def _stock_reference_rasterizer():
    """The UNMODIFIED reference rasterizer, if the operator has installed it under baseline/_ref (its sources are absent
    from /root/reference, so normally there is none).  Returns the imported module or None."""
    ref_dir = os.path.join(ROOT, "baseline", "_ref")
    if not os.path.isdir(os.path.join(ref_dir, "diff_gaussian_rasterization")):
        return None
    saved = list(sys.path)
    try:
        sys.path.insert(0, ref_dir)
        for name in [m for m in sys.modules if m.split(".")[0] == "diff_gaussian_rasterization"]:
            del sys.modules[name]
        import diff_gaussian_rasterization as stock
        if os.path.realpath(os.path.dirname(stock.__file__)).startswith(os.path.realpath(ref_dir)) and hasattr(stock, "_C"):
            return stock
    except Exception:
        pass
    finally:
        sys.path[:] = saved
    return None


def run_reference_cuda(a, stock, syn):
    """--impl reference with a stock install present: the reference's own CUDA rasterizer through its own Python API,
    one view per step, same scene / cameras / metric (kind "reference-cuda")."""
    import torch
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
    torch.cuda.set_device(dev)
    scene = {k: v.to(dev).requires_grad_(True) for k, v in syn.make_scene(a.gaussians, seed=0, log_scale_mean=LOG_SCALE_MEAN).items()}
    V, H, W = a.views_per_rank, a.height, a.width
    cams = []
    for i in range(V):
        R, T = syn.sphere_pose(i, 3.0)
        fovx = math.radians(60.0)
        fovy = 2.0 * math.atan(math.tan(fovx / 2) * H / W)
        wvt, full, center = syn.camera_matrices(R, T, fovx, fovy)
        cams.append((fovx, fovy, wvt.to(dev), full.to(dev), center.to(dev)))
    gen = torch.Generator().manual_seed(1234)
    gts = [torch.rand(3, H, W, generator=gen).to(dev) for _ in range(V)]
    bg = torch.zeros(3, device=dev)

    def one(i):
        fovx, fovy, wvt, full, center = cams[i % V]
        rs = stock.GaussianRasterizationSettings(image_height=H, image_width=W, tanfovx=math.tan(fovx * 0.5), tanfovy=math.tan(fovy * 0.5),
                                                 bg=bg, scale_modifier=1.0, viewmatrix=wvt, projmatrix=full, sh_degree=a.sh_degree,
                                                 campos=center, prefiltered=False, debug=False, antialiasing=False)
        out = stock.GaussianRasterizer(raster_settings=rs)(
            means3D=scene["means3D"], means2D=torch.zeros_like(scene["means3D"], requires_grad=True), shs=scene["shs"],
            colors_precomp=None, opacities=scene["opacities"], scales=scene["scales"], rotations=scene["rotations"], cov3D_precomp=None)
        (out[0].clamp(0, 1) - gts[i % V]).abs().mean().backward()

    for i in range(max(a.warmup, 3) * V):
        one(i)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(a.steps * V):
        one(i)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    value = a.steps * V * H * W / 1e6 / (ms / 1e3)
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": 1, "steps": a.steps, "warmup": max(a.warmup, 3),
            "ms_per_step": ms / a.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "config": workload_config(a, 1),
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": 0, "kind": "reference-cuda",
                             "sample": f"{V} views per step through the stock diff_gaussian_rasterization in baseline/_ref (GPU)"},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def run_reference(a):
    """--impl reference: the path's CPU implementation on the host cores, one view per step (bounded sample)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    syn = _load_synthetic()
    stock = _stock_reference_rasterizer()
    if stock is not None:
        return run_reference_cuda(a, stock, syn)
    from oracle.c_oracle import set_threads
    if hasattr(os, "sched_setaffinity"):
        try:                            # launchers may start the process on one NUMA node: the CPU arm gets every core of the box
            os.sched_setaffinity(0, range(os.cpu_count() or 1))
        except OSError:
            pass
    nthreads = set_threads(len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1))
    scene = syn.make_scene(a.gaussians, seed=0, log_scale_mean=LOG_SCALE_MEAN)
    R, T = syn.sphere_pose(0, 3.0)
    cam = BenchCamera(a.width, a.height, math.radians(60.0), R, T, "cpu", camera_matrices=syn.camera_matrices)
    cs = oracle_settings(cam, a.sh_degree)
    times, nthreads = cpu_reference_pass(scene, cs, a.warmup + a.steps)
    timed = times[a.warmup:]
    total = sum(timed)
    mpix = a.width * a.height / 1e6
    value = mpix * len(timed) / total
    sample = "1 full view (forward+backward) per step"
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": a.gpus, "steps": a.steps,
            "warmup": a.warmup, "ms_per_step": 1e3 * total / len(timed), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": workload_config(a, max(1, a.gpus)),
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": nthreads, "kind": "port", "sample": sample,
                             "host_cpus": os.cpu_count()},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0,
            "note": "CPU port of the path (oracle/gs_oracle.c, OpenMP); the reference's CUDA rasterizer sources "
                    "are absent from /root/reference so its own implementation cannot be built or timed"}
    print(json.dumps(line), flush=True)


def main():
    a = parse()
    if a.impl == "reference":
        run_reference(a)
        return
    if a.workload == "train6m":
        sys.path.insert(0, os.path.join(ROOT, "tools"))
        import train_bench
        return train_bench.bench_line(a)
    import torch
    import torch.distributed as dist
    from gaussian_renderer.synthetic import make_scene   # the oracle is only loaded by the cpu_baseline leg below
    import diff_gaussian_rasterization as dgr
    from gaussian_renderer import AsyncCapacity, GradientBucket, pin_to_gpu_numa_node, render, render_views_backward

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the rasterizer has no CPU path (use --impl reference for the CPU port)")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    pinned_cores = None if a.no_pin else pin_to_gpu_numa_node(local)
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    for kv in os.environ.get("GS_OPTS", "").split(","):      # tuning knobs for A/B runs, e.g. GS_OPTS=sort_small=1
        if "=" in kv:
            dgr.set_option(kv.split("=")[0], int(kv.split("=")[1]))
    if world != a.gpus and rank == 0:
        print(f"# note: --gpus {a.gpus} but WORLD_SIZE {world}; using {world}", file=sys.stderr)
    grad_chunks = max(1, a.grad_chunks)

    torch.manual_seed(0)
    scene = make_scene(a.gaussians, seed=0, log_scale_mean=LOG_SCALE_MEAN)
    if a.optimizer:
        from types import SimpleNamespace
        from gaussian_store import GaussianModel
        sc = {k: v.to(dev) for k, v in scene.items()}
        pc = GaussianModel(int(round(math.sqrt(sc["shs"].shape[1]))) - 1)
        pc.active_sh_degree = a.sh_degree
        op = sc["opacities"].clamp(1e-6, 1 - 1e-6).reshape(-1, 1)
        pc.create_from_tensors(sc["means3D"], sc["shs"][:, :1].contiguous(), sc["shs"][:, 1:].contiguous(), torch.log(sc["scales"]),
                               sc["rotations"], torch.log(op / (1 - op)), 1.0)
        pc.training_setup(SimpleNamespace(position_lr_init=0.00016, position_lr_final=0.0000016, position_lr_delay_mult=0.01,
                                          position_lr_max_steps=30000, feature_lr=0.0025, opacity_lr=0.025, scaling_lr=0.005,
                                          rotation_lr=0.001, percent_dense=0.01))      # arguments/__init__.py:77-89
        del sc
        bucket = pc.gradient_bucket()          # the store's gradient buffer IS the all-reduce bucket
    else:
        pc = BenchGaussians(scene, a.sh_degree, dev)
        bucket = GradientBucket(pc.parameters())
    peer_bucket = None
    if a.reduce == "peer" and world > 1 and not a.optimizer and a.api == "views" and not a.no_batch:
        from gaussian_renderer.peer import PeerGradientBucket
        peer_bucket = PeerGradientBucket({"means3D": pc._xyz, "shs": pc._shs, "opacities": pc._opacity, "scales": pc._scaling,
                                          "rotations": pc._rotation})
    pipe = Pipe()
    bg = torch.zeros(3, device=dev)
    V, H, W = a.views_per_rank, a.height, a.width
    cams = [BenchCamera(W, H, math.radians(60.0), *view_pose(rank * V + i, 3.0), dev) for i in range(V)]
    gen = torch.Generator().manual_seed(1234 + rank)
    gt_host = [torch.rand(3, H, W, generator=gen).pin_memory() for _ in range(V)]
    gt_dev = [g.to(dev) for g in gt_host]
    mpix_step = V * world * H * W / 1e6
    capacity = None if (a.sync or a.api != "views" or a.no_batch) else AsyncCapacity(dev)

    # e2e leg: per-view host inputs.  The 24.9 MB target image of view i is copied from pinned memory on a side
    # stream into one of two staging buffers when view i STARTS, so the copy overlaps that view's forward kernels;
    # the loss kernel waits for it through an event.  Camera matrices (140 B) go on the compute stream.
    copy_stream = torch.cuda.Stream(device=dev)
    NS = V                          # one staging buffer per view of the step (the batched path starts all views at once)
    stage = [torch.empty(3, H, W, device=dev) for _ in range(NS)]
    copied = [torch.cuda.Event() for _ in range(NS)]
    consumed = [torch.cuda.Event() for _ in range(NS)]
    for e in consumed:
        e.record()

    class HostCams:
        def __iter__(self):
            for i, cam in enumerate(cams):
                cam.upload(dev)
                with torch.cuda.stream(copy_stream):
                    copy_stream.wait_event(consumed[i % NS])         # last step's loss kernel is done with the buffer
                    stage[i % NS].copy_(gt_host[i], non_blocking=True)
                    copied[i % NS].record(copy_stream)
                yield cam

    loss_host = torch.zeros(1024, 1).pin_memory()
    step_counter = [0]
    last = {}                       # per-view losses and radii the latest step returned (--dump-outputs)

    def step(host_inputs: bool):
        if a.api != "views":
            bucket.zero_()
        pending = []
        if a.api == "views":
            def loss_fn(img, _invdepth, i, grad_out=None):      # the gradient goes straight into the batch's buffer (no copy)
                if a.loss == "l1":
                    fused = lambda x, y: dgr.l1_loss_and_grad(x, y, grad_out=grad_out)
                else:
                    fused = lambda x, y: dgr.photometric_loss_and_grad(x, y, 0.2, grad_out=grad_out)[:2]
                if host_inputs:
                    torch.cuda.current_stream(dev).wait_event(copied[i % NS])
                    res = fused(img, stage[i % NS])      # fused loss (train.py:120-126) + gradient
                    consumed[i % NS].record()
                    return res
                return fused(img, gt_dev[i])

            def on_chunk(_c, p0, p1):      # rows [p0, p1) of every gradient are final: reduce them while the next chunk computes
                pending.extend(bucket.all_reduce_rows(p0, p1))
            chunked = world > 1 and grad_chunks > 1 and not a.no_batch and peer_bucket is None
            if peer_bucket is not None:
                peer_bucket.begin_step()
            out = render_views_backward(HostCams() if host_inputs else cams, pc, pipe, bg, loss_fn, loss_returns_grad=True,
                                        batched=not a.no_batch, overwrite=True,   # first chunk writes the bucket: no zeroing pass
                                        capacity=capacity, grad_chunks=grad_chunks if chunked else 1,
                                        on_grad_chunk=on_chunk if chunked else None,
                                        peers=peer_bucket.table() if peer_bucket is not None else None)
            last["losses"], last["radii"] = out["losses"], [out["radii_max"]]
            total = out["losses"].sum()
            if peer_bucket is not None:
                peer_bucket.finish()        # barrier + in-place all-gather of the owned rows: every rank holds the summed gradient
            elif chunked:
                pending.extend(bucket.all_reduce_rest())     # the narrow parameters: one collective behind the last chunk
                GradientBucket.wait_all(pending)
            else:
                bucket.all_reduce()
        else:
            total = torch.zeros((), device=dev)
            last["losses"], last["radii"] = [], []
            for i, cam in enumerate(cams):
                if host_inputs:
                    cam.upload(dev)
                    gt = gt_host[i].to(dev, non_blocking=True)
                else:
                    gt = gt_dev[i]
                pkg = render(cam, pc, pipe, bg)
                loss = (pkg["render"] - gt).abs().mean()
                loss.backward()
                total += loss.detach()
                last["losses"].append(loss.detach())
                last["radii"].append(pkg["radii"])
            bucket.all_reduce()
        if a.optimizer:
            pc.update_learning_rate(pc.step_count + 1)
            pc.optimizer_step()
        if host_inputs:
            # device -> host read of the step's result: an asynchronous copy into pinned memory every step (the host does
            # not stall on it; all of them have landed when the timed region's final synchronize returns)
            slot = loss_host[step_counter[0] % loss_host.shape[0]]
            slot.copy_(total.reshape(1), non_blocking=True)
            step_counter[0] += 1
        return None

    step_stats = {}

    def timed(host_inputs: bool, steps: int):
        """K steps between barrier + synchronize on both sides; CUDA events; max over ranks.  Also the wall time the HOST
        needed to enqueue the K steps (how far it runs ahead of the device)."""
        gc.collect()
        gc.disable()        # a generation-2 collection in the launch thread is a multi-ms stall that every rank then waits for
        try:
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize()
            marks = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
            sampler.hold()
            t0 = time.perf_counter()
            marks[0].record()
            for k in range(steps):
                step(host_inputs)
                marks[k + 1].record()
            host_ms = (time.perf_counter() - t0) * 1e3
            sampler.release()
            torch.cuda.synchronize()
            sampler.draining = False
            if world > 1:
                dist.barrier()
        finally:
            gc.enable()
            sampler.clear.set()
            sampler.draining = False
        per_step = [marks[k].elapsed_time(marks[k + 1]) for k in range(steps)]
        step_stats[host_inputs] = {"min": round(min(per_step), 3), "median": round(statistics.median(per_step), 3),
                                   "max": round(max(per_step), 3), "slowest_step": int(max(range(steps), key=per_step.__getitem__)),
                                   "host_enqueue_ms_per_step": round(host_ms / steps, 3)}
        ms = torch.tensor([marks[0].elapsed_time(marks[steps])], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
            # every rank's own view of the region (outside the timing): which launch thread fell behind, if any
            mine = torch.tensor([host_ms / steps, float(step_stats[host_inputs]["slowest_step"]), max(per_step),
                                 statistics.median(per_step)], device=dev, dtype=torch.float32)
            every = [torch.empty_like(mine) for _ in range(world)]
            dist.all_gather(every, mine)
            rows = [[round(float(x), 3) for x in t.tolist()] for t in every]
            step_stats[host_inputs]["ranks"] = {"host_enqueue_ms_per_step": [r[0] for r in rows], "slowest_step": [int(r[1]) for r in rows],
                                                "max": [r[2] for r in rows], "median": [r[3] for r in rows]}
        return float(ms.item())

    def measured(host_inputs: bool):
        """One timed leg.  The sync-free path validates its instance capacity AFTER the region (one read of the running
        maximum); a region that overflowed rendered from truncated lists and is re-run with the grown capacity."""
        runs = []
        for _try in range(3):
            ms = timed(host_inputs, a.steps)
            ok = capacity is None or capacity.check()
            if world > 1:
                flag = torch.tensor([0 if ok else 1], device=dev)
                dist.all_reduce(flag, op=dist.ReduceOp.MAX)
                ok = int(flag.item()) == 0
            runs.append({"ms_total": round(ms, 3), **step_stats[host_inputs], "capacity_ok": ok})
            if ok:
                break
            step(host_inputs)       # synchronous-equivalent warm step with the new capacity
        return ms, runs

    # ---- device-resident leg ----
    # the sampler starts BEFORE the warm-up: nvidia-smi's own start-up disturbs the driver for a second or two
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    # untimed warm-up: at least 3 steps (contract) and at least 5 so that buffer sizes / the caching allocator settle
    # (the first step of the sync-free path is synchronous and learns the instance capacity)
    # ... and 32: the one straggler step of this round's N=8 runs (17 ms among 8.6 ms ones, DESIGN.md section 5) sat in the FIRST
    # timed region of a fresh box, a dozen steps into the process's life; a quarter of a second of extra warm-up costs nothing
    warmup_run = max(a.warmup, 32)
    for _ in range(warmup_run):
        step(False)
    torch.cuda.synchronize()
    dgr.set_option("time_kernels", 1)
    dgr.kernel_time("", reset=True)
    dgr.reset_launch_count()
    sampler.mark("start")
    ms_total, attempts = measured(False)
    sampler.mark("end")
    launches = dgr.launch_count() // len(attempts)
    bwd_ms, bwd_n = dgr.kernel_time("render_bwd")
    fwd_ms, fwd_n = dgr.kernel_time("render_fwd", reset=True)
    dgr.set_option("time_kernels", 0)
    clocks = sampler.stop() if rank == 0 else None
    value = mpix_step * a.steps / (ms_total / 1e3)
    if a.dump_outputs and rank == 0:      # before the next leg's steps overwrite the gradients
        dump_outputs(a.dump_outputs, last, pc, with_params=a.optimizer)

    # ---- end-to-end leg (host inputs) ----
    for _ in range(max(a.warmup, 3)):
        step(True)
    ms_e2e, e2e_attempts = measured(True)
    e2e_value = mpix_step * a.steps / (ms_e2e / 1e3)
    h2d = V * (3 * H * W * 4 + 4 * 35)
    d2h = 4

    # ---- drop-in single-view leg: GaussianRasterizer.forward + loss.backward() per camera (train.py:111-142) ----
    single_view = None
    if not a.no_single_view and not a.optimizer:
        sv_params = pc.parameters()

        def one_view(i):
            for p in sv_params:          # optimizer.zero_grad(set_to_none=True) of train.py:186: autograd then assigns the fresh
                p.grad = None            # gradient tensors instead of adding them into existing ones (one pass less over 236 MB)
            pkg = render(cams[i % V], pc, pipe, bg)
            (pkg["render"] - gt_dev[i % V]).abs().mean().backward()
        for i in range(2 * V):
            one_view(i)
        torch.cuda.synchronize()
        n_sv = a.steps * V
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        gc.collect(); gc.disable()
        e0.record()
        for i in range(n_sv):
            one_view(i)
        e1.record()
        torch.cuda.synchronize()
        gc.enable()
        sv_ms = e0.elapsed_time(e1) / n_sv
        # where the time goes (separate, untimed pass): this library's kernels per view; the rest of ms_per_view is torch's own
        # kernels (zeros, clamp, |x - y|.mean() and its backward, nonzero) and launch gaps behind the two host synchronisations
        # of the drop-in contract (the instance-count read-back and render()'s visibility_filter = (radii > 0).nonzero())
        dgr.set_option("time_kernels", 2)
        dgr.kernel_time("", reset=True)
        for i in range(V):
            one_view(i)
        torch.cuda.synchronize()
        sv_kernels = {}
        for name in ("preprocess_fwd", "sort_hist", "sort_scatter", "scan_reduce", "scan_partials", "scan_apply", "emit", "tile_ranges",
                     "tile_order", "render_fwd", "render_bwd", "preprocess_bwd"):
            t, n = dgr.kernel_time(name)
            sv_kernels[name] = round(t / V, 4)
        sv_kernels["sum"] = round(sum(sv_kernels.values()), 4)
        dgr.kernel_time("", reset=True)
        dgr.set_option("time_kernels", 0)
        if peer_bucket is not None:
            peer_bucket.begin_step()
        else:
            bucket = GradientBucket(sv_params)      # the legs after this one write into the bucket again
        single_view = {"value": H * W / 1e6 / (sv_ms / 1e3), "unit": UNIT, "ms_per_view": sv_ms, "views_timed": n_sv,
                       "library_kernel_ms_per_view": sv_kernels,
                       "api": "gaussian_renderer.render() -> GaussianRasterizer.forward + loss.backward(), one camera per iteration, "
                              "per rank (not aggregated over ranks)"}

    # ---- instance statistics of every view of the step + per-kernel breakdown (outside the timed regions) ----
    def view_stats(cam):
        with torch.no_grad():
            rs = dgr.GaussianRasterizationSettings(H, W, math.tan(cam.FoVx * 0.5), math.tan(cam.FoVy * 0.5), bg, 1.0,
                                                   cam.world_view_transform, cam.full_proj_transform, a.sh_degree,
                                                   cam.camera_center, False, False, False)
            _, radii, _, pack = dgr._forward_impl(pc.get_xyz.detach(), pc.get_features.detach(), None, pc.get_opacity.detach().reshape(-1),
                                                  pc.get_scaling.detach(), pc.get_rotation.detach(), None, rs)
            sv = dgr.state_views(pack, H, W)
            lens = (sv["ranges"][:, 1] - sv["ranges"][:, 0]).float()
            nc = sv["n_contrib"]
            gy, gx = (H + 15) // 16, (W + 15) // 16
            pad = torch.zeros(gy * 16, gx * 16, dtype=nc.dtype, device=dev)
            pad[:H, :W] = nc
            tile_max = pad.view(gy, 16, gx, 16).permute(0, 2, 1, 3).reshape(gy * gx, 256).max(dim=1).values
            return {"P_visible": int((radii > 0).sum().item()), "D": int(pack["num_rendered"]), "D_visited_bwd": int(tile_max.sum().item()),
                    "tile_list_mean": float(lens.mean().item()), "tile_list_max": int(lens.max().item()),
                    "n_contrib_mean": float(nc.float().mean().item())}
    per_view = [view_stats(c) for c in cams]
    stats = dict(per_view[0])
    stats["all_views"] = {"D": [p["D"] for p in per_view], "D_visited_bwd": [p["D_visited_bwd"] for p in per_view]}
    dgr.set_option("time_kernels", 2)
    dgr.kernel_time("", reset=True)
    for _ in range(2):
        step(False)
    torch.cuda.synchronize()
    breakdown = {}
    for name in ("preprocess_fwd", "sort_hist", "sort_rowscan", "sort_scatter", "scan_reduce", "scan_partials",
                 "scan_apply", "count_max", "emit", "tile_ranges", "ranges_from_counts", "tile_order", "render_fwd", "render_bwd",
                 "preprocess_bwd", "adam_step"):
        t, n = dgr.kernel_time(name)
        breakdown[name] = round(t / (2 * V), 4)
    dgr.kernel_time("", reset=True)
    dgr.set_option("time_kernels", 0)

    if world > 1:
        dist.barrier()
    if peer_bucket is not None:
        torch.cuda.synchronize()
        peer_bucket.close()
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel (render_bwd); byte counts per DESIGN.md section 4 ----
    # One launch blends all V views of the step.  Algorithmic bytes: per visited instance id 4 + record 48 + 10 float atomics 40;
    # per pixel n_contrib 4 + dL/dcolor 12 + forward colour 12.  Forward: id 4 + record 48; per pixel colour 12 + depth 4 + T 4 + count 4.
    npix = H * W
    batched_launch = a.api == "views" and not a.no_batch
    dv_sum = sum(p["D_visited_bwd"] for p in per_view)
    views_per_launch = V if batched_launch else 1
    bytes_bwd = (dv_sum * (4 + 48 + 40) + V * npix * 28) * views_per_launch // V
    bytes_fwd = (dv_sum * (4 + 48) + V * npix * 24) * views_per_launch // V
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_kind = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6.65 TB/s (B200_PROFILING.md)"
    traffic, prof = None, {}
    try:
        prof = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        traffic = prof.get("render_bwd_dram_bytes_per_launch")
    except Exception:
        pass
    bwd_avg_ms = bwd_ms / max(1, bwd_n)
    fwd_avg_ms = fwd_ms / max(1, fwd_n)
    achieved = bytes_bwd / (bwd_avg_ms * 1e-3) / 1e9 if bwd_avg_ms > 0 else 0.0
    roofline = {"kernel": "render_bwd", "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": traffic, "peak_kind": peak_kind,
                "algorithmic_bytes_per_launch": bytes_bwd, "views_per_launch": views_per_launch, "avg_launch_ms": bwd_avg_ms,
                "launches_timed": bwd_n,
                # what actually bounds the blend kernels (DESIGN.md section 4): warp instructions issued (ncu count of the
                # committed capture) over the live launch time, against 148 SMs x 4 schedulers x the sampled SM clock
                "issue": (lambda wi, ms, mhz: None if not (wi and ms and mhz) else
                          {"warp_instructions_per_launch": wi, "achieved_ginstr_s": wi / ms / 1e6,
                           "peak_ginstr_s": 148 * 4 * mhz / 1e3, "frac": (wi / ms / 1e6) / (148 * 4 * mhz / 1e3)})(
                    prof.get("render_bwd_warp_instructions_per_launch"), bwd_avg_ms, (clocks or {}).get("sm_mhz")),
                "render_fwd": {"avg_launch_ms": fwd_avg_ms, "algorithmic_bytes_per_launch": bytes_fwd,
                               "achieved": bytes_fwd / (fwd_avg_ms * 1e-3) / 1e9 if fwd_avg_ms > 0 else 0.0,
                               "frac": (bytes_fwd / (fwd_avg_ms * 1e-3) / 1e9 / peak) if fwd_avg_ms > 0 else 0.0}}

    cpu = None
    if not a.no_cpu_baseline and world == 1:
        from oracle.c_oracle import set_threads
        if hasattr(os, "sched_setaffinity"):
            try:                        # the GPU legs ran pinned to the GPU's NUMA node; the CPU port gets every core of the box
                os.sched_setaffinity(0, range(os.cpu_count() or 1))
            except OSError:
                pass
        set_threads(len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1))
        cs = oracle_settings(cams[0], a.sh_degree)
        t0 = time.perf_counter()
        times, nthreads = cpu_reference_pass(scene, cs, 1)
        reps = int(max(0, min(3, (a.cpu_baseline_seconds - (time.perf_counter() - t0)) // max(times[0], 1e-3))))
        if reps > 0:
            more, _ = cpu_reference_pass(scene, cs, reps)
            times += more
        cpu = {"value": (H * W / 1e6) * len(times) / sum(times), "unit": UNIT, "cores": nthreads, "kind": "port",
               "sample": f"{len(times)} full view(s) of the same workload, forward+backward, oracle/gs_oracle.c",
               "host_cpus": os.cpu_count()}

    cfg = workload_config(a, world)
    cfg.update({"sync_free": capacity is not None, "grad_chunks": grad_chunks if world > 1 else 1,
                "reduction": "fused reduce-scatter over peer memory + all-gather" if peer_bucket is not None else "one NCCL all-reduce",
                "pinned_cores": None if not pinned_cores else f"{pinned_cores[0]}-{pinned_cores[-1]} ({len(pinned_cores)})",
                "instance_capacity": None if capacity is None else capacity.capacity})
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": a.steps, "warmup": max(a.warmup, 3), "warmup_run": warmup_run,
            "ms_per_step": ms_total / a.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": cfg, "roofline": roofline,
            "cpu_baseline": cpu, "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d,
                                         "d2h_bytes_per_step": d2h, "ms_per_step": ms_e2e / a.steps,
                                         "d2h_is": "the step's loss scalar (float32)",
                                         "h2d_is": "per view: 3xHxW float32 target image + camera matrices, from pinned host memory"},
            "single_view": single_view,
            "gpu_launches": launches, "clocks": clocks,
            "step_ms": {"resident": step_stats.get(False), "e2e": step_stats.get(True)},
            "attempts": {"resident": attempts, "e2e": e2e_attempts,
                         "rule": "one timed region per leg; it is repeated only if the sync-free path's instance capacity turned out "
                                 "too small (capacity_ok false), never because of timing"},
            "scene_stats": stats, "kernel_ms_per_view": breakdown}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
