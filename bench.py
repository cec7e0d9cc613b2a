#!/usr/bin/env python
"""bench.py -- BASELINE.json's metric on BASELINE.json's config.

    python bench.py --gpus N --steps K --warmup W            # our CUDA path
    python bench.py --impl reference --gpus N --steps K ...   # the reference's CPU path (oracle port)
    python bench.py --gpus 1 --steps K --warmup W --dump-outputs DIR   # + what the last timed step computed, as .npy

Workload (config.workload): BASELINE.json configs[2] -- 1 006 065 Gaussians (the test_garden crop tiled
3x3, SURVEY.md section 8(d)), one 1920x1080 view per GPU, SH degree 3, dense (packed=False).
A "step" is one pass of the hot path: rasterization() forward (fused projection + SH, tile intersection,
radix sort, offsets, compositing) + L1 loss against a target image + backward to all five parameter
tensors; at N > 1 every rank renders its own view of the replicated scene and the Gaussian gradients are
all-reduced over NVLink by the library's own row-sparse kernel (NCCL where there is no symmetric memory; view-axis
data parallelism, weak scaling).  The optimizer is outside the path.

Printed line (rank 0): metric = rendered views/s (fwd+bwd), ms_per_step = train-step ms,
value = device-resident timing, e2e = same step with the per-step host->device copy of the camera and
the target image (uint8 HWC, converted on the device inside the timed region) from pinned memory, double-buffered on
a copy stream, and the device->host read of the loss inside the timed region.
roofline = dominant kernel (compositing backward) algorithmic bytes / CUDA-event time vs the measured
HBM peak; cpu_baseline = the CPU oracle port timed on this box's host cores.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

W_IMG, H_IMG, SH_DEGREE, SCENE_GRID = 1920, 1080, 3, 3
METRIC = "rendered views/sec, fwd+bwd train step (1M Gaussians, 1080p, SH3)"
UNIT = "views/s"


def workload_config(n_gpus: int) -> dict:
    return {
        "workload": "BASELINE configs[2]: synthetic 1M Gaussians (test_garden crop tiled 3x3 = 1006065), "
        "1 view 1920x1080 per GPU, SH3, packed=False, near=0.01 far=1e10 eps2d=0.3",
        "step": "rasterization fwd + L1 loss (fused l1_loss) + bwd to means/quats/scales/opacities/SH"
        + (" + all-reduce (SUM) of the Gaussian grads over NVLink" if n_gpus > 1 else ""),
        "views_per_step": n_gpus,
        "parallelism": f"view-axis DP x{n_gpus} (replicated Gaussians)" if n_gpus > 1 else "single GPU",
        "l2": "inputs (236 MB of Gaussian parameters + 25 MB target) exceed the 126 MB L2; no explicit flush",
    }


# --------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""

    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True,
            )
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def wait_ready(self, timeout: float = 5.0) -> None:
        """Blocks until nvidia-smi has delivered its first sample (its start-up is then over)."""
        t0 = time.time()
        while self.proc is not None and not self.rows and time.time() - t0 < timeout:
            time.sleep(0.02)

    def mark(self) -> None:
        """Samples taken before this call (nvidia-smi start-up, warm-up steps) are not reported."""
        self.first = len(self.rows)

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        rows = self.rows[getattr(self, "first", 0):] or self.rows
        for r in rows:
            try:
                sm.append(float(r[0]))
                mx = float(r[1])
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


def measured_peak_gbs() -> tuple[float, str]:
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


DUMP_ROWS = 65536  # Gaussians whose gradients --dump-outputs writes (the full SH gradient alone is 193 MB)


def dump_outputs(out_dir: str, render_colors, render_alphas, loss, grads: dict) -> None:
    """Writes what the timed step returns to its caller as float32 DIR/<name>.npy: render_colors, render_alphas, loss
    and v_<param>, the gradients of a fixed seeded sample of DUMP_ROWS Gaussians (their indices in gaussian_rows.npy,
    float64); about 50 MB at the default workload.  The inputs are seeded, so two builds can be compared file by file."""
    import torch

    os.makedirs(out_dir, exist_ok=True)
    n = grads["means"].shape[0]
    rows = np.sort(np.random.RandomState(0).choice(n, min(DUMP_ROWS, n), replace=False))
    idx = torch.from_numpy(rows).to(grads["means"].device)
    arrays = {"render_colors": render_colors, "render_alphas": render_alphas, "loss": loss.reshape(1)}
    arrays.update({"v_" + k: g[idx] for k, g in grads.items()})
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a.detach().float().cpu().numpy())
    np.save(os.path.join(out_dir, "gaussian_rows.npy"), rows.astype(np.float64))


def build_scene():
    from tests import scene

    sc = scene.make_scene(scene_grid=SCENE_GRID, sh_degree=SH_DEGREE)
    Ks = scene.rescale_K(sc["Ks"], sc["width"], sc["height"], W_IMG, H_IMG)
    return sc, Ks


# --------------------------------------------------------------------------------------------
def _host_threads() -> int:
    """Threads the OpenMP C oracle will really use.  torch.distributed.run exports OMP_NUM_THREADS=1 to its workers
    (round 1: the CPU arm under torchrun ran single-threaded while claiming 128 cores), so the arm sets the variable
    itself -- before libgomp is initialised -- and reports omp_get_max_threads()."""
    import ctypes

    want = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    os.environ["OMP_NUM_THREADS"] = str(want)
    os.environ.setdefault("OMP_PROC_BIND", "false")
    try:
        gomp = ctypes.CDLL("libgomp.so.1")
        gomp.omp_set_num_threads(want)
        return int(gomp.omp_get_max_threads())
    except OSError:
        return want


CPU_ARM_MAX_STEPS, CPU_ARM_MAX_WARMUP = 20, 5  # ~2 s per view on a 128-core host: the whole arm stays within ~1 min


def run_cpu_reference(steps: int, warmup: int, n_gpus: int, as_main_line: bool):
    """The reference's CPU implementation of the path: the C oracle port (oracle/), all host cores.
    One timed unit = fwd+bwd of ONE full view of the workload.  A step at N GPUs is N views; the host's throughput in
    views/s does not depend on N, so the arm times single views (a bounded sample: 1/N of a step) and reports
    value = views/s, ms_per_step = N x the per-view time."""
    threads = _host_threads()
    from oracle import gso

    gso.build()
    sc, Ks = build_scene()
    rng = np.random.RandomState(0)
    target = rng.random_sample((1, H_IMG, W_IMG, 3)).astype(np.float32)

    def step():
        fwd, _ = gso.rasterization_fwd_bwd(
            sc["means"], sc["quats"], sc["scales"], sc["opacities"], sc["sh"], sc["viewmats"][:1], Ks[:1], W_IMG, H_IMG,
            SH_DEGREE, None, None,
        )
        v_rc = np.sign(fwd["render_colors"] - target).astype(np.float32) / target.size
        gso.rasterization_fwd_bwd(
            sc["means"], sc["quats"], sc["scales"], sc["opacities"], sc["sh"], sc["viewmats"][:1], Ks[:1], W_IMG, H_IMG,
            SH_DEGREE, v_rc, np.zeros((1, H_IMG, W_IMG, 1), np.float32),
        )

    for _ in range(warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    dt = (time.perf_counter() - t0) / max(steps, 1)
    base = {
        "value": 1.0 / dt, "unit": UNIT, "cores": threads, "kind": "port",
        "sample": f"{steps} x one full 1080p view of the 1M-Gaussian workload (= 1/{n_gpus} of a step at {n_gpus} GPU(s)), "
        "fwd (twice: loss needs the render) + bwd, C oracle port, OpenMP threads = cores",
    }
    if not as_main_line:
        return base
    cfg = workload_config(n_gpus)
    cfg["reference_arm"] = f"CPU port on {threads} OpenMP threads, rank 0 only; steps/warm-up capped at {CPU_ARM_MAX_STEPS}/{CPU_ARM_MAX_WARMUP}"
    line = {
        "impl": "reference", "metric": METRIC, "value": 1.0 / dt, "unit": UNIT, "n_gpus": n_gpus, "steps": steps,
        "warmup": warmup, "ms_per_step": n_gpus * dt * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic", "config": cfg, "cpu_baseline": base,
        "e2e": {"value": 1.0 / dt, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# --------------------------------------------------------------------------------------------
def run_ref_cuda(params, vm, K, target, steps: int):
    """Extra information (not the contract's reference arm): the REAL reference's CUDA kernels
    (oracle/_ref/gsplat_ref.so, built by oracle/build_ref.py with the reference's release flags for
    sm_100a) chained as its orchestrator chains them (csrc/Rendering.cpp:976-1447) on the same inputs,
    forward ops + the matching *_bwd ops called by hand (no autograd / Python overhead -> a lower bound
    on the reference's train step).  Returns None when the library is absent."""
    import torch

    from oracle import refcuda

    if not refcuda.available():
        return None
    try:
        R = refcuda.load_ops()
        means, quats, scales, opac, sh = (params[k].detach() for k in ("means", "quats", "scales", "opacities", "sh"))
        tw, th = (W_IMG + 15) // 16, (H_IMG + 15) // 16
        op_cn = opac[None].contiguous()

        def step():
            radii, m2, dep, con, _ = R.projection_ewa_3dgs_fused(means, None, quats, scales, opac, vm, K, W_IMG, H_IMG, 0.3, 0.01, 1e10, 0.0, False, 0)
            valid = (radii > 0).all(-1)
            raw = R.spherical_harmonics(SH_DEGREE, means, vm, sh, valid, None, None, None, None)
            col = torch.clamp_min(raw + 0.5, 0.0)
            tpg, ids, fl = R.intersect_tile(m2, radii, dep, con, op_cn, None, None, 1, 16, tw, th, True, False)
            off = R.intersect_offset(ids, 1, tw, th)
            rc, ra, _, last = R.rasterize_to_pixels_3dgs(m2, con, col, op_cn, None, None, W_IMG, H_IMG, 16, off, fl, False, False)
            diff = rc - target
            loss = diff.abs().mean()
            v_rc = torch.sign(diff) / diff.numel()
            v_ra = torch.zeros_like(ra)
            rb = R.rasterize_to_pixels_3dgs_bwd(m2, con, col, op_cn, None, None, off, fl, ra, last, W_IMG, H_IMG, 16, False, v_rc, v_ra, False)
            v_col = rb[3] * (col > 0)
            sb = R.spherical_harmonics_bwd(SH_DEGREE, means, vm, sh, valid, None, None, None, None, v_col, True, False, False)
            pb = R.projection_ewa_3dgs_fused_bwd(means, None, quats, scales, vm, K, W_IMG, H_IMG, 0.3, 0, radii, con, None, rb[1], torch.zeros_like(dep), rb[2], None, False)
            v_means = pb[0] + sb[1]
            v_op = rb[4].sum(0)
            return loss, v_means, v_op, fl

        for _ in range(3):
            out = step()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            out = step()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / steps
        return {
            "what": "HAND-CHAINED: reference gsplat v1.6.0 CUDA kernels (sm_100a, -use_fast_math), ops called one by one, "
            "no autograd overhead (not the reference's stock path: see ref_cuda_stock)",
            "ms_per_step": ms, "views_per_s": 1e3 / ms, "n_isects": int(out[3].numel()),
        }
    except Exception as e:  # noqa: BLE001
        return {"error": f"{type(e).__name__}: {e}"[:300]}


# --------------------------------------------------------------------------------------------
def run_ref_cuda_stock(params, vm, K, target, steps: int, scale_mul: float = 1.0):
    """The reference's STOCK path on the same step: the unmodified Python package installed in baseline/_ref
    (baseline/install_ref.py) -- gsplat.rasterization() -> torch.ops.gsplat.rasterization_3dgs
    (csrc/Rendering.cpp:745-1481, fused assemble_proj_features, the reference's registered autograd) -- plus the
    torch L1 loss and loss.backward().  This is the comparator north_star's 1.5x target is about; `ref_cuda`
    (hand-chained ops) stays beside it as a lower bound without autograd overhead."""
    import torch

    try:
        from oracle import refcuda

        if not refcuda.package_available():
            return None
        gsplat = refcuda.import_package()
        p = {k: v.detach().clone().requires_grad_(True) for k, v in params.items()}
        scales = p["scales"] if scale_mul == 1.0 else (p["scales"].detach() * scale_mul).requires_grad_(True)

        def step():
            for t in list(p.values()) + [scales]:
                t.grad = None
            rc, ra, meta = gsplat.rasterization(
                p["means"], p["quats"], scales, p["opacities"], p["sh"], vm, K, W_IMG, H_IMG, sh_degree=SH_DEGREE, packed=False,
            )
            loss = (rc - target).abs().mean()
            loss.backward()
            return meta

        for _ in range(3):
            meta = step()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            meta = step()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / steps
        return {
            "path": "gsplat.rasterization() (baseline/_ref, unmodified reference v1.6.0: rasterization_3dgs orchestrator + its autograd) "
            "+ torch L1 + backward",
            "ms_per_step": ms, "views_per_s": 1e3 / ms, "n_isects": int(meta["flatten_ids"].numel()),
        }
    except Exception as e:  # noqa: BLE001
        return {"error": f"{type(e).__name__}: {e}"[:300]}


def run_big_s(params, vm, K, target, steps: int, scale_mul: float = 4.0):
    """Second driver-timed workload (VERDICT round 1, item 4): the same scene with the Gaussians' scales x4 -- about
    9x the tile intersections (S = 20 M instead of 2.3 M), the regime of trained 1080p scenes, where the tile
    intersection / sort stage and the record pack weigh as much as compositing.  Same step as the headline
    (rasterization fwd + fused L1 + bwd), ours and the reference's stock path, CUDA events."""
    import torch

    import gsplat_b200

    p = {k: v.detach().clone().requires_grad_(True) for k, v in params.items()}
    scales = (p["scales"].detach() * scale_mul).requires_grad_(True)

    def step():
        for t in list(p.values()) + [scales]:
            t.grad = None
        rc, _, meta = gsplat_b200.rasterization(
            p["means"], p["quats"], scales, p["opacities"], p["sh"], vm, K, W_IMG, H_IMG, sh_degree=SH_DEGREE, packed=False,
        )
        gsplat_b200.l1_loss(rc, target).backward()
        return meta

    for _ in range(3):
        meta = step()
    torch.cuda.synchronize()
    e = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    e[0].record()
    for _ in range(steps):
        meta = step()
    e[1].record()
    with torch.no_grad():
        for _ in range(steps):
            gsplat_b200.rasterization(
                p["means"], p["quats"], scales, p["opacities"], p["sh"], vm, K, W_IMG, H_IMG, sh_degree=SH_DEGREE, packed=False,
            )
    e[2].record()
    torch.cuda.synchronize()
    out = {
        "workload": f"BASELINE configs[2] scene with scales x{scale_mul:g} (1 006 065 Gaussians, 1 view 1920x1080, SH3)",
        "n_isects": int(meta["flatten_ids"].numel()),
        "ms_per_step": e[0].elapsed_time(e[1]) / steps, "fwd_only_ms": e[1].elapsed_time(e[2]) / steps,
    }
    del p, scales, meta
    torch.cuda.empty_cache()
    ref = run_ref_cuda_stock(params, vm, K, target, steps, scale_mul=scale_mul)
    out["ref_cuda_stock_ms_per_step"] = None if not ref else ref.get("ms_per_step", ref.get("error"))
    if ref and ref.get("ms_per_step"):
        out["speedup_vs_ref_cuda_stock"] = ref["ms_per_step"] / out["ms_per_step"]
    return out


# DefaultStrategy.grow_grad2d of the cfg5 runs.  The reference's default (2e-4) is tuned for real captures; on the synthetic
# targets the densification statistic is much smaller (tools/trainer_bench.py --grad-stats at the first refinement:
# median 1.4e-7, p95 2.3e-5, p99 9.2e-5), so 2e-4 would grow the scene by 0.3 % per refinement instead of cfg5's 1M -> 3M
TRAINER_GROW_GRAD2D = 1e-5


def run_trainer_bench(steps: int):
    """cfg5 (BASELINE configs[4]): the simple_trainer.py loop on both backends of the installed reference package,
    default and MCMC strategies (tools/trainer_bench.py, one subprocess per run).  Returns the `trainer` object."""
    import subprocess as sp

    tool = os.path.join(ROOT, "tools", "trainer_bench.py")
    out = {}
    arms = (("ref", ["--backend", "reference"]), ("ours", ["--backend", "b200"]),
            ("ours_raster_only", ["--backend", "b200", "--no-fused-losses"]),
            ("ref_with_our_fused_ssim", ["--backend", "reference", "--fused-ssim-only"]))
    for strat in ("default", "mcmc"):
        runs = {}
        for name, flags in arms:
            try:
                extra = ["--grow-grad2d", str(TRAINER_GROW_GRAD2D)] if strat == "default" else []
                r = sp.run([sys.executable, tool, *flags, "--strategy", strat, "--steps", str(steps), "--breakdown", *extra],
                           capture_output=True, text=True, timeout=900)
                line = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
                runs[name] = json.loads(line[-1]) if line else {"error": (r.stderr or r.stdout)[-400:]}
            except Exception as e:  # noqa: BLE001
                runs[name] = {"error": f"{type(e).__name__}: {e}"[:300]}
        ref = runs["ref"]

        def ratio(key, a):
            return (a[key] / ref[key]) if ("error" not in a and "error" not in ref and a.get(key) and ref.get(key)) else None

        pick = lambda key: {k: v.get(key) for k, v in runs.items()}  # noqa: E731
        out[strat] = {
            "it_per_s": pick("it_per_s_total"), "it_per_s_at_1M": pick("it_per_s_at_1M"),
            "speedup_total": {k: ratio("it_per_s_total", v) for k, v in runs.items() if k != "ref"},
            "speedup_at_1M": {k: ratio("it_per_s_at_1M", v) for k, v in runs.items() if k != "ref"},
            "n_gaussians_end": pick("n_gaussians_end"), "n_isects_last": pick("n_isects_last"),
            "breakdown_ms": pick("breakdown_ms"),
            "final_loss": {k: (v.get("loss_hist") or [[None, None]])[-1][1] for k, v in runs.items()},
            "steps": steps, "untimed_warm_steps": ref.get("untimed_warm_steps"), "schedule": runs["ours"].get("schedule"),
            "errors": {k: v["error"] for k, v in runs.items() if "error" in v} or None,
        }
    out["what"] = ("examples/simple_trainer.py:795-1198 restated on synthetic 1080p targets (tools/trainer_bench.py): 1M -> 3M "
                   "Gaussians, L1 + SSIM, 6 fused Adam, reference strategies; `ref` = unmodified package (no third-party fused_ssim "
                   "in this image: its ssim_loss runs the torch conv2d path), `ours` = same package after gsplat_b200.dropin.apply() "
                   "(rasterization + fused SSIM), `ours_raster_only` = drop-in with the package's own torch SSIM kept, "
                   "`ref_with_our_fused_ssim` = the reference's rasterization with only the fused SSIM swapped in (what the reference "
                   "would do with its third-party fused_ssim hook): ours / ref_with_our_fused_ssim isolates the rasterizer")
    return out


# --------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-trainer", action="store_true", help="skip the cfg5 trainer-loop runs (about 2 minutes)")
    ap.add_argument("--trainer-steps", type=int, default=700)
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        if rank == 0:
            run_cpu_reference(max(1, min(args.steps, CPU_ARM_MAX_STEPS)), min(args.warmup, CPU_ARM_MAX_WARMUP), args.gpus, True)
        return

    import torch
    import torch.distributed as dist

    import gsplat_b200
    from gsplat_b200 import distributed as D
    from gsplat_b200 import ops

    assert torch.cuda.is_available(), "bench.py needs a GPU (no CPU fallback exists)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        # NCCL_DEBUG is left as the launcher set it (the driver reads NCCL's communicator lines); the gradient
        # all-reduce data plane is our own kernel over symmetric memory, NCCL only carries barriers / small metadata
        dist.init_process_group("nccl", device_id=dev)
    n_gpus = world

    sc, Ks = build_scene()
    N = sc["means"].shape[0]
    params = {
        k: torch.from_numpy(sc[k]).to(dev).requires_grad_(True) for k in ("means", "quats", "scales", "opacities", "sh")
    }
    cam = rank % sc["viewmats"].shape[0]
    vm_host = torch.from_numpy(sc["viewmats"][cam : cam + 1].copy()).pin_memory()
    K_host = torch.from_numpy(Ks[cam : cam + 1].copy()).pin_memory()
    rng = np.random.RandomState(100 + rank)
    target_host = torch.from_numpy(rng.random_sample((1, H_IMG, W_IMG, 3)).astype(np.float32)).pin_memory()
    vm_dev, K_dev, target_dev = vm_host.to(dev), K_host.to(dev), target_host.to(dev)
    # e2e ships the target image the way datasets store it -- uint8 HWC, 6.2 MB instead of 24.9 MB of float32 -- and
    # converts it on the device INSIDE the timed region: measured on this pool the pinned H2D path gives ~17 GB/s, so the
    # float32 image (1.48 ms per copy) was what bounded e2e, not the step (GSB200_E2E_TARGET=f32 restores it)
    e2e_u8 = os.environ.get("GSB200_E2E_TARGET", "u8") != "f32"
    target_host_u8 = (target_host * 255.0).round().clamp_(0, 255).to(torch.uint8).pin_memory() if e2e_u8 else None
    loss_host = torch.empty((), dtype=torch.float32).pin_memory()
    h2d_bytes = vm_host.numel() * 4 + K_host.numel() * 4 + (target_host_u8.numel() if e2e_u8 else target_host.numel() * 4)
    d2h_bytes = 4
    grad_names = ("means", "quats", "scales", "opacities", "sh")

    # N > 1: the gradient all-reduce is our own kernel over NVSwitch peer memory (csrc/nvls.cu): the fused backward
    # writes the gradients straight into a symmetric buffer, one launch reduces it in place on every rank.
    # NCCL (coalesced, in place) is the fallback when the system has no symmetric / multicast memory.
    arena, allreduce_kind = None, "none"
    if world > 1:
        allreduce_kind = "nccl (coalesced, in place)"
        if os.environ.get("GSB200_ALLREDUCE", "own") != "nccl":
            try:
                arena = D.NvlsGradArena({k: params[k] for k in grad_names})
                ops.set_gradient_allocator(arena.allocator)
                allreduce_kind = f"own kernel over symmetric memory ({arena.algo}, {arena.blocks} blocks)"
            except Exception as e:  # noqa: BLE001
                if rank == 0:
                    print(f"[bench] symmetric-memory all-reduce unavailable ({type(e).__name__}: {e}); using NCCL", file=sys.stderr)

    def all_reduce_grads():
        if arena is not None:
            arena.all_reduce()
        else:
            D.all_reduce_gaussian_grads([params[k] for k in grad_names], coalesced=True)

    # e2e input pipeline: every step's camera + target image are copied from pinned host memory inside
    # the timed region, double-buffered on a side stream so that the copy of step i+1 overlaps the compute
    # of step i (what a DataLoader with pin_memory + non_blocking does); step i waits for ITS copy.
    copy_stream = torch.cuda.Stream(device=dev)
    dev_in = [
        (torch.empty_like(vm_dev), torch.empty_like(K_dev),
         torch.empty(target_dev.shape, dtype=torch.uint8, device=dev) if e2e_u8 else torch.empty_like(target_dev))
        for _ in range(2)
    ]
    copy_done = [torch.cuda.Event(), torch.cuda.Event()]
    consumed = [torch.cuda.Event(), torch.cuda.Event()]

    def issue_copy(slot: int):
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(consumed[slot])  # the previous user of this slot has finished
            dev_in[slot][0].copy_(vm_host, non_blocking=True)
            dev_in[slot][1].copy_(K_host, non_blocking=True)
            dev_in[slot][2].copy_(target_host_u8 if e2e_u8 else target_host, non_blocking=True)
            copy_done[slot].record(copy_stream)

    last_out = {}  # outputs of the latest step, kept only for --dump-outputs

    def step(e2e: bool, slot: int = 0):
        if e2e:
            torch.cuda.current_stream().wait_event(copy_done[slot])
            vm, K, tgt = dev_in[slot]
            if e2e_u8:
                tgt = tgt.to(torch.float32).mul_(1.0 / 255.0)  # uint8 -> [0, 1] float on the device, part of the timed step
        else:
            vm, K, tgt = vm_dev, K_dev, target_dev
        for p in params.values():
            p.grad = None
        rc, ra, meta = gsplat_b200.rasterization(
            params["means"], params["quats"], params["scales"], params["opacities"], params["sh"], vm, K, W_IMG, H_IMG,
            sh_degree=SH_DEGREE, packed=False,
        )
        loss = gsplat_b200.l1_loss(rc, tgt)  # == (rc - tgt).abs().mean(), fused (losses.py)
        loss.backward()
        if world > 1:
            all_reduce_grads()  # the 59 floats / Gaussian (SURVEY.md section 8e), one launch, in place
        if args.dump_outputs:
            last_out.update(render_colors=rc, render_alphas=ra, loss=loss)
        if e2e:
            consumed[slot].record()
            loss_host.copy_(loss.detach(), non_blocking=True)
        return meta

    host_issue_ms = {}

    def timed(e2e: bool, steps: int) -> float:
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        t_host = time.perf_counter()
        if e2e:
            for c in consumed:
                c.record()
            issue_copy(0)  # the first copy is inside the timed region too
            for i in range(steps):
                if i + 1 < steps:
                    issue_copy((i + 1) & 1)
                step(True, i & 1)
        else:
            for _ in range(steps):
                step(False)
        e1.record()
        host_issue_ms[e2e] = (time.perf_counter() - t_host) * 1e3 / steps  # host time to ISSUE a step (diagnostic)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    # nvidia-smi is started, and waited for, BEFORE the warm-up: its start-up (NVML init touches every GPU of the
    # box) must not fall into the timed region; it then polls GPU 0 every 100 ms; only samples taken after the
    # warm-up are reported
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        sampler.wait_ready()
    if world > 1:
        dist.barrier()
    for c in consumed:
        c.record()
    for i in range(max(args.warmup, 3)):  # the warm-up runs right before the timed region: clocks are up
        meta = step(False)
        issue_copy(i & 1)
        step(True, i & 1)
    torch.cuda.synchronize()
    if rank == 0:
        sampler.mark()
    ms_dev = timed(False, args.steps)
    ms_e2e = timed(True, args.steps)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, **last_out, grads={k: params[k].grad for k in grad_names})

    # ---- N > 1 diagnostics (outside the timed regions): where a DP step spends its time on every rank, and the
    # same job (world views / step over the same Gaussians, every gradient summed over all views) laid out the
    # reference's way -- Gaussians sharded across ranks, projected rows exchanged by all-to-all, no all-reduce.
    dp_info = None
    if world > 1:
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
        comp, comm, nccl = [], [], []
        for _ in range(5):
            dist.barrier()
            torch.cuda.synchronize()
            ev[0].record()
            for p in params.values():
                p.grad = None
            rc, _, _ = gsplat_b200.rasterization(
                params["means"], params["quats"], params["scales"], params["opacities"], params["sh"], vm_dev, K_dev, W_IMG,
                H_IMG, sh_degree=SH_DEGREE, packed=False,
            )
            gsplat_b200.l1_loss(rc, target_dev).backward()
            ev[1].record()
            all_reduce_grads()
            ev[2].record()
            D.all_reduce_gaussian_grads([params[k] for k in grad_names], coalesced=True)  # NCCL on the same payload
            ev[3].record()
            torch.cuda.synchronize()
            comp.append(ev[0].elapsed_time(ev[1]))
            comm.append(ev[1].elapsed_time(ev[2]))
            nccl.append(ev[2].elapsed_time(ev[3]))
        mine = torch.tensor([sorted(comp)[2], sorted(comm)[2], sorted(nccl)[2]], device=dev)
        allr = [torch.empty_like(mine) for _ in range(world)]
        dist.all_gather(allr, mine)
        # ---- correctness of the N > 1 data plane, checked in the run the driver times (VERDICT round 1, item 7)
        checks = {}
        for p in params.values():
            p.grad = None
        rc, _, _ = gsplat_b200.rasterization(
            params["means"], params["quats"], params["scales"], params["opacities"], params["sh"], vm_dev, K_dev, W_IMG, H_IMG,
            sh_degree=SH_DEGREE, packed=False,
        )
        gsplat_b200.l1_loss(rc, target_dev).backward()
        want = {k: params[k].grad.detach().clone() for k in grad_names}
        for w in want.values():
            dist.all_reduce(w, op=dist.ReduceOp.SUM)  # NCCL on copies of the very same per-rank gradients
        if arena is not None:
            arena.stats.zero_() if getattr(arena, "stats", None) is not None else None
        all_reduce_grads()
        torch.cuda.synchronize()
        err = torch.tensor([max(float((params[k].grad - want[k]).abs().max()) for k in grad_names)], device=dev)
        mag = torch.tensor([max(float(want[k].abs().max()) for k in grad_names)], device=dev)
        dist.all_reduce(err, op=dist.ReduceOp.MAX)
        dist.all_reduce(mag, op=dist.ReduceOp.MAX)
        checks["own_allreduce_vs_nccl_max_abs"] = float(err.item())
        checks["grad_max_abs"] = float(mag.item())
        if arena is not None and getattr(arena, "stats", None) is not None:
            moved = arena.stats.clone()
            dist.all_reduce(moved)
            checks["allreduce_payload_fraction_moved"] = float(moved.item()) * 16 / float(sum(params[k].numel() for k in grad_names) * 4)
        del want
        ops.set_gradient_allocator(None)
        bounds = [int(round(i * N / world)) for i in range(world + 1)]
        shard = {k: params[k].detach()[bounds[rank] : bounds[rank + 1]].clone().requires_grad_(True) for k in params}

        def sharded_step(packed):
            for p in shard.values():
                p.grad = None
            rc, _, _ = gsplat_b200.rasterization(
                shard["means"], shard["quats"], shard["scales"], shard["opacities"], shard["sh"], vm_dev, K_dev, W_IMG, H_IMG,
                sh_degree=SH_DEGREE, packed=packed, distributed=True,
            )
            gsplat_b200.l1_loss(rc, target_dev).backward()

        # gaussian-sharded render of this rank's camera must equal the single-GPU render of all gaussians, bit for bit
        with torch.no_grad():
            rc_full, ra_full, _ = gsplat_b200.rasterization(
                params["means"], params["quats"], params["scales"], params["opacities"], params["sh"], vm_dev, K_dev, W_IMG, H_IMG,
                sh_degree=SH_DEGREE, packed=False,
            )
            rc_sh, ra_sh, _ = gsplat_b200.rasterization(
                shard["means"], shard["quats"], shard["scales"], shard["opacities"], shard["sh"], vm_dev, K_dev, W_IMG, H_IMG,
                sh_degree=SH_DEGREE, packed=False, distributed=True,
            )
            same = torch.tensor([int(torch.equal(rc_full, rc_sh) and torch.equal(ra_full, ra_sh))], device=dev)
            dist.all_reduce(same, op=dist.ReduceOp.MIN)
            checks["sharded_vs_single_bitexact"] = bool(same.item())
            del rc_full, ra_full, rc_sh, ra_sh
        sharded = {}
        for packed in (False, True):
            for _ in range(3):
                sharded_step(packed)
            dist.barrier()
            torch.cuda.synchronize()
            ev[0].record()
            for _ in range(args.steps):
                sharded_step(packed)
            ev[1].record()
            torch.cuda.synchronize()
            dist.barrier()
            ms_sh = torch.tensor([ev[0].elapsed_time(ev[1])], device=dev)
            dist.all_reduce(ms_sh, op=dist.ReduceOp.MAX)
            sharded["packed" if packed else "dense"] = {
                "value": n_gpus * args.steps / (float(ms_sh.item()) * 1e-3), "unit": UNIT,
                "ms_per_step": float(ms_sh.item()) / args.steps,
            }
        dp_info = {
            "per_rank_compute_ms": [round(float(t[0]), 3) for t in allr],
            "per_rank_allreduce_ms": [round(float(t[1]), 3) for t in allr],
            "per_rank_nccl_allreduce_ms": [round(float(t[2]), 3) for t in allr],
            "allreduce": allreduce_kind + (f" [{arena.last_kind}]" if arena is not None and getattr(arena, "last_kind", None) else ""),
            "exposed_allreduce_ms": round(ms_dev / args.steps - max(float(t[0]) for t in allr), 3),
            "compute_skew_ms": round(max(float(t[0]) for t in allr) - min(float(t[0]) for t in allr), 3),
            "checks": checks,
            "allreduce_bytes_per_rank": int(sum(params[k].numel() for k in grad_names) * 4),
            "gaussian_sharded": dict(
                what="same job with rasterization(distributed=True): Gaussians sharded, all-to-all of the projected rows "
                "(dense: all C*N rows; packed: only the visible rows of the compacting projection), no all-reduce",
                **sharded,
            ),
        }

    # ---- roofline of the dominant kernels, timed alone with CUDA events on the launching stream
    S = int(meta["flatten_ids"].numel())
    P, T = W_IMG * H_IMG, meta["tile_width"] * meta["tile_height"]
    det = {k: meta[k].detach().requires_grad_(True) for k in ("means2d", "conics")}
    with torch.no_grad():
        colors = ops.fused_project_sh(
            params["means"], params["quats"], params["scales"], params["opacities"], params["sh"], vm_dev, K_dev, W_IMG,
            H_IMG, SH_DEGREE,
        )[4]
    colors = colors.detach().requires_grad_(True)
    opac = meta["opacities"].detach().contiguous().requires_grad_(True)
    v_rc = torch.randn((1, H_IMG, W_IMG, 3), device=dev)

    def time_kernel(fn, reps=10):
        fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / reps

    def raster_fwd():
        return ops.rasterize_to_pixels(
            det["means2d"], det["conics"], colors, opac, W_IMG, H_IMG, 16, meta["isect_offsets"], meta["flatten_ids"]
        )

    ms_rfwd = time_kernel(raster_fwd)
    rc_keep, _ = raster_fwd()

    def raster_bwd():
        torch.autograd.grad((rc_keep,), (det["means2d"], det["conics"], colors, opac), (v_rc,), retain_graph=True)

    ms_rbwd = time_kernel(raster_bwd)
    peak, peak_src = measured_peak_gbs()
    bytes_fwd, bytes_bwd = 40 * S + 20 * P + 4 * T, 76 * S + 24 * P + 4 * T
    traffic = None
    tp = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    if os.path.exists(tp):
        try:
            traffic = json.load(open(tp)).get("raster_bwd_dram_bytes")
        except Exception:
            traffic = None
    achieved = bytes_bwd / (ms_rbwd * 1e-3) / 1e9
    roofline = {
        "kernel": "raster_bwd2_kernel<3,false,4,pipe> (+ zero-init of the gradient records)", "bound": "hbm", "achieved": achieved,
        "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
        "algorithmic_bytes": bytes_bwd, "ms": ms_rbwd, "n_isects": S,
        "note": "compositing is FP32/MUFU-bound, not HBM-bound (SURVEY.md section 8d): the HBM fraction is reported as "
        "required, pair throughput below is the meaningful figure",
        "raster_fwd": {"ms": ms_rfwd, "achieved": bytes_fwd / (ms_rfwd * 1e-3) / 1e9, "algorithmic_bytes": bytes_fwd},
        # compute-side figure (SURVEY.md section 8d): candidate (pixel, gaussian) pairs = 256 per (tile, gaussian)
        # intersection; the kernels are instruction-issue bound (profiles/r02_v7_ncu.md: 77 % / 93 % issue-active)
        "pairs": {
            "candidate_pairs": 256 * S,
            "bwd_gpairs_per_s": 256 * S / (ms_rbwd * 1e-3) / 1e9,
            "fwd_gpairs_per_s": 256 * S / (ms_rfwd * 1e-3) / 1e9,
            "issue_peak_ginst_per_s": 148 * 4 * 1.965,
            "issue_evidence": "profiles/r02_v7_ncu.md (smsp__issue_active 77 % / 93 %, smsp__inst_executed: 418 M backward, 251 M forward)",
        },
    }

    if rank == 0:
        cpu_base, ref_cuda, ref_stock, trainer, big_s = None, None, None, None, None
        if n_gpus == 1:
            ref_cuda = run_ref_cuda(params, vm_dev, K_dev, target_dev, args.steps)
            ref_stock = run_ref_cuda_stock(params, vm_dev, K_dev, target_dev, args.steps)
            try:
                big_s = run_big_s(params, vm_dev, K_dev, target_dev, args.steps)
            except Exception as e:  # noqa: BLE001
                big_s = {"error": f"{type(e).__name__}: {e}"[:300]}
            if not args.no_trainer:
                del colors, opac, rc_keep, det
                torch.cuda.empty_cache()
                trainer = run_trainer_bench(args.trainer_steps)
        if n_gpus == 1 and not args.no_cpu_baseline:
            cpu_base = run_cpu_reference(2, 1, 1, False)
        line = {
            "metric": METRIC, "value": n_gpus * args.steps / (ms_dev * 1e-3), "unit": UNIT, "n_gpus": n_gpus,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_dev / args.steps,
            "host_issue_ms_per_step": host_issue_ms.get(False),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": dict(workload_config(n_gpus), **({"allreduce": allreduce_kind} if n_gpus > 1 else {})),
            "e2e": {
                "value": n_gpus * args.steps / (ms_e2e * 1e-3), "unit": UNIT, "ms_per_step": ms_e2e / args.steps,
                "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": d2h_bytes,
                "host_issue_ms_per_step": host_issue_ms.get(True),
                "input": ("target image shipped as uint8 HWC from pinned memory and converted to float on the device inside "
                          "the timed region" if e2e_u8 else "target image shipped as float32 HWC from pinned memory"),
            },
            # our own kernels per step (profiles/r02_v9_launches.csv): project_sh_fwd (+ tile counts + row records),
            # publish_totals, depth_key_rows_bounded, isect_emit_coop, isect_offsets_tilekeys, pack_rows, tile_order,
            # raster_fwd, l1 partial/final/bwd, raster_bwd2, project_sh_bwd (= 13; the cub select / scan / radix-sort launches
            # made by the library are not counted); timed region = `steps` device-resident + `steps` e2e steps
            "gpu_launches": args.steps * 2 * (13 + (1 if arena is not None else 0)),
            "clocks": clocks, "roofline": roofline, "cpu_baseline": cpu_base, "ref_cuda_stock": ref_stock,
            "ref_cuda": ref_cuda, "big_s": big_s, "trainer": trainer, "dp": dp_info,
        }
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
