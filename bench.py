#!/usr/bin/env python
"""bench.py — the hot path of BASELINE.json measured on its own configurations.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config 2|3|4|5] [--batch B] [--full]
                    [--dump-outputs DIR]

--config (default 2 = configs[1], the configuration the metric is quoted on):
  2  rgbd_imagenet_adm_128_large_cfg, unconditional view, DDPM 1000 steps + classifier-free guidance 0.5, batch 16 / GPU
  3  config 2 + a second view: viewset `random`, device warp, rgbd_imagenet_adm_128_large_cond (InpaintCFG) 50 guided DDIM steps
  4  viewset `3x9`: 27 views / sample (26 conditional views, 351 source-view rasterisations), device warp
  5  rgbd_imagenet_adm_256_128_small_sr (SuperResCFG), 256x256, 50 DDIM steps + guidance, batch 8 / GPU
Synthetic class labels, synthetic seeded N(0, 1/fan_in) weights (the reference zero-initialises its last layers), synthetic
smooth RGBD source views for the warp phase.

One bench "step" = ONE denoising step of the whole batch of every network the configuration runs (batch-2N UNet forward
with both guidance halves + fused eps mix + x_{t-1} update; configs 3/4: one step of the unconditional AND one of the
conditional model).  The steps of a sample are homogeneous (same kernels, same shapes; only the table row differs), so

    seconds / sample-batch = n_uncond_steps * t_uncond + n_cond_views * 50 * t_cond + t_warp        (stated in `config`)

with t_warp the device time of the complete warp sequence of the view set (add_view + aggregate for every view), measured
on its own with CUDA events.  `--full` runs the complete pipeline instead (one bench step = one finished sample batch).

N>1: launched by torchrun, one rank per GPU; samples shard by batch (no data-path collective), weights are packed on rank 0
and broadcast once with NCCL.  Timing: CUDA events on the launching stream, barrier + synchronize on both sides, max
over ranks.  `--impl reference`: the reference's CPU path (oracle port; the Python reference cannot travel to the GPU
box) on the host cores, same configuration, bounded sample.

`--dump-outputs DIR`: after the timed steps, rank 0 writes what the last timed step returned, as float32 DIR/<name>.npy:
uncond_/cond_pred_x_prev and uncond_/cond_pred_x_0 per network, or `samples` under --full.  Inputs and weights are seeded,
so two builds run with the same arguments can be compared output for output.  Above 64 MiB in all, every array keeps the
same seeded choice of batch entries.
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

_BASE = dict(out_channels=4, num_res_blocks=2, num_groups=32, num_heads=None, num_head_channels=64, dropout=0.0,
             channel_mult=[1, 1, 2, 3, 4])
MODELS = {   # backbone args of the reference's configs/*.json
    "L": dict(_BASE, image_size=128, in_channels=4, model_channels=256, num_classes=1000, has_null_class=True,
              attention_resolutions=[32, 16, 8], use_fp16=False),       # rgbd_imagenet_adm_128_large_cfg
    "Lc": dict(_BASE, image_size=128, in_channels=10, model_channels=256, num_classes=1000, has_null_class=True,
               attention_resolutions=[32, 16, 8], use_fp16=True),       # rgbd_imagenet_adm_128_large_cond
    "SR": dict(_BASE, image_size=256, in_channels=8, model_channels=128, num_classes=1000, has_null_class=True,
               attention_resolutions=[64, 32, 16], use_fp16=True),      # rgbd_imagenet_adm_256_128_small_sr
}
GFLOP_PER_FORWARD = {"L": 613.8, "Lc": 614.2, "SR": 697.8}        # per sample (SURVEY.md §8d)
GUIDANCE = 0.5            # README.md:90 evaluation protocol
DENOISE_STEPS = 1000
COND_STEPS = 50
WARP_KW = dict(fov=45, near=0.6, far=5, atol=0.03, rtol=0.03, erode_rgb=3)      # inference/sample.py:258-263
DUMP_LIMIT = 64 << 20     # bytes written by --dump-outputs

WORKLOADS = {
    2: dict(name="rgbd_imagenet_adm_128_large_cfg uncond, DDPM 1000 steps + classifier-free guidance 0.5 (BASELINE configs[1])",
            batch=16, views=1, uncond="L", cond=None),
    3: dict(name="imagenet128 uncond+cond iterative, viewset=random (2 views), 1000 DDPM + 50 DDIM steps, guidance 0.5 (BASELINE configs[2])",
            batch=16, views=2, uncond="L", cond="Lc"),
    4: dict(name="viewset=3x9 (27 views / sample, 26 conditional views x 50 DDIM steps), on-device RGBD warp, guidance 0.5 (BASELINE configs[3])",
            batch=16, views=27, uncond="L", cond="Lc"),
    5: dict(name="rgbd_imagenet_adm_256_128_small_sr super-resolution, 256x256, 50 DDIM steps + guidance 0.5 (BASELINE configs[4])",
            batch=8, views=1, uncond=None, cond="SR"),
}


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d.get("hbm_gbs", 6650.0), tf_burst=d.get("bf16_tflops", 1590.0),
                    tf_sust=d.get("bf16_tflops_sustained", 1400.0), src="measured (MEASURED_PEAKS.json)")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sust=1400.0, src="fallback (B200_PROFILING.md)")


def synth_rgbd(rng, n=128):
    """Smooth synthetic RGBD view in [0,1] (z-buffer depth): a height field with one foreground blob."""
    yy, xx = np.mgrid[0:n, 0:n] / n
    z = 0.55 + 0.08 * np.sin(6.0 * xx + rng.uniform(0, 6)) * np.cos(5.0 * yy + rng.uniform(0, 6))
    cx, cy, r = rng.uniform(0.35, 0.65), rng.uniform(0.35, 0.65), rng.uniform(0.15, 0.25)
    z = np.where((xx - cx) ** 2 + (yy - cy) ** 2 < r ** 2, z - 0.18, z)
    rgb = np.stack([0.5 + 0.5 * np.sin(9 * xx + i) * np.cos(7 * yy - i) for i in range(3)], axis=-1)
    return np.concatenate([rgb, z[..., None]], axis=-1).astype(np.float32)


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons.  The process is started BEFORE the warm-up (nvidia-smi needs ~0.2 s to
    deliver its first row) and every row is stamped when it arrives; `stop()` keeps the rows that fall inside the timed region
    marked by `mark_start()` .. `stop()` (short regions: the rows closest to it)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.rows, self.proc, self.index = [], None, index
        self.t0 = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), [c.strip() for c in line.split(",")]))

    def mark_start(self):
        self.t0 = time.perf_counter()

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        t1 = time.perf_counter()
        time.sleep(0.12)                      # let the row that covers the end of the region arrive
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        t0 = self.t0 if self.t0 is not None else 0.0
        inside = [r for (t, r) in self.rows if t0 <= t <= t1 + 0.12]
        if not inside and self.rows:          # region shorter than the sampling period: the rows nearest to it
            inside = [r for (t, r) in sorted(self.rows, key=lambda tr: abs(tr[0] - 0.5 * (t0 + t1)))[:2]]
        sm, mx, reasons = [], [], set()
        for r in inside:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
                for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def dump_outputs(out_dir, tensors):
    """Writes each [B, ...] tensor as float32 <out_dir>/<name>.npy; above DUMP_LIMIT in all, the same seeded choice of batch
    entries from each."""
    arrays = {k: v.detach().float().cpu().numpy() for k, v in tensors.items()}
    total = sum(a.nbytes for a in arrays.values())
    n = min(a.shape[0] for a in arrays.values())
    keep = slice(None)
    if total > DUMP_LIMIT:
        keep = np.sort(np.random.default_rng(0).choice(n, max(1, n * DUMP_LIMIT // total), replace=False))
        print(f"[bench] --dump-outputs: {total / 2**20:.0f} MiB > {DUMP_LIMIT >> 20} MiB, keeping batch entries {keep.tolist()}",
              file=sys.stderr)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a[keep])


def seconds_per_batch(wl, t_u, t_c, t_warp):
    """Composition rule of the module docstring (seconds per finished sample batch)."""
    s = 0.0
    if wl["uncond"]:
        s += DENOISE_STEPS * t_u
    if wl["cond"]:
        s += max(wl["views"] - 1, 1 if wl["uncond"] is None else 0) * COND_STEPS * t_c
    return s + t_warp


# ----------------------------------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the CPU oracle port of the reference path (the Python reference cannot travel)
# ----------------------------------------------------------------------------------------------------------------------
def pick_threads(unit):
    """Thread count that is actually fastest for `unit()` (one UNet forward of the configuration's first network at batch 1) on
    this host: oversubscribed SMT threads slow oneDNN down, and a single-conv probe is too noisy (it picked 16 in one process
    and 32 in the next on the same box, a 1.6x difference in the result).  One warm run + two timed runs per candidate."""
    avail = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    best, cores = None, 1
    for nt in sorted({min(avail, c) for c in (8, 16, 32, 64)}):
        torch.set_num_threads(nt)
        unit()
        t0 = time.perf_counter()
        unit(); unit()
        dt = time.perf_counter() - t0
        if best is None or dt < best * 0.93:       # prefer fewer threads unless clearly faster
            best, cores = dt, nt
    torch.set_num_threads(cores)
    return cores


def cpu_reference(config, steps, warmup, budget_s):
    """Times the CPU oracle port on a bounded sample of the workload: `steps` denoising steps of each network at batch 1
    (after >= `warmup` warm steps, at least one), plus — configs 3/4 — one CPU warp (mesh build + software rasteriser +
    aggregate_conditions) per distinct source count.  Returns (samples_per_s, description dict)."""
    from oracle import sampler_ref, unet_ref
    wl = WORKLOADS[config]
    tb = sampler_ref.Tables(sampler_ref.get_betas("linear", 1000))
    g = torch.Generator().manual_seed(0)
    phases = [k for k in ("uncond", "cond") if wl[k]]
    cores = None
    per_phase_budget = budget_s * (0.85 if wl["views"] == 1 else 0.7) / len(phases)
    times, counts = {}, {}
    for ph in phases:
        key = wl[ph]
        cfg = MODELS[key]
        sd = unet_ref.make_synthetic_state_dict(cfg, seed=1234 if ph == "uncond" else 4321)
        model = lambda x, t, c: unet_ref.unet_forward(cfg, sd, x, t, c)
        S = cfg["image_size"]
        x = torch.randn(1, 4, S, S, generator=g)
        classes = torch.tensor([7])
        if cores is None:
            xin = torch.randn(1, cfg["in_channels"], S, S, generator=g)
            cores = pick_threads(lambda: model(xin, torch.tensor([500]), classes))
        if key == "Lc":
            y = torch.randn(1, 4, S, S, generator=g); m = (torch.rand(1, 1, S, S, generator=g) > 0.3).float()
        elif key == "SR":
            y = torch.randn(1, 4, S // 2, S // 2, generator=g)
        state = {"x": x}

        def one(i):
            xx = state["x"]
            if key == "L":
                t = torch.tensor([999 - i])
                eps = sampler_ref.cfg_eps(model, xx, t, classes, GUIDANCE)
                state["x"], _ = sampler_ref.ddpm_step(tb, xx, t, eps, torch.randn(xx.shape, generator=g))
                return
            t = torch.tensor([1000 - 20 * i]); tp = t - 20
            if key == "Lc":
                z = torch.randn(1, 4, S, S, generator=g)
                inp = sampler_ref.make_inpaint_inputs(xx, y, m, m, z[:, :3], z[:, 3:])
                eps = sampler_ref.cond_eps(model, inp, t - 1, classes, GUIDANCE)
                state["x"], _ = sampler_ref.ddim_step(tb, xx, t, tp, eps, torch.zeros_like(xx), replace_rgb=(0.1, y[:, :3], m),
                                                      replace_depth=(0.2, y[:, 3:], m), constrain_depth=(0.5, y[:, 3:]))
            else:
                eps = sampler_ref.cond_eps(model, sampler_ref.make_sr_inputs(xx, y), t - 1, classes, GUIDANCE)
                state["x"], _ = sampler_ref.ddim_step(tb, xx, t, tp, eps, torch.zeros_like(xx))

        t0 = time.perf_counter(); one(0); first = time.perf_counter() - t0          # cold step: never timed
        n_warm = max(1, min(warmup, int(per_phase_budget * 0.25 / max(first, 1e-3))))
        for i in range(n_warm):
            one(1 + i)
        n = max(1, min(steps, int(per_phase_budget * 0.6 / max(first, 1e-3))))
        t0 = time.perf_counter()
        for i in range(n):
            one(1 + n_warm + i)
        times[ph] = (time.perf_counter() - t0) / n
        counts[ph] = n
        del sd
    t_warp = 0.0
    warp_note = ""
    if wl["views"] > 1:
        from oracle import warp_ref
        rng = np.random.default_rng(0)
        views = [warp_ref.view_on_sphere(0.0, 0.0), warp_ref.view_on_sphere(0.15, 0.0)]      # the first two cameras of the view set
        kw = dict(WARP_KW)
        rgbd = synth_rgbd(rng)
        t0 = time.perf_counter()
        mesh = warp_ref.depth_to_mesh(warp_ref.linearize_depth(rgbd[:, :, 3:], kw["near"], kw["far"]), fov=kw["fov"],
                                      modelview=np.asarray(views[0], np.float64), atol=kw["atol"], rtol=kw["rtol"], erode_rgb=kw["erode_rgb"])
        t_mesh = time.perf_counter() - t0
        rend = warp_ref.SoftwareAggregationRenderer(384, 128)
        t0 = time.perf_counter()
        warp_ref.aggregate_conditions(rend, [mesh], [rgbd[:, :, :3]], np.asarray(views[1], np.float64), **kw)
        t_agg1 = time.perf_counter() - t0
        # the software renderer rasterises every source view for every target: cost is linear in the source count
        V = wl["views"]
        t_warp = V * t_mesh + t_agg1 * sum(range(1, V))
        warp_note = f"; CPU warp: 1 mesh build ({t_mesh * 1e3:.0f} ms) + 1 aggregate with 1 source ({t_agg1 * 1e3:.0f} ms), scaled linearly to {sum(range(1, V))} source-view rasterisations"
    sec = seconds_per_batch(wl, times.get("uncond", 0.0), times.get("cond", 0.0), t_warp)      # batch 1
    desc = {"cores": cores, "kind": "port",
            "sample": ", ".join(f"{counts[ph]} {wl[ph]} denoising steps (guidance, 2 forwards each)" for ph in phases) +
                      f" at batch 1, fp32 torch CPU, {cores} threads" + warp_note,
            "ms_per_step": {ph: times[ph] * 1e3 for ph in phases}}
    return 1.0 / sec, desc


def run_reference(args):
    if int(os.environ.get("RANK", "0")) != 0:
        return
    value, desc = cpu_reference(args.config, args.steps, max(args.warmup, 1), budget_s=120.0)
    wl = WORKLOADS[args.config]
    line = {
        "impl": "reference", "metric": "128x128 RGBD multiview samples/sec", "value": value, "unit": "samples/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": sum(desc["ms_per_step"].values()),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": wl["name"] + " — CPU oracle port of the reference path", "batch": 1,
                   "denoise_steps_per_sample": DENOISE_STEPS if wl["uncond"] else COND_STEPS,
                   "timed_unit": "one denoising step of each network (2 UNet forwards each)", "phase_ms": desc["ms_per_step"]},
        "cpu_baseline": {"value": value, "unit": "samples/s", "cores": desc["cores"], "kind": "port", "sample": desc["sample"]},
        "e2e": {"value": value, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ----------------------------------------------------------------------------------------------------------------------
def _ncu_traffic():
    """DRAM bytes of ONE named launch of the dominant conv kernel (the 128x128 256->256 conv with fp32 + fp16 outputs and
    residual) from the committed `ncu --set full` capture, or (None, None)."""
    import glob
    files = sorted(glob.glob(os.path.join(ROOT, "profiles", "ncu_full_*_conv_summary.json")))
    if not files:
        return None, None
    unit = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
    best = None
    for k in json.load(open(files[-1])):
        try:
            b = 0.0
            for key in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
                v, u = k[key].split()
                b += float(v.replace(",", "")) * unit[u]
            if best is None or b > best:
                best = b           # the residual conv (conv2) is the larger of the two captured launches
        except (KeyError, ValueError):
            continue
    if best is None:
        return None, None
    return best, f"{os.path.relpath(files[-1], ROOT)}: the 128x128 256->256 conv2 launch (fp32 + fp16 outputs + fp32 residual; algorithmic 1.61 GB)"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=2, choices=[2, 3, 4, 5])
    ap.add_argument("--batch", type=int, default=None, help="samples per GPU (default: the configuration's, 16 / 8)")
    ap.add_argument("--full", action="store_true", help="one bench step = a complete sample batch (all steps, all views)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned as float32 DIR/<name>.npy (module docstring)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        return run_reference(args)
    args.warmup = max(args.warmup, 3) if not args.full else args.warmup
    wl = WORKLOADS[args.config]
    B = args.batch or wl["batch"]

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))

    # CPU baseline first (rank 0, N=1 only): same procedure as the reference arm, before this process touches the GPU, so the
    # thread probe and the warm-up steps see an idle host
    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        v, desc = cpu_reference(args.config, 5, 3, budget_s=120.0)     # same procedure and sample as `--impl reference --steps 5 --warmup 3`
        cpu = {"value": v, "unit": "samples/s", "cores": desc["cores"], "kind": "port", "sample": desc["sample"]}

    assert torch.cuda.is_available(), "bench.py needs a GPU (no CPU fallback in the product path)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = None
    if world > 1:
        import torch.distributed as dist_
        dist = dist_
        dist.init_process_group("nccl", device_id=dev)

    from ivid_b200 import _lib
    import ivid_b200.backbones as backbones
    import ivid_b200.frameworks as frameworks
    import ivid_b200.samplers as samplers
    from ivid_b200.inference.sample import build_modelviews, sample_all
    from ivid_b200.rgbd_3d import DeviceWarp
    from oracle import unet_ref   # only for the synthetic weight generator + cpu_baseline leg

    bcast_ms = []

    def make_net(key, seed):
        cfg = MODELS[key]
        net = backbones.AdmUnet2d(**cfg)
        if rank == 0:
            net.load_state_dict(unet_ref.make_synthetic_state_dict(cfg, seed=seed))
        net = net.cuda()
        net.repack()
        if world > 1:
            # weights: packed on rank 0, ONE NCCL broadcast of the device arena over NVLink (sample.py:186-195 loads per rank)
            ptr, nbytes = net.weight_arena()

            class _Arena:
                __cuda_array_interface__ = {"shape": (nbytes,), "typestr": "|u1", "data": (ptr, False), "version": 3}
            arena = torch.as_tensor(_Arena(), device=dev)
            torch.cuda.synchronize(); dist.barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); dist.broadcast(arena, src=0); e1.record(); torch.cuda.synchronize()
            bcast_ms.append(e0.elapsed_time(e1))
        return net

    gen = torch.Generator().manual_seed(1000 + rank)
    classes_host = (torch.arange(B) + rank * B) % 1000
    classes = classes_host.to(dev)
    fw_u = fw_c = s_u = s_c = None
    if wl["uncond"]:
        fw_u = frameworks.ClassifierFreeGuidance(make_net(wl["uncond"], 1234), timesteps=1000, beta_schedule="linear", p_uncond=0.1)
        s_u = samplers.DdpmSampler(fw_u)
    if wl["cond"] == "Lc":
        fw_c = frameworks.InpaintCFG(make_net("Lc", 4321), timesteps=1000, beta_schedule="linear")
        s_c = samplers.DdimSampler(fw_c)
    elif wl["cond"] == "SR":
        fw_c = frameworks.SuperResCFG(make_net("SR", 4321), timesteps=1000, beta_schedule="linear")
        s_c = samplers.DdimSampler(fw_c)
    S = MODELS[wl["uncond"] or wl["cond"]]["image_size"]
    x_host = torch.randn(B, 4, S, S, generator=gen).pin_memory()
    x = x_host.to(dev)

    # conditional-model inputs: the condition maps of a real warp of synthetic source views (configs 3/4), low-res RGBD (5)
    rng = np.random.default_rng(7 + rank)
    cond_kw, cond_host = {}, {}
    warp = None
    views = build_modelviews("3x9", 1) if wl["views"] > 1 else None
    src = None
    if wl["cond"] == "Lc":
        src = torch.from_numpy(np.stack([synth_rgbd(rng).transpose(2, 0, 1) * 2 - 1 for _ in range(B)])).float().to(dev)
        warp = DeviceWarp(B, image_size=128, ssaa=3, max_views=max(wl["views"], 2), device=local)
        warp.add_view(src, views[0], **WARP_KW)
        c7 = warp.aggregate(views[1], **WARP_KW)
        y = (c7[:, 0:4] * 2 - 1).contiguous(); m = c7[:, 4:5].contiguous(); mr = c7[:, 5:6].contiguous(); cv = (c7[:, 6:7] * 2 - 1).contiguous()
        cond_kw = dict(y=y, mask=m, mask_rgb=mr, replace_rgb=(0.1, y[:, :3].contiguous(), mr), replace_depth=(0.2, y[:, 3:].contiguous(), m),
                       constrain_depth=(0.5, cv))
        cond_host = {k: v.cpu().pin_memory() for k, v in dict(y=y, mask=m, mask_rgb=mr, convex=cv).items()}
    elif wl["cond"] == "SR":
        y = torch.randn(B, 4, S // 2, S // 2, generator=gen).to(dev)
        cond_kw = dict(y=y)
        cond_host = {"y": y.cpu().pin_memory()}
    kw = {"strength": GUIDANCE}
    last = {}     # network -> the latest step's result (pred_x_prev, pred_x_0), for --dump-outputs

    def step_u(xc, i):
        last["uncond"] = s_u._native_step(xc, (DENOISE_STEPS - 1 - i) % DENOISE_STEPS, 0, classes, False, 0.0, kw, None, None)
        return last["uncond"].pred_x_prev

    def step_c(xc, i):
        k = i % COND_STEPS
        last["cond"] = s_c._native_step(xc, 1000 - 20 * k, 980 - 20 * k, classes, False, 0.0, dict(kw, **cond_kw), None, None)
        return last["cond"].pred_x_prev

    def full_batch():
        if args.config == 2:
            return s_u.sample(B, noise=x, classes=classes, strength=GUIDANCE, verbose=False).samples
        if args.config == 5:
            return s_c.sample(B, noise=x, classes=classes, steps=COND_STEPS, strength=GUIDANCE, verbose=False, **cond_kw).samples
        mvs = build_modelviews("random", B, rng=np.random.default_rng(3)) if args.config == 3 else views
        # every finished sample's views: [B, V, 4, H, W]
        return torch.stack([out[2] for out in sample_all(fw_u, fw_c, B, DENOISE_STEPS, COND_STEPS, mvs,
                                                         classes=[int(c) for c in classes_host], guidance=GUIDANCE,
                                                         batchsize=B, **WARP_KW)])

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    ev = lambda: torch.cuda.Event(enable_timing=True)
    # ---- warm-up ----
    clocks = ClockSampler(local) if rank == 0 else None
    if clocks:
        clocks.start()
    xu = xc = x
    for i in range(args.warmup):
        if args.full:
            xu = full_batch()
        else:
            if s_u: xu = step_u(xu, i)
            if s_c: xc = step_c(xc, i)
    # ---- timed region: K steps ----
    barrier()
    if clocks:
        clocks.mark_start()
    e0, e1 = ev(), ev()
    marks = []
    e0.record()
    for i in range(args.steps):
        if args.full:
            xu = full_batch()
            continue
        a = ev(); a.record()
        if s_u: xu = step_u(xu, args.warmup + i)
        b = ev(); b.record()
        if s_c: xc = step_c(xc, args.warmup + i)
        c = ev(); c.record()
        marks.append((a, b, c))
    e1.record()
    barrier()
    ms_total = e0.elapsed_time(e1)
    clk = clocks.stop() if clocks else None
    t_u = sum(a.elapsed_time(b) for a, b, _ in marks) / max(len(marks), 1) / 1e3
    t_c = sum(b.elapsed_time(c) for _, b, c in marks) / max(len(marks), 1) / 1e3
    finite = bool(torch.isfinite(xu).all() and torch.isfinite(xc).all())
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"samples": xu} if args.full else
                     {f"{net}_{k}": r[k] for net, r in last.items() for k in ("pred_x_prev", "pred_x_0")})

    # ---- the warp sequence of the view set (device time, CUDA events; configs 3/4, not under --full) ----
    t_warp, warp_info = 0.0, None
    if warp is not None and not args.full:
        V = wl["views"]
        reps = 2
        agg_ms, add_ms = [], []
        for rep in range(reps + 1):                      # first repetition = warm-up
            warp.reset()
            a_tot = d_tot = 0.0
            for j in range(V):
                if j > 0:
                    a, b = ev(), ev(); a.record(); c7 = warp.aggregate(views[j], **WARP_KW); b.record(); torch.cuda.synchronize()
                    a_tot += a.elapsed_time(b)
                a, b = ev(), ev(); a.record(); warp.add_view(src, views[j], **WARP_KW); b.record(); torch.cuda.synchronize()
                d_tot += a.elapsed_time(b)
            if rep > 0:
                agg_ms.append(a_tot); add_ms.append(d_tot)
        t_warp = (min(agg_ms) + min(add_ms)) / 1e3
        # algorithmic bytes (SURVEY §8d): per (sample, target) with j sources: j*(4*128^2*4 + 384^2*8*2) + 7*128^2*4
        alg = sum(B * (j * (4 * 128 * 128 * 4 + 384 * 384 * 16) + 7 * 128 * 128 * 4) for j in range(1, V))
        warp_info = {"aggregate_ms_total": min(agg_ms), "add_view_ms_total": min(add_ms), "source_view_rasterisations": B * sum(range(1, V)),
                     "algorithmic_GB": alg / 1e9, "achieved_GBs": alg / 1e9 / (min(agg_ms) / 1e3),
                     "frac_of_hbm_peak": alg / 1e9 / (min(agg_ms) / 1e3) / _peaks()["hbm"], "mask_coverage_last_view": float(c7[:, 4].mean())}

    def reduce_max(v):
        if dist is None:
            return v
        tt = torch.tensor([v], device=dev, dtype=torch.float64)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        return float(tt.item())
    ms_total, t_u, t_c, t_warp = reduce_max(ms_total), reduce_max(t_u), reduce_max(t_c), reduce_max(t_warp)
    ms_per_step = ms_total / args.steps
    if args.full:
        value = world * B / (ms_per_step / 1e3)
    else:
        value = world * B / seconds_per_batch(wl, t_u, t_c, t_warp)

    # ---- e2e: the public API call a user makes, host buffers, H2D + D2H inside the timed region ----
    out_host = torch.empty(B, 4, S, S).pin_memory()
    t_host = torch.full((B,), 500, dtype=torch.int64)

    def to_dev(d):
        return {k: v.to(dev, non_blocking=True) for k, v in d.items()}

    def e2e_u():
        r = s_u.sample_once(x_host.to(dev, non_blocking=True), t_host.to(dev, non_blocking=True), classes_host.to(dev, non_blocking=True),
                            strength=GUIDANCE)
        out_host.copy_(r.pred_x_prev, non_blocking=True)
        torch.cuda.current_stream().synchronize()

    def e2e_c():
        xd = x_host.to(dev, non_blocking=True); cd = classes_host.to(dev, non_blocking=True)
        td = t_host.to(dev, non_blocking=True)
        h = to_dev(cond_host)
        if wl["cond"] == "Lc":
            r = s_c.sample_once(xd, td, td - 20, cd, strength=GUIDANCE, y=h["y"], mask=h["mask"], mask_rgb=h["mask_rgb"],
                                replace_rgb=(0.1, h["y"][:, :3], h["mask_rgb"]), replace_depth=(0.2, h["y"][:, 3:], h["mask"]),
                                constrain_depth=(0.5, h["convex"]))
        else:
            r = s_c.sample_once(xd, td, td - 20, cd, strength=GUIDANCE, y=h["y"])
        out_host.copy_(r.pred_x_prev, non_blocking=True)
        torch.cuda.current_stream().synchronize()

    if args.full:
        e2e_value, h2d, d2h = value, x_host.numel() * 4 + classes_host.numel() * 8, out_host.numel() * 4
        e2e_api = "same run: DdpmSampler / DdimSampler.sample (sample_all for the multiview configurations) from host noise, samples read back"
    else:
        for _ in range(2):
            if s_u: e2e_u()
            if s_c: e2e_c()
        barrier()
        tu = tc = 0.0
        for _ in range(args.steps):
            t0 = time.perf_counter()
            if s_u: e2e_u()
            t1 = time.perf_counter()
            if s_c: e2e_c()
            t2 = time.perf_counter()
            tu += t1 - t0; tc += t2 - t1
        barrier()
        tu, tc = reduce_max(tu / args.steps), reduce_max(tc / args.steps)
        e2e_value = world * B / seconds_per_batch(wl, tu, tc, t_warp)
        nb = lambda t: t.numel() * t.element_size()
        h2d = (nb(x_host) + nb(classes_host) + nb(t_host)) * (int(bool(s_u)) + int(bool(s_c))) + sum(nb(v) for v in cond_host.values())
        d2h = nb(out_host) * (int(bool(s_u)) + int(bool(s_c)))
        e2e_api = "Ddpm/DdimSampler.sample_once(x_t, t[, t_prev], classes, strength[, y, mask, ...]) from pinned host tensors, x_{t-1} read back to host"

    # ---- roofline of the dominant kernel (per-launch CUDA events inside the library, one profiled step) ----
    L = _lib.lib()
    net_p = (fw_u or fw_c).backbone
    key_p = wl["uncond"] or wl["cond"]
    _lib.check(L.ivid_unet_profile_begin(net_p._handle))
    (step_u if s_u else step_c)(x, 1)
    buf = ctypes.create_string_buffer(1 << 19)
    _lib.check(L.ivid_unet_profile_end(net_p._handle, buf, len(buf)))
    prof = json.loads(buf.value.decode())
    per_op = prof.pop("_ops", None)
    if per_op is not None and rank == 0:
        # outside the tree, which may be read-only
        path = os.path.join(tempfile.gettempdir(), f"ivid_per_op_profile_c{args.config}.json")
        with open(path, "w") as f:
            json.dump(per_op, f)
        print(f"[bench] per-launch profile: {path}", file=sys.stderr)
    peaks = _peaks()
    dom = max((k for k in prof if k.startswith("conv_gemm")), key=lambda k: prof[k]["ms"])
    d = prof[dom]
    ach = d["flops"] / (d["ms"] * 1e-3) / 1e12
    step_ms_prof = sum(v["ms"] for v in prof.values())
    traffic, traffic_src = _ncu_traffic()
    roofline = {"bound": "tensor", "kernel": dom, "achieved": ach, "peak": peaks["tf_sust"], "unit": "TFLOP/s",
                "frac": ach / peaks["tf_sust"], "traffic": traffic, "traffic_unit": "DRAM bytes of the named launch", "traffic_source": traffic_src,
                "peak_source": peaks["src"] + ", bf16/fp16 dense sustained", "model": key_p,
                "launches_per_step": d["launches"], "kernel_share_of_step": d["ms"] / step_ms_prof,
                "families": {k: {"launches": v["launches"], "ms": round(v["ms"], 4),
                                 "tflops": (v["flops"] / (v["ms"] * 1e-3) / 1e12) if v["ms"] > 0 else None,
                                 "gbs": (v["bytes"] / (v["ms"] * 1e-3) / 1e9) if v["ms"] > 0 else None} for k, v in prof.items()}}
    if warp_info:
        roofline["warp"] = dict(warp_info, bound="hbm", peak=peaks["hbm"], unit="GB/s")
    kernels_per_forward = sum(v["launches"] for v in prof.values()) + 3       # "embed" ops = 3 + 2 kernels
    # one step = (memset + kernels) replayed as ONE CUDA graph + set_step + class fill + fused step kernel
    launches_per_step = (kernels_per_forward + 3) * (int(bool(s_u)) + int(bool(s_c)))

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return

    nets = [k for k in (wl["uncond"], wl["cond"]) if k]
    model_tf = None
    if not args.full:
        fl = 0.0
        if s_u: fl += 2 * B * GFLOP_PER_FORWARD[wl["uncond"]] / 1e3
        if s_c: fl += 2 * B * GFLOP_PER_FORWARD[wl["cond"]] / 1e3
        model_tf = fl / (t_u + t_c)
    line = {
        "metric": "128x128 RGBD multiview samples/sec", "value": value, "unit": "samples/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "fp16 tensor-core operands, fp32 accumulate / residual stream / GroupNorm / softmax / sampler",
        "data": "synthetic",
        "config": {"workload": wl["name"], "config_id": args.config, "models": nets,
                   "batch_per_gpu": B, "global_batch": B * world, "views_per_sample": wl["views"],
                   "denoise_steps_per_sample": {"uncond": DENOISE_STEPS if s_u else 0, "cond_per_view": COND_STEPS if s_c else 0},
                   "timed_unit": "complete sample batch (all steps, all views)" if args.full else
                                 "one denoising step of the batch of each network (batch-2N UNet forward + fused guidance mix / x_{t-1} update)",
                   "composition": None if args.full else "seconds/batch = 1000*t_uncond + (views-1)*50*t_cond + t_warp (module docstring)",
                   "phase_ms": None if args.full else {"uncond_step": t_u * 1e3, "cond_step": t_c * 1e3, "warp_sequence": t_warp * 1e3},
                   "unet_step_ms": None if args.full else (t_u or t_c) * 1e3,
                   "model_tflops_per_s": model_tf,
                   "parallelism": f"dp{world} (samples sharded by batch, no data-path collective)",
                   "l2": "per-step working set (0.84 GB weights + >2 GB activations) exceeds the 126 MB L2; no flush needed",
                   "weights_broadcast_ms": bcast_ms or None, "finite": finite},
        "roofline": roofline,
        "e2e": {"value": e2e_value, "unit": "samples/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "api": e2e_api},
        "gpu_launches": launches_per_step * args.steps * ((DENOISE_STEPS if s_u else COND_STEPS) if args.full else 1),
        "gpu_kernels_per_unet_forward": kernels_per_forward,
        "clocks": clk,
    }
    if cpu:
        line["cpu_baseline"] = cpu
    print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
