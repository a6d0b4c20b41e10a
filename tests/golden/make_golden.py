"""Generate the golden fixtures under tests/golden/ by running the UNMODIFIED reference (imported from /root/reference,
build container only) and pin the oracle restatement (oracle/*.py) against it.

    python tests/golden/make_golden.py            # writes tests/golden/*.npz, asserts oracle == reference

The fixtures are small (tiny UNet configs, a few steps) and are what the GPU box compares against — /root/reference
does not exist there.  Weights are not stored: they are regenerated from numpy PCG64 seeds
(oracle.unet_ref.make_synthetic_state_dict).
"""
from __future__ import annotations

import json
import os
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
REF = os.environ.get("IVID_REF", "/root/reference")
sys.path.insert(0, ROOT)

# easydict shim: the only import of the reference's diffusion package that is missing here (SURVEY.md §8c)
if "easydict" not in sys.modules:
    m = types.ModuleType("easydict")

    class EasyDict(dict):
        def __init__(self, d=None, **kw):
            super().__init__()
            for k, v in dict(d or {}, **kw).items():
                self[k] = v

        def __getattr__(self, k):
            try:
                return self[k]
            except KeyError as e:
                raise AttributeError(k) from e

        def __setattr__(self, k, v):
            self[k] = v

    m.EasyDict = EasyDict
    sys.modules["easydict"] = m
sys.path.insert(0, REF)

import diffusion.backbones as ref_backbones   # noqa: E402
import diffusion.frameworks as ref_frameworks  # noqa: E402
import diffusion.samplers as ref_samplers      # noqa: E402

from oracle import sampler_ref, unet_ref       # noqa: E402

TINY = dict(image_size=32, in_channels=4, model_channels=64, out_channels=4, num_res_blocks=1,
            attention_resolutions=[16, 8], channel_mult=[1, 2, 2], num_classes=10, has_null_class=True,
            num_groups=32, num_heads=None, num_head_channels=64, dropout=0.0, use_fp16=False)
TINY_COND = dict(TINY, in_channels=10)
TINY_SR = dict(TINY, in_channels=8, image_size=32, attention_resolutions=[8])


def ref_model(cfg, sd):
    args = {k: v for k, v in cfg.items()}
    net = ref_backbones.AdmUnet2d(**args)
    missing = net.load_state_dict(sd, strict=True)
    net.eval()
    return net


def rel(a, b):
    return float((a - b).norm() / b.norm().clamp_min(1e-30))


class FixedNoise:
    """Replays a queue of pre-drawn tensors through torch.randn_like inside the reference code."""

    def __init__(self, queue):
        self.queue = list(queue)
        self.orig = torch.randn_like

    def __enter__(self):
        def fake(x, *a, **k):
            t = self.queue.pop(0)
            assert t.shape == x.shape, (t.shape, x.shape)
            return t
        torch.randn_like = fake
        return self

    def __exit__(self, *exc):
        torch.randn_like = self.orig


def main():
    torch.manual_seed(0)
    torch.set_num_threads(8)
    out = {}
    rng = np.random.default_rng(7)

    # ---------------- schedule known-answer values (SURVEY.md Appendix C) ----------------
    betas = sampler_ref.get_betas("linear", 1000)
    fw = ref_frameworks.GaussianDiffusion(torch.nn.Identity(), timesteps=1000, beta_schedule="linear") if False else None
    ref_betas = ref_frameworks.utils.get_betas_by_name("linear", 1000).astype(np.float64)
    assert np.array_equal(betas, ref_betas)
    tb = sampler_ref.Tables(betas)

    class _FW:  # minimal framework surface the reference samplers read (.betas)
        pass
    f = _FW(); f.betas = ref_betas; f.timesteps = 1000
    rd = ref_samplers.DdpmSampler(f)
    ri = ref_samplers.DdimSampler(f)
    for name in ["alphas_cumprod", "alphas_cumprod_prev", "sqrt_recip_alphas_cumprod", "sqrt_recipm1_alphas_cumprod",
                 "posterior_variance", "posterior_log_variance_clipped", "posterior_mean_coef1", "posterior_mean_coef2"]:
        assert np.array_equal(getattr(tb, name), getattr(rd, name)), name
        out["sched_" + name] = getattr(rd, name)
    assert np.array_equal(tb.alphas_cumprod, ri.alphas_cumprod)
    out["sched_betas"] = ref_betas

    # ---------------- UNet forward: oracle vs reference, tiny configs ----------------
    for tag, cfg in [("tiny", TINY), ("tiny_cond", TINY_COND), ("tiny_sr", TINY_SR)]:
        sd = unet_ref.make_synthetic_state_dict(cfg, seed=1234)
        net = ref_model(cfg, sd)
        assert list(net.state_dict().keys()) == list(unet_ref.unet_param_shapes(cfg).keys()), "state-dict key order"
        N = 3
        x = torch.from_numpy(rng.standard_normal((N, cfg["in_channels"], cfg["image_size"], cfg["image_size"])).astype(np.float32))
        t = torch.tensor([999, 500, 3])
        classes = torch.tensor([1, -1, 7])
        with torch.no_grad():
            y_ref = net(x, t, classes)
            y_ref_none = net(x, t, None)
        y_or = unet_ref.unet_forward(cfg, sd, x, t, classes)
        y_or_none = unet_ref.unet_forward(cfg, sd, x, t, None)
        e1, e2 = rel(y_or, y_ref), rel(y_or_none, y_ref_none)
        print(f"[{tag}] oracle vs reference forward: rel {e1:.2e} (classes) {e2:.2e} (None); eps std {float(y_ref.std()):.3f}")
        assert e1 < 2e-6 and e2 < 2e-6
        # x is not stored: these are the first draws of the seed-7 stream, and tests/conftest.py regenerates them
        out[f"{tag}_t"] = t.numpy(); out[f"{tag}_classes"] = classes.numpy()
        out[f"{tag}_eps"] = y_ref.numpy(); out[f"{tag}_eps_none"] = y_ref_none.numpy()
        out[f"{tag}_cfg"] = np.frombuffer(json.dumps(cfg).encode(), dtype=np.uint8)

    # ---------------- state-dict schema of the real configs ----------------
    for name in ["rgbd_imagenet_adm_128_large_cfg", "rgbd_imagenet_adm_128_large_cond",
                 "rgbd_singlecategory_adm_128_small", "rgbd_imagenet_adm_256_128_small_sr"]:
        cfg = json.load(open(os.path.join(REF, "configs", name + ".json")))["backbone"]["args"]
        with torch.device("meta"):
            net = ref_backbones.AdmUnet2d(**cfg)
        keys = [(k, tuple(v.shape)) for k, v in net.state_dict().items()]
        mine = list(unet_ref.unet_param_shapes(cfg).items())
        assert keys == mine, name
        print(f"[schema] {name}: {len(keys)} keys match")
        out[f"schema_{name}"] = np.frombuffer(json.dumps([[k, list(s)] for k, s in keys]).encode(), dtype=np.uint8)
        out[f"schemacfg_{name}"] = np.frombuffer(json.dumps(cfg).encode(), dtype=np.uint8)

    # ---------------- sampler steps: reference classes with injected noise ----------------
    cfg = TINY
    sd = unet_ref.make_synthetic_state_dict(cfg, seed=1234)
    net = ref_model(cfg, sd)
    fwk = ref_frameworks.ClassifierFreeGuidance(net, timesteps=1000, beta_schedule="linear", p_uncond=0.1)
    N, S = 2, cfg["image_size"]
    x_t = torch.from_numpy(rng.standard_normal((N, 4, S, S)).astype(np.float32))
    classes = torch.tensor([3, 5])
    model = lambda x, t, c: unet_ref.unet_forward(cfg, sd, x, t, c)
    # DDPM
    ddpm = ref_samplers.DdpmSampler(fwk)
    for ti in [999, 1, 0]:
        z = torch.from_numpy(rng.standard_normal((N, 4, S, S)).astype(np.float32))
        t = torch.tensor([ti] * N)
        with FixedNoise([z]):
            r = ddpm.sample_once(x_t, t, classes, strength=0.5)
        eps = sampler_ref.cfg_eps(model, x_t, t, classes, 0.5)
        xp, x0 = sampler_ref.ddpm_step(tb, x_t, t, eps, z)
        e = rel(xp, r.pred_x_prev)
        print(f"[ddpm t={ti}] oracle vs reference x_prev rel {e:.2e}")
        assert e < 2e-6 and rel(x0, r.pred_x_0) < 2e-6
        out[f"ddpm_t{ti}_noise"] = z.numpy(); out[f"ddpm_t{ti}_xprev"] = r.pred_x_prev.numpy(); out[f"ddpm_t{ti}_x0"] = r.pred_x_0.numpy()
    out["step_x_t"] = x_t.numpy(); out["step_classes"] = classes.numpy()

    # DDIM with the multiview guidance on the conditional (10-channel) model
    cfgc = TINY_COND
    sdc = unet_ref.make_synthetic_state_dict(cfgc, seed=4321)
    netc = ref_model(cfgc, sdc)
    fwc = ref_frameworks.InpaintCFG(netc, timesteps=1000, beta_schedule="linear", p_uncond=0.1)
    ddim = ref_samplers.DdimSampler(fwc)
    y = torch.from_numpy(rng.uniform(-1, 1, (N, 4, S, S)).astype(np.float32))
    mask = torch.from_numpy((rng.uniform(size=(N, 1, S, S)) < 0.7).astype(np.float32))
    mask_rgb = mask * torch.from_numpy((rng.uniform(size=(N, 1, S, S)) < 0.8).astype(np.float32))
    convex = torch.from_numpy(rng.uniform(-1, 1, (N, 1, S, S)).astype(np.float32))
    modelc = lambda x, t, c: unet_ref.unet_forward(cfgc, sdc, x, t, c)
    for (tt, tp) in [(1000, 980), (20, 0)]:
        zs = [torch.from_numpy(rng.standard_normal((N, 3, S, S)).astype(np.float32)),
              torch.from_numpy(rng.standard_normal((N, 1, S, S)).astype(np.float32)),
              torch.from_numpy(rng.standard_normal((N, 4, S, S)).astype(np.float32))]
        t = torch.tensor([tt] * N); t_prev = torch.tensor([tp] * N)
        kw = dict(y=y, mask=mask, mask_rgb=mask_rgb, replace_rgb=(0.1, y[:, :3], mask_rgb), replace_depth=(0.2, y[:, 3:], mask),
                  constrain_depth=(0.5, convex))
        with FixedNoise(list(zs)):
            r = ddim.sample_once(x_t, t, t_prev, classes, strength=0.5, **kw)
        ci = sampler_ref.make_inpaint_inputs(x_t, y, mask, mask_rgb, zs[0], zs[1])
        eps = sampler_ref.cond_eps(modelc, ci, t - 1, classes, 0.5)
        xp, x0 = sampler_ref.ddim_step(tb, x_t, t, t_prev, eps, zs[2], replace_rgb=(0.1, y[:, :3], mask_rgb),
                                       replace_depth=(0.2, y[:, 3:], mask), constrain_depth=(0.5, convex))
        e = rel(xp, r.pred_x_prev)
        print(f"[ddim t={tt}->{tp}] oracle vs reference x_prev rel {e:.2e}")
        assert e < 2e-6 and rel(x0, r.pred_x_0) < 2e-6
        out[f"ddim_t{tt}_noise_rgb"] = zs[0].numpy(); out[f"ddim_t{tt}_noise_d"] = zs[1].numpy()
        out[f"ddim_t{tt}_xprev"] = r.pred_x_prev.numpy()
    out["ddim_y"] = y.numpy(); out["ddim_mask"] = mask.numpy(); out["ddim_mask_rgb"] = mask_rgb.numpy(); out["ddim_convex"] = convex.numpy()

    # SuperResCFG cond inputs
    xs = torch.from_numpy(rng.standard_normal((N, 4, 32, 32)).astype(np.float32))
    ys = torch.from_numpy(rng.uniform(-1, 1, (N, 4, 16, 16)).astype(np.float32))
    fws = ref_frameworks.SuperResCFG(ref_model(TINY_SR, unet_ref.make_synthetic_state_dict(TINY_SR, seed=1234)),
                                     timesteps=1000, beta_schedule="linear")
    ci_ref = fws.make_cond_inputs(xs, ys)
    assert torch.equal(ci_ref, sampler_ref.make_sr_inputs(xs, ys))
    out["sr_x"] = xs.numpy(); out["sr_y"] = ys.numpy(); out["sr_cond_inputs"] = ci_ref.numpy()

    np.savez_compressed(os.path.join(HERE, "unet_sampler_golden.npz"), **out)
    sz = os.path.getsize(os.path.join(HERE, "unet_sampler_golden.npz"))
    print(f"wrote unet_sampler_golden.npz ({sz/1024:.0f} KiB)")


if __name__ == "__main__":
    main()
