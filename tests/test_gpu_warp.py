"""GPU parity of the CUDA warp (mesh build, visibility-buffer rasteriser, deferred shading + aggregation, post-filters)
against the warp oracle (oracle/warp_ref.py + oracle/raster_ref.c), through the C ABI and the rgbd_3d mirror classes.

Integer / byte work is compared bit-exactly (faces, flags, coverage masks, LANCZOS on 8-bit colour, votes, erosion);
floating-point images within tolerances written at each assert."""
import os

import numpy as np
import pytest
import torch

import ivid_b200.rgbd_3d as rgbd_3d
from conftest import ROOT
from oracle import warp_ref

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def wg():
    return np.load(os.path.join(ROOT, "tests", "golden", "warp_golden.npz"))


def _params(wg):
    near, far, fov, atol, rtol, erode = wg["params"]
    return dict(fov=float(fov), near=float(near), far=float(far), atol=float(atol), rtol=float(rtol), erode_rgb=int(erode))


def _model_space(rgbd01):
    return torch.from_numpy(rgbd01.transpose(2, 0, 1)[None] * 2 - 1).float().cuda()


def _oracle_inputs(ms_tensor):
    """what sample.py hands to rgbd_3d: rgbd = samples.cpu().numpy().transpose(0,2,3,1) * 0.5 + 0.5 (float32)"""
    return ms_tensor.cpu().numpy().transpose(0, 2, 3, 1) * 0.5 + 0.5


def _oracle_meshes(wg, rgbds01, k):
    p = _params(wg)
    ms, cs = [], []
    for i in range(k):
        ms.append(warp_ref.depth_to_mesh(warp_ref.linearize_depth(rgbds01[i][:, :, 3:], p["near"], p["far"]), fov=p["fov"],
                                         modelview=wg["views"][i], atol=p["atol"], rtol=p["rtol"], erode_rgb=p["erode_rgb"]))
        cs.append(rgbds01[i][:, :, :3])
    return ms, cs


def test_mesh_build_matches_oracle(wg):
    p = _params(wg)
    dw = rgbd_3d.DeviceWarp(batch=2, image_size=128, ssaa=3, max_views=4)
    x = torch.cat([_model_space(wg["rgbd0"]), _model_space(wg["rgbd1"])], 0)
    dw.add_view(x, [wg["views"][0], wg["views"][1]], **p)
    r01 = _oracle_inputs(x)
    for b in range(2):
        m = warp_ref.depth_to_mesh(warp_ref.linearize_depth(r01[b][:, :, 3:], p["near"], p["far"]), fov=p["fov"], modelview=wg["views"][b],
                                   atol=p["atol"], rtol=p["rtol"], erode_rgb=p["erode_rgb"])
        vb_ref = warp_ref.mesh_vertex_buffer(m)
        vb, faces, col = dw.get_mesh(b, 0)
        assert np.array_equal(faces, m.faces.astype(np.uint32)), "triangulation (diagonal choice) must match exactly"
        assert np.array_equal(vb[:, 8], vb_ref[:, 8]), "discontinuity / padding / erosion flags must match exactly"
        assert np.array_equal(vb[:, 6:8], vb_ref[:, 6:8])
        dpos = np.abs(vb[:, :3] - vb_ref[:, :3]).max(); dn = np.abs(vb[:, 3:6] - vb_ref[:, 3:6]).max()
        print(f"[parity] mesh sample {b}: max |dpos| {dpos:.2e}, max |dnormal| {dn:.2e}, flags/faces/uv exact")
        assert dpos <= 2.5e-7 and dn <= 2.5e-7          # float32 rounding of float64 math (1 ulp at |x| <= 2)
        assert np.array_equal(col, r01[b][:, :, :3])


def test_numpy_facing_depth_to_mesh(wg):
    p = _params(wg)
    d = warp_ref.linearize_depth(wg["rgbd0"][:, :, 3:], p["near"], p["far"])
    m = rgbd_3d.utils.depth_to_mesh(d, padding="frustum", fov=p["fov"], modelview=wg["views"][1], atol=p["atol"], rtol=p["rtol"],
                                    erode_rgb=p["erode_rgb"], cal_normal=True)
    ref = warp_ref.depth_to_mesh(d, fov=p["fov"], modelview=wg["views"][1], atol=p["atol"], rtol=p["rtol"], erode_rgb=p["erode_rgb"])
    assert np.array_equal(m.faces, ref.faces) and np.array_equal(m.vertices.flag, ref.vertices.flag.astype(np.float32))
    assert np.abs(m.vertices.position - ref.vertices.position).max() < 2.5e-7
    with pytest.raises(NotImplementedError):
        rgbd_3d.utils.depth_to_mesh(d, padding="bogus", modelview=wg["views"][1])
    # tolerances left at None (the reference's defaults): no discontinuity test at all, hence no erosion either; a single None
    # counts as 0 (utils.py:227-229)
    for at, rt in ((None, None), (0.03, None), (None, 0.03)):
        m = rgbd_3d.utils.depth_to_mesh(d, padding="frustum", fov=p["fov"], modelview=wg["views"][1], atol=at, rtol=rt,
                                        erode_rgb=p["erode_rgb"], cal_normal=True)
        ref = warp_ref.depth_to_mesh(d, fov=p["fov"], modelview=wg["views"][1], atol=at, rtol=rt, erode_rgb=p["erode_rgb"])
        assert np.array_equal(m.vertices.flag, ref.vertices.flag.astype(np.float32)), (at, rt)
        if at is None and rt is None:
            assert set(np.unique(m.vertices.flag)) <= {0.0, 2.0}


def _raw_compare(tag, got, ref):
    mc_eq = (got["mask_color"] == ref["mask_color"]).mean(); md_eq = (got["mask_depth"] == ref["mask_depth"]).mean()
    both = (got["mask_depth"] & ref["mask_depth"])[..., 0]
    dz = np.abs(got["depth"] - ref["depth"])[both]
    dc = np.abs(got["color"] - ref["color"])[(got["mask_color"] & ref["mask_color"])[..., 0]]
    print(f"[parity] {tag}: mask_color agree {mc_eq:.6f}, mask_depth agree {md_eq:.6f}, depth max {dz.max():.2e} p99.9 "
          f"{np.quantile(dz, 0.999):.2e}, color max {dc.max():.2e} p99.9 {np.quantile(dc, 0.999):.2e}")
    return mc_eq, md_eq, dz, dc


def test_render_matches_oracle_and_golden(wg):
    """AggregationRenderer.render on oracle-built meshes (identical inputs on both sides)."""
    p = _params(wg)
    rgbds = [wg["rgbd0"], wg["rgbd1"]]
    ms, cs = _oracle_meshes(wg, rgbds, 2)
    ref_r = warp_ref.SoftwareAggregationRenderer(384, 128)
    gpu_r = rgbd_3d.AggregationRenderer(384, 128)
    for j in range(2):
        target = wg["views"][j + 1]
        ref = ref_r.render(ms[: j + 1], cs[: j + 1], target, p["fov"], is_autoregressive=True)
        got = gpu_r.render(ms[: j + 1], cs[: j + 1], target, p["fov"], is_autoregressive=True)
        mc_eq, md_eq, dz, dc = _raw_compare(f"render target {j} ({j + 1} source views)", got, ref)
        assert mc_eq == 1.0 and md_eq == 1.0, "coverage / visibility must match the oracle exactly (integer edge functions)"
        assert np.quantile(dz, 0.999) < 1e-4 and np.quantile(dc, 0.999) < 1e-4
    # the committed golden (cross-machine pin of the same quantities): full mask, depth at the SSAA centre samples
    g_md = np.unpackbits(wg["raw1_mask_depth"])[: 384 * 384].reshape(384, 384, 1).astype(bool)
    assert (got["mask_depth"] == g_md).mean() > 0.9999
    both = (got["mask_depth"] & g_md)[1::3, 1::3, 0]
    assert np.abs(got["depth"][1::3, 1::3] - wg["raw1_depth_centre"])[both].max() < 1e-3


def test_postfilter_bit_exact_on_oracle_render(wg):
    """aggregate_conditions' post-filters on the SAME raw render: 8-bit LANCZOS (Pillow fixed point), votes, depth_edge,
    erosion and products must be bit-identical to the reference's PIL / cv2 / numpy code path."""
    p = _params(wg)
    ms, cs = _oracle_meshes(wg, [wg["rgbd0"], wg["rgbd1"]], 2)

    class Replay:     # hands the oracle's raw render to the reference-equivalent numpy post-processing
        render_size = 384
        def __init__(self, raw): self.raw = raw
        def render(self, *a, **k): return self.raw
    raw = warp_ref.SoftwareAggregationRenderer(384, 128).render(ms, cs, wg["views"][2], p["fov"], is_autoregressive=True)
    ref = warp_ref.aggregate_conditions(Replay(raw), ms, cs, wg["views"][2], fov=p["fov"], near=p["near"], far=p["far"], atol=p["atol"],
                                        rtol=p["rtol"], erode_rgb=p["erode_rgb"])
    gpu_r = rgbd_3d.AggregationRenderer(384, 128)
    gpu_r._last_raw = tuple(torch.from_numpy(np.ascontiguousarray(a.astype(np.float32))).cuda() for a in
                            (raw.color, raw.depth[..., 0], raw.mask_color[..., 0], raw.mask_depth[..., 0]))
    gpu_r.render = lambda *a, **k: None
    got = rgbd_3d.utils.aggregate_conditions(gpu_r, ms, cs, wg["views"][2], **{k: p[k] for k in ("fov", "near", "far", "atol", "rtol", "erode_rgb")})
    for k in ["mask", "mask_rgb", "depth", "depth_convex"]:
        assert np.array_equal(got[k], np.asarray(ref[k], np.float32)), k
    assert np.array_equal(got["color"], np.asarray(ref["color"]).astype(np.float32)), "LANCZOS(8-bit) * mask_rgb"
    print("[parity] post-filters: color / depth / mask / mask_rgb / depth_convex bit-identical")


def test_device_pipeline_end_to_end(wg):
    """The device-resident path the sampling loop uses (add_view x2 -> aggregate) vs the whole oracle pipeline."""
    p = _params(wg)
    dw = rgbd_3d.DeviceWarp(batch=1, image_size=128, ssaa=3, max_views=4)
    xs = [_model_space(wg["rgbd0"]), _model_space(wg["rgbd1"])]
    r01 = [_oracle_inputs(x)[0] for x in xs]
    ms, cs = _oracle_meshes(wg, r01, 2)
    rend = warp_ref.SoftwareAggregationRenderer(384, 128)
    for j in range(2):
        dw.add_view(xs[j], wg["views"][j], **p)
        cond = dw.aggregate(wg["views"][j + 1], **p)[0].permute(1, 2, 0).cpu().numpy()
        ref = warp_ref.aggregate_conditions(rend, ms[: j + 1], cs[: j + 1], wg["views"][j + 1], **p)
        m_eq = (cond[:, :, 4:5] == ref["mask"]).mean(); mr_eq = (cond[:, :, 5:6] == ref["mask_rgb"]).mean()
        agree = (cond[:, :, 4] == ref["mask"][:, :, 0])
        dd = np.abs(cond[:, :, 3:4] - ref["depth"])[agree]; dc = np.abs(cond[:, :, :3] - ref["color"])
        print(f"[parity] device warp target {j}: mask agree {m_eq:.5f}, mask_rgb agree {mr_eq:.5f}, depth max {dd.max():.2e}, "
              f"color max {dc.max():.3f} ({(dc > 1.5 / 255).mean():.2e} of pixels off by more than one 8-bit step)")
        assert m_eq > 0.999 and mr_eq > 0.999
        assert dd.max() < 1e-4 and (dc > 1.5 / 255).mean() < 1e-3


def test_self_reprojection_property_gpu(wg):
    """Size-independent property: view 0 rendered from its own camera returns its own colours and depth."""
    p = _params(wg)
    dw = rgbd_3d.DeviceWarp(batch=1, image_size=128, ssaa=3, max_views=2)
    x = _model_space(wg["rgbd0"])
    dw.add_view(x, wg["views"][0], **p)
    color, depth, mc, md = dw.render_raw(wg["views"][0], p["fov"])
    r01 = _oracle_inputs(x)[0]
    rec = color[0].cpu().numpy().reshape(128, 3, 128, 3, 3)[:, 1, :, 1]
    assert np.abs(rec - r01[:, :, :3]).max() < 1e-6
    z = depth[0].cpu().numpy()[1::3, 1::3]
    assert np.abs(z - warp_ref.linearize_depth(r01[:, :, 3], p["near"], p["far"])).max() < 2e-3
    assert float(md.mean()) > 0.95


def test_numeric_padding_mesh_matches_oracle(wg):
    """depth_to_mesh(depth, 32, ...) of inference/utils.py:load_scene (free-view rendering)."""
    p = _params(wg)
    d = warp_ref.linearize_depth(wg["rgbd1"][:, :, 3:], p["near"], p["far"])
    m = rgbd_3d.utils.depth_to_mesh(d, 32, p["fov"], wg["views"][1], atol=p["atol"], rtol=p["rtol"], erode_rgb=p["erode_rgb"], cal_normal=True)
    ref = warp_ref.depth_to_mesh(d, fov=p["fov"], modelview=wg["views"][1], atol=p["atol"], rtol=p["rtol"], erode_rgb=p["erode_rgb"], padding=32)
    assert np.array_equal(m.faces, ref.faces) and np.array_equal(m.vertices.flag, ref.vertices.flag.astype(np.float32))
    assert np.array_equal(m.vertices.uv, ref.vertices.uv.astype(np.float32))
    pos_ref = ref.vertices.position.astype(np.float32)
    dpos = np.abs(m.vertices.position - pos_ref)
    print(f"[parity] numeric-padding mesh: max |dpos| {dpos.max():.2e} (|pos| up to {np.abs(pos_ref).max():.2f}), flags/faces/uv exact")
    assert (dpos <= np.spacing(np.abs(pos_ref))).all(), "positions within one float32 ulp of the float64 reference math"
    assert np.abs(m.vertices.normal - ref.vertices.normal).max() <= 2.5e-7


def test_free_view_render_matches_oracle(wg, tmp_path):
    """inference/render.py path: save_scene -> load_scene (re-mesh with padding 32) -> AggregationRenderer(640, 128, near=0.1)
    from two trajectory cameras -> LANCZOS / depth colour map, against the same pipeline on the oracle."""
    from ivid_b200.inference import load_scene, load_scene_views, save_scene, swing_trajectory
    from ivid_b200.inference.render import SSAA, resolve_frame
    from ivid_b200.utils import edict
    p = _params(wg)
    views = [edict(depth=warp_ref.linearize_depth(wg[f"rgbd{i}"][:, :, 3:], p["near"], p["far"]).astype(np.float32), fov=p["fov"],
                   modelview=wg["views"][i]) for i in range(2)]
    colors = [wg[f"rgbd{i}"][:, :, :3] for i in range(2)]
    path = os.path.join(tmp_path, "scene.npz")
    save_scene(path, views, colors)
    meshes, cols = load_scene(path)                                   # defaults atol = rtol = 0.03, erode_rgb = 3
    stored = load_scene_views(path)
    ms_ref = [warp_ref.depth_to_mesh(v.depth, fov=v.fov, modelview=np.asarray(v.modelview), atol=0.03, rtol=0.03, erode_rgb=3, padding=32)
              for v in stored]
    targets = [swing_trajectory(8)[1], swing_trajectory(8)[5]]
    gpu_r = rgbd_3d.AggregationRenderer(128 * SSAA, 128, near=0.1, far=200)
    ref_r = warp_ref.SoftwareAggregationRenderer(128 * SSAA, 128, near=0.1, far=200)
    got = gpu_r.render(meshes, cols, targets)
    assert isinstance(got, list) and len(got) == 2
    for j, t in enumerate(targets):
        ref = ref_r.render(ms_ref, [v.color for v in stored], t)
        mc_eq, md_eq, dz, dc = _raw_compare(f"free-view frame {j} (640x640, 2 source views)", got[j], ref)
        assert mc_eq > 0.9999 and md_eq > 0.9999       # meshes differ by <= 1 float32 ulp: a handful of edge pixels may flip
        assert np.quantile(dz, 0.999) < 1e-3 and np.quantile(dc, 0.999) < 1e-3
        c8, d8 = resolve_frame(got[j], 128)
        c8r, d8r = resolve_frame(ref, 128)
        assert c8.shape == (128, 128, 3) and d8.shape == (128, 128, 3) and c8.dtype == np.uint8
        off = (np.abs(c8.astype(int) - c8r.astype(int)) > 1).mean()
        print(f"[parity] free-view frame {j}: resolved colour pixels off by more than one 8-bit step: {off:.2e}")
        assert off < 1e-3
        assert (d8 != d8r).mean() < 1e-2
    # the device-side resolve (8-bit LANCZOS kernels + depth colour table) is bit-identical to the host numpy / PIL / cv2 steps
    from ivid_b200.inference.render import depth_colour_table
    cd, dd = gpu_r.render_resolved(meshes, cols, targets, lut=depth_colour_table())
    for j in range(2):
        c8, d8 = resolve_frame(got[j], 128)
        assert np.array_equal(cd[j], c8), "device LANCZOS resolve differs from PIL"
        assert np.array_equal(dd[j], d8), "device depth colour map differs from colorize_depth"


def test_unpadded_mesh_and_simple_renderer_match_oracle(wg):
    """depth_to_mesh(padding=None, cal_normal=False) and SimpleRenderer.render (training-pair warp building blocks)."""
    fov = float(wg["params"][2])
    d = warp_ref.linearize_depth(wg["rgbd0"][:, :, 3:], 0.5, 100)
    for pad in (None, 128):
        m = rgbd_3d.utils.depth_to_mesh(d, padding=pad, fov=fov, modelview=wg["views"][1], atol=0.02, rtol=0.02)
        ref = warp_ref.depth_to_mesh(d, fov=fov, modelview=wg["views"][1], atol=0.02, rtol=0.02, padding=pad, cal_normal=False)
        assert "normal" not in m.vertices
        assert np.array_equal(m.faces, ref.faces) and np.array_equal(m.vertices.flag, ref.vertices.flag.astype(np.float32)), pad
        assert np.array_equal(m.vertices.uv, ref.vertices.uv.astype(np.float32))
        pos_ref = ref.vertices.position.astype(np.float32)
        assert (np.abs(m.vertices.position - pos_ref) <= np.spacing(np.abs(pos_ref))).all(), "positions within one float32 ulp"
        got = rgbd_3d.SimpleRenderer(384, 128, near=0.1, far=200).render(ref, wg["rgbd0"][:, :, :3], wg["views"][2], fov)
        want = warp_ref.SoftwareSimpleRenderer(384, 128, near=0.1, far=200).render(ref, wg["rgbd0"][:, :, :3], wg["views"][2], fov)
        assert np.array_equal(got.mask, want.mask), "coverage / alpha must match the oracle exactly on identical meshes"
        assert np.array_equal(got.color, want.color.astype(np.float32))
        dz = np.abs(got.depth - want.depth)
        print(f"[parity] SimpleRenderer (padding={pad}): mask / colour exact, depth max rel {float((dz / want.depth).max()):.2e}")
        assert (dz / want.depth).max() < 1e-5


def test_forward_backward_warp_matches_oracle_and_golden(wg):
    """rgbd_3d.utils.forward_backward_warp (datasets/base.py:238 call shape: padding = image_size, near 0.5, far 100) against
    the oracle pipeline and the fixture produced by the unmodified reference function."""
    fov = float(wg["params"][2])
    r = rgbd_3d.utils.forward_backward_warp(rgbd_3d.SimpleRenderer(384, 128, near=0.1, far=200), wg["rgbd0"], wg["views"][2],
                                            modelview0=wg["views"][0], padding=128, fov=fov, near=0.5, far=100)
    ref = warp_ref.forward_backward_warp(warp_ref.SoftwareSimpleRenderer(384, 128, near=0.1, far=200), wg["rgbd0"], wg["views"][2],
                                         modelview0=wg["views"][0], padding=128, fov=fov, near=0.5, far=100)
    for name, want in (("oracle", ref), ("reference golden", {k: wg[f"fbw_{k}"] for k in ("color", "depth", "mask")})):
        m_ne = (r.mask != np.asarray(want["mask"], np.float32)).mean()
        agree = (r.mask == np.asarray(want["mask"], np.float32))[..., 0]
        dd = np.abs(r.depth - np.asarray(want["depth"], np.float32))[agree].max()
        dc = np.abs(r.color - np.asarray(want["color"], np.float32))[agree]
        print(f"[parity] forward_backward_warp vs {name}: mask differs on {m_ne:.2e} of pixels, depth max {dd:.2e}, colour max {dc.max():.4f} "
              f"({(dc > 1.5 / 255).mean():.2e} off by more than one 8-bit step), kept {float(r.mask.mean()):.3f}")
        assert m_ne < 1e-3 and dd < 1e-5 and (dc > 1.5 / 255).mean() < 1e-3
    # size-independent property: warping to the SAME camera and back keeps almost everything and reproduces the input
    same = rgbd_3d.utils.forward_backward_warp(rgbd_3d.SimpleRenderer(384, 128, near=0.1, far=200), wg["rgbd0"], wg["views"][0],
                                               modelview0=wg["views"][0], padding=128, fov=fov, near=0.5, far=100)
    keep = same.mask[..., 0] > 0
    assert keep.mean() > 0.9
    assert np.abs(same.depth[..., 0] - wg["rgbd0"][:, :, 3])[keep].max() < 1e-5
    assert np.quantile(np.abs(same.color - wg["rgbd0"][:, :, :3])[keep], 0.95) <= 2.0 / 255 + 1e-6


def test_aggregate_is_deterministic_under_load():
    """Size-independent property at the benchmark shape (batch 16, 9 source views, 384^2 visibility buffers, every SM busy):
    the same aggregate issued repeatedly returns the same bits (64-bit atomicMin visibility + exact integer coverage leave no
    room for order dependence; the warp-cooperative big-triangle path must not race on its shared-memory table)."""
    from ivid_b200.inference import build_modelviews
    B, V = 16, 9
    rng = np.random.default_rng(0)
    yy, xx = np.mgrid[0:128, 0:128] / 128

    def synth():
        z = 0.55 + 0.08 * np.sin(6.0 * xx + rng.uniform(0, 6)) * np.cos(5.0 * yy + rng.uniform(0, 6))
        cx, cy, r = rng.uniform(0.35, 0.65), rng.uniform(0.35, 0.65), rng.uniform(0.15, 0.25)
        z = np.where((xx - cx) ** 2 + (yy - cy) ** 2 < r ** 2, z - 0.18, z)
        rgb = np.stack([0.5 + 0.5 * np.sin(9 * xx + i) * np.cos(7 * yy - i) for i in range(3)], axis=-1)
        return np.concatenate([rgb, z[..., None]], axis=-1).astype(np.float32)

    views = build_modelviews("3x9", 1)
    kw = dict(fov=45, near=0.6, far=5, atol=0.03, rtol=0.03, erode_rgb=3)
    w = rgbd_3d.DeviceWarp(B, image_size=128, ssaa=3, max_views=V + 1)
    for j in range(V):
        x = torch.from_numpy(np.stack([synth().transpose(2, 0, 1) * 2 - 1 for _ in range(B)])).float().cuda()
        w.add_view(x, views[j], **kw)
    first = [t.clone() for t in _cond_tensors(w.aggregate(views[V], **kw))]
    for _ in range(25):
        again = _cond_tensors(w.aggregate(views[V], **kw))
        for a, b in zip(first, again):
            assert torch.equal(a, b), "aggregate is not reproducible"
    assert float(first[0].abs().sum()) > 0


def _cond_tensors(cond):
    if isinstance(cond, dict):
        return [v for _, v in sorted(cond.items()) if torch.is_tensor(v)]
    if torch.is_tensor(cond):
        return [cond]
    return [v for v in cond if torch.is_tensor(v)]
