"""Pin oracle/warp_ref.py against the reference's own rgbd_3d/utils.py (build container only) and write the warp
golden fixture tests/golden/warp_golden.npz.

rgbd_3d/utils.py is imported by file path with stubbed `glm` (numpy-backed: inverse/mat3, mathematical orientation),
`plyfile` and `easydict`; rgbd_3d/__init__.py (which pulls in moderngl) is bypassed.  The reference's
aggregate_conditions is then run unmodified with the oracle's software renderer standing in for the OpenGL
AggregationRenderer, which pins every numpy / cv2 / PIL step; the GL rasteriser itself stays unpinned.
"""
from __future__ import annotations

import importlib.util
import os
import sys
import types

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
REF = os.environ.get("IVID_REF", "/root/reference")
sys.path.insert(0, ROOT)

from oracle import warp_ref  # noqa: E402


def _stub_modules():
    glm = types.ModuleType("glm")
    glm.inverse = lambda m: np.linalg.inv(np.asarray(m, dtype=np.float64)).astype(np.float32)
    glm.mat3 = lambda m: np.asarray(m)[:3, :3]
    sys.modules["glm"] = glm
    sys.modules["plyfile"] = types.ModuleType("plyfile")
    ed = types.ModuleType("easydict")

    class EasyDict(dict):
        def __init__(self, d=None, **kw):
            super().__init__()
            for k, v in dict(d or {}, **kw).items():
                self[k] = v
        __getattr__ = dict.__getitem__
        __setattr__ = dict.__setitem__
    ed.EasyDict = EasyDict
    sys.modules["easydict"] = ed


def load_ref_utils():
    _stub_modules()
    spec = importlib.util.spec_from_file_location("ref_rgbd_utils", os.path.join(REF, "rgbd_3d", "utils.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def synthetic_rgbd(rng, n=128):
    """Smooth random height field with a foreground blob (depth discontinuities) — z-buffer depth in (0,1), RGB in [0,1]."""
    yy, xx = np.mgrid[0:n, 0:n] / n
    z = 0.55 + 0.08 * np.sin(6.0 * xx + rng.uniform(0, 6)) * np.cos(5.0 * yy + rng.uniform(0, 6))
    cx, cy, r = rng.uniform(0.35, 0.65), rng.uniform(0.35, 0.65), rng.uniform(0.15, 0.25)
    blob = (xx - cx) ** 2 + (yy - cy) ** 2 < r ** 2
    z = np.where(blob, z - 0.18 - 0.05 * np.cos(8 * xx), z)
    rgb = np.stack([0.5 + 0.5 * np.sin(9 * xx + i) * np.cos(7 * yy - i) for i in range(3)], axis=-1)
    rgb = np.where(blob[..., None], 1.0 - rgb, rgb)
    return np.concatenate([rgb, z[..., None]], axis=-1).astype(np.float32)


def main():
    ref = load_ref_utils()
    rng = np.random.default_rng(5)
    out = {}
    near, far, fov, atol, rtol, erode_rgb = 0.6, 5.0, 45, 0.03, 0.03, 3    # inference/sample.py:258-263
    views = [warp_ref.view_on_sphere(0.0, 0.0), warp_ref.view_on_sphere(0.15, 0.0), warp_ref.view_on_sphere(-0.3, 0.15)]
    rgbds = [synthetic_rgbd(rng) for _ in range(2)]

    # --- mesh building ---
    meshes_ref, meshes_or = [], []
    for rgbd, mv in zip(rgbds, views[:2]):
        d_lin_ref = ref.linearize_depth(rgbd[:, :, 3:], near, far)
        d_lin = warp_ref.linearize_depth(rgbd[:, :, 3:], near, far)
        assert np.array_equal(d_lin, d_lin_ref)
        m_ref = ref.depth_to_mesh(d_lin_ref, padding="frustum", fov=fov, modelview=mv, atol=atol, rtol=rtol, erode_rgb=erode_rgb, cal_normal=True)
        m_or = warp_ref.depth_to_mesh(d_lin, fov=fov, modelview=mv, atol=atol, rtol=rtol, erode_rgb=erode_rgb)
        for k in ["position", "normal", "uv", "flag"]:
            assert np.array_equal(m_ref.vertices[k], m_or.vertices[k]), k
        assert np.array_equal(m_ref.faces, m_or.faces)
        meshes_ref.append(m_ref); meshes_or.append(m_or)
    print("[pin] linearize_depth / depth_to_mesh (position, normal, uv, flag, faces): bit-identical to the reference")
    assert np.array_equal(ref.project_depth(np.linspace(0.1, 7, 50), near, far), warp_ref.project_depth(np.linspace(0.1, 7, 50), near, far))
    dd = rng.uniform(0.3, 0.8, (64, 64, 1))
    assert np.array_equal(ref.depth_edge(dd, atol, rtol), warp_ref.depth_edge(dd, atol, rtol))

    # --- aggregate_conditions: reference post-processing around the software renderer ---
    colors = [r[:, :, :3] for r in rgbds]
    rend = warp_ref.SoftwareAggregationRenderer(128 * 3, 128)
    for j, target in enumerate([views[1], views[2]]):
        ms, cs = meshes_or[: j + 1], colors[: j + 1]
        c_ref = ref.aggregate_conditions(rend, meshes_ref[: j + 1], cs, target, fov=fov, near=near, far=far, atol=atol, rtol=rtol, erode_rgb=erode_rgb)
        c_or = warp_ref.aggregate_conditions(rend, ms, cs, target, fov=fov, near=near, far=far, atol=atol, rtol=rtol, erode_rgb=erode_rgb)
        for k in ["color", "depth", "mask", "mask_rgb", "depth_convex"]:
            assert np.array_equal(c_ref[k], c_or[k]), k
            out[f"cond{j}_{k}"] = np.asarray(c_ref[k], dtype=np.float32)
        cover = float(c_ref["mask"].mean())
        print(f"[pin] aggregate_conditions target {j}: identical to the reference post-processing; mask coverage {cover:.3f}")
        if j == 1:   # raw 384x384 render of the two-source-view case: the full depth mask, and the depth at the 3x3 SSAA
            #          centre samples (the pixels aggregate_conditions reads), which keeps the fixture under 1 MB
            raw = rend.render(ms, cs, target, fov, is_autoregressive=True)
            out["raw1_depth_centre"] = np.ascontiguousarray(raw.depth[1::3, 1::3])
            out["raw1_mask_depth"] = np.packbits(raw.mask_depth)
    # self-reprojection property: a view rendered from its own camera reproduces its own colours / depth
    raw = rend.render(meshes_or[:1], colors[:1], views[0], fov, is_autoregressive=True)
    rec = np.array(raw.color).reshape(128, 3, 128, 3, 3)[:, 1, :, 1]
    err = np.abs(rec - colors[0]).max()
    zerr = np.abs(raw.depth[1::3, 1::3, 0] - warp_ref.linearize_depth(rgbds[0][:, :, 3], near, far)).max()
    print(f"[prop] self-reprojection: max colour err {err:.2e}, max depth err {zerr:.2e}")
    assert err < 1e-6 and zerr < 2e-3

    # --- numeric padding (inference/utils.py:load_scene -> depth_to_mesh(depth, 32, ...), free-view rendering) ---
    meshes_pad = []
    for rgbd, mv in zip(rgbds, views[:2]):
        d_lin = warp_ref.linearize_depth(rgbd[:, :, 3:], near, far)
        m_ref = ref.depth_to_mesh(d_lin, 32, fov, mv, atol=atol, rtol=rtol, erode_rgb=erode_rgb, cal_normal=True)
        m_or = warp_ref.depth_to_mesh(d_lin, fov=fov, modelview=mv, atol=atol, rtol=rtol, erode_rgb=erode_rgb, padding=32)
        for k in ["position", "normal", "uv", "flag"]:
            assert np.array_equal(m_ref.vertices[k], m_or.vertices[k]), k
        assert np.array_equal(m_ref.faces, m_or.faces)
        meshes_pad.append(m_or)
    print("[pin] depth_to_mesh(padding=32): bit-identical to the reference")
    for i, m in enumerate(meshes_pad):
        vb = warp_ref.mesh_vertex_buffer(m)
        out[f"meshpad{i}_colsum"] = vb.astype(np.float64).sum(0)
        out[f"meshpad{i}_abssum"] = np.abs(vb.astype(np.float64)).sum(0)
        out[f"meshpad{i}_flaghist"] = np.bincount(vb[:, 8].astype(np.int64), minlength=8)
        out[f"meshpad{i}_faces_sum"] = np.array([m.faces.astype(np.int64).sum(), (m.faces.astype(np.int64) * np.arange(1, 4)).sum()])

    # --- training-pair warp (datasets/base.py:219-238): SimpleRenderer(384, 128, near=0.1, far=200) + forward_backward_warp
    #     with padding = image_size; the reference's numpy / PIL steps run unmodified around the software SimpleRenderer ---
    simple = warp_ref.SoftwareSimpleRenderer(128 * 3, 128, near=0.1, far=200)
    d_lin = warp_ref.linearize_depth(rgbds[0][:, :, 3:], 0.5, 100)
    for pad_arg, cal in [(None, False), (128, False)]:
        m_ref = ref.depth_to_mesh(d_lin, padding=pad_arg, fov=fov, modelview=views[1], atol=0.02, rtol=0.02)
        m_or = warp_ref.depth_to_mesh(d_lin, fov=fov, modelview=views[1], atol=0.02, rtol=0.02, padding=pad_arg, cal_normal=cal)
        for k in ["position", "uv", "flag"]:
            assert np.array_equal(m_ref.vertices[k], m_or.vertices[k]), (pad_arg, k)
        assert np.array_equal(m_ref.faces, m_or.faces) and "normal" not in m_or.vertices
    fb_ref = ref.forward_backward_warp(simple, rgbds[0], views[2], modelview0=views[0], padding=128, fov=fov, near=0.5, far=100)
    fb_or = warp_ref.forward_backward_warp(simple, rgbds[0], views[2], modelview0=views[0], padding=128, fov=fov, near=0.5, far=100)
    for k in ["color", "depth", "mask"]:
        assert np.array_equal(fb_ref[k], fb_or[k]), k
        out[f"fbw_{k}"] = np.asarray(fb_ref[k], dtype=np.float32)
    print(f"[pin] depth_to_mesh(padding=None / 128, no normals) and forward_backward_warp: identical to the reference around the "
          f"software SimpleRenderer; surviving mask {float(fb_ref['mask'].mean()):.3f}")

    for i, r in enumerate(rgbds):
        out[f"rgbd{i}"] = r
    out["views"] = np.stack(views)
    out["params"] = np.array([near, far, fov, atol, rtol, erode_rgb], dtype=np.float64)
    for i, m in enumerate(meshes_or):
        vb = warp_ref.mesh_vertex_buffer(m)
        # vertex buffers are regenerated by the oracle in-test; the fixture pins them through column sums + flag histogram
        out[f"mesh{i}_colsum"] = vb.astype(np.float64).sum(0)
        out[f"mesh{i}_abssum"] = np.abs(vb.astype(np.float64)).sum(0)
        out[f"mesh{i}_flaghist"] = np.bincount(vb[:, 8].astype(np.int64), minlength=8)
        out[f"mesh{i}_faces_sum"] = np.array([m.faces.astype(np.int64).sum(), (m.faces.astype(np.int64) * np.arange(1, 4)).sum()])
    np.savez_compressed(os.path.join(HERE, "warp_golden.npz"), **out)
    print(f"wrote warp_golden.npz ({os.path.getsize(os.path.join(HERE, 'warp_golden.npz')) / 1024:.0f} KiB)")


if __name__ == "__main__":
    main()
