"""Host-side glue of the composed trainer steps (sugar_b200/steps.py) on the CPU: the recipe of
sugar_trainers/coarse_sdf.py:506-716 run end to end with the reference's PyTorch op chains (oracle/) and a stand-in
rasterizer, through the loader bench.py's reference arm uses (no import of the package, no CUDA library mapped)."""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


class FakeRasterizerModule:
    """Differentiable stand-in with the module's surface: image = mean colour (+ zero-weight terms so that every
    input receives a gradient), radii = 1."""

    class GaussianRasterizationSettings:
        def __init__(self, **kw):
            self.__dict__.update(kw)

    class GaussianRasterizer:
        def __init__(self, st):
            self.st = st

        def __call__(self, means3D, means2D, opacities, scales, rotations, shs=None, colors_precomp=None):
            H, W = self.st.image_height, self.st.image_width
            c = colors_precomp if colors_precomp is not None else shs[:, 0]
            z = 0 * (opacities.sum() + scales.sum() + rotations.sum() + means3D.sum())
            return (c.mean(0)[:, None, None] + z).expand(3, H, W) + 0 * self.st.bg[:, None, None], \
                torch.ones(means3D.shape[0], dtype=torch.int32)


def test_coarse_sdf_step_recipe_runs_and_reaches_every_parameter():
    import bench
    import bench_workloads as bw
    from oracle import field_oracle as fo
    before = set(sys.modules)   # other tests in this process may have imported the package themselves
    steps = bw._load_steps_without_package()
    assert not any(m == "sugar_b200" or m.startswith("sugar_b200.") for m in set(sys.modules) - before)
    scenes = bench.load_scenes()
    sc = scenes.make_scene(500, 64, 48, seed=0)
    cam = steps.camera_from_scene(sc, "cpu")
    ops = bw.reference_ops(torch, FakeRasterizerModule)
    leaf = lambda t: t.clone().requires_grad_(True)
    raw = dict(points=leaf(torch.from_numpy(sc.means3D)), sh_dc=leaf(torch.from_numpy(sc.shs[:, :1].copy())),
               sh_rest=leaf(torch.from_numpy(sc.shs[:, 1:].copy())),
               densities=leaf(torch.logit(torch.from_numpy(sc.opacities).clamp(1e-4, 1 - 1e-4))),
               scales=leaf(torch.from_numpy(sc.scales).log()), quaternions=leaf(torch.from_numpy(sc.rotations) * 1.3))
    knn = fo.knn_idx(raw["points"].detach(), 16)
    g = torch.Generator().manual_seed(1)
    loss, stats = steps.coarse_sdf_step(raw, cam, torch.rand(3, 48, 64), knn, ops, n_samples=2000, generator=g)
    assert np.isfinite(float(loss)) and stats["visible"] == 500 and 0 < stats["sampled_gaussians"] <= 500
    for k, v in raw.items():
        assert v.grad is not None and bool(torch.isfinite(v.grad).all()), k
    assert float(raw["quaternions"].grad.abs().max()) > 0 and float(raw["densities"].grad.abs().max()) > 0


def test_depth_lookup_uses_the_rasterizer_pixel_convention():
    """grid_sample(align_corners=False) on the rasterizer's NDC == bilinear lookup at ndc2Pix pixel coordinates
    (auxiliary.h:41-44): a depth map that is linear in the pixel coordinates is reproduced exactly."""
    import bench
    import bench_workloads as bw
    steps = bw._load_steps_without_package()
    scenes = bench.load_scenes()
    W, H = 64, 48
    sc = scenes.make_scene(400, W, H, seed=2, frac_behind=0.0, lateral=0.8)
    cam = steps.camera_from_scene(sc, "cpu")
    ys, xs = torch.meshgrid(torch.arange(H, dtype=torch.float32), torch.arange(W, dtype=torch.float32), indexing="ij")
    depth = 2.0 + 0.1 * xs + 0.03 * ys
    pts = torch.from_numpy(sc.means3D)
    hom = pts @ cam.projmatrix[:3, :] + cam.projmatrix[3, :]
    ndc = hom[:, :2] / (hom[:, 3:4] + 1e-7)
    px, py = ((ndc[:, 0] + 1) * W - 1) * 0.5, ((ndc[:, 1] + 1) * H - 1) * 0.5
    inside = (px > 0) & (px < W - 1) & (py > 0) & (py < H - 1)
    got = steps.depth_lookup(depth, pts, cam.projmatrix)
    want = 2.0 + 0.1 * px + 0.03 * py
    assert inside.sum() > 100 and torch.allclose(got[inside], want[inside], atol=1e-4)
