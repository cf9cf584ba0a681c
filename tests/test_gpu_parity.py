"""GPU parity tests (run on the B200 box): sugar_b200 CUDA path vs
  (1) the UNMODIFIED reference CUDA build: what it computed on a B200 from the same seeded inputs
      (tests/golden/reference_build.npz: digests of the arrays held bit-exact, sampled gradients);
  (2) the CPU oracle (oracle/raster_oracle.c).

Tolerances.  Everything the reference computes before blending and every integer/index output
(radii, tiles_touched, depths, means2D, conic, sort keys, sorted ids, ranges, n_contrib) must be
BIT-EXACT.  The forward image and final_T are also bit-exact against the reference build (same
rounding order, same libdevice expf).  Gradients are sums whose order is nondeterministic in the
reference (fp32 atomics), so they are compared per tensor as |a-b|_inf / |b|_inf <= 1e-4
(BASELINE.json: "gradients within 1e-4 rel").  One documented exception: for surface-aligned Gaussians with a
1e-6 axis (case mesh_bound) the reference's per-Gaussian chain amplifies one-ulp differences of the blend
accumulators ~300x into dL_dscales / dL_drotations (the reference differs from itself by up to 3e-5 run to
run); those tensors are held to 5x the measured sensitivity to 1e-6 accumulator noise instead.
"""
import numpy as np
import pytest

import helpers as h

pytestmark = pytest.mark.gpu

GRAD_RTOL = 1e-4

CASES = [
    # name, P, W, H, camera, use_sh, sh_degree, cov_precomp, bg
    ("sh3_posed", 4000, 200, 120, "posed", True, 3, False, (0.0, 0.0, 0.0)),
    ("sh2_identity", 3000, 160, 96, "identity", True, 2, False, (1.0, 1.0, 1.0)),
    ("sh0_posed", 2000, 129, 67, "posed", True, 0, False, (0.2, 0.4, 0.6)),
    ("colors_posed", 4000, 200, 120, "posed", False, 0, False, (0.1, 0.2, 0.3)),
    ("covpre_posed", 2000, 96, 64, "posed", False, 0, True, (0.0, 0.0, 0.0)),
    ("mesh_bound", 3000, 160, 96, "posed", True, 3, False, (0.0, 0.0, 0.0)),
    ("big_splats", 600, 160, 96, "identity", False, 0, False, (0.0, 0.0, 0.0)),
    # dense tiles: ~6k-30k instances per tile -> exercises the 8192-word sort class and the global
    # radix fallback (tiles above 8192 instances)
    ("dense_tiles", 120000, 64, 48, "posed", False, 0, False, (0.0, 0.0, 0.0)),
    ("mid_tiles", 35000, 64, 48, "posed", True, 1, False, (0.5, 0.5, 0.5)),
    # every Gaussian at the same camera depth: all sort keys of a tile tie on depth, order = Gaussian id
    ("coplanar", 20000, 160, 96, "identity", False, 0, False, (0.0, 0.0, 0.0)),
    # two thin depth shells: very skewed per-tile depth histogram (bucket sort falls back to merge)
    ("two_shells", 60000, 128, 96, "identity", False, 0, False, (0.0, 0.0, 0.0)),
]


def _scene(name, P, W, H, camera):
    from sugar_b200 import scenes
    kw = {}
    if name == "mesh_bound":
        kw["mesh_bound"] = True
    if name == "big_splats":
        kw["px_sigma"] = 25.0
    if name == "coplanar":
        kw["zrange"] = (5.0, 5.0)
        kw["frac_behind"] = 0.0
    if name == "two_shells":
        kw["px_sigma"] = 0.8
    if name in ("dense_tiles", "mid_tiles"):
        kw["px_sigma"] = 0.8
        kw["lateral"] = 0.9
    sc = scenes.make_scene(P, W, H, seed=len(name) * 7 + P % 13, camera=camera, **kw)
    if name == "two_shells":  # snap depths onto two thin shells (identity camera: depth == z)
        m = sc.means3D.copy()
        front = m[:, 2] > 0.3
        shell = np.where(np.arange(P) % 2 == 0, 3.0, 7.0) + (np.arange(P) % 7) * 1e-6
        m[front, 2] = shell[front].astype(np.float32)
        sc = sc._replace(means3D=m)
    return sc


def _cov_from_oracle(sc):
    fw, _ = h.run_oracle(sc, np.zeros(3, np.float32), use_sh=False)
    return fw["cov3D"].copy()


def compared_state(radii, st, use_sh):
    """The forward state held bit-identical to the reference build's, as {name: (array, failure message)}; per-Gaussian
    arrays only where radii > 0 (the reference leaves the others unwritten).  `st`: _C.inspect_state of ours or
    helpers.decode_ref_state of the reference."""
    vis = radii > 0
    out = {"tiles_touched": (st["tiles_touched"][vis], "tiles_touched differ"),
           "depths": (st["depths"][vis], "depths not bit-exact"),
           "means2D": (st["means2D"][vis], "means2D not bit-exact"),
           "conic_opacity": (st["conic_opacity"][vis], "conic/opacity not bit-exact")}
    if use_sh:
        out["clamped"] = (st["clamped"][vis].bool(), "clamp flags differ")
        out["rgb"] = (st["rgb"][vis], "SH colours not bit-exact")
    out.update(keys=(st["keys"], "sorted 64-bit keys differ"), point_list=(st["point_list"], "sorted Gaussian ids differ"),
               ranges=(st["ranges"], "tile ranges differ"), n_contrib=(st["n_contrib"], "n_contrib differs"),
               final_T=(st["final_T"], "final_T not bit-exact"))
    return out


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_matches_reference_build(case):
    """Against what the reference build computed on the same seeded inputs (helpers.RefGolden)."""
    name, P, W, H, camera, use_sh, deg, covpre, bg = case
    from sugar_b200 import diff_gaussian_rasterization as ours, scenes
    from sugar_b200 import _C
    ref = h.RefGolden("parity." + name)
    sc = _scene(name, P, W, H, camera)
    dL = scenes.upstream_grad(W, H)
    cov3D = _cov_from_oracle(sc) if covpre else None
    opts = dict(use_sh=use_sh, sh_degree=deg, use_cov_precomp=covpre, cov3D=cov3D)
    a = h.run_module(ours, sc, bg, None, **opts)
    st = _C.inspect_state(P, W, H, a["num_rendered"], a["geom"], a["binning"], a["img"])

    assert a["num_rendered"] == ref.num_rendered
    assert ref.same("radii", a["radii"]), "radii differ"
    for k, (x, msg) in compared_state(a["radii"], st, use_sh).items():
        assert ref.same(k, x), msg
    assert ref.same("color", a["color"]), "image not bit-exact"

    # backward
    a = h.run_module(ours, sc, bg, dL, **opts)
    assert set(a["grads"]) == ref.grad_names
    bad, sens = [], None
    for k in sorted(ref.grad_names):
        err, noise = ref.grad_err(k, a["grads"][k]), ref.noise(k)  # noise: the reference's own atomics, run to run
        # 1e-4, except where the reference cannot reproduce itself to 2e-5 (surface-aligned
        # Gaussians with a 1e-6 axis: cancellation in the scale/rotation chain): there 5x its noise, or
        # 5x what 1e-6 relative noise on the blend accumulators (= fp32 summation order) does to this
        # tensor through the reference's own per-Gaussian chain (helpers.grad_sensitivity, CPU oracle).
        if err > max(GRAD_RTOL, 5.0 * noise):
            if sens is None:
                sens = h.grad_sensitivity(sc, bg, dL, **opts)
            if err > 5.0 * sens.get(k, 0.0):
                bad.append(f"grad {k}: rel err {err:.3e} (reference run-to-run {noise:.1e}, "
                           f"sensitivity to 1e-6 accumulator noise {sens.get(k, 0.0):.1e})")
    assert not bad, "; ".join(bad)


@pytest.mark.parametrize("case", CASES[:5], ids=[c[0] for c in CASES[:5]])
def test_matches_cpu_oracle(case):
    name, P, W, H, camera, use_sh, deg, covpre, bg = case
    from sugar_b200 import diff_gaussian_rasterization as ours, scenes
    from sugar_b200 import _C
    sc = _scene(name, P, W, H, camera)
    dL = scenes.upstream_grad(W, H)
    cov3D = _cov_from_oracle(sc) if covpre else None
    opts = dict(use_sh=use_sh, sh_degree=deg, use_cov_precomp=covpre, cov3D=cov3D)
    fw, bw = h.run_oracle(sc, np.asarray(bg, np.float32), dL, **opts)
    a = h.run_module(ours, sc, bg, dL, **opts)
    a0 = h.run_module(ours, sc, bg, None, **opts)
    st = {k: v.cpu().numpy() for k, v in _C.inspect_state(P, W, H, a0["num_rendered"], a0["geom"], a0["binning"],
                                                           a0["img"]).items()}
    assert a["num_rendered"] == fw["num_rendered"]
    assert np.array_equal(a["radii"].cpu().numpy(), fw["radii"])
    vis = fw["radii"] > 0
    assert np.array_equal(st["tiles_touched"][vis].astype(np.uint32), fw["tiles_touched"][vis])
    assert np.array_equal(st["depths"][vis].view(np.uint32), fw["depths"][vis].view(np.uint32))
    assert np.array_equal(st["means2D"][vis].view(np.uint32), fw["means2D"][vis].view(np.uint32))
    assert np.array_equal(st["conic_opacity"][vis].view(np.uint32), fw["conic_opacity"][vis].view(np.uint32))
    assert np.array_equal(st["keys"].view(np.uint64), fw["keys"])
    assert np.array_equal(st["point_list"].view(np.uint32), fw["point_list"])
    assert np.array_equal(st["ranges"].view(np.uint32), fw["ranges"])
    # glibc expf vs MUFU.EX2: alpha may differ in the last ulp, so a pair sitting exactly on the
    # 1/255 or T<1e-4 threshold can flip; allow a handful of pixels to differ by one contributor.
    nc = st["n_contrib"].view(np.uint32)
    flips = int((nc != fw["n_contrib"]).sum())
    assert flips <= max(2, W * H // 5000), f"{flips} n_contrib mismatches"
    img = a["color"].cpu().numpy()
    d = np.abs(img - fw["color"])
    assert np.quantile(d, 0.999) < 2e-6 and d.max() < 5e-3, (float(np.quantile(d, 0.999)), float(d.max()))
    names = dict(means3D="dL_dmeans3D", means2D="dL_dmeans2D", opacities="dL_dopacity", shs="dL_dsh",
                 colors_precomp="dL_dcolors", scales="dL_dscales", rotations="dL_drotations", cov3D_precomp="dL_dcov3D")
    for k, g in a["grads"].items():
        err = h.rel_err(g.cpu().numpy().reshape(bw[names[k]].shape), bw[names[k]])
        assert err <= 5e-4, f"grad {k}: rel err vs oracle {err:.3e}"


def test_mark_visible_and_empty():
    import torch
    from sugar_b200 import diff_gaussian_rasterization as ours, scenes
    from oracle import raster_oracle as ro
    sc = scenes.make_scene(5000, 64, 48, seed=3, camera="posed", frac_behind=0.3)
    t = h.to_torch(sc)
    st = ours.GaussianRasterizationSettings(48, 64, sc.tanfovx, sc.tanfovy, torch.zeros(3, device="cuda"), 1.0,
                                            t["viewmatrix"], t["projmatrix"], 0, t["campos"], False, False)
    r = ours.GaussianRasterizer(st)
    got = r.markVisible(t["means3D"]).cpu().numpy()
    assert np.array_equal(got, ro.mark_visible(sc.means3D, sc.viewmatrix, sc.projmatrix))
    # P == 0: zeros, nothing launched (rasterize_points.cu:81)
    e = torch.zeros((0, 3), device="cuda")
    color, radii = r(means3D=e, means2D=e, opacities=torch.zeros((0, 1), device="cuda"),
                     colors_precomp=e, scales=e, rotations=torch.zeros((0, 4), device="cuda"))
    assert color.shape == (3, 48, 64) and float(color.abs().sum()) == 0.0 and radii.numel() == 0
    with pytest.raises(Exception):
        r(means3D=t["means3D"], means2D=t["means3D"], opacities=t["opacities"])


def test_full_size_properties():
    """BASELINE config sizes: properties that need no oracle (sortedness, conservation, idempotence)."""
    import torch
    from sugar_b200 import diff_gaussian_rasterization as ours, scenes, _C
    P, W, H = 1_000_000, 1920, 1080
    sc = scenes.make_scene(P, W, H, seed=0)
    a = h.run_module(ours, sc, (0, 0, 0), scenes.upstream_grad(W, H), use_sh=True, sh_degree=3)
    a0 = h.run_module(ours, sc, (0, 0, 0), None, use_sh=True, sh_degree=3)
    st = _C.inspect_state(P, W, H, a0["num_rendered"], a0["geom"], a0["binning"], a0["img"])
    R = a0["num_rendered"]
    assert int(st["tiles_touched"].sum()) == R
    keys = st["keys"]
    assert bool((keys[1:] >= keys[:-1]).all()), "keys not sorted"
    eq = keys[1:] == keys[:-1]
    pl = st["point_list"].long()
    assert bool((pl[1:][eq] > pl[:-1][eq]).all()), "ties not in Gaussian-index order"
    rng = st["ranges"].long()
    assert int((rng[:, 1] - rng[:, 0]).sum()) == R
    assert torch.equal(a["color"], a0["color"]), "forward not deterministic"
    assert bool(torch.isfinite(a["color"]).all())
    for k, g in a["grads"].items():
        assert bool(torch.isfinite(g).all()), k
    ref = h.RefGolden("full_size")
    assert ref.num_rendered == R
    assert ref.same("radii", a["radii"])
    assert ref.same("color", a["color"]), "1M/1080p image not bit-exact"
    for k in ref.grad_names:
        err = ref.grad_err(k, a["grads"][k])
        assert err <= GRAD_RTOL, f"grad {k}: rel err {err:.3e}"


def _run_raw(mod, t, sc, bg, dL, sh_degree, shs, device="cuda"):
    """Call GaussianRasterizer of `mod` on explicit torch tensors (for layout / alignment variants)."""
    import torch
    leaf = lambda x: x.detach().requires_grad_(True)
    means3D, opac, scales, rots, shs = (leaf(x) for x in (t["means3D"], t["opacities"], t["scales"], t["rotations"], shs))
    means2D = torch.zeros_like(means3D, requires_grad=True)
    st = mod.GaussianRasterizationSettings(sc.height, sc.width, sc.tanfovx, sc.tanfovy,
                                           torch.tensor(bg, dtype=torch.float32, device=device), 1.0, t["viewmatrix"],
                                           t["projmatrix"], sh_degree, t["campos"], False, False)
    color, radii = mod.GaussianRasterizer(st)(means3D=means3D, means2D=means2D, opacities=opac, shs=shs, scales=scales,
                                              rotations=rots)
    (color * torch.from_numpy(dL).to(device)).sum().backward()
    return color.detach(), radii.detach(), dict(means3D=means3D.grad, opacities=opac.grad, scales=scales.grad,
                                                rotations=rots.grad, shs=shs.grad, means2D=means2D.grad)


SH_LAYOUTS = [(16, 3), (9, 2), (4, 1), (1, 0), (16, 1)]


def run_sh_layout(mod, M, deg):
    """The inputs of test_sh_layouts_and_misaligned_inputs through `mod` -> (color, radii, grads)."""
    from sugar_b200 import scenes
    P, W, H = 3001, 150, 90
    sc = scenes.make_scene(P + 1, W, H, seed=40 + M, camera="posed")
    dL = scenes.upstream_grad(W, H)
    t = h.to_torch(sc)
    # slices that start one row into a larger allocation: contiguous but NOT 16-byte aligned (except rotations)
    tt = {k: (v[1:] if k in ("means3D", "scales", "rotations", "opacities", "shs") else v) for k, v in t.items()}
    shs = tt["shs"][:, :M, :].contiguous() if M != 16 else tt["shs"]
    assert tt["means3D"].data_ptr() % 16 != 0
    return _run_raw(mod, tt, sc, (0.2, 0.1, 0.3), dL, deg, shs)


@pytest.mark.parametrize("M,deg", SH_LAYOUTS)
def test_sh_layouts_and_misaligned_inputs(M, deg):
    """Stored SH count M != 16 (rows not 16-byte multiples -> 4-byte cp.async path) and inputs that start at a
    12-byte offset (no TMA bulk copy possible -> plain staging path); forward bit-exact, grads 1e-4 against
    what the reference build computed on the same inputs."""
    from sugar_b200 import diff_gaussian_rasterization as ours
    ref = h.RefGolden(f"sh_layout.{M}_{deg}")
    a = run_sh_layout(ours, M, deg)
    assert ref.same("radii", a[1])
    assert ref.same("color", a[0]), "image not bit-exact"
    assert set(a[2]) == ref.grad_names
    for k in ref.grad_names:
        err = ref.grad_err(k, a[2][k])
        assert err <= GRAD_RTOL, f"grad {k}: {err:.2e}"


def test_debug_flag_and_argument_errors():
    import torch
    from sugar_b200 import diff_gaussian_rasterization as ours, scenes, _lib
    sc = scenes.make_scene(500, 64, 48, seed=2)
    out = h.run_module(ours, sc, (0, 0, 0), scenes.upstream_grad(64, 48), use_sh=True, sh_degree=3, debug=True)
    assert bool(torch.isfinite(out["color"]).all())
    t = h.to_torch(sc)
    st = ours.GaussianRasterizationSettings(48, 64, sc.tanfovx, sc.tanfovy, torch.zeros(3, device="cuda"), 1.0,
                                            t["viewmatrix"], t["projmatrix"], 3, t["campos"], False, False)
    r = ours.GaussianRasterizer(st)
    with pytest.raises(Exception, match="excatly one"):
        r(means3D=t["means3D"], means2D=t["means3D"], opacities=t["opacities"], shs=t["shs"],
          colors_precomp=t["colors_precomp"], scales=t["scales"], rotations=t["rotations"])
    with pytest.raises(Exception, match="exactly one"):
        r(means3D=t["means3D"], means2D=t["means3D"], opacities=t["opacities"], shs=t["shs"], scales=t["scales"])
    with pytest.raises(RuntimeError, match="num_points, 3"):
        r(means3D=t["means3D"].reshape(-1), means2D=t["means3D"], opacities=t["opacities"], shs=t["shs"],
          scales=t["scales"], rotations=t["rotations"])
    with pytest.raises(_lib.SgrError):  # sh_degree 3 needs 16 coefficients
        r(means3D=t["means3D"], means2D=t["means3D"], opacities=t["opacities"], shs=t["shs"][:, :4].contiguous(),
          scales=t["scales"], rotations=t["rotations"])
    with pytest.raises(Exception):      # CPU tensors: no CPU path
        cpu = {k: v.cpu() for k, v in t.items()}
        st2 = st._replace(bg=torch.zeros(3), viewmatrix=cpu["viewmatrix"], projmatrix=cpu["projmatrix"], campos=cpu["campos"])
        ours.GaussianRasterizer(st2)(means3D=cpu["means3D"], means2D=cpu["means3D"], opacities=cpu["opacities"],
                                     shs=cpu["shs"], scales=cpu["scales"], rotations=cpu["rotations"])


def test_headline_size_linear_properties():
    """3M Gaussians / 1920x1080 (the bench workload): background linearity through final_T and linearity of
    the backward in the upstream gradient -- properties that need no element-wise reference
    (helpers.check_linear_properties; the same checker runs on the CPU oracle in test_oracle_properties.py)."""
    from sugar_b200 import diff_gaussian_rasterization as ours, scenes
    P, W, H = 3_000_000, 1920, 1080
    sc = scenes.make_scene(P, W, H, seed=0)

    def run(bg, dL):
        o = h.run_module(ours, sc, bg, dL, use_sh=True, sh_degree=3)
        grads = None if dL is None else {k: v.cpu().numpy() for k, v in o["grads"].items()}
        return o["color"].cpu().numpy(), o["radii"].cpu().numpy(), grads
    h.check_linear_properties(run, W, H, tol_img=1e-5, tol_grad=1e-4)
