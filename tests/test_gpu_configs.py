"""Element-wise parity with the UNMODIFIED reference CUDA build at every rasterizer configuration BASELINE.json
names, through the public module, against what that build computed on a B200 from the same seeded inputs
(tests/golden/reference_build.npz: digests of the arrays held bit-exact, sampled gradients):

    C2        100k Gaussians,   800x800,  SH degree 2
    C3          1M Gaussians, 1920x1080,  SH degree 3      (also tests/test_gpu_parity.py::test_full_size_properties)
    headline    3M Gaussians, 1920x1080,  SH degree 3      (the workload bench.py times)
    C4          3M mesh-bound (flat first axis, refine.py), 1600x1200, SH degree 3
    C5          6M Gaussians, 3840x2160,  SH degree 3      (one view of the 8-view batch)

Bars: num_rendered, radii, n_contrib equal; image and final_T bit-identical; every gradient
|a-b|_inf / |b|_inf <= 1e-4 (BASELINE.json).  Mesh-bound Gaussians (a 1e-6 axis) are the documented
exception for dL_dscales / dL_drotations: there the reference's own per-Gaussian chain amplifies the fp32
summation-order noise of the blend accumulators by ~1e3, so those two tensors are held to 5x the larger
of (the reference's own run-to-run difference, stored with its gradients; the chain's measured sensitivity to
1e-6 accumulator noise on a 1/64-area sample of the same distribution -- helpers.grad_sensitivity, CPU oracle).

Also here: the capacity-overflow re-run of the forward (rasterizer_impl.cu:281-317 sizes the binning
buffers after a host wait; ours guesses and must re-run binning when the guess was too small) and two
forwards in flight on two streams.
"""
import numpy as np
import pytest

import helpers as h

pytestmark = pytest.mark.gpu

GRAD_RTOL = 1e-4

CONFIGS = [
    # id, P, W, H, sh_degree, mesh_bound
    ("c2_100k_800x800_sh2", 100_000, 800, 800, 2, False),
    ("c3_1m_1080p_sh3", 1_000_000, 1920, 1080, 3, False),
    ("headline_3m_1080p_sh3", 3_000_000, 1920, 1080, 3, False),
    ("c4_3m_meshbound_1600x1200_sh3", 3_000_000, 1600, 1200, 3, True),
    ("c5_6m_4k_sh3", 6_000_000, 3840, 2160, 3, False),
]


# forward state held bit-identical at every configuration: name -> failure message
CONFIG_STATE = {"n_contrib": "n_contrib differs", "final_T": "final_T not bit-exact",
                "point_list": "sorted Gaussian ids differ", "keys": "sorted 64-bit keys differ",
                "ranges": "tile ranges differ"}


@pytest.mark.parametrize("cfg", CONFIGS, ids=[c[0] for c in CONFIGS])
def test_baseline_config_matches_reference_build(cfg):
    """Against what the reference build computed on the same seeded inputs (helpers.RefGolden)."""
    name, P, W, H, deg, mesh = cfg
    from sugar_b200 import _C, diff_gaussian_rasterization as ours, scenes
    ref = h.RefGolden("config." + name)
    sc = scenes.make_scene(P, W, H, seed=0, mesh_bound=mesh)
    dL = scenes.upstream_grad(W, H)
    bg = (0.0, 0.0, 0.0)
    a = h.run_module(ours, sc, bg, dL, use_sh=True, sh_degree=deg)
    assert a["num_rendered"] == ref.num_rendered
    assert ref.same("radii", a["radii"]), "radii differ"
    assert ref.same("color", a["color"]), "image not bit-exact"
    st = _C.inspect_state(P, W, H, a["num_rendered"], a["geom"], a["binning"], a["img"])
    for k, msg in CONFIG_STATE.items():
        assert ref.same(k, st[k]), msg
    del st
    assert set(a["grads"]) == ref.grad_names
    errs = {k: ref.grad_err(k, a["grads"][k]) for k in ref.grad_names}
    bad = {k: e for k, e in errs.items() if e > GRAD_RTOL}
    if bad and mesh:
        small = scenes.make_scene(P // 64, W // 8, H // 8, seed=0, mesh_bound=True)
        sens = h.grad_sensitivity(small, bg, scenes.upstream_grad(W // 8, H // 8), use_sh=True, sh_degree=deg)
        bad = {k: e for k, e in bad.items()
               if k not in ("scales", "rotations") or e > 5.0 * max(ref.noise(k), sens.get(k, 0.0))}
    assert not bad, f"{name}: gradient rel err over the bar: {bad} (all: {errs})"


def _forward_state(mod, sc, ctx=None):
    from sugar_b200 import _C
    if ctx is None:
        return h.run_module(mod, sc, (0.1, 0.2, 0.3), None, use_sh=True, sh_degree=3)
    with _C.use_context(ctx):
        return h.run_module(mod, sc, (0.1, 0.2, 0.3), None, use_sh=True, sh_degree=3)


def test_capacity_overflow_reruns_binning():
    """A capacity hint far below the true instance count: the guarded first attempt must be a no-op and the
    re-run (exact size) must give the same keys / ids / ranges / image as a run without any hint."""
    import torch
    from sugar_b200 import _C, diff_gaussian_rasterization as ours, scenes
    P, W, H = 200_000, 640, 360
    sc = scenes.make_scene(P, W, H, seed=11, camera="posed")
    dL = scenes.upstream_grad(W, H)
    cold = _C.Context()                       # no hint: waits for the count like the reference
    a = _forward_state(ours, sc, cold)
    R = a["num_rendered"]
    assert R > (1 << 16)
    key = (torch.cuda.current_device(), H, W)
    assert cold.capacity_hint[key] >= R       # the next view's optimistic capacity
    tiny = _C.Context()
    tiny.capacity_hint[key] = 1 << 12         # forces the overflow path
    with _C.use_context(tiny):
        b = h.run_module(ours, sc, (0.1, 0.2, 0.3), dL, use_sh=True, sh_degree=3)
    assert b["num_rendered"] == R and tiny.capacity_hint[key] >= R
    sa = _C.inspect_state(P, W, H, R, a["geom"], a["binning"], a["img"])
    sb = _C.inspect_state(P, W, H, R, b["geom"], b["binning"], b["img"])
    for k in ("keys", "point_list", "ranges", "n_contrib", "tiles_touched"):
        assert torch.equal(sa[k], sb[k]), k
    assert torch.equal(a["color"], b["color"]) and torch.equal(a["radii"], b["radii"])
    # backward after a re-run forward reads the right ranges: compare with a hinted (no overflow) run
    with _C.use_context(cold):
        c = h.run_module(ours, sc, (0.1, 0.2, 0.3), dL, use_sh=True, sh_degree=3)
    for k in c["grads"]:
        assert h.rel_err(b["grads"][k].cpu().numpy(), c["grads"][k].cpu().numpy()) <= GRAD_RTOL, k
    # a hint that is too small by ONE instance overflows too; one that is exact does not change anything
    for cap in (R - 1, R):
        ctx = _C.Context()
        ctx.capacity_hint[key] = cap
        d = _forward_state(ours, sc, ctx)
        assert d["num_rendered"] == R and torch.equal(d["color"], a["color"]), cap


def test_two_forwards_in_flight_on_two_streams():
    """Two different views enqueued back to back on two streams (per-call pinned slot + event on the C
    side): each must report its own instance count and image."""
    import torch
    from sugar_b200 import _C, diff_gaussian_rasterization as ours, scenes
    sc1 = scenes.make_scene(150_000, 640, 360, seed=21, camera="posed")
    sc2 = scenes.make_scene(60_000, 640, 360, seed=22, camera="posed", px_sigma=3.0)
    want1, want2 = _forward_state(ours, sc1, _C.Context()), _forward_state(ours, sc2, _C.Context())
    assert want1["num_rendered"] != want2["num_rendered"]
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    c1, c2 = _C.Context(), _C.Context()
    torch.cuda.synchronize()
    for _ in range(3):
        with torch.cuda.stream(s1):
            g1 = _forward_state(ours, sc1, c1)
        with torch.cuda.stream(s2):
            g2 = _forward_state(ours, sc2, c2)
        torch.cuda.synchronize()
        assert g1["num_rendered"] == want1["num_rendered"] and g2["num_rendered"] == want2["num_rendered"]
        assert torch.equal(g1["color"], want1["color"]) and torch.equal(g2["color"], want2["color"])


@pytest.mark.parametrize("scene_kw", [dict(), dict(px_sigma=6.0), dict(mesh_bound=True), dict(px_sigma=0.6)],
                         ids=["default", "large", "flat", "tiny"])
def test_footprint_masks_are_conservative_and_tight(scene_kw):
    """The per-instance footprint masks (which 8x4 blocks of its tile a splat can reach, computed once in the
    scatter kernel and used by both blend kernels to skip work) must never clear a block that holds a pixel
    passing the reference's alpha test (forward.cu:333-347), and should not be much looser than the truth."""
    import torch
    from sugar_b200 import _C, diff_gaussian_rasterization as ours, scenes
    P, W, H = 20_000, 320, 192
    sc = scenes.make_scene(P, W, H, seed=5, camera="posed", **scene_kw)
    a = h.run_module(ours, sc, (0, 0, 0), None, use_sh=True, sh_degree=1)
    R = a["num_rendered"]
    st = _C.inspect_state(P, W, H, R, a["geom"], a["binning"], a["img"])
    gx = (W + 15) // 16
    tile = (st["keys"] >> 32).long()
    ids = st["point_list"].long()
    fp = st["footprint"].long()
    m2, co = st["means2D"][ids], st["conic_opacity"][ids]
    ty, tx = tile // gx, tile % gx
    px = (tx[:, None, None] * 16 + torch.arange(16, device="cuda")[None, None, :]).float()   # [R,1,16]
    py = (ty[:, None, None] * 16 + torch.arange(16, device="cuda")[None, :, None]).float()   # [R,16,1]
    dx, dy = m2[:, 0, None, None] - px, m2[:, 1, None, None] - py
    power = -0.5 * (co[:, 0, None, None] * dx * dx + co[:, 2, None, None] * dy * dy) - co[:, 1, None, None] * dx * dy
    alpha = torch.clamp(co[:, 3, None, None] * torch.exp(power), max=0.99)
    hit = (power <= 0) & (alpha >= 1.0 / 255.0)                                              # [R,16(y),16(x)]
    blocks = hit.view(R, 4, 4, 2, 8).any(dim=4).any(dim=2)                                   # [R, band, half]
    truth = (blocks.long() * (1 << (torch.arange(4, device="cuda")[:, None] * 2 + torch.arange(2, device="cuda")[None, :]))).sum((1, 2))
    missed = truth & ~fp
    assert int((missed != 0).sum()) == 0, "a footprint mask clears a block that holds a contributing pixel"
    pop = lambda v: sum(((v >> b) & 1) for b in range(8)).sum().item()
    assert pop(fp) <= 1.25 * pop(truth) + 64, (pop(fp), pop(truth))
    assert int((fp == 0).sum()) > 0  # some instances are dead in their tile (the rect is 3 sigma_max wide)


def test_unpacked_instance_lists_give_identical_results():
    """P > 2^24 Gaussians cannot carry the footprint mask next to the id; the blend kernels then compute it
    while staging.  SGR_FORCE_UNPACKED_IDS=1 selects that format at any P (read once per process, hence the
    subprocess): image, radii and gradients must equal the packed format's."""
    import os
    import subprocess
    import sys
    import tempfile
    import torch
    from sugar_b200 import diff_gaussian_rasterization as ours, scenes
    code = r'''
import sys, numpy as np, torch
sys.path.insert(0, %r); sys.path.insert(0, %r + "/tests")
import helpers as h
from sugar_b200 import diff_gaussian_rasterization as ours, scenes
sc = scenes.make_scene(60000, 480, 270, seed=9, camera="posed")
o = h.run_module(ours, sc, (0.2, 0.1, 0.0), scenes.upstream_grad(480, 270), use_sh=True, sh_degree=3)
np.savez(sys.argv[1], color=o["color"].cpu().numpy(), radii=o["radii"].cpu().numpy(), R=o["num_rendered"],
         **{"g_" + k: v.cpu().numpy() for k, v in o["grads"].items()})
''' % (h.ROOT, h.ROOT)
    with tempfile.TemporaryDirectory() as d:
        out = os.path.join(d, "u.npz")
        env = dict(os.environ, SGR_FORCE_UNPACKED_IDS="1")
        subprocess.run([sys.executable, "-c", code, out], check=True, env=env, timeout=600)
        u = np.load(out)
    sc = scenes.make_scene(60000, 480, 270, seed=9, camera="posed")
    p = h.run_module(ours, sc, (0.2, 0.1, 0.0), scenes.upstream_grad(480, 270), use_sh=True, sh_degree=3)
    assert int(u["R"]) == p["num_rendered"]
    assert np.array_equal(u["radii"], p["radii"].cpu().numpy())
    assert np.array_equal(u["color"].view(np.int32), p["color"].cpu().numpy().view(np.int32))
    for k, g in p["grads"].items():
        assert h.rel_err(u["g_" + k], g.cpu().numpy()) <= GRAD_RTOL, k
