"""Shared test plumbing: run the same seeded scene through (a) the sugar_b200 CUDA path,
(b) the CPU oracle, (c) the unmodified reference CUDA build in oracle/_ref (when present), or
compare with what (c) computed on a B200, stored in tests/golden/reference_build.npz."""
import hashlib
import importlib
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF_DIR = os.path.join(ROOT, "oracle", "_ref")
REF_GOLDEN = os.path.join(ROOT, "tests", "golden", "reference_build.npz")
GRAD_SAMPLE, GRAD_TOP = 128, 32   # elements of each gradient kept in REF_GOLDEN: a fixed spread + the largest


def scene_kwargs(sc, use_sh=True, use_cov_precomp=False, sh_degree=3, cov3D=None):
    kw = dict(means3D=sc.means3D, opacities=sc.opacities, viewmatrix=sc.viewmatrix, projmatrix=sc.projmatrix,
              campos=sc.campos, W=sc.width, H=sc.height, tanfovx=sc.tanfovx, tanfovy=sc.tanfovy, sh_degree=sh_degree)
    if use_sh:
        kw["shs"] = sc.shs
    else:
        kw["colors_precomp"] = sc.colors_precomp
    if use_cov_precomp:
        kw["cov3D_precomp"] = cov3D
    else:
        kw["scales"] = sc.scales
        kw["rotations"] = sc.rotations
    return kw


def run_oracle(sc, bg, dL=None, **opts):
    from oracle import raster_oracle as ro
    kw = scene_kwargs(sc, **opts)
    fw = ro.forward(bg=bg, **kw)
    bw = ro.backward(fw, dL) if dL is not None else None
    return fw, bw


def have_ref():
    return os.path.exists(os.path.join(REF_DIR, "diff_gaussian_rasterization", "_C.so"))


def load_ref_module():
    """Import the reference build under its own name without shadowing ours."""
    if "diff_gaussian_rasterization_ref" in sys.modules:
        return sys.modules["diff_gaussian_rasterization_ref"]
    import torch  # noqa: F401  (the extension links libtorch)
    spec = importlib.util.spec_from_file_location(
        "diff_gaussian_rasterization_ref", os.path.join(REF_DIR, "diff_gaussian_rasterization", "__init__.py"),
        submodule_search_locations=[os.path.join(REF_DIR, "diff_gaussian_rasterization")])
    mod = importlib.util.module_from_spec(spec)
    sys.modules["diff_gaussian_rasterization_ref"] = mod
    spec.loader.exec_module(mod)
    return mod


def _numpy(x):
    return x.detach().cpu().numpy() if hasattr(x, "detach") else np.asarray(x)


def digest(x):
    """sha256 of an array's shape, dtype and bytes, integer and bool arrays widened to int64 first (torch.equal compares
    integers by value across dtypes): equal digests <=> equal integer arrays / bit-identical float arrays."""
    a = _numpy(x)
    a = np.ascontiguousarray(a.astype(np.int64) if a.dtype.kind in "biu" else a)
    return hashlib.sha256(repr(a.shape).encode() + a.dtype.str.encode() + a.tobytes()).hexdigest()


def sample_index(numel, n=GRAD_SAMPLE):
    """n flat indices spread over [0, numel) by Fibonacci hashing: integer arithmetic, the same on every platform."""
    k = np.arange(n, dtype=np.uint64) * np.uint64(0x9E3779B97F4A7C15)
    return np.unique(k % np.uint64(max(numel, 1))).astype(np.int64)


def _grad_index(numel, top):
    return np.unique(np.concatenate([sample_index(numel), np.asarray(top, np.int64)]))


def record_reference(rec, prefix, num_rendered=None, same=None, grads=None, grads2=None):
    """Add to `rec` (name -> array, saved as REF_GOLDEN) what RefGolden(prefix) reads back: the sha256 digests of `same`
    (the arrays a test holds bit-identical) and of each gradient its shape, |.|_inf, values at sample_index() and at its
    GRAD_TOP largest elements and, given `grads2` (a second run of the reference), its run-to-run rel err."""
    import torch
    if num_rendered is not None:
        rec[f"{prefix}.num_rendered"] = np.int64(num_rendered)
    if same:
        rec[f"{prefix}.sha256"] = np.array([(k, digest(x)) for k, x in same.items()], dtype="S64")
    if not grads:
        return
    names = sorted(grads)
    shape, stats, top, values = [], [], [], []
    for k in names:
        flat = grads[k].detach().reshape(-1)
        t = flat.abs().topk(min(GRAD_TOP, flat.numel())).indices.cpu().numpy()
        idx = torch.from_numpy(_grad_index(flat.numel(), t)).to(flat.device)
        shape.append(list(grads[k].shape) + [-1] * (4 - grads[k].dim()))
        stats.append((flat.abs().max().item(), rel_err(_numpy(grads2[k]), _numpy(grads[k])) if grads2 is not None else np.nan))
        top.append(np.pad(t, (0, GRAD_TOP - t.size), constant_values=-1))
        values.append(flat[idx].cpu().numpy())
    rec[f"{prefix}.grads"] = np.array(names)
    rec[f"{prefix}.grad_shape"] = np.array(shape, np.int64)
    rec[f"{prefix}.grad_stats"] = np.array(stats, np.float64)      # |ref|_inf, run-to-run rel err
    rec[f"{prefix}.grad_top"] = np.array(top, np.int32)
    rec[f"{prefix}.grad_values"] = np.concatenate(values).astype(np.float32)


_GOLDEN = {}


class RefGolden:
    """What the unmodified reference CUDA build computed for one test case on a B200 (written by record_reference,
    tests/golden/make_reference_build_golden.py)."""

    def __init__(self, prefix):
        if not _GOLDEN:
            with np.load(REF_GOLDEN) as z:
                _GOLDEN.update((k, z[k]) for k in z.files)
        self.prefix = prefix
        assert any(k.startswith(prefix + ".") for k in _GOLDEN), f"{prefix} not in {REF_GOLDEN}"
        self.digests = {n.decode(): d.decode() for n, d in self.get("sha256", np.zeros((0, 2), "S64"))}
        self.grad_names = {str(k) for k in self.get("grads", [])}
        self._grads, off = {}, 0
        for i, k in enumerate(self.get("grads", [])):
            shape = tuple(int(v) for v in self["grad_shape"][i] if v >= 0)
            top = self["grad_top"][i]
            idx = _grad_index(int(np.prod(shape)), top[top >= 0])
            self._grads[str(k)] = (shape, idx, self["grad_values"][off:off + idx.size], *self["grad_stats"][i])
            off += idx.size

    def __getitem__(self, k):
        return _GOLDEN[f"{self.prefix}.{k}"]

    def get(self, k, default=None):
        return _GOLDEN.get(f"{self.prefix}.{k}", default)

    @property
    def num_rendered(self):
        return int(self["num_rendered"])

    def same(self, k, x):
        """x equals the reference's array k bit for bit."""
        return digest(x) == self.digests[k]

    def grad_err(self, k, g):
        """|g - ref|_inf / |ref|_inf of gradient k over the reference's stored elements."""
        shape, idx, values, absmax, _ = self._grads[k]
        assert tuple(g.shape) == shape, f"grad {k}: shape {tuple(g.shape)}, reference {shape}"
        d = np.abs(_numpy(g).reshape(-1)[idx].astype(np.float64) - values).max()
        return float(d / max(absmax, 1e-30))

    def noise(self, k):
        """The reference's own run-to-run rel err of gradient k (fp32 atomics)."""
        return float(self._grads[k][4])


def to_torch(sc, device="cuda"):
    import torch
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(device)
    return {k: t(getattr(sc, k)) for k in ("means3D", "scales", "rotations", "opacities", "shs", "colors_precomp",
                                           "viewmatrix", "projmatrix", "campos")}


def run_module(mod, sc, bg, dL=None, use_sh=True, use_cov_precomp=False, sh_degree=3, cov3D=None, device="cuda",
               debug=False):
    """Run GaussianRasterizer of `mod` (ours or the reference build).  Returns dict with image, radii, grads and
    the saved opaque buffers."""
    import torch
    t = to_torch(sc, device)
    leaf = lambda x: x.clone().requires_grad_(True)
    means3D = leaf(t["means3D"]); opac = leaf(t["opacities"])
    means2D = torch.zeros_like(means3D, requires_grad=True)
    settings = mod.GaussianRasterizationSettings(
        image_height=sc.height, image_width=sc.width, tanfovx=sc.tanfovx, tanfovy=sc.tanfovy,
        bg=torch.from_numpy(np.asarray(bg, np.float32)).to(device), scale_modifier=1.0, viewmatrix=t["viewmatrix"],
        projmatrix=t["projmatrix"], sh_degree=sh_degree, campos=t["campos"], prefiltered=False, debug=debug)
    rast = mod.GaussianRasterizer(raster_settings=settings)
    kw = {}
    leaves = dict(means3D=means3D, means2D=means2D, opacities=opac)
    if use_sh:
        leaves["shs"] = kw["shs"] = leaf(t["shs"])
    else:
        leaves["colors_precomp"] = kw["colors_precomp"] = leaf(t["colors_precomp"])
    if use_cov_precomp:
        leaves["cov3D_precomp"] = kw["cov3D_precomp"] = leaf(torch.from_numpy(cov3D).to(device))
    else:
        leaves["scales"] = kw["scales"] = leaf(t["scales"])
        leaves["rotations"] = kw["rotations"] = leaf(t["rotations"])
    color, radii = rast(means3D=means3D, means2D=means2D, opacities=opac, **kw)
    out = dict(color=color.detach(), radii=radii.detach())
    fn = color.grad_fn
    saved = fn.saved_tensors if fn is not None else None
    if saved is not None:
        out["geom"], out["binning"], out["img"] = saved[7], saved[8], saved[9]
        out["num_rendered"] = fn.num_rendered
    if dL is not None:
        (color * torch.from_numpy(dL).to(device)).sum().backward()
        out["grads"] = {k: v.grad.detach() for k, v in leaves.items() if v.grad is not None}
    return out


def decode_ref_state(out, P, W, H):
    """Decode the reference's GeometryState / BinningState / ImageState chunks
    (rasterizer_impl.cu:155-194: 128-byte aligned bump allocation, in this order)."""
    import torch
    R = out["num_rendered"]

    def carve(buf, specs):
        base = buf.data_ptr()
        off = 0
        res = {}
        for name, dtype, count in specs:
            addr = (base + off + 127) & ~127
            off = addr - base
            nbytes = count * torch.empty((), dtype=dtype).element_size()
            res[name] = buf[off:off + nbytes].view(dtype)
            off += nbytes
        return res
    g = carve(out["geom"], [("depths", torch.float32, P), ("clamped", torch.uint8, 3 * P),
                            ("internal_radii", torch.int32, P), ("means2D", torch.float32, 2 * P),
                            ("cov3D", torch.float32, 6 * P), ("conic_opacity", torch.float32, 4 * P),
                            ("rgb", torch.float32, 3 * P), ("tiles_touched", torch.int32, P)])
    b = carve(out["binning"], [("point_list", torch.int32, R), ("point_list_unsorted", torch.int32, R),
                               ("keys", torch.int64, R)])
    i = carve(out["img"], [("final_T", torch.float32, W * H), ("n_contrib", torch.int32, W * H),
                           ("ranges", torch.int32, 2 * W * H)])
    T = ((W + 15) // 16) * ((H + 15) // 16)
    return dict(depths=g["depths"], clamped=g["clamped"].view(P, 3), means2D=g["means2D"].view(P, 2),
                cov3D=g["cov3D"].view(P, 6), conic_opacity=g["conic_opacity"].view(P, 4), rgb=g["rgb"].view(P, 3),
                tiles_touched=g["tiles_touched"], point_list=b["point_list"], keys=b["keys"],
                final_T=i["final_T"].view(H, W), n_contrib=i["n_contrib"].view(H, W),
                ranges=i["ranges"][:2 * T].view(T, 2))


def rel_err(a, b):
    """|a-b|_inf / |b|_inf (per-tensor relative error, SURVEY section 7 'hard parts')."""
    a = np.asarray(a, np.float64); b = np.asarray(b, np.float64)
    d = np.abs(a - b).max() if a.size else 0.0
    return d / max(np.abs(b).max() if b.size else 0.0, 1e-30)


def grad_sensitivity(sc, bg, dL, eps=1e-6, **opts):
    """Conditioning probe for the per-Gaussian backward chain (CPU oracle): relative change (|.|_inf / |g|_inf)
    of each returned gradient when the blend accumulators dL_dmeans2D / dL_dconic are perturbed by `eps`
    relative noise, i.e. by what fp32 summation order alone does to them.  For surface-aligned Gaussians
    with a 1e-6 axis, eps = 1e-6 moves dL_drotations by ~1e-4: there a fixed 1e-4 bar measures the
    conditioning of the reference's formula, not the implementation."""
    import ctypes as C
    from oracle import raster_oracle as ro
    fw, bw = run_oracle(sc, np.asarray(bg, np.float32), dL, **opts)
    L, i, _p = ro.lib(), fw["_in"], ro._p
    P, W, H, M, D = fw["P"], fw["W"], fw["H"], fw["M"], fw["D"]
    cov3Ds = i["cov3D_precomp"] if i["cov3D_precomp"] is not None else fw["cov3D"]

    def chain(dm2d, dconic):
        g = dict(means3D=np.zeros((P, 3), np.float32), cov3D_precomp=np.zeros((P, 6), np.float32),
                 shs=np.zeros((P, max(M, 1), 3), np.float32), scales=np.zeros((P, 3), np.float32),
                 rotations=np.zeros((P, 4), np.float32))
        L.oracle_preprocess_backward(
            C.c_int(P), C.c_int(D), C.c_int(M), _p(i["means3D"]), _p(fw["radii"]), _p(i["shs"]), _p(fw["clamped"]),
            _p(i["scales"]), _p(i["rotations"]), C.c_float(i["scale_modifier"]), _p(cov3Ds), _p(i["viewmatrix"]),
            _p(i["projmatrix"]), C.c_int(W), C.c_int(H), C.c_float(i["tanfovx"]), C.c_float(i["tanfovy"]),
            _p(i["campos"]), _p(dm2d), _p(dconic), _p(bw["dL_dcolors"].copy()), _p(g["means3D"]), _p(g["cov3D_precomp"]),
            _p(g["shs"]), _p(g["scales"]), _p(g["rotations"]))
        return g
    base = chain(bw["dL_dmeans2D"].copy(), bw["dL_dconic"].copy())
    rng = np.random.default_rng(0)
    noisy = lambda a: (a * (1 + eps * rng.standard_normal(a.shape))).astype(np.float32)
    pert = chain(noisy(bw["dL_dmeans2D"]), noisy(bw["dL_dconic"]))
    return {k: float(np.abs(pert[k] - base[k]).max() / max(np.abs(base[k]).max(), 1e-30)) for k in base}


def check_linear_properties(run, W, H, tol_img=1e-5, tol_grad=1e-4):
    """Size-independent invariants of the rasterizer, for any implementation behind
    run(bg, dL) -> (color f32[3,H,W], radii, {name: grad} or None), all numpy:
      * the background enters as  image(bg) = image(0) + final_T * bg  with one final_T for the three channels
        (forward.cu:361-367), and radii do not depend on it;
      * the backward is linear in the upstream image gradient.
    The CPU suite runs it on the oracle (small), the GPU suite on the CUDA path at the headline size."""
    from sugar_b200 import scenes
    c0, r0, _ = run((0.0, 0.0, 0.0), None)
    c1, r1, _ = run((1.0, 1.0, 1.0), None)
    T = c1 - c0
    assert np.abs(T[0] - T[1]).max() <= tol_img and np.abs(T[0] - T[2]).max() <= tol_img
    assert T.min() >= -tol_img and T.max() <= 1.0 + tol_img
    bg2 = np.array([0.25, 0.5, 1.0], np.float32)
    c2, r2, _ = run(tuple(float(v) for v in bg2), None)
    assert np.abs(c2 - (c0 + T[0][None] * bg2[:, None, None])).max() <= 2 * tol_img
    assert np.array_equal(r0, r1) and np.array_equal(r0, r2)
    d1, d2 = scenes.upstream_grad(W, H, seed=1), scenes.upstream_grad(W, H, seed=2)
    a, b = 0.75, -1.5
    g1, g2 = run((0.0, 0.0, 0.0), d1)[2], run((0.0, 0.0, 0.0), d2)[2]
    g12 = run((0.0, 0.0, 0.0), (a * d1 + b * d2).astype(np.float32))[2]
    assert set(g1) == set(g12) and len(g12) >= 5
    for k in g12:
        err = rel_err(g12[k], a * g1[k] + b * g2[k])
        assert err <= tol_grad, f"backward not linear in dL for {k}: {err:.2e}"
