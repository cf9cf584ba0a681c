"""Record what the UNMODIFIED reference CUDA build (oracle/_ref, made by oracle/build_ref.py) computes for every
GPU test that compares with it, as tests/golden/reference_build.npz (helpers.record_reference / RefGolden).

Needs a B200 and oracle/_ref:   python tests/golden/make_reference_build_golden.py OUT.npz
Inputs are not stored: the tests regenerate them from their seeds (sugar_b200.scenes, numpy PCG64) or read
tests/golden/render_wrapper.npz.  Arrays the tests hold bit-exact are stored as sha256 digests; gradients as
a fixed sample plus their largest elements and |.|_inf (each file under tests/ stays far below 1 MB).
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def main(out_path):
    import torch
    import helpers as h
    import test_gpu_configs as tc
    import test_gpu_parity as tp
    from sugar_b200 import scenes
    ref = h.load_ref_module()
    rec = {}

    for name, P, W, H, camera, use_sh, deg, covpre, bg in tp.CASES:
        sc = tp._scene(name, P, W, H, camera)
        cov3D = tp._cov_from_oracle(sc) if covpre else None
        opts = dict(use_sh=use_sh, sh_degree=deg, use_cov_precomp=covpre, cov3D=cov3D)
        b = h.run_module(ref, sc, bg, None, **opts)
        rs = h.decode_ref_state(b, P, W, H)
        same = {k: x for k, (x, _) in tp.compared_state(b["radii"], rs, use_sh).items()}
        same.update(radii=b["radii"], color=b["color"])
        dL = scenes.upstream_grad(W, H)
        gb, gb2 = (h.run_module(ref, sc, bg, dL, **opts)["grads"] for _ in range(2))
        h.record_reference(rec, "parity." + name, b["num_rendered"], same, gb, gb2)
        print("parity", name, "R =", b["num_rendered"], flush=True)

    P, W, H = 1_000_000, 1920, 1080
    b = h.run_module(ref, scenes.make_scene(P, W, H, seed=0), (0, 0, 0), scenes.upstream_grad(W, H), use_sh=True,
                     sh_degree=3)
    h.record_reference(rec, "full_size", b["num_rendered"], dict(radii=b["radii"], color=b["color"]), b["grads"])
    print("full_size R =", b["num_rendered"], flush=True)

    for M, deg in tp.SH_LAYOUTS:
        color, radii, grads = tp.run_sh_layout(ref, M, deg)
        h.record_reference(rec, f"sh_layout.{M}_{deg}", None, dict(radii=radii, color=color), grads)
    print("sh layouts", tp.SH_LAYOUTS, flush=True)

    for name, P, W, H, deg, mesh in tc.CONFIGS:
        sc = scenes.make_scene(P, W, H, seed=0, mesh_bound=mesh)
        dL = scenes.upstream_grad(W, H)
        b = h.run_module(ref, sc, (0.0, 0.0, 0.0), dL, use_sh=True, sh_degree=deg)
        rs = h.decode_ref_state(b, P, W, H)
        same = {k: rs[k] for k in tc.CONFIG_STATE}
        same.update(radii=b["radii"], color=b["color"])
        gb2 = h.run_module(ref, sc, (0.0, 0.0, 0.0), dL, use_sh=True, sh_degree=deg)["grads"] if mesh else None
        h.record_reference(rec, "config." + name, b["num_rendered"], same, b["grads"], gb2)
        print("config", name, "R =", b["num_rendered"], flush=True)
        del b, rs, same, gb2
        torch.cuda.empty_cache()

    g = np.load(os.path.join(ROOT, "tests", "golden", "render_wrapper.npz"))
    t = lambda k: torch.from_numpy(g[k]).cuda()
    H, W = (int(v) for v in g["hw"])
    st = ref.GaussianRasterizationSettings(
        image_height=H, image_width=W, tanfovx=float(g["tanfov"][0]), tanfovy=float(g["tanfov"][1]), bg=t("bg"),
        scale_modifier=1.0, viewmatrix=t("viewmatrix"), projmatrix=t("projmatrix"), sh_degree=int(g["sh_degree"]),
        campos=t("campos"), prefiltered=False, debug=False)
    m3 = t("means3D")
    img, radii = ref.GaussianRasterizer(st)(means3D=m3, means2D=torch.zeros_like(m3), opacities=t("opacities"),
                                            colors_precomp=t("colors_precomp"), scales=t("scales"), rotations=t("rotations"))
    h.record_reference(rec, "render", same=dict(image=img, radii=radii))

    rec["device"] = np.array(torch.cuda.get_device_name(0))
    rec["torch"] = np.array(torch.__version__)
    np.savez_compressed(out_path, **rec)
    print("wrote", out_path, os.path.getsize(out_path), "bytes;", rec["device"], "torch", rec["torch"])


if __name__ == "__main__":
    main(sys.argv[1])
