"""Generates tests/golden/ref_raster_views.npz and tests/golden/ref_raster_full_size.npz: what the UNMODIFIED reference
rasterizer (oracle/_ref/libref_dgr.so, built by oracle/build_ref.sh from the reference sources) renders on a B200 for the
inputs of the parity tests in tests/test_gpu_raster.py and tests/test_gpu_pipeline.py, which compare against these files.

    python tests/golden/make_ref_parity_golden.py OUT_DIR      # on a B200, with oracle/_ref built

Exact outputs (radii, tiles touched, the full-precision transmittance frame) are stored as sha256 digests, images as the
fixed pixel sample of tests/raster_compare.fixed_sample (the first N of a longer sample are the sample of N, so the arrays
may be shortened afterwards), per-Gaussian values for a fixed sample of the visible Gaussians.  Every case carries the
digest of its inputs."""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from gs2mesh_b200 import camera as cam  # noqa: E402
from gs2mesh_b200 import scene  # noqa: E402
from oracle import oracle as orc  # noqa: E402
from tests import test_gpu_pipeline as tp  # noqa: E402
from tests import test_gpu_raster as tr  # noqa: E402
from tests.raster_compare import digest, fixed_sample, sample_image  # noqa: E402

N_PIXELS_VIEWS = 2048  # pixels kept per frame of the small parity cases
N_PIXELS_FULL = 1024  # per frame of the full-size cases
N_GAUSSIANS = 512  # visible Gaussians kept for the per-Gaussian comparison


def small_cases(dev):
    out = {}
    for n, W, H, seed in tr.REF_CASES + [tr.PINNED_CASE]:
        key = tr.case_key(n, W, H, seed)
        g, vt = tr._case(n, W, H, seed)
        inp = tr._np_inputs(g, vt)
        t = lambda a: None if a is None else torch.as_tensor(np.ascontiguousarray(a, dtype=np.float32)).to(dev)
        ref = orc.ref_forward_torch(t(inp["means3D"]), t(inp["opacities"]).reshape(-1), t(inp["view"]), t(inp["proj"]),
                                    t(inp["campos"]), W, H, inp["tan_fovx"], inp["tan_fovy"], t(inp["bg"]), shs=t(inp["shs"]),
                                    scales=t(inp["scales"]), rotations=t(inp["rotations"]), sh_degree=inp["sh_degree"],
                                    scale_modifier=inp["scale_modifier"], want_geometry=True)
        ref = {k: (v.cpu().numpy() if hasattr(v, "cpu") else v) for k, v in ref.items()}
        c = dict(inputs_sha256=tr.inputs_sha256(inp), radii_sha256=digest(ref["radii"]), num_rendered=ref["num_rendered"],
                 color=sample_image(ref["color"], N_PIXELS_VIEWS), final_T=sample_image(ref["final_T"], N_PIXELS_VIEWS))
        if (n, W, H, seed) == tr.PINNED_CASE:
            vis = np.flatnonzero(ref["radii"] > 0)
            gi = vis[fixed_sample(len(vis), N_GAUSSIANS)]
            c.update(tiles_touched_sha256=digest(ref["tiles_touched"].astype(np.uint32)),
                     **{k: ref[k][gi] for k in ("depths", "xy", "conic_opacity", "rgb")})
        out.update({f"{key}__{k}": np.asarray(v) for k, v in c.items()})
        print("views", key, ref["num_rendered"], flush=True)
    return out


def full_size_cases(dev):
    out = {}
    for case, cfg in tp.FULL_SIZE_CASES.items():
        W, H = cfg["width"], cfg["height"]
        cloud = scene.make_gaussians(cfg["num_points"], seed=1)
        rigs, _ = scene.make_stereo_cameras(8, W, H, layout=cfg["layout"], principal_point=cfg.get("principal_point"))
        up = lambda a: torch.as_tensor(np.ascontiguousarray(a, dtype=np.float32)).to(dev)
        g = dict(xyz=up(cloud.xyz), op=up(cloud.opacity).reshape(-1), sh=up(cloud.features), sc=up(cloud.scaling),
                 ro=up(cloud.rotation))
        for side, name in enumerate(("left", "right")):
            vt = cam.view_transforms_from_camera(rigs[tp.FULL_SIZE_VIEW][name])
            rec = np.asarray(vt.packed(), np.float32)
            rt = up(rec)
            ref = orc.ref_forward_torch(g["xyz"], g["op"], rt[0:16], rt[16:32], rt[32:35], W, H, vt.tan_fovx, vt.tan_fovy,
                                        torch.zeros(3, device=dev), shs=g["sh"], scales=g["sc"], rotations=g["ro"], sh_degree=3)
            T = ref["final_T"].cpu().numpy()
            c = dict(inputs_sha256=tp.full_size_inputs_sha256(cloud, rec), num_rendered=ref["num_rendered"],
                     final_T_sha256=digest(T + np.float32(0)), color=sample_image(ref["color"].cpu().numpy(), N_PIXELS_FULL),
                     final_T=sample_image(T, N_PIXELS_FULL))
            out.update({f"{case}-side{side}__{k}": np.asarray(v) for k, v in c.items()})
            print("full size", case, side, ref["num_rendered"], flush=True)
        del g
        torch.cuda.empty_cache()
    return out


def main():
    out_dir = sys.argv[1]
    os.makedirs(out_dir, exist_ok=True)
    if not orc.ref_available():
        raise SystemExit("oracle/_ref/libref_dgr.so is missing: build it with oracle/build_ref.sh first")
    dev = torch.device("cuda", 0)
    np.savez_compressed(os.path.join(out_dir, "ref_raster_views.npz"), **small_cases(dev))
    np.savez_compressed(os.path.join(out_dir, "ref_raster_full_size.npz"), **full_size_cases(dev))


if __name__ == "__main__":
    main()
