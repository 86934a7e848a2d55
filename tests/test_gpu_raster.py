"""GPU parity tests of the rasterizer: CUDA path (through the C ABI) vs the CPU oracle and vs the
UNMODIFIED reference rasterizer built for sm_100a, same seeded inputs.  The reference's outputs were recorded on a B200
(tests/golden/make_ref_parity_golden.py -> tests/golden/ref_raster_views.npz): exact outputs as digests, images as a
fixed sample of their pixels.

Tolerance (north_star): 1e-4 relative fp32 per pixel, with an outlier budget for pixels where a
hard threshold of the algorithm flips (see tests/raster_compare.py).  Integer outputs (radii,
instance counts, sort order effects) are exact.
"""
import ctypes as C

import numpy as np
import pytest

from gs2mesh_b200 import camera as cam
from gs2mesh_b200 import scene
from tests.raster_compare import compare_images, digest, fixed_sample, inputs_digest, load_ref_golden, sample_image

pytestmark = pytest.mark.gpu

REF_CASES = [(3000, 320, 240, 0), (10000, 640, 480, 1), (777, 250, 130, 2)]  # (num_points, W, H, seed)
PINNED_CASE = (4000, 320, 240, 5)

BUDGET = 1e-4  # fraction of values allowed outside 1e-4 (hard thresholds flip on rounding); on these small frames one flipped
               # pixel is already 4e-6 .. 1e-5 of the values.  Full-size frames: tests/test_gpu_pipeline.py (4e-5, observed 4e-6)
MAX_ERR = 0.05  # ceiling on the size of any single outlier (observed on B200: <= 3e-3)


def _case(num_points, W, H, seed=0, view=0, n_views=4, sh_degree=3):
    g = scene.make_gaussians(num_points, seed=seed, sh_degree=sh_degree)
    rigs, _ = scene.make_stereo_cameras(n_views, W, H)
    vt = cam.view_transforms_from_camera(rigs[view]["left"])
    return g, vt


def _np_inputs(g, vt, **over):
    d = dict(means3D=g.xyz, opacities=g.opacity, view=vt.world_view, proj=vt.full_proj, campos=vt.cam_center, W=vt.width,
             H=vt.height, tan_fovx=vt.tan_fovx, tan_fovy=vt.tan_fovy, bg=np.zeros(3, np.float32), shs=g.features,
             scales=g.scaling, rotations=g.rotation, sh_degree=g.sh_degree, scale_modifier=1.0)
    d.update(over)
    return {k: v for k, v in d.items() if v is not None or k in ()}


def _ours(dev, inp, flags=None, **kw):
    import torch

    from gs2mesh_b200 import rasterizer as rast

    t = lambda a: None if a is None else torch.as_tensor(np.ascontiguousarray(a, dtype=np.float32)).to(dev)
    out = rast.rasterize_forward(
        means3D=t(inp["means3D"]), opacities=t(inp["opacities"]).reshape(-1), viewmatrix=t(inp["view"]), projmatrix=t(inp["proj"]),
        campos=t(inp["campos"]), bg=t(inp["bg"]), width=inp["W"], height=inp["H"], tan_fovx=inp["tan_fovx"],
        tan_fovy=inp["tan_fovy"], shs=t(inp.get("shs")), colors_precomp=t(inp.get("colors_precomp")), scales=t(inp.get("scales")),
        rotations=t(inp.get("rotations")), cov3D_precomp=t(inp.get("cov3D_precomp")), sh_degree=inp["sh_degree"],
        scale_modifier=inp["scale_modifier"], flags=rast.DEFAULT_FLAGS if flags is None else flags, want_counts=True, **kw)
    torch.cuda.synchronize()
    return {k: (v.cpu().numpy() if v is not None else None) for k, v in out.items()}


def case_key(num_points, W, H, seed):
    return f"{num_points}-{W}-{H}-{seed}"


def inputs_sha256(inp):
    return inputs_digest(inp["means3D"], inp["opacities"], inp["shs"], inp["scales"], inp["rotations"], inp["view"], inp["proj"],
                         inp["campos"], inp["bg"], [inp["W"], inp["H"], inp["tan_fovx"], inp["tan_fovy"], inp["sh_degree"],
                                                    inp["scale_modifier"]])


def _ref(num_points, W, H, seed, inp):
    """The reference rasterizer's recorded outputs for this case (see the module docstring)."""
    return load_ref_golden("ref_raster_views.npz", case_key(num_points, W, H, seed), inputs_sha256(inp))


def _assert_parity(a, b, what, budget=BUDGET):
    r = compare_images(a, b)
    assert r["frac_bad"] <= budget, (what, r)
    assert r["median"] <= 1e-6, (what, r)
    assert r["max_err"] <= MAX_ERR, (what, r)


def _oracle_best(oracle, inp):
    o = oracle.forward(**inp)
    of = oracle.forward(fma=True, **inp)
    return o, of


@pytest.mark.parametrize("num_points,W,H,seed", [(3000, 320, 240, 0), (10000, 640, 480, 1), (777, 250, 130, 2)])
def test_cuda_matches_cpu_oracle(oracle, gsb_lib, cuda_device, num_points, W, H, seed):
    g, vt = _case(num_points, W, H, seed)
    inp = _np_inputs(g, vt)
    ours = _ours(cuda_device, inp)
    o, of = _oracle_best(oracle, inp)
    np.testing.assert_array_equal(ours["radii"], o["radii"])
    assert int(ours["counts"][1]) == o["num_rendered"]  # reference-equivalent instance count
    assert int(ours["counts"][0]) <= o["num_rendered"]
    best = min((compare_images(ours["color"], x["color"]) for x in (o, of)), key=lambda r: r["frac_bad"])
    assert best["frac_bad"] <= BUDGET and best["median"] <= 1e-6, best
    _assert_parity(ours["final_T"], o["final_T"], "final_T")
    _assert_parity(ours["depth"], o["depth"], "depth")


@pytest.mark.parametrize("num_points,W,H,seed", REF_CASES)
def test_cuda_matches_reference_rasterizer(gsb_lib, cuda_device, num_points, W, H, seed):
    g, vt = _case(num_points, W, H, seed)
    inp = _np_inputs(g, vt)
    ref = _ref(num_points, W, H, seed, inp)
    n = ref["final_T"].size
    from gs2mesh_b200 import _lib

    rect = _ours(cuda_device, inp, flags=0)  # reference rectangle binning
    assert digest(rect["radii"]) == ref["radii_sha256"]
    assert int(rect["counts"][0]) == ref["num_rendered"] == int(rect["counts"][1])
    _assert_parity(sample_image(rect["color"], n), ref["color"], "color(rect)")
    _assert_parity(sample_image(rect["final_T"], n), ref["final_T"], "final_T(rect)")
    ours = _ours(cuda_device, inp, flags=_lib.RASTER_EXACT_TILE_CULL)
    _assert_parity(sample_image(ours["color"], n), ref["color"], "color(exact)")
    assert int(ours["counts"][1]) == ref["num_rendered"]


def test_oracle_is_pinned_by_reference_rasterizer(oracle):
    """Pins the CPU restatement itself: oracle vs the reference binary on the same inputs,
    per-Gaussian intermediates included (for a fixed sample of the visible Gaussians)."""
    g, vt = _case(*PINNED_CASE[:3], seed=PINNED_CASE[3])
    inp = _np_inputs(g, vt)
    ref = _ref(*PINNED_CASE, inp)
    pre = oracle.preprocess(g.xyz, g.opacity, vt.world_view, vt.full_proj, vt.cam_center, vt.width, vt.height, vt.tan_fovx,
                            vt.tan_fovy, shs=g.features, scales=g.scaling, rotations=g.rotation)
    assert digest(pre["radii"]) == ref["radii_sha256"]
    assert digest(pre["tiles_touched"]) == ref["tiles_touched_sha256"]
    vis = np.flatnonzero(pre["radii"] > 0)  # == the reference's visible set: the radii are equal
    gi = vis[fixed_sample(len(vis), len(ref["depths"]))]
    np.testing.assert_allclose(pre["depths"][gi], ref["depths"], rtol=1e-6)
    np.testing.assert_allclose(pre["xy"][gi], ref["xy"], rtol=1e-5, atol=1e-4)
    np.testing.assert_allclose(pre["conic_opacity"][gi], ref["conic_opacity"], rtol=2e-4, atol=1e-6)
    np.testing.assert_allclose(pre["rgb"][gi], ref["rgb"], rtol=1e-5, atol=2e-6)
    o, of = _oracle_best(oracle, inp)
    assert o["num_rendered"] == ref["num_rendered"]
    n = ref["final_T"].size
    best = min((compare_images(sample_image(x["color"], n), ref["color"]) for x in (o, of)), key=lambda r: r["frac_bad"])
    assert best["frac_bad"] <= BUDGET, best


def test_exact_tile_cull_is_bit_identical_to_rectangle_binning(gsb_lib, cuda_device):
    from gs2mesh_b200 import _lib

    for seed, (n, W, H) in enumerate([(5000, 400, 300), (20000, 640, 480)]):
        g, vt = _case(n, W, H, seed=10 + seed)
        inp = _np_inputs(g, vt)
        rect = _ours(cuda_device, inp, flags=0)
        exact = _ours(cuda_device, inp, flags=_lib.RASTER_EXACT_TILE_CULL)
        for k in ("color", "depth", "final_T", "radii"):
            np.testing.assert_array_equal(rect[k], exact[k], err_msg=k)
        assert exact["counts"][0] < rect["counts"][0]
        assert exact["counts"][1] == rect["counts"][1] == rect["counts"][0]


def test_binned_sort_equals_reference_shaped_sort(gsb_lib, cuda_device):
    """Default pipeline (depth-sort the P Gaussians, emit instances in that order, stable radix split on
    the tile id) against the validation path that keeps the reference's shape (global stable radix sort on
    (tile, depth) of keys emitted in Gaussian order): identical blend order => bit-identical images.
    The dense cases put tens of thousands of instances into single tiles."""
    from gs2mesh_b200 import _lib

    for n, W, H, seed in [(6000, 320, 240, 60), (20000, 96, 64, 61), (60000, 64, 48, 62), (5, 40, 40, 63), (4097, 1000, 30, 64)]:
        g, vt = _case(n, W, H, seed=seed)
        inp = _np_inputs(g, vt)
        for cull in (0, _lib.RASTER_EXACT_TILE_CULL):
            ref = _ours(cuda_device, inp, flags=cull | _lib.RASTER_CUB_SORT)
            new = _ours(cuda_device, inp, flags=cull)
            for k in ("color", "depth", "final_T", "radii"):
                np.testing.assert_array_equal(ref[k], new[k], err_msg=f"{k} n={n} cull={cull}")
            np.testing.assert_array_equal(ref["counts"][:2], new["counts"][:2])
            assert new["counts"][2] == 0


def test_async_mode_reports_overflow_in_status_word(gsb_lib, cuda_device):
    import torch

    from gs2mesh_b200 import rasterizer as rast

    g, vt = _case(3000, 320, 240, seed=0)
    dev = cuda_device
    t = lambda a: torch.as_tensor(np.ascontiguousarray(a, dtype=np.float32)).to(dev)
    status = torch.zeros(4, dtype=torch.int64).pin_memory()
    kw = dict(means3D=t(g.xyz), opacities=t(g.opacity).reshape(-1), viewmatrix=t(vt.world_view), projmatrix=t(vt.full_proj),
              campos=t(vt.cam_center), bg=torch.zeros(3, device=dev), width=320, height=240, tan_fovx=vt.tan_fovx,
              tan_fovy=vt.tan_fovy, shs=t(g.features), scales=t(g.scaling), rotations=t(g.rotation), sh_degree=3)
    sync = rast.rasterize_forward(**kw, want_counts=True)
    torch.cuda.synchronize()
    out = rast.rasterize_forward(**kw, async_mode=True, counts_out=status)
    torch.cuda.synchronize()
    assert status[2] == 0 and status[0] == sync["counts"][0].item() and status[1] == sync["counts"][1].item()
    assert torch.equal(out["color"], sync["color"])


def _raw_call(gsb_lib, dev, g, vt, cap, flags, status=None):
    """Direct C-ABI call with an explicit binning capacity."""
    import torch

    from gs2mesh_b200 import _lib

    t = lambda a: torch.as_tensor(np.ascontiguousarray(a, dtype=np.float32)).to(dev)
    P, W, H = g.xyz.shape[0], vt.width, vt.height
    ten = dict(m=t(g.xyz), o=t(g.opacity).reshape(-1), sh=t(g.features), s=t(g.scaling), r=t(g.rotation), v=t(vt.world_view),
               p=t(vt.full_proj), c=t(vt.cam_center), bg=torch.zeros(3, device=dev), col=torch.zeros(3, H, W, device=dev))
    ws = torch.empty(gsb_lib.gsb_raster_workspace_bytes(P, W, H, cap), dtype=torch.uint8, device=dev)
    a = _lib.GsbRasterArgs(P=P, sh_degree=3, sh_coeffs=16, width=W, height=H, background=_lib.ptr(ten["bg"]),
                           means3D=_lib.ptr(ten["m"]), shs=_lib.ptr(ten["sh"]), opacities=_lib.ptr(ten["o"]), scales=_lib.ptr(ten["s"]),
                           rotations=_lib.ptr(ten["r"]), scale_modifier=1.0, viewmatrix=_lib.ptr(ten["v"]), projmatrix=_lib.ptr(ten["p"]),
                           cam_pos=_lib.ptr(ten["c"]), tan_fovx=vt.tan_fovx, tan_fovy=vt.tan_fovy, flags=flags, out_color=_lib.ptr(ten["col"]),
                           num_rendered=_lib.ptr(status), workspace=_lib.ptr(ws), workspace_bytes=ws.numel(), max_instances=cap)
    rc = gsb_lib.gsb_raster_forward(C.byref(a), None)
    torch.cuda.synchronize()
    return rc, ten["col"], (ten, ws)


def test_undersized_workspace_async_flags_frame_and_stays_in_bounds(gsb_lib, cuda_device):
    import torch

    from gs2mesh_b200 import _lib

    g, vt = _case(3000, 320, 240, seed=0)
    status = torch.zeros(4, dtype=torch.int64).pin_memory()
    rc, _, _ = _raw_call(gsb_lib, cuda_device, g, vt, 1000, _lib.RASTER_ASYNC, status)
    assert rc == _lib.GSB_OK and status[2] == 1 and status[0] > 1000
    need = int(status[0])
    status.zero_()
    rc, col, _ = _raw_call(gsb_lib, cuda_device, g, vt, need, _lib.RASTER_ASYNC, status)
    assert rc == _lib.GSB_OK and status[2] == 0 and status[0] == need
    rc2, col2, _ = _raw_call(gsb_lib, cuda_device, g, vt, need + 12345, 0, None)
    assert rc2 == _lib.GSB_OK and torch.equal(col, col2)


def test_fast_exp_stays_inside_parity_budget(oracle, gsb_lib, cuda_device):
    """GSB_RASTER_FAST_EXP (ex2.approx in the blend loop, the Renderer's default) vs the reference
    rasterizer / oracle: still within 1e-4 relative with the same outlier budget."""
    from gs2mesh_b200 import _lib

    for n, W, H, seed in [(10000, 640, 480, 1), (3000, 320, 240, 0)]:
        g, vt = _case(n, W, H, seed)
        inp = _np_inputs(g, vt)
        fast = _ours(cuda_device, inp, flags=_lib.RASTER_EXACT_TILE_CULL | _lib.RASTER_FAST_EXP)
        exact = _ours(cuda_device, inp, flags=_lib.RASTER_EXACT_TILE_CULL)
        r = compare_images(fast["color"], exact["color"])
        assert r["frac_bad"] <= BUDGET and r["median"] <= 1e-6, r
        ref = _ref(n, W, H, seed, inp)
        k = ref["final_T"].size
        _assert_parity(sample_image(fast["color"], k), ref["color"], "fast-exp color vs reference")
        _assert_parity(sample_image(fast["final_T"], k), ref["final_T"], "fast-exp final_T vs reference")
        o = oracle.forward(**inp)
        _assert_parity(fast["depth"], o["depth"], "fast-exp depth vs oracle")


@pytest.mark.parametrize("fast", [False, True])
def test_blend_kernel_variants_agree(gsb_lib, cuda_device, fast):
    """dual (the reference's exponent expression) vs table (default: log2-domain exponent from per-column / per-row terms, packed
    f32x2, predicated accumulation): same thresholds of forward.cu:336-353, same instance lists; alpha differs by rounding
    (~1e-6 relative), so the images agree like against the reference.  Without GSB_RASTER_FAST_EXP both names run the dual
    kernel with full-precision expf: bit-identical."""
    from gs2mesh_b200 import _lib

    for n, W, H, seed in [(10000, 640, 480, 1), (3000, 333, 250, 5)]:  # 333x250: ragged tiles on both axes
        g, vt = _case(n, W, H, seed)
        inp = _np_inputs(g, vt)
        base = _lib.RASTER_EXACT_TILE_CULL | (_lib.RASTER_FAST_EXP if fast else 0)
        outs = {name: _ours(cuda_device, inp, flags=base | _lib.RASTER_RENDER_IMPL(name)) for name in _lib.RENDER_IMPLS}
        ref, out = outs["dual"], outs["table"]
        np.testing.assert_array_equal(out["counts"], ref["counts"])
        if fast:
            for k in ("color", "final_T", "depth"):
                cmp = compare_images(out[k], ref[k])
                assert cmp["frac_bad"] <= BUDGET and cmp["median"] <= 2e-6, (k, cmp)
            assert np.abs(out["color"] - ref["color"]).max() > 0  # they are different kernels
        else:
            for k in ("color", "final_T", "depth"):
                np.testing.assert_array_equal(out[k], ref[k], err_msg=k)
        legacy = _ours(cuda_device, inp, flags=base | _lib.RASTER_RENDER_IMPL(2))  # a removed variant's number selects dual
        np.testing.assert_array_equal(legacy["color"], ref["color"])


def test_sh_staging_variants_agree(gsb_lib, cuda_device):
    """scalar / 16-byte / padded-slot staging of the SH block (also without TMA and on the ragged last warp).  The two
    register-fed variants run the same instructions and are bit-identical; the scalar variant evaluates the same
    expression from shared-memory operands, where ptxas fuses one multiply-add differently: colours within 2 ulp,
    everything that decides binning and blending order identical."""
    from gs2mesh_b200 import _lib

    g, vt = _case(4099, 320, 240, seed=22)
    inp = _np_inputs(g, vt)
    for extra in (0, _lib.RASTER_NO_TMA):
        outs = {m: _ours(cuda_device, inp, flags=_lib.RASTER_EXACT_TILE_CULL | extra | _lib.RASTER_SH_MODE(m)) for m in _lib.SH_MODES}
        for k in ("color", "depth", "final_T", "radii", "counts"):
            np.testing.assert_array_equal(outs["padded"][k], outs["vec"][k], err_msg=k)
        for k in ("depth", "final_T", "radii", "counts"):
            np.testing.assert_array_equal(outs["scalar"][k], outs["vec"][k], err_msg=k)
        np.testing.assert_allclose(outs["scalar"]["color"], outs["vec"]["color"], rtol=3e-7, atol=3e-7)


def test_tma_staging_equals_plain_loads(gsb_lib, cuda_device):
    from gs2mesh_b200 import _lib

    g, vt = _case(4099, 320, 240, seed=21)  # 4099 = 128*32 + 3: exercises the ragged last warp
    inp = _np_inputs(g, vt)
    a = _ours(cuda_device, inp, flags=_lib.RASTER_EXACT_TILE_CULL)
    b = _ours(cuda_device, inp, flags=_lib.RASTER_EXACT_TILE_CULL | _lib.RASTER_NO_TMA)
    for k in ("color", "depth", "final_T", "radii", "counts"):
        np.testing.assert_array_equal(a[k], b[k], err_msg=k)


@pytest.mark.parametrize("deg", [0, 1, 2, 3])
def test_sh_degrees(oracle, gsb_lib, cuda_device, deg):
    g, vt = _case(2000, 200, 160, seed=30 + deg)
    inp = _np_inputs(g, vt, sh_degree=deg)
    ours = _ours(cuda_device, inp)
    o, of = _oracle_best(oracle, inp)
    best = min((compare_images(ours["color"], x["color"]) for x in (o, of)), key=lambda r: r["frac_bad"])
    assert best["frac_bad"] <= BUDGET, best


def test_optional_input_variants(oracle, gsb_lib, cuda_device):
    """colors_precomp instead of SHs, cov3D_precomp instead of scale/rotation, white background,
    scale_modifier != 1 (the optional-argument combinations of __init__.py:191-207)."""
    g, vt = _case(2500, 256, 192, seed=40)
    base = _np_inputs(g, vt)
    pre = oracle.preprocess(g.xyz, g.opacity, vt.world_view, vt.full_proj, vt.cam_center, vt.width, vt.height, vt.tan_fovx,
                            vt.tan_fovy, shs=g.features, scales=g.scaling, rotations=g.rotation)
    rng = np.random.default_rng(0)
    variants = {
        "colors_precomp": dict(base, shs=None, colors_precomp=rng.uniform(0, 1, (2500, 3)).astype(np.float32)),
        "cov3D_precomp": dict(base, scales=None, rotations=None, cov3D_precomp=pre["cov3d"]),
        "white_bg": dict(base, bg=np.ones(3, np.float32)),
        "scale_modifier": dict(base, scale_modifier=0.5),
    }
    for name, inp in variants.items():
        inp = {k: v for k, v in inp.items() if v is not None}
        ours = _ours(cuda_device, inp)
        o, of = _oracle_best(oracle, inp)
        np.testing.assert_array_equal(ours["radii"], o["radii"], err_msg=name)
        best = min((compare_images(ours["color"], x["color"]) for x in (o, of)), key=lambda r: r["frac_bad"])
        assert best["frac_bad"] <= BUDGET, (name, best)


def test_edge_sizes(oracle, gsb_lib, cuda_device):
    """Empty scene, single Gaussian, one full warp, one-past-a-warp, image smaller than a tile."""
    for n, W, H in [(0, 64, 48), (1, 64, 48), (32, 100, 70), (33, 100, 70), (50, 10, 7)]:
        g, vt = _case(max(n, 1), W, H, seed=50 + n)
        inp = _np_inputs(g, vt, bg=np.array([0.2, 0.4, 0.6], np.float32))
        if n == 0:
            for k in ("means3D", "opacities", "shs", "scales", "rotations"):
                inp[k] = inp[k][:0]
        ours = _ours(cuda_device, inp)
        o = oracle.forward(**inp)
        assert int(ours["counts"][1]) == o["num_rendered"]
        _assert_parity(ours["color"], o["color"], f"color n={n}", budget=1e-3)
        _assert_parity(ours["final_T"], o["final_T"], f"final_T n={n}", budget=1e-3)


def test_workspace_too_small_is_reported(gsb_lib, cuda_device):
    import torch

    from gs2mesh_b200 import _lib

    g, vt = _case(3000, 320, 240, seed=0)
    for flags in (0, _lib.RASTER_CUB_SORT):
        rc, _, _ = _raw_call(gsb_lib, cuda_device, g, vt, 1000, flags)
        assert rc == _lib.GSB_ERR_WORKSPACE
        need = gsb_lib.gsb_raster_required_instances()
        assert need > 1000 and b"instances" in gsb_lib.gsb_last_error()
        rc, col, _ = _raw_call(gsb_lib, cuda_device, g, vt, need, flags)
        assert rc == _lib.GSB_OK and torch.isfinite(col).all() and float(col.mean()) > 0.01


def test_invalid_argument_combinations(gsb_lib, cuda_device):
    import torch

    import sys, os
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "gs2mesh_b200", "compat"))
    from diff_gaussian_rasterization import GaussianRasterizationSettings, GaussianRasterizer

    g, vt = _case(100, 64, 48)
    dev = cuda_device
    t = lambda a: torch.as_tensor(np.ascontiguousarray(a, dtype=np.float32)).to(dev)
    rs = GaussianRasterizationSettings(image_height=48, image_width=64, tanfovx=vt.tan_fovx, tanfovy=vt.tan_fovy, bg=torch.zeros(3, device=dev),
                                       scale_modifier=1.0, viewmatrix=t(vt.world_view), projmatrix=t(vt.full_proj), sh_degree=3,
                                       campos=t(vt.cam_center), prefiltered=False, debug=False)
    r = GaussianRasterizer(rs)
    with pytest.raises(Exception, match="excatly one of either SHs"):
        r(t(g.xyz), None, t(g.opacity), scales=t(g.scaling), rotations=t(g.rotation))
    with pytest.raises(Exception, match="exactly one of either scale/rotation"):
        r(t(g.xyz), None, t(g.opacity), shs=t(g.features), scales=t(g.scaling))
    with pytest.raises(RuntimeError, match="num_points, 3"):
        r(t(g.xyz).reshape(-1), None, t(g.opacity), shs=t(g.features), scales=t(g.scaling), rotations=t(g.rotation))
    with torch.no_grad():
        color, radii = r(t(g.xyz), None, t(g.opacity), shs=t(g.features), scales=t(g.scaling), rotations=t(g.rotation))
    assert color.shape == (3, 48, 64) and radii.shape == (100,) and radii.dtype == torch.int32
    vis = r.markVisible(t(g.xyz))
    z = (np.c_[g.xyz, np.ones(100)] @ vt.world_view.astype(np.float64))[:, 2]
    np.testing.assert_array_equal(vis.cpu().numpy(), z > 0.2)


def test_compat_module_runs_reference_render_function_shape(gsb_lib, cuda_device):
    """`gaussian_renderer.render`'s call sequence (gaussian_renderer/__init__.py:36-93) through the
    drop-in module gives the same image as the low-level entry point."""
    import torch

    import sys, os
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "gs2mesh_b200", "compat"))
    from diff_gaussian_rasterization import GaussianRasterizationSettings, GaussianRasterizer

    g, vt = _case(3000, 320, 240, seed=0)
    dev = cuda_device
    t = lambda a: torch.as_tensor(np.ascontiguousarray(a, dtype=np.float32)).to(dev)
    rs = GaussianRasterizationSettings(image_height=240, image_width=320, tanfovx=vt.tan_fovx, tanfovy=vt.tan_fovy, bg=torch.zeros(3, device=dev),
                                       scale_modifier=1.0, viewmatrix=t(vt.world_view), projmatrix=t(vt.full_proj), sh_degree=3,
                                       campos=t(vt.cam_center), prefiltered=False, debug=True)
    with torch.no_grad():
        img, radii = GaussianRasterizer(raster_settings=rs)(means3D=t(g.xyz), means2D=torch.zeros_like(t(g.xyz)), shs=t(g.features),
                                                            colors_precomp=None, opacities=t(g.opacity), scales=t(g.scaling),
                                                            rotations=t(g.rotation), cov3D_precomp=None)
    ours = _ours(dev, _np_inputs(g, vt))
    np.testing.assert_array_equal(img.cpu().numpy(), ours["color"])
    np.testing.assert_array_equal(radii.cpu().numpy(), ours["radii"])


def test_image_to_u8_matches_cv2_rule(gsb_lib, cuda_device):
    import torch

    from gs2mesh_b200 import rasterizer as rast

    rng = np.random.default_rng(0)
    img = rng.uniform(-0.1, 1.1, (3, 37, 53)).astype(np.float32)
    img[0, 0, :6] = [0.5 / 255, 1.5 / 255, 2.5 / 255, 254.5 / 255, 1.0, 0.0]  # ties round to even
    got = rast.image_to_u8(torch.as_tensor(img).to(cuda_device)).cpu().numpy()
    want = np.clip(np.rint(np.transpose(img, (1, 2, 0)) * np.float32(255.0)), 0, 255).astype(np.uint8)
    np.testing.assert_array_equal(got, want)
