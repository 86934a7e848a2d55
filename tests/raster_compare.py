"""Shared parity metric for rasterizer images (north_star: 1e-4 relative fp32).

A pixel is "bad" if |a-b| > 1e-4 * max(1, |b|).  The pipeline has hard thresholds
(alpha < 1/255, T < 1e-4, power > 0, ceil / floor in the tile rectangle) that a 1-ulp
difference in expf or an FMA contraction can flip for isolated pixels (SURVEY.md section 7,
"Branch-boundary parity"), so comparisons carry an explicit outlier budget instead of a max.
"""
import hashlib
import math
import os

import numpy as np

TOL = 1e-4
OBSERVED = {"n": 0, "frac_bad": 0.0, "frac_bad_rel": 0.0, "max_err": 0.0, "max_err_rel": 0.0}  # worst over this session's comparisons


REL_FLOOR = 0.05  # colours live in [0,1]: "relative" below this magnitude is measured against the floor


def compare_images(a, b):
    """frac_bad / max_err: |a-b| / max(1, |b|) (the round-1 criterion, absolute for colours in [0,1]);
    frac_bad_rel / max_err_rel: TRUE relative error |a-b| / max(REL_FLOOR, |b|) -- north_star's "1e-4 relative fp32" read
    per pixel, with a floor so that black pixels (b ~ 0, rounding noise ~1e-8) do not divide by zero."""
    a = np.asarray(a, np.float64)
    b = np.asarray(b, np.float64)
    diff = np.abs(a - b)
    err = diff / np.maximum(1.0, np.abs(b))
    rel = diff / np.maximum(REL_FLOOR, np.abs(b))
    bad = err > TOL
    bad_rel = rel > TOL
    n = max(err.size, 1)
    OBSERVED["n"] += 1
    for k, v in (("frac_bad", bad.sum() / n), ("frac_bad_rel", bad_rel.sum() / n), ("max_err", err.max() if err.size else 0.0),
                 ("max_err_rel", rel.max() if rel.size else 0.0)):
        OBSERVED[k] = max(OBSERVED[k], float(v))
    return dict(frac_bad=float(bad.sum() / n), max_err=float(err.max()) if err.size else 0.0, n_bad=int(bad.sum()),
                median=float(np.median(err)) if err.size else 0.0, frac_bad_rel=float(bad_rel.sum() / n),
                max_err_rel=float(rel.max()) if rel.size else 0.0, p9999_rel=float(np.quantile(rel, 0.9999)) if rel.size else 0.0)


def fixed_sample(n_total, n):
    """Indices of an evenly spread, fixed sample of n of n_total values (a golden-ratio lattice, no RNG involved).
    The first m indices of a sample of n are the sample of m, so a stored sample can be shortened without re-running."""
    step = int(n_total * 0.6180339887498949) | 1
    while math.gcd(step, n_total) != 1:
        step += 2
    return (np.arange(min(n, n_total), dtype=np.int64) * step) % n_total


def digest(*arrays):
    """sha256 over dtype, shape and bytes: stands in for an exact comparison with an array too large to store."""
    h = hashlib.sha256()
    for a in arrays:
        a = np.ascontiguousarray(a)
        h.update(f"{a.dtype.str}{a.shape}".encode())
        h.update(a.tobytes())
    return h.hexdigest()


def inputs_digest(*arrays):
    """digest() of rasterizer inputs as the float32 values the kernels receive."""
    return digest(*(np.ascontiguousarray(a, dtype=np.float32).reshape(-1) for a in arrays))


REF_GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def load_ref_golden(file_name, key, inputs_sha256):
    """One case of the reference rasterizer's stored outputs (tests/golden/make_ref_parity_golden.py): exact outputs as
    digests (`*_sha256`), images as the fixed_sample() of their pixels.  Fails if the case's inputs are no longer the ones
    the outputs were recorded for."""
    with np.load(os.path.join(REF_GOLDEN_DIR, file_name)) as z:
        case = {k[len(key) + 2:]: z[k] for k in z.files if k.startswith(key + "__")}
    assert case, f"no case {key} in tests/golden/{file_name}"
    for k in [k for k in case if k.endswith("_sha256")]:
        case[k] = str(case[k])
    assert case["inputs_sha256"] == inputs_sha256, f"inputs of {key} differ from those tests/golden/{file_name} was made from"
    return case


def sample_image(img, n):
    """[C,H,W] or [H,W] -> the fixed_sample() of n pixels, [C,n] or [n]."""
    img = np.asarray(img)
    flat = img.reshape(img.shape[0], -1) if img.ndim == 3 else img.reshape(-1)
    return flat[..., fixed_sample(flat.shape[-1], n)]


def load_golden_case(path):
    z = np.load(path)
    inputs = dict(means3D=z["means3D"], opacities=z["opacities"], view=z["view"], proj=z["proj"], campos=z["campos"],
                  W=int(z["W"]), H=int(z["H"]), tan_fovx=float(z["tan_fovx"]), tan_fovy=float(z["tan_fovy"]), bg=z["bg"],
                  sh_degree=int(z["sh_degree"]), scale_modifier=float(z["scale_modifier"]))
    for k_npz, k_arg in (("shs", "shs"), ("colors_precomp", "colors_precomp"), ("scales", "scales"), ("rotations", "rotations"),
                         ("cov3D_precomp", "cov3D_precomp")):
        if k_npz in z.files:
            inputs[k_arg] = z[k_npz]
    return dict(inputs=inputs, color=z["color"], radii=z["radii"], num_rendered=int(z["num_rendered"]), final_T=z["final_T"])
