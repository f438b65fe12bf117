"""Double-precision referee for the blend kernels: a ctypes front end of tests/native/blend_f64.c and the per-pixel /
per-Gaussian comparisons with their error-model tolerances.

`reference(...)` takes the records the library blends (means2D, conic + opacity, colour, depth), the sorted
`point_list` and the tile `ranges` — from `bloomscene_b200.debug.state_views` on the GPU or `Oracle.state()` on the
CPU — and recomputes the forward and the ten blend-backward sums of every Gaussian in double (see the C file's header
for the rules and the guard bands of the two threshold tests).  `check_forward` / `check_backward` compare an
implementation's outputs with it element by element and return a report with the worst error-to-bound ratio.

`pixel_scene` builds a scene whose footprints are placed in pixel coordinates: a camera at the origin looking down +z
(identity view matrix), precomputed colours and 3D covariances whose only non-zero block is xy, so that the 2D
covariance is (f / z)^2 Sigma_xy + 0.3 I exactly in real arithmetic."""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "native", "blend_f64.c")
EPS = 2.0 ** -24

# Forward: rho (per pixel, in units of EPS, computed by the C side) bounds T's relative error: 2 EPS per blended record
# (1 - alpha and the product) plus alpha's own error amplified by alpha / (1 - alpha); rho >= 2 n_contrib.  A colour or
# depth term c alpha T also carries its alpha's error (da_max: the largest over the pixel's records, <= ~50) and two
# roundings (alpha * c, the fma into the running sum, whose error is <= EPS per step relative to sum |terms|, i.e. <= rho
# again), covered by the factor 2:
#   |T - T64| <= KAPPA_F EPS (1 + rho) T64
#   |C - C64| <= KAPPA_F EPS (1 + rho + da_max) (sum |c alpha T| + |bg| T);  depth: D / acc with D and acc alike.
KAPPA_F = 2.0  # must equal KAPPA_F in blend_f64.c (used there to match undecided pixels)
# Backward, per Gaussian and slot: |g - s64| <= KAPPA_B EPS (1 + L) M, M the sum of |terms| (every factor of every term
# by its absolute value, (c - beta) bounded by |c| + |beta|).  The error sources of one term, in units of EPS:
#   - T recovered back to front from T_final by division (blend_bwd.cu:361-365): T_final carries the forward's rho,
#     each of the chain's divisions adds 2 (rcp.approx <= 1 ulp, the product); both are <= rho of the pixel (rho >= 2 n);
#   - beta, the behind-colour recurrence: one fma per record behind, <= rho again;
#   - G and alpha: da = 0.5 Eq + 4 (the q error model of the C file; da_g is the Gaussian's largest).  It is ~50 for
#     compact footprints but grows where |a| dx^2 + |c| dy^2 + 2 |b| |dx dy| >> q, i.e. along thin needles;
#   - the products forming the slot (o, a dx + b dy, ...): <= 6;
#   - the summation: 8 rows per lane, 2 shuffle levels, then one float atomic per 8x8 block: <= 12 + blocks.
# So L = rho_max (the largest rho of the pixels the Gaussian contributes to; >= 2 (1 + deepest list position)) + da_g +
# blocks, and KAPPA_B = 16 covers 3 rho + da + 18 + blocks for every L >= 3 (one pixel, one block).
KAPPA_B = 16.0

_lib = None


class _In(C.Structure):
    _fields_ = [("P", C.c_int), ("W", C.c_int), ("H", C.c_int)] + [
        (n, C.c_void_p) for n in ("means2D", "conic_opacity", "colors", "depths", "point_list", "ranges", "bg", "dL_dpix",
                                  "dL_ddepth", "impl_T", "impl_n")] + [
        ("mutation", C.c_int), ("mut_a", C.c_int), ("mut_b", C.c_int)]


class _Out(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("T", "color", "depth", "acc", "n_contrib", "rho", "color_mag", "depth_mag",
                                          "da_max", "pix_state", "g", "m", "L", "rho_max", "da_g", "blocks", "excluded")] + [
        ("stats", C.c_longlong * 4)]


MUTATIONS = {"drop_pair": 1, "drop_block": 2, "row_shift": 3, "double_record": 4, "drop_partial_group": 5,
             "skip_first_live": 6}
PIX_DECIDED, PIX_RESOLVED, PIX_EXCLUDED, PIX_MISMATCH = 0, 1, 2, 3


def _build_dir():
    d = os.path.join(HERE, "native", "_build")
    try:
        os.makedirs(d, exist_ok=True)
        if os.access(d, os.W_OK):
            return d
    except OSError:
        pass
    d = os.path.join(tempfile.gettempdir(), "blend_f64_build_%d" % os.getuid())
    os.makedirs(d, exist_ok=True)
    return d


def lib():
    global _lib
    if _lib is None:
        out = os.path.join(_build_dir(), "libblendf64.so")
        if not os.path.exists(out) or os.path.getmtime(out) < os.path.getmtime(SRC):
            tmp = out + ".%d.tmp" % os.getpid()
            subprocess.run(["gcc", "-O2", "-std=c99", "-fPIC", "-shared", "-ffp-contract=off", SRC, "-o", tmp, "-lm"],
                           check=True)
            os.replace(tmp, out)
        L = C.CDLL(out)
        L.bf64_run.argtypes = [C.POINTER(_In), C.POINTER(_Out)]
        L.bf64_run.restype = C.c_int
        _lib = L
    return _lib


def _np(a, dtype):
    if a is None:
        return None
    if hasattr(a, "detach"):
        a = a.detach().cpu().numpy()
    return np.ascontiguousarray(a, dtype=dtype)


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def reference(state, W, H, bg, dL_dpix, dL_ddepth=None, impl_T=None, impl_n=None, mutation=None, mut_a=-1, mut_b=-1):
    """state: means2D [P,2], conic_opacity [P,4], colors [P,3], depths [P], point_list [R], ranges [tiles,2]."""
    f32, u32 = np.float32, np.uint32
    arr = {"means2D": _np(state["means2D"], f32), "conic_opacity": _np(state["conic_opacity"], f32),
           "colors": _np(state["colors"], f32), "depths": _np(state["depths"], f32),
           "point_list": _np(state["point_list"], np.int64).astype(u32), "ranges": _np(state["ranges"], np.int64).astype(u32),
           "bg": _np(bg, f32), "dL_dpix": _np(dL_dpix, f32).reshape(3, H, W),
           "dL_ddepth": None if dL_ddepth is None else _np(dL_ddepth, f32).reshape(H, W),
           "impl_T": None if impl_T is None else _np(impl_T, f32).reshape(H * W),
           "impl_n": None if impl_n is None else _np(impl_n, np.int64).astype(u32).reshape(H * W)}
    P = arr["means2D"].shape[0]
    assert arr["ranges"].shape == (((W + 15) // 16) * ((H + 15) // 16), 2)
    if arr["point_list"].size == 0:
        arr["point_list"] = np.zeros(1, u32)
    inp = _In(P, W, H, *[_p(arr[k]) for k in ("means2D", "conic_opacity", "colors", "depths", "point_list", "ranges", "bg",
                                               "dL_dpix", "dL_ddepth", "impl_T", "impl_n")],
              MUTATIONS[mutation] if mutation else 0, int(mut_a), int(mut_b))
    npix = W * H
    out = {"T": np.zeros(npix), "color": np.zeros((3, H, W)), "depth": np.zeros(npix), "acc": np.zeros(npix),
           "n_contrib": np.zeros(npix, u32), "rho": np.zeros(npix), "color_mag": np.zeros((3, H, W)),
           "depth_mag": np.zeros(npix), "da_max": np.zeros(npix), "pix_state": np.zeros(npix, np.int32), "g": np.zeros((P, 10)),
           "m": np.zeros((P, 10)), "L": np.zeros(P, np.int32), "rho_max": np.zeros(P), "da_g": np.zeros(P), "blocks": np.zeros(P, np.int32),
           "excluded": np.zeros(P, np.uint8)}
    o = _Out(*[_p(out[n]) for n, _ in _Out._fields_[:-1]])
    assert lib().bf64_run(C.byref(inp), C.byref(o)) == 0
    out["stats"] = {"pairs_evaluated": o.stats[0], "pairs_contributing": o.stats[1], "undecided": o.stats[2],
                    "pixels_excluded": o.stats[3]}
    out["excluded"] = out["excluded"].astype(bool)
    out["depth"] = out["depth"].reshape(H, W)
    out["depth_mag"] = out["depth_mag"].reshape(H, W)
    out["W"], out["H"] = W, H
    return out


def _ratio(err, tol):
    """err / tol elementwise, with 0/0 = 0 and x/0 = inf."""
    err, tol = np.asarray(err, np.float64), np.asarray(tol, np.float64)
    with np.errstate(divide="ignore", invalid="ignore"):
        r = np.where(err == 0, 0.0, err / tol)
    return np.nan_to_num(r, nan=np.inf)


def check_forward(ref, T=None, n_contrib=None, color=None, depth=None):
    """Per pixel, over the pixels the referee did not exclude.  Returns {"worst": max err/bound, "fail": #pixels over,
    "excluded": #pixels, "n_contrib_mismatch": #pixels}."""
    W, H = ref["W"], ref["H"]
    keep = (ref["pix_state"] != PIX_EXCLUDED).reshape(H, W)
    rho = ref["rho"].reshape(H, W)
    scale = KAPPA_F * EPS * (1.0 + rho)
    scale_c = KAPPA_F * EPS * (1.0 + rho + ref["da_max"].reshape(H, W))
    ratios, rep = [], {"excluded": int((~keep).sum()), "n_contrib_mismatch": 0}
    if n_contrib is not None:
        n = np.asarray(n_contrib).reshape(H, W).astype(np.int64)
        bad = (n != ref["n_contrib"].reshape(H, W).astype(np.int64)) & keep
        rep["n_contrib_mismatch"] = int(bad.sum())
        ratios.append(np.where(bad, np.inf, 0.0))
    if T is not None:
        T64 = ref["T"].reshape(H, W)
        ratios.append(_ratio(np.abs(np.asarray(T, np.float64).reshape(H, W) - T64), scale * T64) * keep)
    if color is not None:
        c = np.asarray(color, np.float64).reshape(3, H, W)
        ratios.append((_ratio(np.abs(c - ref["color"]), scale_c * ref["color_mag"]) * keep).max(axis=0))
    if depth is not None:
        d = np.asarray(depth, np.float64).reshape(H, W)
        dm = ref["depth_mag"]
        checked = keep & np.isfinite(dm)  # depth gate undecided: value not checked (only counted)
        ratios.append(_ratio(np.abs(d - ref["depth"]), scale_c * np.where(np.isfinite(dm), dm, 0.0)) * checked)
        rep["depth_gate_undecided"] = int((keep & ~np.isfinite(dm)).sum())
    r = np.max(np.stack(ratios), axis=0) if ratios else np.zeros((H, W))
    rep["worst"] = float(r.max(initial=0.0))
    rep["fail"] = int((r > 1.0).sum())
    return rep


def backward_bound(ref):
    """KAPPA_B EPS (1 + L) M per Gaussian and slot, L = rho_max + da_g + blocks (see KAPPA_B)."""
    L = ref["rho_max"] + ref["da_g"] + ref["blocks"]
    return KAPPA_B * EPS * (1.0 + L)[:, None] * ref["m"]


def check_backward(ref, g, slots=range(10), scale=None):
    """g: [P, len(slots)] the implementation's sums for `slots` (scale: per-slot factor already applied to g, e.g. the
    0.5 W of dL_dmeans2D; the bound is scaled alike).  Over the Gaussians the referee did not exclude."""
    slots = list(slots)
    g = np.asarray(g, np.float64).reshape(-1, len(slots))
    s = np.ones(len(slots)) if scale is None else np.asarray(scale, np.float64)
    want = ref["g"][:, slots] * s
    tol = backward_bound(ref)[:, slots] * np.abs(s)
    keep = ~ref["excluded"]
    r = _ratio(np.abs(g - want), tol) * keep[:, None]
    worst = np.unravel_index(int(np.argmax(r)), r.shape) if r.size else (0, 0)
    return {"worst": float(r.max(initial=0.0)), "fail": int((r > 1.0).any(axis=1).sum()), "excluded": int((~keep).sum()),
            "worst_at": (int(worst[0]), slots[int(worst[1])]) if r.size else None}


# ---- scenes placed in pixel coordinates ---------------------------------------------------------------------------

def pixel_scene(W, H, u, v, cov2, opacity, color, z):
    """Gaussians centred at pixel (u, v) with 2D covariance cov2 = (sxx, sxy, syy) in pixels^2 (including the 0.3
    low-pass the preprocess adds; needs cov2 - 0.3 I >= 0), opacity, colour [.,3] and view depth z.
    Returns (scene dict for the rasterizer / oracle, camera)."""
    import torch

    from workload import synthetic

    cam = synthetic.yaw_camera(W, H, 0.0)
    u, v, z, opacity = (np.asarray(x, np.float64).reshape(-1) for x in (u, v, z, opacity))
    cov2 = np.asarray(cov2, np.float64).reshape(-1, 3)
    n = u.size
    fx, fy = W / (2.0 * cam.tanfovx), H / (2.0 * cam.tanfovy)
    ndc_x, ndc_y = (2.0 * u + 1.0) / W - 1.0, (2.0 * v + 1.0) / H - 1.0
    means = np.stack([ndc_x * z * cam.tanfovx, ndc_y * z * cam.tanfovy, z], 1)
    cov3 = np.zeros((n, 6))
    cov3[:, 0] = (cov2[:, 0] - 0.3) * (z / fx) ** 2
    cov3[:, 1] = cov2[:, 1] * (z / fx) * (z / fy)
    cov3[:, 3] = (cov2[:, 2] - 0.3) * (z / fy) ** 2
    t = lambda a: torch.tensor(np.asarray(a, np.float32))
    scene = {"means3D": t(means), "opacities": t(opacity.reshape(-1, 1)), "colors_precomp": t(np.asarray(color).reshape(-1, 3)),
             "cov3D_precomp": t(cov3)}
    return scene, cam


def needle_cov(sigma_major, sigma_minor, theta):
    """(sxx, sxy, syy) of an ellipse with the given standard deviations (pixels), major axis at angle theta."""
    c, s = np.cos(theta), np.sin(theta)
    a, b = sigma_major ** 2, sigma_minor ** 2
    return np.array([a * c * c + b * s * s, (a - b) * c * s, a * s * s + b * c * c])


def oracle_state(scene, cam, bg, dL_dpix, dL_ddepth=None):
    """Forward + backward (f64 sums) of the CPU oracle on a pixel_scene; returns (state for reference(), outputs)."""
    from oracle import oracle as orc

    o = orc.Oracle()
    R, color, depth, radii = o.forward(W=cam.image_width, H=cam.image_height, tanfovx=cam.tanfovx, tanfovy=cam.tanfovy,
                                       bg=bg, viewmatrix=cam.viewmatrix, projmatrix=cam.projmatrix, campos=cam.campos,
                                       sh_degree=0, means3D=scene["means3D"], opacities=scene["opacities"],
                                       colors_precomp=scene.get("colors_precomp"), shs=scene.get("shs"),
                                       scales=scene.get("scales"), rotations=scene.get("rotations"),
                                       cov3D_precomp=scene.get("cov3D_precomp"))
    return oracle_outputs(o, color, depth, radii, scene.get("colors_precomp"), dL_dpix, dL_ddepth)


def oracle_outputs(o, color, depth, radii, colors_precomp, dL_dpix, dL_ddepth=None):
    st = o.state()
    grads = o.backward(dL_dpix, dL_ddepth, f64_sums=True)
    colors = st["rgb"] if colors_precomp is None else _np(colors_precomp, np.float32)
    state = {"means2D": st["means2D"], "conic_opacity": st["conic_opacity"], "colors": colors, "depths": st["depths"],
             "point_list": st["point_list"], "ranges": st["ranges"]}
    outs = {"final_T": st["final_T"], "n_contrib": st["n_contrib"], "color": color, "depth": depth, "radii": radii,
            "grads": grads}
    return state, outs
