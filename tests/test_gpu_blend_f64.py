"""GPU: the blend kernels pixel by pixel and Gaussian by Gaussian against the double-precision referee
(tests/blend_f64.py).

Forward and backward run through the C-ABI (as in test_gpu_c_abi.py).  The forward's own state — records, point list,
ranges, final T, n_contrib — feeds the referee; the backward's scratch allocation is the blend accumulator (12 floats
per Gaussian, ACCUM_STRIDE), which the preprocess backward only reads, so after the call it holds all ten blend sums,
including the conic sums that no public output exposes.  Every case reports its worst error-to-bound ratio and the
number of pixels / Gaussians the referee excluded (zero on the constructed scenes)."""
import ctypes as C
import math

import numpy as np
import pytest
import torch

import blend_f64 as bf
import parity_lib as pl
from test_gpu_c_abi import ALLOC, Arena, FwdState, Gaussians, Grads, View, _lib, _ptr
from workload import synthetic

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
BG = (0.3, -0.2, 0.8)
LIST_LENGTHS = [1, 7, 8, 9, 31, 32, 33, 127, 128, 129, 255, 256, 257, 511, 512, 513]


def run_gpu(scene, cam, bg, dL_dpix, dL_ddepth=None, sh_degree=0):
    """Forward + backward of one view through the C-ABI.  Returns the forward state (for the referee), the outputs
    and the blend accumulator [P, 12]."""
    from bloomscene_b200.debug import state_views

    lib = _lib()
    lib.brs_backward.argtypes = [C.POINTER(View), C.POINTER(Gaussians), C.c_void_p, C.POINTER(FwdState), C.c_void_p,
                                 C.c_void_p, C.POINTER(Grads), ALLOC, C.c_void_p, C.c_void_p]
    W, H = cam.image_width, cam.image_height
    t = {k: (None if v is None else v.to(DEV).contiguous()) for k, v in scene.items()}
    P = t["means3D"].shape[0]
    M = 0 if t.get("shs") is None else t["shs"].shape[1]
    bg_t = torch.tensor(bg, dtype=torch.float32, device=DEV)
    vm, pm, cp = (x.to(DEV).contiguous() for x in (cam.viewmatrix, cam.projmatrix, cam.campos))
    view = View(W, H, cam.tanfovx, cam.tanfovy, 1.0, sh_degree, M, 0, 0, _ptr(bg_t), _ptr(vm), _ptr(pm), _ptr(cp))
    g = Gaussians(P, _ptr(t["means3D"]), _ptr(t["opacities"]), _ptr(t.get("shs")), _ptr(t.get("colors_precomp")),
                  _ptr(t.get("scales")), _ptr(t.get("rotations")), _ptr(t.get("cov3D_precomp")))
    color = torch.empty(3, H, W, device=DEV)
    depth = torch.empty(1, H, W, device=DEV)
    radii = torch.empty(P, dtype=torch.int32, device=DEV)
    arena, state = Arena(), FwdState()
    stream = torch.cuda.current_stream().cuda_stream
    rc = lib.brs_forward(C.byref(view), C.byref(g), color.data_ptr(), depth.data_ptr(), radii.data_ptr(), arena.fn, None,
                         C.byref(state), stream)
    assert rc == 0, lib.brs_error_string(rc)
    torch.cuda.synchronize()
    R = state.num_rendered
    empty = torch.zeros(16, dtype=torch.uint8, device=DEV)
    sv = state_views(pl.ours()._C, arena.buffers[0], arena.buffers.get(1, empty), arena.buffers[2], P, R, W, H)
    rec = sv["records"].cpu().numpy()
    fstate = {"means2D": rec[:, 0:2], "conic_opacity": rec[:, 4:8], "colors": rec[:, 8:11], "depths": rec[:, 11],
              "point_list": sv["point_list"].cpu().numpy().astype(np.int64) if R else np.zeros(0, np.int64),
              "ranges": sv["ranges"].cpu().numpy().astype(np.int64)}
    outs = {"final_T": sv["final_T"].cpu().numpy().copy(), "n_contrib": sv["n_contrib"].cpu().numpy().copy(),
            "color": color.cpu().numpy(), "depth": depth.cpu().numpy(), "radii": radii.cpu().numpy()}

    dpix = torch.as_tensor(np.asarray(dL_dpix, np.float32), device=DEV).contiguous()
    ddep = None if dL_ddepth is None else torch.as_tensor(np.asarray(dL_ddepth, np.float32), device=DEV).contiguous()
    shapes = {"dL_dmeans2D": (P, 3), "dL_dcolors": (P, 3), "dL_dopacity": (P, 1), "dL_dmeans3D": (P, 3),
              "dL_dcov3D": (P, 6), "dL_dsh": (P, max(M, 1), 3), "dL_dscales": (P, 3), "dL_drotations": (P, 4)}
    gout = {k: torch.full(s, float("nan"), device=DEV) for k, s in shapes.items()}
    grads = Grads(*[gout[k].data_ptr() if (k != "dL_dsh" or M > 0) else None for k in shapes], 0,
                  1 if ddep is not None else 0, depth.data_ptr() if ddep is not None else None)
    n_scratch = len(arena.scratch)
    rc = lib.brs_backward(C.byref(view), C.byref(g), radii.data_ptr(), C.byref(state), dpix.data_ptr(), _ptr(ddep),
                          C.byref(grads), arena.fn, None, stream)
    assert rc == 0, lib.brs_error_string(rc)
    torch.cuda.synchronize()
    assert len(arena.scratch) == n_scratch + 1  # the backward's one scratch allocation: the blend accumulator
    accum = arena.scratch[-1][:P * 12 * 4].view(torch.float32).view(P, 12).cpu().numpy().copy()
    outs["grads"] = {k: v.cpu().numpy() for k, v in gout.items()}
    return fstate, outs, accum


def check_public_outputs_are_slot_scalings(outs, accum, W, H):
    """preprocess_bwd.cu:163-167: dL_dmeans2D = (slot0 * (0.5f W), slot1 * (0.5f H), 0), dL_dopacity = slot5,
    dL_dcolors = slots 6..8 (colours precomputed), bit for bit, for every rendered Gaussian; zeros otherwise."""
    f = np.float32
    vis = outs["radii"] > 0
    g = outs["grads"]
    m2 = g["dL_dmeans2D"]
    assert np.array_equal(m2[vis, 0], accum[vis, 0] * f(f(0.5) * f(W)))
    assert np.array_equal(m2[vis, 1], accum[vis, 1] * f(f(0.5) * f(H)))
    assert not m2[:, 2].any() and not m2[~vis].any()
    assert np.array_equal(g["dL_dopacity"][vis, 0], accum[vis, 5])
    assert not g["dL_dopacity"][~vis].any()


def check_case(what, scene, cam, bg=BG, seed=0, depth="off", sh_degree=0, exclusions_allowed=0.0, report=None):
    """depth: "off" (colour gradient only), "both" (colour + depth) or "only" (depth gradient, zero colour gradient)."""
    W, H = cam.image_width, cam.image_height
    rng = np.random.default_rng(seed)
    dpix = rng.standard_normal((3, H, W)).astype(np.float32)
    if depth == "only":
        dpix[:] = 0
    ddep = rng.standard_normal((1, H, W)).astype(np.float32) if depth != "off" else None
    fstate, outs, accum = run_gpu(scene, cam, bg, dpix, ddep, sh_degree)
    check_public_outputs_are_slot_scalings(outs, accum, W, H)
    ref = bf.reference(fstate, W, H, np.asarray(bg, np.float32), dpix, ddep, impl_T=outs["final_T"],
                       impl_n=outs["n_contrib"])
    fw = bf.check_forward(ref, outs["final_T"], outs["n_contrib"], outs["color"], outs["depth"])
    slots = list(range(10)) if ddep is not None else list(range(9))
    bw = bf.check_backward(ref, accum[:, slots], slots)
    if ddep is None:
        assert not accum[:, 9:].any()  # slot 9 only with the depth gradient; 10, 11 never written
    P = accum.shape[0]
    line = ("%s: forward worst %.3g, backward worst %.3g, pixels excluded %d/%d, Gaussians excluded %d/%d, "
            "pairs contributing %d" % (what, fw["worst"], bw["worst"], fw["excluded"], W * H, bw["excluded"], P,
                                       ref["stats"]["pairs_contributing"]))
    print(line)
    if report is not None:
        report.append(line)
    assert fw["n_contrib_mismatch"] == 0, (what, fw)
    assert fw["fail"] == 0, (what, fw)
    assert bw["fail"] == 0, (what, bw)
    assert fw["excluded"] <= exclusions_allowed * W * H, (what, fw)
    assert bw["excluded"] <= exclusions_allowed * P, (what, bw)
    return ref, outs


def _tile_scene(n, opacity, seed, W=16, H=16, spread=(2.0, 8.0), centre_box=(0.0, 16.0)):
    rng = np.random.default_rng(seed)
    u, v = rng.uniform(*centre_box, n), rng.uniform(*centre_box, n)
    cov = np.stack([bf.needle_cov(a, b, t) for a, b, t in
                    zip(rng.uniform(*spread, n), rng.uniform(spread[0], spread[1], n), rng.uniform(0, np.pi, n))])
    op = opacity(rng, n) if callable(opacity) else np.full(n, opacity)
    z = 1.0 + rng.permutation(n) * 0.003
    return bf.pixel_scene(W, H, u, v, cov, op, rng.uniform(-0.1, 1.1, (n, 3)), z)


@pytest.mark.parametrize("n", LIST_LENGTHS)
def test_list_lengths_low_opacity(n):
    """One 16 x 16 tile, n broad Gaussians of low opacity: every pixel blends (nearly) the whole list, so the batch
    (256 forward / 128 backward), ballot chunk (32), group (8) and double-buffer edges are all hit."""
    scene, cam = _tile_scene(n, lambda r, k: r.uniform(0.006, 0.012, k), seed=n, spread=(8.0, 14.0))
    _, outs = check_case("list length %d" % n, scene, cam, seed=n)
    # no pixel saturates, and the deepest pixel blends (nearly) the whole list
    assert outs["n_contrib"].max() >= 0.9 * n and (outs["final_T"] > 1e-4).all()


@pytest.mark.parametrize("n", LIST_LENGTHS)
def test_list_lengths_saturating(n):
    """The same lengths with opacities that saturate pixels at varying list positions: n_contrib differs between the
    two pixels of a lane, between the warps of a tile, and from the list length (tile max < n)."""
    if n < 255:  # dense and opaque enough that the shorter lists saturate too
        scene, cam = _tile_scene(n, lambda r, k: r.uniform(0.3, 0.99, k), seed=1000 + n, spread=(2.0, 9.0))
    else:  # saturation between list positions ~100 and ~250: the tile's max(n_contrib) straddles the 128-record batch
        scene, cam = _tile_scene(n, lambda r, k: r.uniform(0.05, 0.95, k), seed=1000 + n, spread=(1.0, 6.0))
    _, outs = check_case("saturating %d" % n, scene, cam, seed=n)
    nc = outs["n_contrib"].reshape(16, 16).astype(np.int64)
    if n >= 31:  # a lane's pixels are rows y and y + 4 of its warp's 8 x 8 block
        assert (nc[0:4] != nc[4:8]).any() and (nc[8:12] != nc[12:16]).any()
    if n >= 127:
        warps = {int(nc[:8, :8].max()), int(nc[:8, 8:].max()), int(nc[8:, :8].max()), int(nc[8:, 8:].max())}
        assert len(warps) > 1 and nc.max() < n


def test_ragged_images():
    """W, H in {1, 4, 5, 8, 12, 13, 16, 17, 33}: partial tiles and blocks, H mod 8 in 1..4 (a lane's second pixel
    outside the image)."""
    sizes = [1, 4, 5, 8, 12, 13, 16, 17, 33]
    k = 0
    for W in sizes:
        for H in sizes:
            k += 1
            scene, cam = _tile_scene(40, lambda r, m: r.uniform(0.05, 0.9, m), seed=2000 + k, W=W, H=H,
                                     spread=(0.6, 5.0), centre_box=(-3.0, max(W, H) + 3.0))
            check_case("ragged %dx%d" % (W, H), scene, cam, seed=k)


def test_confined_and_straddling_footprints():
    W, H = 48, 40
    u, v, cov, op = [], [], [], []

    def add(x, y, c, o):
        u.append(x), v.append(y), cov.append(c), op.append(o)

    add(5.0, 5.0, [0.31, 0.0, 0.31], 0.02)         # one pixel
    add(20.0, 3.0, [60.0, 0.0, 0.31], 0.02)        # one row
    add(27.5, 27.5, [2.0, 0.0, 2.0], 0.02)         # one 8x8 block (pixels 24..31)
    for x, y in [(7.5, 12.0), (15.5, 20.0), (16.0, 16.0), (31.5, 31.5), (8.0, 7.5), (23.5, 8.0)]:
        add(x, y, [3.0, 0.5, 2.0], 0.6)            # straddling warp-block and tile boundaries
    for x, y in [(-3.0, 10.0), (W + 2.0, 20.0), (12.0, -4.0), (30.0, H + 3.0), (-2.0, -2.0)]:
        add(x, y, [9.0, -2.0, 6.0], 0.8)           # centres outside the image
    n = len(u)
    scene, cam = bf.pixel_scene(W, H, u, v, np.array(cov), op, np.random.default_rng(3).uniform(0, 1, (n, 3)),
                                1.0 + np.arange(n) * 0.1)
    ref, outs = check_case("confined footprints", scene, cam, seed=3)
    blocks = ref["blocks"]
    assert blocks[0] == 1 and blocks[2] == 1  # one pixel, one block: contributes in exactly one 8x8 block
    assert (ref["g"][:3] != 0).any(axis=1).all()


def test_culling_edge_needles():
    """Needles at 0..180 degrees in 10 degree steps with aspect ratios up to about 1:300, opacities from
    (1/255)(1 + 1e-4) to 1.7, and ellipses whose 1/255 level set grazes a block corner."""
    W, H = 96, 96
    rng = np.random.default_rng(11)
    u, v, cov, op = [], [], [], []
    opac = [(1 / 255) * (1 + 1e-4), 0.01, 0.3, 1.0, 1.7]
    for i, deg in enumerate(range(0, 181, 10)):
        for j, major in enumerate([3.0, 30.0, 165.0]):
            u.append(rng.uniform(10, W - 10)), v.append(rng.uniform(10, H - 10))
            cov.append(bf.needle_cov(major, 0.56, math.radians(deg)))
            op.append(opac[(i + j) % len(opac)])
    # grazing: circle of sigma s whose alpha = 1/255 radius r = s sqrt(2 ln(255 o)) passes the corner pixel (39, 39)
    # of block [32, 39]^2 at distances r (1 +- 1e-4, 1e-3) along the diagonal
    for k, rel in enumerate([-1e-3, -1e-4, 0.0, 1e-4, 1e-3]):
        s, o = 1.5, 0.4
        r = s * math.sqrt(2 * math.log(255 * o)) * (1 + rel)
        d = r / math.sqrt(2)
        u.append(39.0 + d), v.append(39.0 + d), cov.append([s * s, 0.0, s * s]), op.append(o)
    n = len(u)
    scene, cam = bf.pixel_scene(W, H, u, v, np.array(cov), op, rng.uniform(0, 1, (n, 3)), 1.0 + rng.permutation(n) * 0.01)
    check_case("culling edge", scene, cam, seed=11)


@pytest.mark.parametrize("depth", ["off", "both", "only"])
def test_background_and_depth_gradient(depth):
    scene, cam = _tile_scene(300, lambda r, k: r.uniform(0.05, 0.9, k), seed=77, W=40, H=24, spread=(0.8, 6.0),
                             centre_box=(-2.0, 42.0))
    check_case("bg + depth=%s" % depth, scene, cam, bg=(0.7, -0.4, 1.3), seed=78, depth=depth)


def test_stacked_views_match_reference():
    """render_views(stack=k) blends several views in one launch (blockIdx.z); it keeps no state, so each view's colour
    and depth are checked per pixel against the referee built from that view's single-view forward state."""
    api = pl.ours()
    scene, _ = _tile_scene(400, lambda r, k: r.uniform(0.05, 0.9, k), seed=91, W=56, H=40, spread=(0.8, 7.0),
                           centre_box=(-2.0, 58.0))
    cams = [synthetic.make_camera(56, 40, synthetic._rot_y(0.02 * k), np.array([0.01 * k, 0.0, 0.05 * k]))
            for k in range(5)]
    bg = torch.tensor(BG, device=DEV)
    rs = [synthetic.raster_settings(c.to(DEV), 0, bg, api.GaussianRasterizationSettings) for c in cams]
    t = {k: v.to(DEV) for k, v in scene.items()}
    color, depth, _ = api.render_views(rs, t["means3D"], t["opacities"], colors_precomp=t["colors_precomp"],
                                       cov3D_precomp=t["cov3D_precomp"], stack=5, streams=1)
    torch.cuda.synchronize()
    zero = np.zeros((3, 40, 56), np.float32)
    for k, cam in enumerate(cams):
        fstate, outs, _ = run_gpu(scene, cam, BG, zero)
        ref = bf.reference(fstate, 56, 40, np.asarray(BG, np.float32), zero, impl_T=outs["final_T"],
                           impl_n=outs["n_contrib"])
        fw = bf.check_forward(ref, color=color[k].cpu().numpy(), depth=depth[k].cpu().numpy())
        print("stacked view %d: forward worst %.3g, pixels excluded %d" % (k, fw["worst"], fw["excluded"]))
        assert fw["fail"] == 0 and fw["excluded"] == 0, (k, fw)


@pytest.mark.parametrize("color", ["sh3", "precomp"])
def test_random_scene_per_colour_mode(color):
    s = synthetic.make_scene(20000, "object", color, -4.0, seed=5)
    cam = synthetic.orbit_camera(256, 192, 0.7)
    scene = {"means3D": s.means3D, "opacities": s.opacities, "shs": s.shs, "colors_precomp": s.colors_precomp,
             "scales": s.scales, "rotations": s.rotations}
    check_case("random %s" % color, scene, cam, seed=6, sh_degree=s.sh_degree, exclusions_allowed=1e-3)


def test_config_A_element_by_element():
    import time

    s = synthetic.config_scene("A")
    cam = synthetic.config_cameras("A")[0]
    scene = {"means3D": s.means3D, "opacities": s.opacities, "shs": s.shs, "colors_precomp": s.colors_precomp,
             "scales": s.scales, "rotations": s.rotations}
    t0 = time.time()
    check_case("config A", scene, cam, seed=12, sh_degree=s.sh_degree, exclusions_allowed=1e-3)
    print("config A: %.1f s including the referee" % (time.time() - t0))
