"""GPU: the preprocess backward kernel Gaussian by Gaussian against the double-precision referee (tests/pbwd_f64.py),
in every launch variant and write mode.

Forward and backward run through the C-ABI (as in test_gpu_c_abi.py / test_gpu_blend_f64.py).  The backward's one
scratch allocation is the blend accumulator, which the preprocess backward only reads: after the call it holds the
per-Gaussian sums that are the referee's input.  The instantiation that ran, preprocess_backward_kernel<VEC, EAGER,
STATS>, is read from the profiler's kernel names and asserted for every case.  Every case prints its worst
error-to-bound ratio and its resolved and excluded counts; the excluded count is zero on the constructed scenes."""
import ctypes as C
import re
import time
from types import SimpleNamespace

import numpy as np
import pytest
import torch

import parity_lib as pl
import pbwd_f64 as pf
from test_gpu_blend_f64 import check_public_outputs_are_slot_scalings
from test_gpu_c_abi import ALLOC, Arena, FwdState, Gaussians, Grads, View, _lib, _ptr
from workload import synthetic
from workload.params import GaussianParams

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
BG = (0.1, 0.2, 0.3)
SHAPES = [1, 2, 31, 32, 33, 63, 64, 127, 128, 129, 255, 257]
PATTERNS = ["even", "odd", "both", "neither", "random", "last_alone"]
NAMES = ["dL_dmeans2D", "dL_dcolors", "dL_dopacity", "dL_dmeans3D", "dL_dcov3D", "dL_dsh", "dL_dscales", "dL_drotations"]
KERNEL = re.compile(r"preprocess_backward_kernel<(\w+), (\w+), (\w+)>")


class DensifyStats(C.Structure):  # brs_densify_stats
    _fields_ = [("grad_norm", C.c_void_p), ("count", C.c_void_p), ("index", C.c_void_p), ("rows", C.c_int)]


def lib():
    L = _lib()
    L.brs_backward_ex.argtypes = [C.POINTER(View), C.POINTER(Gaussians), C.c_void_p, C.POINTER(FwdState), C.c_void_p,
                                  C.c_void_p, C.POINTER(Grads), C.POINTER(DensifyStats), ALLOC, C.c_void_p, C.c_void_p]
    return L


class Variants:
    """Collects the preprocess_backward_kernel instantiations launched inside the block."""

    def __enter__(self):
        self.prof = torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA])
        self.prof.__enter__()
        return self

    def __exit__(self, *exc):
        torch.cuda.synchronize()
        self.prof.__exit__(*exc)
        self.ran = []
        for ev in self.prof.events():
            m = KERNEL.search(ev.name)
            if m:
                self.ran.append(tuple(x == "true" for x in m.groups()))
        return False


def camera(W=64, H=48):
    return synthetic.make_camera(W, H, np.eye(3), np.zeros(3))


def visible_mask(P, pattern, rng):
    i = np.arange(P)
    return {"even": i % 2 == 0, "odd": i % 2 == 1, "both": np.ones(P, bool), "neither": np.zeros(P, bool),
            "random": rng.random(P) < 0.5, "last_alone": (i == P - 1)}[pattern]


def make_scene(P, vis, rng, cam, D=3, M=16, cov_precomp=False, colors=False):
    """P Gaussians in front of the camera where vis, behind the near plane (culled) elsewhere; |q| in [0.5, 2];
    colour channels negative, near zero and positive."""
    import test_pbwd_f64 as tp

    gs = tp.edge_gaussians(rng, P, cam, D, 0 if colors else M)
    tz = rng.uniform(1.0, 6.0, P)
    t = np.stack([rng.uniform(-0.9, 0.9, P) * cam.tanfovx * tz, rng.uniform(-0.9, 0.9, P) * cam.tanfovy * tz, tz], 1)
    t[~vis, 2] = -1.0
    gs["means3D"] = pf.view_to_world(cam, t)
    gs["scales"] = (np.exp(rng.normal(-3.5, 0.6, (P, 3))) * tz[:, None] / 3).astype(np.float32)
    if cov_precomp:
        gs["cov3D_precomp"] = tp.covariance(gs["scales"], gs["rotations"])
    if not colors and M:
        # recompute the DC term for the new positions: targets straddle 0
        d = gs["means3D"].astype(np.float64) - np.asarray(cam.campos, np.float64)
        b = tp.sh_basis(D, d / np.linalg.norm(d, axis=1, keepdims=True))
        k = (D + 1) ** 2
        shs = gs["shs"].astype(np.float64)
        rest = np.einsum("nk,nkc->nc", b[:, 1:k], shs[:, 1:k])
        target = rng.uniform(-0.8, 1.2, (P, 3))
        shs[:, 0] = (target - 0.5 - rest) / 0.28209479177387814
        gs["shs"] = shs.astype(np.float32)
    if colors:
        gs["colors_precomp"] = rng.uniform(0, 1, (P, 3)).astype(np.float32)
    gs["opacities"] = rng.uniform(0.05, 0.9, (P, 1)).astype(np.float32)
    return {k: torch.from_numpy(np.ascontiguousarray(v)) for k, v in gs.items()
            if not (cov_precomp and k in ("scales", "rotations"))}


def run(scene, cam, D, seed=0, depth=False, mod=1.0, variant="lazy", shs_offset=False, dsh_offset=False, stats=False,
        bucket=None, frozen=()):
    """Forward + backward through the C-ABI.  variant "lazy": marks forgotten between forward and backward; "eager":
    a forward of the same (P, W, H) with every Gaussian visible runs first.  bucket: accumulate into a
    GaussianParams gradient bucket (frozen names get NULL sinks).  Returns (Problem, outputs, the accumulator); the
    Problem takes the forward records' colours as the colour-clamp hint."""
    from bloomscene_b200.debug import state_views

    L = lib()
    W, H = cam.image_width, cam.image_height
    t = {k: v.to(DEV).contiguous() for k, v in scene.items()}
    P = t["means3D"].shape[0]
    M = t["shs"].shape[1] if "shs" in t else 0
    bg = torch.tensor(BG, device=DEV)
    vm, pm, cp = (x.to(DEV).contiguous() for x in (cam.viewmatrix, cam.projmatrix, cam.campos))
    view = View(W, H, cam.tanfovx, cam.tanfovy, mod, D, M, 0, 0, _ptr(bg), _ptr(vm), _ptr(pm), _ptr(cp))
    g = Gaussians(P, _ptr(t["means3D"]), _ptr(t["opacities"]), _ptr(t.get("shs")), _ptr(t.get("colors_precomp")),
                  _ptr(t.get("scales")), _ptr(t.get("rotations")), _ptr(t.get("cov3D_precomp")))
    stream = torch.cuda.current_stream().cuda_stream
    color = torch.empty(3, H, W, device=DEV)
    depth_img = torch.empty(1, H, W, device=DEV)
    radii = torch.empty(P, dtype=torch.int32, device=DEV)
    if variant == "eager":
        warm = dict(t, means3D=torch.tensor([[0.0, 0.0, 3.0]], device=DEV).expand(P, 3).contiguous())
        gw = Gaussians(P, _ptr(warm["means3D"]), _ptr(t["opacities"]), _ptr(t.get("shs")), _ptr(t.get("colors_precomp")),
                       _ptr(t.get("scales")), _ptr(t.get("rotations")), _ptr(t.get("cov3D_precomp")))
        rc = L.brs_forward(C.byref(view), C.byref(gw), color.data_ptr(), depth_img.data_ptr(), radii.data_ptr(),
                           Arena().fn, None, C.byref(FwdState()), stream)
        assert rc == 0, L.brs_error_string(rc)
    arena, state = Arena(), FwdState()
    rc = L.brs_forward(C.byref(view), C.byref(g), color.data_ptr(), depth_img.data_ptr(), radii.data_ptr(), arena.fn,
                       None, C.byref(state), stream)
    assert rc == 0, L.brs_error_string(rc)
    torch.cuda.synchronize()
    if variant == "lazy":
        L.brs_reset_marks()
    R = state.num_rendered
    empty = torch.zeros(16, dtype=torch.uint8, device=DEV)
    sv = state_views(pl.ours()._C, arena.buffers[0], arena.buffers.get(1, empty), arena.buffers[2], P, R, W, H)
    rec_colors = sv["records"][:, 8:11].cpu().numpy().copy()

    rng = np.random.default_rng(seed)
    dpix = torch.as_tensor(rng.standard_normal((3, H, W)).astype(np.float32), device=DEV)
    ddep = torch.as_tensor(rng.standard_normal((1, H, W)).astype(np.float32), device=DEV) if depth else None
    gb = t
    if shs_offset:  # the same coefficients 4 bytes past a 16-byte boundary
        raw = torch.empty(P * M * 3 + 1, device=DEV)
        raw[1:].copy_(t["shs"].reshape(-1))
        gb = dict(t, shs=raw[1:].view(P, M, 3))
        assert gb["shs"].data_ptr() % 16 == 4
    gbwd = Gaussians(P, _ptr(gb["means3D"]), _ptr(gb["opacities"]), _ptr(gb.get("shs")), _ptr(gb.get("colors_precomp")),
                     _ptr(gb.get("scales")), _ptr(gb.get("rotations")), _ptr(gb.get("cov3D_precomp")))
    shapes = {"dL_dmeans2D": (P, 3), "dL_dcolors": (P, 3), "dL_dopacity": (P, 1), "dL_dmeans3D": (P, 3),
              "dL_dcov3D": (P, 6), "dL_dsh": (P, max(M, 1), 3), "dL_dscales": (P, 3), "dL_drotations": (P, 4)}
    if bucket is None:
        out = {k: torch.full(s, float("nan"), device=DEV) for k, s in shapes.items()}
        if dsh_offset:
            raw = torch.full((P * max(M, 1) * 3 + 1,), float("nan"), device=DEV)
            out["dL_dsh"] = raw[1:].view(P, max(M, 1), 3)
            assert out["dL_dsh"].data_ptr() % 16 == 4
        ptrs = [out[k].data_ptr() if (k != "dL_dsh" or M > 0) else None for k in NAMES]
        acc_mode = 0
    else:
        out = {"dL_dmeans2D": torch.full((P, 3), float("nan"), device=DEV)}
        sink = {"dL_dmeans3D": "means3D", "dL_dopacity": "opacities", "dL_dsh": "shs", "dL_dscales": "scales",
                "dL_drotations": "rotations", "dL_dcolors": "colors_precomp", "dL_dcov3D": "cov3D_precomp"}
        ptrs = [out["dL_dmeans2D"].data_ptr()] + [
            None if (sink[k] in frozen or sink[k] not in bucket.tensors) else bucket.tensors[sink[k]].grad.data_ptr()
            for k in NAMES[1:]]
        acc_mode = 1
    grads = Grads(*ptrs, acc_mode, 1 if depth else 0, depth_img.data_ptr() if depth else None)
    st = None
    if stats:
        norm = torch.zeros(P, device=DEV)
        cnt = torch.zeros(P, device=DEV)
        st = DensifyStats(norm.data_ptr(), cnt.data_ptr(), None, P)
    n_scratch = len(arena.scratch)
    rc = L.brs_backward_ex(C.byref(view), C.byref(gbwd), radii.data_ptr(), C.byref(state), dpix.data_ptr(), _ptr(ddep),
                           C.byref(grads), C.byref(st) if st else None, arena.fn, None, stream)
    assert rc == 0, L.brs_error_string(rc)
    torch.cuda.synchronize()
    assert len(arena.scratch) == n_scratch + 1  # the backward's one scratch allocation: the blend accumulator
    accum = arena.scratch[-1][:P * 12 * 4].view(torch.float32).view(P, 12).cpu().numpy().copy()
    rad = radii.cpu().numpy()
    pb = pf.Problem(W, H, cam.tanfovx, cam.tanfovy, cam.viewmatrix, cam.projmatrix, cam.campos, scene["means3D"], rad,
                    accum, sh_degree=D, shs=scene.get("shs"), scales=scene.get("scales"),
                    rotations=scene.get("rotations"), cov3D_precomp=scene.get("cov3D_precomp"), scale_modifier=mod,
                    depth_gradient=depth, color_hint=rec_colors if "shs" in scene else None)
    outs = {"radii": rad, "grads": {k: v.cpu().numpy().copy() for k, v in out.items()}}
    if st is not None:
        outs["stats"] = (norm.cpu().numpy(), cnt.cpu().numpy())
    return pb, outs, accum


def check_plain(what, pb, outs, accum, report=None):
    """Plain mode: public outputs are the slot scalings, visible rows are within bound, culled rows are exactly 0."""
    g = outs["grads"]
    check_public_outputs_are_slot_scalings(outs, accum, pb.W, pb.H)
    vis = pb.visible
    for k in NAMES:
        if k == "dL_dsh" and pb.M == 0:
            continue
        assert not np.isnan(g[k]).any(), (what, k)
        assert not g[k][~vis].any(), (what, k)
    rep = pf.check(pb, pf.pack(pb, g["dL_dmeans3D"], g["dL_dcov3D"], g["dL_dscales"], g["dL_drotations"],
                                g["dL_dsh"] if pb.M else None))
    line = "%s: %s" % (what, pf.describe(rep))
    if report is not None:
        report.append(line)
    else:
        print(line)
    assert rep["fail"] == 0, (what, rep["first_fail"], pf.element_name(rep["fail_elem"]), rep["worst"])
    return rep


# (variant, M, D, shs_offset, dsh_offset, expected (VEC, EAGER))
VARIANTS = {"lazy_vec": ("lazy", 16, 3, False, False, (True, False)),
            "eager_vec": ("eager", 16, 3, False, False, (True, True)),
            "fallback_m1": ("lazy", 1, 0, False, False, (False, False)),
            "fallback_m4": ("eager", 4, 1, False, False, (False, False)),
            "fallback_m9": ("lazy", 9, 2, False, False, (False, False)),
            "fallback_shs_offset": ("eager", 16, 3, True, False, (False, False)),
            "fallback_dsh_offset": ("lazy", 16, 3, False, True, (False, False))}


@pytest.mark.parametrize("name", list(VARIANTS))
def test_plain_mode_every_shape_and_pattern(name):
    """P in SHAPES x visibility patterns within lane pairs (even only, odd only, both, neither, random, the last
    Gaussian of the array alone), in one launch variant each."""
    variant, M, D, so, do, want = VARIANTS[name]
    cam = camera()
    worst, resolved, excluded, n = 0.0, 0, 0, 0
    lines = []
    with Variants() as v:
        for P in SHAPES:
            for k, pattern in enumerate(PATTERNS):
                rng = np.random.default_rng(1000 * P + k)
                vis = visible_mask(P, pattern, rng)
                scene = make_scene(P, vis, rng, cam, D=D, M=M)
                pb, outs, accum = run(scene, cam, D, seed=P + k, depth=(k % 2 == 1), variant=variant, shs_offset=so,
                                      dsh_offset=do)
                assert np.array_equal(pb.visible, vis), (P, pattern)
                rep = check_plain("%s P=%d %s" % (name, P, pattern), pb, outs, accum, lines)
                worst, resolved, excluded, n = max(worst, rep["worst"]), resolved + rep["resolved"], excluded + rep[
                    "excluded"], n + 1
    print("%s (VEC=%s, EAGER=%s): %d cases, worst %.3g, resolved %d, excluded %d" % (name, want[0], want[1], n, worst,
                                                                                      resolved, excluded))
    assert len(v.ran) == n and set(v.ran) == {want + (False,)}, (name, set(v.ran))
    assert excluded == 0


@pytest.mark.parametrize("opt", ["cov3D_precomp", "scale_modifier", "precomputed_colours"])
@pytest.mark.parametrize("depth", [False, True])
def test_plain_mode_options(opt, depth):
    cam = camera(80, 56)
    rng = np.random.default_rng(5)
    P = 257
    vis = rng.random(P) < 0.7
    scene = make_scene(P, vis, rng, cam, D=3, M=16, cov_precomp=opt == "cov3D_precomp",
                       colors=opt == "precomputed_colours")
    if opt == "precomputed_colours":
        scene.pop("shs", None)
    with Variants() as v:
        pb, outs, accum = run(scene, cam, 3, seed=9, depth=depth, mod=1.7 if opt == "scale_modifier" else 1.0)
    rep = check_plain("%s depth=%s" % (opt, depth), pb, outs, accum)
    assert rep["excluded"] == 0 and rep["checked"] == vis.sum()
    assert v.ran == [(opt != "precomputed_colours", False, False)]
    if opt == "precomputed_colours":
        assert np.array_equal(outs["grads"]["dL_dcolors"][vis], accum[vis, 6:9])


@pytest.mark.parametrize("variant", ["lazy", "eager"])
def test_densify_stats_do_not_change_gradients(variant):
    """The STATS instantiations share everything else: gradients bit-identical with and without brs_densify_stats."""
    cam = camera()
    rng = np.random.default_rng(31)
    P = 129
    scene = make_scene(P, rng.random(P) < 0.6, rng, cam)
    with Variants() as v:
        pb0, o0, a0 = run(scene, cam, 3, seed=3, depth=True, variant=variant)
        pb1, o1, a1 = run(scene, cam, 3, seed=3, depth=True, variant=variant, stats=True)
    eager = variant == "eager"
    assert v.ran == [(True, eager, False), (True, eager, True)]
    # the blend backward's float atomics may add in another order in the second call: rows whose accumulator is
    # bit-identical must give bit-identical gradient rows (most rows of these small Gaussians touch one 8x8 block)
    same = (a0 == a1).all(axis=1)
    assert same[pb1.visible].mean() > 0.5
    for k in NAMES:
        assert np.array_equal(o0["grads"][k][same], o1["grads"][k][same]), k
    check_plain("stats %s" % variant, pb1, o1, a1)
    vis = pb1.visible
    assert np.array_equal(o1["stats"][1], vis.astype(np.float32))


@pytest.mark.parametrize("P", [128, 129, 130, 131])
def test_accumulate_mode_bucket_alignment(P):
    """Accumulate into a GaussianParams bucket: P % 4 in {0..3} covers the rotation slice's 16-byte alignment (even P:
    red.v4) and the SH slice's (P % 4 == 0: VEC).  Invisible rows stay bit-identical, visible rows add the gradient
    (got - fill within bound plus u |got|), a second backward adds again, and NULL sinks leave their slices alone."""
    cam = camera()
    rng = np.random.default_rng(40 + P)
    vis = rng.random(P) < 0.6
    vis[-1] = True
    scene = make_scene(P, vis, rng, cam)
    sc = synthetic.Scene(scene["means3D"], scene["scales"], scene["rotations"], scene["opacities"], scene["shs"], None, 3)
    u = 2.0 ** -24
    for frozen in [(), ("scales", "rotations", "shs")]:
        params = GaussianParams(sc.to(DEV))
        fill = torch.randn(params.grad_bucket.shape, device=DEV) * 0.01
        params.grad_bucket.copy_(fill)
        names = [n for n in params.names]
        before = {n: params.tensors[n].grad.cpu().numpy().copy() for n in names}
        with Variants() as v:
            pb, outs, accum = run(scene, cam, 3, seed=P, depth=True, variant="lazy", bucket=params, frozen=frozen)
        # VEC needs dL_dsh 16-byte aligned: the SH slice starts at 11 P floats; a frozen (NULL) SH sink is no constraint
        assert v.ran == [(P % 4 == 0 or "shs" in frozen, False, False)], (P, v.ran)
        after = {n: params.tensors[n].grad.cpu().numpy().copy() for n in names}
        for n in names:
            assert np.array_equal(after[n][~vis], before[n][~vis]), n
            if n in frozen:
                assert np.array_equal(after[n], before[n]), n
        m2 = outs["grads"]["dL_dmeans2D"]
        assert np.array_equal(m2[vis, 0], accum[vis, 0] * np.float32(np.float32(0.5) * np.float32(cam.image_width)))
        d = {n: after[n].astype(np.float64) - before[n] for n in names}
        assert np.array_equal(after["opacities"][vis, 0], (before["opacities"][vis, 0] + accum[vis, 5]).astype(np.float32))
        got = pf.pack(pb, d["means3D"], np.zeros((P, 6)), None if "scales" in frozen else d["scales"],
                      None if "rotations" in frozen else d["rotations"], None if "shs" in frozen else d["shs"])
        slack = u * np.abs(pf.pack(pb, after["means3D"], np.zeros((P, 6)), after["scales"], after["rotations"],
                                   after["shs"])).astype(np.float64)
        vd, _, _ = pf.evaluate(pb, "double")
        # dL_dcov3D has no sink when scales + rotations are given, and frozen sinks have no gradient: those columns
        # hold the reference rounded to float, so only the added gradients are compared
        cols = list(range(3)) + ([] if "scales" in frozen else list(range(9, 12))) + \
            ([] if "rotations" in frozen else list(range(12, 16))) + ([] if "shs" in frozen else list(range(16, pb.n)))
        full = vd.astype(np.float32)
        full[:, cols] = got[:, cols]
        rep = pf.check(pb, full, slack=slack)
        print("accumulate P=%d frozen=%s: %s" % (P, frozen or "-", pf.describe(rep)))
        assert rep["fail"] == 0 and rep["excluded"] == 0, (P, frozen, rep["first_fail"], pf.element_name(rep["fail_elem"]))
        # a second backward into the same bucket adds again (its own blend sums: their float atomics may add in
        # another order)
        pb, _, _ = run(scene, cam, 3, seed=P, depth=True, variant="lazy", bucket=params, frozen=frozen)
        vd, _, _ = pf.evaluate(pb, "double")
        again = {n: params.tensors[n].grad.cpu().numpy().copy() for n in names}
        for n in names:
            assert np.array_equal(again[n][~vis], before[n][~vis]), n
            if n in frozen:
                assert np.array_equal(again[n], before[n]), n
        d2 = {n: again[n].astype(np.float64) - after[n] for n in names}
        got2 = pf.pack(pb, d2["means3D"], np.zeros((P, 6)), None if "scales" in frozen else d2["scales"],
                       None if "rotations" in frozen else d2["rotations"], None if "shs" in frozen else d2["shs"])
        full2 = vd.astype(np.float32)
        full2[:, cols] = got2[:, cols]
        slack2 = u * np.abs(pf.pack(pb, again["means3D"], np.zeros((P, 6)), again["scales"], again["rotations"],
                                    again["shs"])).astype(np.float64)
        rep2 = pf.check(pb, full2, slack=slack2)
        print("accumulate again P=%d frozen=%s: %s" % (P, frozen or "-", pf.describe(rep2)))
        assert rep2["fail"] == 0 and rep2["excluded"] == 0, (P, frozen, rep2["first_fail"], pf.element_name(rep2["fail_elem"]))


def test_accumulate_mode_cov3D_precomp_and_colours():
    """Accumulate mode with cov3D_precomp and precomputed colours: the dL_dcov3D and dL_dcolors sinks receive the
    gradients of the visible rows, nothing else moves."""
    cam = camera()
    rng = np.random.default_rng(77)
    P = 131
    vis = rng.random(P) < 0.6
    scene = make_scene(P, vis, rng, cam, cov_precomp=True, colors=True)
    scene.pop("shs", None)
    fill = {"means3D": torch.randn(P, 3, device=DEV), "opacities": torch.randn(P, 1, device=DEV),
            "colors_precomp": torch.randn(P, 3, device=DEV), "cov3D_precomp": torch.randn(P, 6, device=DEV)}

    bucket = SimpleNamespace(tensors={k: SimpleNamespace(grad=v) for k, v in fill.items()})
    before = {k: v.cpu().numpy().copy() for k, v in fill.items()}
    pb, outs, accum = run(scene, cam, 0, seed=4, bucket=bucket)
    after = {k: v.cpu().numpy().copy() for k, v in fill.items()}
    for k in fill:
        assert np.array_equal(after[k][~vis], before[k][~vis]), k
    assert np.array_equal(after["colors_precomp"][vis], (before["colors_precomp"][vis] + accum[vis, 6:9]).astype(np.float32))
    d = {k: after[k].astype(np.float64) - before[k] for k in fill}
    got = pf.pack(pb, d["means3D"], d["cov3D_precomp"])
    slack = 2.0 ** -24 * np.abs(pf.pack(pb, after["means3D"], after["cov3D_precomp"])).astype(np.float64)
    rep = pf.check(pb, got, slack=slack)
    print("accumulate cov3D_precomp + colours: %s" % pf.describe(rep))
    assert rep["fail"] == 0 and rep["excluded"] == 0


@pytest.mark.parametrize("color", ["sh3", "precomp"])
def test_random_scene_per_colour_mode(color):
    s = synthetic.make_scene(20000, "object", color, -4.0, seed=5)
    cam = synthetic.orbit_camera(256, 192, 0.7)
    scene = {"means3D": s.means3D, "opacities": s.opacities, "scales": s.scales, "rotations": s.rotations}
    if s.shs is not None:
        scene["shs"] = s.shs
    else:
        scene["colors_precomp"] = s.colors_precomp
    for depth in (False, True):
        pb, outs, accum = run(scene, cam, s.sh_degree, seed=6, depth=depth)
        rep = check_plain("random %s depth=%s" % (color, depth), pb, outs, accum)
        assert rep["excluded"] <= 1e-4 * rep["checked"]


@pytest.mark.parametrize("config", ["A", "C"])
def test_config_element_by_element(config):
    s = synthetic.config_scene(config)
    cam = synthetic.config_cameras(config)[0]
    scene = {"means3D": s.means3D, "opacities": s.opacities, "scales": s.scales, "rotations": s.rotations}
    if s.shs is not None:
        scene["shs"] = s.shs
    else:
        scene["colors_precomp"] = s.colors_precomp
    t0 = time.time()
    pb, outs, accum = run(scene, cam, s.sh_degree, seed=12)
    rep = check_plain("config %s" % config, pb, outs, accum)
    print("config %s: %.1f s including the referee" % (config, time.time() - t0))
    assert rep["excluded"] <= 1e-4 * rep["checked"]
