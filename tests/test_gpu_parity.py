"""GPU parity tests (pytest -m gpu on a B200).

Three independent checkers for the CUDA library, all driven through the public binding / C-ABI:
  1. stored records of the reference-parity cases (tests/golden/parity/*.npz, the `ref` fixture) — bit-exact
     integers and per-Gaussian intermediates, colour/depth <= 1e-5, gradients rel-L2 <= 1e-4, so the tests need
     no reference build.  The committed records were taken on a B200 from this library, with product code unchanged
     since the build that passed these tests against the reference's own CUDA rasterizer (profiles/r02_pytest_gpu.log);
     tests/golden/make_golden_parity.py records new ones only from that reference build, compared live;
  2. golden vectors captured from that reference (tests/golden/*.npz) — same bars;
  3. the CPU oracle (oracle/rasterizer_oracle.c) on small scenes, and size-independent properties at
     BASELINE.json's full sizes (sorted keys, range partition, bg linearity, determinism).
"""
import math

import numpy as np
import pytest
import torch

import parity_lib as pl
from workload import synthetic

pytestmark = pytest.mark.gpu

DEV = "cuda:0"


@pytest.fixture
def ref(request):
    """The stored results of the reference-parity comparisons of this test (parity_lib.Recorded)."""
    rec = pl.Recorded(request.node.name)
    failed = request.session.testsfailed
    yield rec
    rec.finish(passed=request.session.testsfailed == failed)  # the call's report is counted before teardown


def _assert_stage_parity(rep):
    for k in ("radii_mismatch", "depth_bits_mismatch", "means2D_mismatch", "conic_opacity_mismatch",
              "tiles_touched_mismatch", "point_list_mismatch", "ranges_mismatch", "sorted_keys_mismatch",
              "n_contrib_mismatch", "final_T_mismatch"):
        if k in rep:
            assert rep[k] == 0, (k, rep)
    assert rep["R_ours"] == rep["R_ref"], rep
    assert rep.get("color_maxabs", 0.0) <= pl.COLOR_TOL, rep
    assert rep.get("depth_maxabs", 0.0) <= pl.COLOR_TOL, rep


def _assert_grad_parity(rep):
    assert rep["radii_mismatch"] == 0
    assert rep["color_maxabs"] <= pl.COLOR_TOL and rep["depth_maxabs"] <= pl.COLOR_TOL, rep
    for k, v in rep.items():
        if k.startswith("grad_"):
            assert v <= pl.GRAD_TOL, (k, rep)  # relative L2 <= 1e-4


CASES = [
    # name, P, kind, color, mu, (W, H), yaw, bg, scale_modifier
    ("p1_tile", 1, "object", "sh0", -2.0, (16, 16), 0.0, (0, 0, 0), 1.0),
    ("p17_ragged", 17, "object", "sh3", -3.0, (17, 33), 0.3, (0.2, 0.5, 0.7), 1.0),
    ("p1000_sh1", 1000, "object", "sh1", -3.5, (130, 70), 1.0, (0, 0, 0), 1.0),
    ("p1000_sh2m16", 1000, "object", "sh2m16", -3.5, (64, 64), 2.0, (1, 1, 1), 1.0),
    ("p5000_sh0m16", 5000, "object", "sh0m16", -3.8, (200, 120), 0.0, (0, 0, 0), 0.7),
    ("p20k_precomp", 20_000, "object", "precomp", -4.0, (256, 256), 0.5, (0.1, 0.1, 0.1), 1.3),
    ("band_mostly_culled", 30_000, "band", "precomp", -4.0, (128, 128), 0.7, (0, 0, 0), 1.0),
    ("A_100k_sh0", 100_000, "object", "sh0", -4.0, (512, 512), 0.0, (0, 0, 0), 1.0),
]


def _make(case):
    name, P, kind, color, mu, (W, H), yaw, bg, mod = case
    scene = synthetic.make_scene(P, kind, color, mu, seed=sum(map(ord, name)) % 1000).to(DEV)
    cam = (synthetic.orbit_camera(W, H, yaw) if kind == "object" else synthetic.yaw_camera(W, H, yaw)).to(DEV)
    return scene, cam, torch.tensor(bg, dtype=torch.float32, device=DEV), mod


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_stages_bit_exact_vs_reference_cuda(case, ref):
    scene, cam, bg, mod = _make(case)
    _assert_stage_parity(pl.stages_vs_record(ref, scene, cam, bg, scale_modifier=mod))


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_autograd_vs_reference_cuda(case, ref):
    scene, cam, bg, mod = _make(case)
    Wc, Wd = (t.to(DEV) for t in synthetic.loss_weights(cam.image_width, cam.image_height))
    _assert_grad_parity(pl.autograd_vs_record(ref, scene, cam, bg, Wc, Wd, scale_modifier=mod))


def test_cov3d_precomp_vs_reference_cuda(ref):
    from golden.make_golden import cov3d_from_scale_rot

    s = synthetic.make_scene(3000, "object", "sh1", -3.6, seed=21)
    cov = cov3d_from_scale_rot(s.scales, s.rotations).to(DEV)
    scene, cam = s.to(DEV), synthetic.orbit_camera(160, 90, 0.4).to(DEV)
    bg = torch.zeros(3, device=DEV)
    Wc, Wd = (t.to(DEV) for t in synthetic.loss_weights(160, 90))
    _assert_stage_parity(pl.stages_vs_record(ref, scene, cam, bg, cov3D=cov))
    _assert_grad_parity(pl.autograd_vs_record(ref, scene, cam, bg, Wc, Wd, cov3D=cov))


def test_full_size_1m_1080p_sh3_vs_reference_cuda(ref):
    """BASELINE.json's headline configuration (config C)."""
    scene = synthetic.config_scene("C").to(DEV)
    cam = synthetic.config_cameras("C")[0].to(DEV)
    bg = torch.zeros(3, device=DEV)
    Wc, Wd = (t.to(DEV) for t in synthetic.loss_weights(cam.image_width, cam.image_height))
    _assert_stage_parity(pl.stages_vs_record(ref, scene, cam, bg))
    _assert_grad_parity(pl.autograd_vs_record(ref, scene, cam, bg, Wc, Wd))


def test_config_D_3m_4k_sh3_vs_reference_cuda(ref):
    """BASELINE.json configs[3]: 3M Gaussians, SH3, 3840x2160 (32 400 tiles, 47 key bits in the reference's
    sort: getHigherMsb, rasterizer_impl.cu:35-50), band scene seen from two yaws of the rotate360 trajectory."""
    scene = synthetic.config_scene("D").to(DEV)
    cams = synthetic.config_cameras("D")
    bg = torch.zeros(3, device=DEV)
    for k in (0, 37):
        cam = cams[k].to(DEV)
        rep = pl.stages_vs_record(ref, scene, cam, bg)
        assert rep["visible"] > 100_000 and rep["R_ref"] > 1_000_000, rep
        _assert_stage_parity(rep)
        torch.cuda.empty_cache()


def test_config_B_500k_precomp_512_vs_reference_cuda(ref):
    """BASELINE.json configs[1]: BloomScene's own working point — 500K neural Gaussians with colors_precomp,
    512x512, rotate360 yaws; ~88 % of the Gaussians are outside any one view (culled)."""
    scene = synthetic.config_scene("B").to(DEV)
    cams = synthetic.config_cameras("B")
    bg = torch.zeros(3, device=DEV)
    Wc, Wd = (t.to(DEV) for t in synthetic.loss_weights(512, 512))
    for k in (0, 29, 60, 101):
        cam = cams[k].to(DEV)
        rep = pl.stages_vs_record(ref, scene, cam, bg)
        assert 0 < rep["visible"] < scene.P // 4, rep
        _assert_stage_parity(rep)
        _assert_grad_parity(pl.autograd_vs_record(ref, scene, cam, bg, Wc, Wd))


def test_edge_cases_vs_reference_cuda(ref):
    mine = pl.ours()
    bg = torch.tensor([0.3, 0.6, 0.9], device=DEV)
    # P == 0: zero image, background NOT composited (rasterize_points.cu:68-82)
    s0 = synthetic.make_scene(0, "object", "precomp", -3.0).to(DEV)
    cam = synthetic.orbit_camera(48, 32, 0.0).to(DEV)
    R, color, depth, radii, *_ = mine._C.rasterize_gaussians(*pl.forward_args(s0, cam, bg))
    assert R == 0 and not color.any() and not depth.any() and radii.numel() == 0
    _assert_stage_parity(pl.stages_vs_record(ref, s0, cam, bg))
    # everything behind the camera: R == 0 but the blend still runs -> image == background
    s = synthetic.make_scene(500, "object", "precomp", -3.0, seed=1)
    s.means3D[:, 2] -= 10.0
    s = s.to(DEV)
    rep = pl.stages_vs_record(ref, s, cam, bg)
    assert rep["R_ours"] == 0 and rep["R_ref"] == 0 and rep["radii_mismatch"] == 0
    R, color, depth, radii, *_ = mine._C.rasterize_gaussians(*pl.forward_args(s, cam, bg))
    assert torch.allclose(color, bg.view(3, 1, 1).expand_as(color)) and not depth.any() and not radii.any()
    Wc, Wd = (t.to(DEV) for t in synthetic.loss_weights(48, 32))
    out = pl.run_autograd(mine, s, cam, bg, Wc, Wd)
    assert all(not g.any() for g in out["grads"].values() if g is not None)
    # a huge opaque Gaussian over the whole screen + saturation (0.99 clamp, T < 1e-4 early stop)
    s = synthetic.make_scene(800, "object", "sh0", -3.0, seed=7)
    s.scales[0] = torch.tensor([0.8, 0.8, 0.8])
    s.means3D[0] = torch.tensor([0.0, 0.0, -1.5])
    s.opacities[:100] = 1.0
    s = s.to(DEV)
    _assert_stage_parity(pl.stages_vs_record(ref, s, cam, bg))
    _assert_grad_parity(pl.autograd_vs_record(ref, s, cam, bg, Wc, Wd))
    # exact depth ties (duplicated Gaussians): stability of the sort decides the order
    b = synthetic.make_scene(400, "object", "sh2", -3.0, seed=6)
    dup = synthetic.Scene(*[None if t is None else torch.cat([t, t]).contiguous() for t in
                            (b.means3D, b.scales, b.rotations, b.opacities, b.shs, b.colors_precomp)], b.sh_degree).to(DEV)
    _assert_stage_parity(pl.stages_vs_record(ref, dup, cam, bg))
    # opacity below 1/255 and above 1: culling boxes must stay conservative
    s = synthetic.make_scene(2000, "object", "precomp", -3.2, seed=8)
    s.opacities[::3] = 0.003
    s.opacities[1::3] = 1.7
    s = s.to(DEV)
    _assert_stage_parity(pl.stages_vs_record(ref, s, cam, bg))
    _assert_grad_parity(pl.autograd_vs_record(ref, s, cam, bg, Wc, Wd))
    # strongly anisotropic Gaussians (needle-like): loose fp32 power evaluation in the reference
    s = synthetic.make_scene(1500, "object", "precomp", -4.0, seed=9)
    s.scales[:, 0] *= 60.0
    s = s.to(DEV)
    _assert_stage_parity(pl.stages_vs_record(ref, s, synthetic.orbit_camera(320, 200, 0.9).to(DEV), bg))


def test_non_finite_inputs_vs_reference_cuda(ref):
    """Non-finite parameters (a diverged optimisation).  Geometry, keys and lists stay bit-identical; a non-finite
    OPACITY or CONIC behaves as in the reference (fminf(0.99, NaN) = 0.99 on both sides, the culling test lets NaNs
    pass).  A non-finite COLOUR is the one documented difference (INTEGRATION.md): the reference poisons the pixels
    the Gaussian contributes to, the branch-free blend poisons the 8x8 pixel blocks it contributes to — a superset,
    and everything outside it is unchanged."""
    mine = pl.ours()
    cam = synthetic.orbit_camera(96, 64, 0.2).to(DEV)
    bg = torch.tensor([0.1, 0.2, 0.3], device=DEV)

    def render(api, s):
        R, color, depth, radii, *_ = api._C.rasterize_gaussians(*pl.forward_args(s, cam, bg))
        torch.cuda.synchronize()
        return R, color, depth, radii

    def record(R, color, depth, radii):
        """counts, radii, where colour and depth are finite (every element), colour and depth values (parity_lib.floats)"""
        return {"R": R, "radii": pl.digest(radii), "color_finite": np.packbits(torch.isfinite(color).cpu().numpy()),
                "depth_finite": np.packbits(torch.isfinite(depth).cpu().numpy()), **pl.floats("color", color),
                **pl.floats("depth", depth)}

    def rendered(s):
        """This library's forward, its record and the reference's record of the same forward."""
        out = render(mine, s)
        m = record(*out)
        return (*out, m, ref.take(m, lambda: record(*render(pl.reference(), s))))

    # opacity / position NaN: identical behaviour
    s = synthetic.make_scene(600, "object", "precomp", -3.2, seed=12)
    s.opacities[20] = float("nan")
    s.opacities[21] = float("inf")
    s.means3D[40, 0] = float("nan")
    s = s.to(DEV)
    rep = pl.stages_vs_record(ref, s, cam, bg)
    assert rep["point_list_mismatch"] == 0 and rep["ranges_mismatch"] == 0 and rep["n_contrib_mismatch"] == 0, rep
    Ro, co, do, ro, m, w = rendered(s)
    assert Ro == int(w["R"]) and pl.rec_mismatch(m, w, "radii") == 0
    assert np.array_equal(m["color_finite"], w["color_finite"])
    assert pl.rec_maxabs(m, w, "color", finite_only=True) <= pl.COLOR_TOL
    assert np.array_equal(m["depth_finite"], w["depth_finite"]) and pl.rec_maxabs(m, w, "depth", finite_only=True) <= pl.COLOR_TOL

    # a NaN / inf opacity BEHIND pixels that have already saturated: the reference never touches a finished pixel
    # (`done`), fminf(0.99, NaN) = 0.99 must not revive it
    s = synthetic.make_scene(900, "object", "precomp", -3.0, seed=14)
    s.means3D[0] = torch.tensor([0.0, 0.0, -1.5])          # a huge opaque Gaussian in front of everything
    s.scales[0] = torch.tensor([0.8, 0.8, 0.8])
    s.opacities[:60] = 1.0
    s.opacities[400] = float("nan")
    s.opacities[401] = float("inf")
    s.opacities[402] = float("-inf")
    s = s.to(DEV)
    rep = pl.stages_vs_record(ref, s, cam, bg)
    assert rep["point_list_mismatch"] == 0 and rep["n_contrib_mismatch"] == 0 and rep["final_T_mismatch"] == 0, rep
    _, co, _, _, m, w = rendered(s)
    assert np.array_equal(m["color_finite"], w["color_finite"]) and pl.rec_maxabs(m, w, "color", finite_only=True) <= pl.COLOR_TOL
    assert (co[torch.isfinite(co)] < 1e30).all()

    # NaN scale -> NaN covariance -> radius (int)NaN = 0 with a one-tile rect.  The reference counts that instance but
    # never writes its key (`if (radii[idx] > 0)`, rasterizer_impl.cu:85) and sorts an uninitialised slot; here the
    # Gaussian is culled: same image as with the Gaussian behind the camera.
    s = synthetic.make_scene(600, "object", "precomp", -3.2, seed=12)
    t = synthetic.make_scene(600, "object", "precomp", -3.2, seed=12)
    s.scales[30, 1] = float("nan")
    t.means3D[30, 2] -= 100.0
    Rs, cs, ds, rs = render(mine, s.to(DEV))
    Rt, ct, dt, rt = render(mine, t.to(DEV))
    assert Rs == Rt and torch.equal(rs, rt) and rs[30] == 0 and torch.equal(cs, ct) and torch.equal(ds, dt)

    # colour NaN / inf: superset within 8x8 blocks
    s = synthetic.make_scene(600, "object", "precomp", -3.2, seed=13)
    s.scales[:] *= 0.5
    s.colors_precomp[5, 1] = float("nan")
    s.colors_precomp[9, 0] = float("inf")
    s = s.to(DEV)
    Ro, co, do, ro, m, w = rendered(s)
    assert Ro == int(w["R"]) and pl.rec_mismatch(m, w, "radii") == 0
    finite_ref = np.unpackbits(w["color_finite"], count=co.numel()).astype(bool).reshape(co.shape)
    bad_ref = ~torch.from_numpy(finite_ref).to(DEV).all(0)
    bad_ours = ~torch.isfinite(co).all(0)
    assert bad_ref.any() and not bad_ref.all()
    assert not (bad_ref & ~bad_ours).any()                       # superset
    H, W = bad_ref.shape
    blocks = torch.nn.functional.max_pool2d(bad_ref[None, None].float(), 8, 8, ceil_mode=True)
    dil = torch.nn.functional.interpolate(blocks, scale_factor=8, mode="nearest")[0, 0, :H, :W] > 0
    assert not (bad_ours & ~dil).any()                           # ... confined to the touched 8x8 blocks
    k = w["color"].size                                          # stored colour elements (a sample of the image)
    good = ~bad_ours.flatten().cpu().numpy()[pl.sample_index(co.numel(), k) % (H * W)]
    assert np.abs(m["color"][:k][good].astype(np.float64) - w["color"][good]).max() <= pl.COLOR_TOL
    assert pl.rec_maxabs(m, w, "depth") <= pl.COLOR_TOL         # depth does not see colours


def test_debug_flag_and_python_api_shapes():
    mine = pl.ours()
    scene = synthetic.make_scene(2000, "object", "sh3", -3.5, seed=2).to(DEV)
    cam = synthetic.orbit_camera(96, 64, 0.1).to(DEV)
    bg = torch.zeros(3, device=DEV)
    a = mine._C.rasterize_gaussians(*pl.forward_args(scene, cam, bg, debug=False))
    b = mine._C.rasterize_gaussians(*pl.forward_args(scene, cam, bg, debug=True))
    assert a[0] == b[0] and torch.equal(a[1], b[1]) and torch.equal(a[2], b[2]) and torch.equal(a[3], b[3])
    assert a[1].shape == (3, 64, 96) and a[2].shape == (1, 64, 96) and a[3].dtype == torch.int32


def test_visible_filter_and_mark_visible(ref):
    mine = pl.ours()
    from bloomscene_b200.rasterizer import GaussianRasterizationSettings as S

    scene = synthetic.make_scene(50_000, "band", "precomp", -3.5, seed=4).to(DEV)
    cam = synthetic.yaw_camera(256, 192, 1.0).to(DEV)
    st = synthetic.raster_settings(cam, 0, torch.zeros(3, device=DEV), S)
    six = torch.cat([scene.scales, scene.scales * 2], dim=1)  # BloomScene passes scaling[:, :3] of a [P,6] tensor
    sliced = six[:, :3]
    assert not sliced.is_contiguous()
    r_mine = mine.GaussianRasterizer(st).visible_filter(scene.means3D, sliced, scene.rotations)
    v_mine = mine.GaussianRasterizer(st).markVisible(scene.means3D)
    got = {"visible_filter": pl.digest(r_mine), "mark_visible": pl.digest(v_mine)}
    want = ref.take(got, lambda: {"visible_filter": pl.digest(pl.reference().GaussianRasterizer(st).visible_filter(scene.means3D, sliced, scene.rotations)),
                                  "mark_visible": pl.digest(pl.reference().GaussianRasterizer(st).markVisible(scene.means3D))})
    assert r_mine.dtype == torch.int32 and pl.rec_mismatch(got, want, "visible_filter") == 0
    fw = mine._C.rasterize_gaussians(*pl.forward_args(scene, cam, torch.zeros(3, device=DEV)))
    assert torch.equal(fw[3], r_mine)
    # fused filter + compaction (SURVEY.md 8f N2): same radii, and the index list torch.nonzero would give
    r2, idx = mine.GaussianRasterizer(st).visible_filter_indices(scene.means3D, sliced, scene.rotations)
    assert torch.equal(r2, r_mine) and idx.dtype == torch.int64
    assert torch.equal(idx, torch.nonzero(r_mine > 0).flatten()) and idx.numel() > 1000
    empty = synthetic.make_scene(700, "object", "precomp", -3.0, seed=1)
    empty.means3D[:, 2] -= 10.0
    r3, idx3 = mine.GaussianRasterizer(st).visible_filter_indices(empty.means3D.to(DEV), empty.scales.to(DEV), empty.rotations.to(DEV))
    assert idx3.numel() == 0 and not r3.any()
    assert v_mine.dtype == torch.bool and pl.rec_mismatch(got, want, "mark_visible") == 0
    assert (v_mine | (r_mine == 0)).all()


def test_sort_pairs_is_a_stable_radix_sort():
    from bloomscene_b200 import _C

    g = torch.Generator(device="cpu").manual_seed(5)
    # sizes on both sides of every tile size (1024 / 2048 / 4096 pairs) and of the capacity thresholds that pick it
    # (128 K and 384 K pairs: 4, 8 or 16 keys per thread, binning.cu sort_items)
    for n, hi in [(0, 32), (1, 32), (33, 32), (1024, 32), (1025, 7), (4096, 9), (4097, 32), (123_457, 13), (131_072, 32),
                  (131_073, 24), (250_001, 32), (393_216, 17), (393_217, 32), (1_000_003, 32), (3_000_000, 15)]:
        keys = torch.randint(0, 2 ** 31 - 1, (n,), generator=g, dtype=torch.int64)
        if hi < 32:
            keys &= (1 << hi) - 1
        if n > 100:
            keys[::5] = keys[0]  # many exact ties
        ko, vo = _C.sort_pairs(keys.to(torch.int32).to(DEV), None, 0, hi)
        rk, ri = torch.sort(keys.to(DEV), stable=True)
        assert torch.equal(ko.long(), rk) and torch.equal(vo.long(), ri), (n, hi)
    # explicit values and a bit sub-range: order inside equal digits must be the input order
    keys = torch.randint(0, 2 ** 20, (50_000,), generator=g, dtype=torch.int64)
    vals = torch.randint(0, 2 ** 31 - 1, (50_000,), generator=g, dtype=torch.int64)
    ko, vo = _C.sort_pairs(keys.to(torch.int32).to(DEV), vals.to(torch.int32).to(DEV), 4, 12)
    digit = (keys >> 4) & 0xFF
    _, ri = torch.sort(digit.to(DEV), stable=True)
    assert torch.equal(vo.long(), vals.to(DEV)[ri]) and torch.equal(ko.long(), keys.to(DEV)[ri])


def test_properties_at_full_size():
    """Size-independent invariants at config C (1M Gaussians, 1080p, SH3) — no reference needed."""
    from bloomscene_b200.debug import state_views

    mine = pl.ours()
    scene = synthetic.config_scene("C").to(DEV)
    cam = synthetic.config_cameras("C")[0].to(DEV)
    W, H = cam.image_width, cam.image_height
    bg0 = torch.zeros(3, device=DEV)
    R, color, depth, radii, geom, binning, img = mine._C.rasterize_gaussians(*pl.forward_args(scene, cam, bg0))
    sv = state_views(mine._C, geom, binning, img, scene.P, R, W, H)
    # ranges partition [0, R) in tile order; keys sorted by (tile, depth bits, id)
    ranges = sv["ranges"].long()
    nonempty = ranges[:, 1] > ranges[:, 0]
    rs = ranges[nonempty]
    assert rs[0, 0] == 0 and rs[-1, 1] == R and torch.equal(rs[1:, 0], rs[:-1, 1])
    tile_of = torch.repeat_interleave(torch.arange(ranges.shape[0], device=DEV), (ranges[:, 1] - ranges[:, 0]).clamp(min=0))
    pl_ids = sv["point_list"].long()
    dk = sv["depth_key"].long() & 0xFFFFFFFF
    keys = (tile_of << 32) | dk[pl_ids]
    assert (keys[1:] >= keys[:-1]).all()
    ties = keys[1:] == keys[:-1]
    assert (pl_ids[1:][ties] > pl_ids[:-1][ties]).all()  # stable: ties keep Gaussian-id order
    # every instance lies inside its Gaussian's tile rectangle; R == sum of rectangle areas
    rect = sv["rect"]
    x0, x1, y0, y1 = rect[:, 0] & 0xFFFF, rect[:, 0] >> 16, rect[:, 1] & 0xFFFF, rect[:, 1] >> 16
    assert int(((x1 - x0) * (y1 - y0)).sum()) == R
    gx = (W + 15) // 16
    tx, ty = tile_of % gx, tile_of // gx
    assert ((tx >= x0[pl_ids]) & (tx < x1[pl_ids]) & (ty >= y0[pl_ids]) & (ty < y1[pl_ids])).all()
    assert ((radii > 0) == (sv["depth_key"] != -1)).all()
    # n_contrib never exceeds the tile's list length; outputs are finite
    n_contrib = sv["n_contrib"].view(H, W)
    lens = (ranges[:, 1] - ranges[:, 0]).view((H + 15) // 16, gx)
    per_pix = lens.repeat_interleave(16, 0)[:H].repeat_interleave(16, 1)[:, :W]
    assert (n_contrib <= per_pix).all()
    assert torch.isfinite(color).all() and torch.isfinite(depth).all() and (depth >= 0).all()
    # determinism of every integer output and of the image across calls
    R2, color2, depth2, radii2, geom2, binning2, img2 = mine._C.rasterize_gaussians(*pl.forward_args(scene, cam, bg0))
    sv2 = state_views(mine._C, geom2, binning2, img2, scene.P, R2, W, H)
    assert R2 == R and torch.equal(radii, radii2) and torch.equal(sv["point_list"], sv2["point_list"])
    assert torch.equal(color, color2) and torch.equal(depth, depth2)
    # background linearity: color(bg) - color(0) == final_T * bg
    bg1 = torch.tensor([0.25, 0.5, 1.0], device=DEV)
    _, color_bg, depth_bg, *_ = mine._C.rasterize_gaussians(*pl.forward_args(scene, cam, bg1))
    T = sv["final_T"].view(1, H, W)
    assert torch.allclose(color_bg - color, T * bg1.view(3, 1, 1), atol=2e-6)
    assert torch.equal(depth_bg, depth)
    # gradients: linear in dL/dpixel (2x upstream gradient -> 2x every gradient, exactly in fp32 up to atomics order)
    Wc, Wd = (t.to(DEV) for t in synthetic.loss_weights(W, H))
    g1 = pl.run_autograd(mine, scene, cam, bg0, Wc, Wd)["grads"]
    g2 = pl.run_autograd(mine, scene, cam, bg0, 2 * Wc, Wd)["grads"]
    for k in g1:
        assert pl.rel_l2(g2[k], 2 * g1[k]) <= 1e-5, k


def test_small_scene_vs_cpu_oracle():
    from oracle import oracle as orc

    mine = pl.ours()
    scene_cpu = synthetic.make_scene(4000, "object", "sh2", -3.4, seed=12)
    cam_cpu = synthetic.orbit_camera(150, 100, 0.8)
    bg = torch.tensor([0.1, 0.3, 0.5])
    Wc, Wd = synthetic.loss_weights(150, 100)
    o = orc.run_scene(scene_cpu, cam_cpu, bg, dL_dcolor=Wc)
    out = pl.run_autograd(mine, scene_cpu.to(DEV), cam_cpu.to(DEV), bg.to(DEV), Wc.to(DEV), Wd.to(DEV))
    assert (out["radii"].cpu().numpy() != o["radii"]).mean() <= 1e-3
    assert np.abs(out["color"].cpu().numpy() - o["color"]).max() <= 1e-4
    assert np.abs(out["depth"].cpu().numpy() - o["depth"]).max() <= 1e-4
    m = {"means3D": "dL_dmeans3D", "means2D": "dL_dmeans2D", "opacities": "dL_dopacity", "scales": "dL_dscales",
         "rotations": "dL_drotations", "shs": "dL_dsh"}
    for k, v in m.items():
        assert pl.rel_l2(out["grads"][k].cpu(), torch.from_numpy(o["grads"][v])) <= 1e-3, k


@pytest.mark.parametrize("color", ["sh3", "precomp"])
def test_grad_sink_accumulates_like_autograd(color):
    """Extension: with `grad_sink` the kernel adds parameter gradients of several views in place; the
    result must equal autograd's own accumulation of the plain path (rel-L2 <= 1e-4, float atomics)."""
    from bloomscene_b200.multiview import GaussianParams, view_sharded_step

    api = pl.ours()
    scene = synthetic.make_scene(6000, "object", color, -3.6, seed=11).to(DEV)
    cams = [synthetic.orbit_camera(176, 112, y).to(DEV) for y in (0.0, 1.1, 2.3)]
    Wc, Wd = [t.to(DEV) for t in synthetic.loss_weights(176, 112)]
    bg = torch.tensor([0.2, 0.1, 0.4], device=DEV)
    loss_fn = lambda c, d, vi: (c * Wc).sum() + (d * Wd).sum()

    class Plain(api.GaussianRasterizer):  # same kernels, reference-style autograd accumulation
        supports_grad_sink = False

    got = GaussianParams(scene)
    want = GaussianParams(scene)
    r1 = view_sharded_step(got, cams, bg, api.GaussianRasterizer, loss_fn)
    r2 = view_sharded_step(want, cams, bg, Plain, loss_fn)
    assert float(r1["loss"]) == pytest.approx(float(r2["loss"]), rel=1e-6)
    for name in got.names:
        g, w = got.tensors[name].grad, want.tensors[name].grad
        assert float(w.abs().max()) > 0, name
        assert pl.rel_l2(g, w) <= pl.GRAD_TOL, (name, pl.rel_l2(g, w))
    # a second step starts from a zeroed bucket again
    view_sharded_step(got, cams, bg, api.GaussianRasterizer, loss_fn)
    for name in got.names:
        assert pl.rel_l2(got.tensors[name].grad, want.tensors[name].grad) <= pl.GRAD_TOL, name


@pytest.mark.gpu
def test_render_views_multi_stream_is_bit_identical_to_single_calls():
    """Forward-only batch render over 4 CUDA streams (band scene, rotate360 yaws) against one call per view."""
    api = pl.ours()
    dev = torch.device("cuda:0")
    scene = synthetic.make_scene(60000, "band", "sh3", -4.6, seed=11).to(dev)
    cams = [synthetic.yaw_camera(320, 192, 0.35 * k).to(dev) for k in range(9)]
    bg = torch.tensor([0.3, 0.2, 0.1], device=dev)
    settings = [synthetic.raster_settings(c, 3, bg, api.GaussianRasterizationSettings) for c in cams]
    color, depth, radii = api.render_views(settings, scene.means3D, scene.opacities, shs=scene.shs, scales=scene.scales,
                                           rotations=scene.rotations, streams=4, keep_radii=True)
    torch.cuda.synchronize()
    assert color.shape == (9, 3, 192, 320) and depth.shape == (9, 1, 192, 320)
    with torch.no_grad():
        for k, rs in enumerate(settings):
            c, r, d = api.GaussianRasterizer(rs)(scene.means3D, torch.zeros_like(scene.means3D), scene.opacities,
                                                 shs=scene.shs, scales=scene.scales, rotations=scene.rotations)
            assert torch.equal(c, color[k]) and torch.equal(d, depth[k]) and torch.equal(r, radii[k])
    assert (radii[0] > 0).sum() > 100


@pytest.mark.parametrize("case", [("sh3", 60000, 320, 192, 9, 4), ("precomp", 30000, 200, 120, 7, 8),
                                  ("sh1", 5000, 130, 70, 5, 2), ("precomp", 200000, 512, 512, 6, 3)],
                         ids=["sh3_320x192_stack4", "precomp_200x120_stack8", "sh1_130x70_stack2", "precomp_512_stack3"])
def test_render_views_stacked_pipeline_is_bit_identical_to_single_calls(case):
    """brs_forward_views: a stack of views as ONE pipeline (one depth sort, one binning chain, one blend launch over
    views * tiles) against one call per view — colour, depth and radii bit for bit.  Ragged image heights (192, 120, 70
    are not multiples of the 128-pixel supertile; 120 and 70 not of the 16-pixel tile), stacks that do not divide the
    number of views, and repeated calls (EXACT first, optimistic afterwards)."""
    color_kind, P, W, H, B, stack = case
    api = pl.ours()
    dev = torch.device("cuda:0")
    scene = synthetic.make_scene(P, "band", color_kind, -4.6, seed=11).to(dev)
    cams = [synthetic.yaw_camera(W, H, 0.35 * k).to(dev) for k in range(B)]
    bg = torch.tensor([0.3, 0.2, 0.1], device=dev)
    settings = [synthetic.raster_settings(c, scene.sh_degree, bg, api.GaussianRasterizationSettings) for c in cams]
    kw = dict(shs=scene.shs, colors_precomp=scene.colors_precomp, scales=scene.scales, rotations=scene.rotations)
    for rep in range(2):
        color, depth, radii = api.render_views(settings, scene.means3D, scene.opacities, keep_radii=True, stack=stack,
                                               streams=1 + rep, **kw)  # one stream, then stacks dealt onto two lanes
        torch.cuda.synchronize()
        assert color.shape == (B, 3, H, W) and depth.shape == (B, 1, H, W)
        with torch.no_grad():
            for k, rs in enumerate(settings):
                c, r, d = api.GaussianRasterizer(rs)(scene.means3D, torch.zeros_like(scene.means3D), scene.opacities, **kw)
                assert torch.equal(r, radii[k]), (rep, k)
                assert torch.equal(c, color[k]) and torch.equal(d, depth[k]), (rep, k)
    assert sum(int((r > 0).sum()) for r in radii) > 100


@pytest.mark.parametrize("color", ["sh2", "precomp"])
def test_opt_in_depth_gradient_vs_cpu_oracle(color):
    """Extension (SURVEY.md 8f N3): with depth_gradient=True the depth image back-propagates through D / acc.
    The CPU oracle implements the same extension (oracle/rasterizer_oracle.c, orc_backward_ex; its
    derivative is pinned by finite differences in tests/test_host_api.py); default stays gradient-free."""
    from oracle import oracle as orc

    api = pl.ours()
    W, H = 150, 100
    scene_cpu = synthetic.make_scene(4000, "object", color, -3.4, seed=21)
    cam_cpu = synthetic.orbit_camera(W, H, 0.5)
    bg = torch.tensor([0.1, 0.3, 0.5])
    Wc, Wd = synthetic.loss_weights(W, H)
    o = orc.run_scene(scene_cpu, cam_cpu, bg)
    ref = o["oracle"].backward(Wc.numpy(), Wd.numpy())
    ref_depth_only = o["oracle"].backward(np.zeros_like(Wc.numpy()), Wd.numpy())
    assert np.abs(ref_depth_only["dL_dmeans3D"]).sum() > 0

    scene, cam = scene_cpu.to(DEV), cam_cpu.to(DEV)
    Wc_d, Wd_d = Wc.to(DEV), Wd.to(DEV)
    settings = synthetic.raster_settings(cam, scene.sh_degree, bg.to(DEV), api.GaussianRasterizationSettings)
    names = ["means3D", "opacities", "scales", "rotations"] + (["shs"] if scene.shs is not None else ["colors_precomp"])
    key = {"means3D": "dL_dmeans3D", "opacities": "dL_dopacity", "scales": "dL_dscales", "rotations": "dL_drotations",
           "shs": "dL_dsh", "colors_precomp": "dL_dcolors", "means2D": "dL_dmeans2D"}

    def run(depth_gradient, use_color=True, sink=False):
        leaves = {n: getattr(scene, n).detach().clone().requires_grad_(True) for n in names}
        m2 = torch.zeros_like(scene.means3D, requires_grad=True)
        sinks = {n: torch.zeros_like(t) for n, t in leaves.items()} if sink else None
        rast = api.GaussianRasterizer(settings, grad_sink=sinks, depth_gradient=depth_gradient)
        color_img, _, depth_img = rast(means3D=leaves["means3D"], means2D=m2, opacities=leaves["opacities"],
                                       shs=leaves.get("shs"), colors_precomp=leaves.get("colors_precomp"),
                                       scales=leaves["scales"], rotations=leaves["rotations"])
        loss = (depth_img * Wd_d).sum() + ((color_img * Wc_d).sum() if use_color else 0.0)
        loss.backward()
        g = {n: (sinks[n] if sink else t.grad) for n, t in leaves.items()}
        g["means2D"] = m2.grad
        return g

    got = run(True)
    for n, t in got.items():
        assert pl.rel_l2(t.cpu(), torch.from_numpy(ref[key[n]]).reshape(t.shape)) <= 1e-3, n
    got = run(True, use_color=False)
    for n, t in got.items():
        r = torch.from_numpy(ref_depth_only[key[n]]).reshape(t.shape)
        if r.abs().sum() > 0:
            assert pl.rel_l2(t.cpu(), r) <= 1e-3, n
        else:
            assert not t.any(), n
    sunk = run(True, sink=True)
    plain = run(True)
    for n in names:
        assert pl.rel_l2(sunk[n], plain[n]) <= 1e-4, n
    # default (reference behaviour): a depth-only loss moves nothing
    off = run(False, use_color=False)
    for n, t in off.items():
        assert t is None or not t.any(), n


def test_fuzz_small_scenes_vs_reference_cuda(ref):
    """Seeded random sweep over sizes the fixed cases do not hit: odd / tiny / non-multiple-of-8 images (the blend
    kernels give every lane the pixels (x, y) and (x, y + 4) of an 8x8 block), Gaussian sizes from sub-pixel to
    screen-filling (saturation, 0.99 clamp), every colour mode, random background and scale modifier."""
    rng = np.random.default_rng(20261017)
    colors = ["sh0", "sh1", "sh2", "sh3", "sh1m16", "precomp"]
    for i in range(28):
        P = int(rng.integers(1, 4000))
        W, H = (int(rng.integers(1, 12)), int(rng.integers(1, 12))) if i % 4 == 0 else (int(rng.integers(9, 150)), int(rng.integers(5, 110)))
        kind = "band" if i % 5 == 4 else "object"
        color = colors[i % len(colors)]
        mu = float(rng.uniform(-4.2, -1.2))
        bg = torch.tensor(rng.uniform(0, 1, 3), dtype=torch.float32, device=DEV)
        mod = float(rng.uniform(0.5, 2.0))
        scene = synthetic.make_scene(P, kind, color, mu, seed=1000 + i).to(DEV)
        cam = (synthetic.orbit_camera(W, H, float(rng.uniform(0, 6.28))) if kind == "object"
               else synthetic.yaw_camera(W, H, float(rng.uniform(0, 6.28)))).to(DEV)
        tag = (i, P, W, H, kind, color, round(mu, 2), round(mod, 2))
        try:
            _assert_stage_parity(pl.stages_vs_record(ref, scene, cam, bg, scale_modifier=mod))
            Wc, Wd = (t.to(DEV) for t in synthetic.loss_weights(W, H, seed=i))
            _assert_grad_parity(pl.autograd_vs_record(ref, scene, cam, bg, Wc, Wd, scale_modifier=mod))
        except AssertionError as e:
            raise AssertionError(f"fuzz case {tag}: {e}") from e


@pytest.mark.parametrize("case", [("precomp", 4000, 320, 200, -2.2, 1.7, "object"), ("sh1", 2500, 256, 256, -1.8, 1.3, "band")],
                         ids=["precomp_320x200", "sh1_256x256"])
def test_gradients_of_screen_filling_gaussians_against_double_precision_sums(case, ref):
    """Where this library and the reference disagree most on a gradient (1e-4 relative L2 and slightly above in a long
    fuzz run, tools/fuzz_vs_reference.py) is a scene of screen-filling Gaussians: the reference adds up to W*H float
    terms per Gaussian into ONE float with atomicAdd (backward.cu:556-575), this library sums 64-pixel blocks first.
    The CPU oracle with its per-Gaussian sums accumulated in double (same fp32 terms, rounded once) is the referee:
    every gradient of this library must be within 1e-5 of it.  Radii, images and gradients are also compared with
    the scene's stored record, as in test_autograd_vs_reference_cuda."""
    from oracle import oracle

    color, P, W, H, mu, mod, kind = case
    scene_c = synthetic.make_scene(P, kind, color, mu, seed=17)
    cam_c = synthetic.orbit_camera(W, H, 0.8) if kind == "object" else synthetic.yaw_camera(W, H, 0.8)
    bg_c = torch.tensor([0.3, 0.5, 0.2])
    Wc, Wd = synthetic.loss_weights(W, H, seed=3)
    o = oracle.run_scene(scene_c, cam_c, bg_c, scale_modifier=mod)
    truth = o["oracle"].backward(Wc.numpy(), f64_sums=True)
    scene, cam, bg = scene_c.to(DEV), cam_c.to(DEV), bg_c.to(DEV)
    zero = torch.zeros_like(Wd).to(DEV)
    a = pl.run_autograd(pl.ours(), scene, cam, bg, Wc.to(DEV), zero, mod)
    assert int((a["radii"] > 0).sum()) > P // 4
    _assert_grad_parity(pl.autograd_vs_record(ref, scene, cam, bg, Wc.to(DEV), zero, mod))
    names = {"means3D": "dL_dmeans3D", "opacities": "dL_dopacity", "scales": "dL_dscales", "rotations": "dL_drotations",
             "shs": "dL_dsh", "colors_precomp": "dL_dcolors", "means2D": "dL_dmeans2D"}
    for k, g in a["grads"].items():
        if g is None:
            continue
        t = torch.from_numpy(truth[names[k]]).to(DEV).reshape(g.shape)
        assert pl.rel_l2(g, t) <= 1e-5, (k, pl.rel_l2(g, t))


def _fwd_ex(_C, scene, cam, bg, mode, mod=1.0, R_cap=0, R1_cap=0, depth_bits=0, report=None):
    return _C.rasterize_gaussians_ex(*pl.forward_args(scene, cam, bg, scale_modifier=mod), mode, R_cap, R1_cap, depth_bits, report)


def _same_forward(_C, a, b, P, W, H):
    from bloomscene_b200.debug import state_views

    Ra, Rb = a[0], b[0]
    assert torch.equal(a[1], b[1]) and torch.equal(a[2], b[2]) and torch.equal(a[3], b[3])
    R = max(Ra, Rb)
    sa, sb = state_views(_C, a[4], a[5], a[6], P, R, W, H), state_views(_C, b[4], b[5], b[6], P, R, W, H)
    for k in ("point_list", "ranges", "n_contrib", "final_T", "depth_key", "rect"):
        assert torch.equal(sa[k], sb[k]), k


def test_forward_modes_are_bit_identical_and_an_overflow_reruns():
    """brs_fwd_options: EXACT (host waits for the counts after preprocess), AUTO (capacities from the high-water
    marks, host waits only after everything is enqueued) and DEFERRED (no host wait) must give identical bits;
    a forward whose capacities were too small must be detected and re-run with the exact sizes."""
    _C = pl.ours()._C
    scene = synthetic.make_scene(20_000, "object", "sh1", -4.2, seed=3).to(DEV)
    cam = synthetic.orbit_camera(272, 208, 0.7).to(DEV)
    bg = torch.tensor([0.1, 0.2, 0.3], device=DEV)
    P, W, H = scene.P, 272, 208
    _C.reset_marks()
    _C.forward_stats(True)
    exact = _fwd_ex(_C, scene, cam, bg, _C.FWD_EXACT)
    first = _fwd_ex(_C, scene, cam, bg, _C.FWD_AUTO)   # marks exist already (EXACT raised them): optimistic
    second = _fwd_ex(_C, scene, cam, bg, _C.FWD_AUTO)
    st = _C.forward_stats(False)
    assert st["exact"] == 1 and st["optimistic"] == 2 and st["overflow_reruns"] == 0, st
    assert exact[0] == first[0] == second[0] > 1000
    _same_forward(_C, exact, first, P, W, H)
    _same_forward(_C, exact, second, P, W, H)
    # same shape, 3x larger Gaussians: ~9x the instances -> the marks' capacity overflows -> re-run
    big_auto = _fwd_ex(_C, scene, cam, bg, _C.FWD_AUTO, mod=3.0)
    st = _C.forward_stats(False)
    assert st["overflow_reruns"] == 1, st
    big_exact = _fwd_ex(_C, scene, cam, bg, _C.FWD_EXACT, mod=3.0)
    assert big_auto[0] == big_exact[0] > 3 * exact[0]
    _same_forward(_C, big_exact, big_auto, P, W, H)
    # the marks were raised: the next optimistic forward fits
    again = _fwd_ex(_C, scene, cam, bg, _C.FWD_AUTO, mod=3.0)
    assert _C.forward_stats(False)["overflow_reruns"] == 1
    _same_forward(_C, big_exact, again, P, W, H)
    # a view with a much wider depth range than the marks have seen (more key bits): re-run as well
    far = synthetic.Scene(scene.means3D.clone(), scene.scales, scene.rotations, scene.opacities, scene.shs, None, scene.sh_degree)
    far.means3D[::7, 2] += 400.0
    far_auto = _fwd_ex(_C, far, cam, bg, _C.FWD_AUTO)
    far_exact = _fwd_ex(_C, far, cam, bg, _C.FWD_EXACT)
    _same_forward(_C, far_exact, far_auto, P, W, H)

    # the visible count is a capacity too (it sizes the depth sort's later passes): marks from a view that sees few
    # Gaussians, then a view that sees many more with FEWER instances each -> only the V capacity overflows -> re-run
    _C.reset_marks()
    away = synthetic.Scene(scene.means3D.clone(), scene.scales, scene.rotations, scene.opacities, scene.shs, None, scene.sh_degree)
    away.means3D[: P - 300, 2] -= 50.0     # all but 300 Gaussians behind the camera
    few = _fwd_ex(_C, away, cam, bg, _C.FWD_EXACT, mod=6.0)
    assert 0 < int((few[3] > 0).sum()) <= 300
    before = _C.forward_stats(False)["overflow_reruns"]
    many_auto = _fwd_ex(_C, scene, cam, bg, _C.FWD_AUTO, mod=0.05)
    assert _C.forward_stats(False)["overflow_reruns"] == before + 1
    many_exact = _fwd_ex(_C, scene, cam, bg, _C.FWD_EXACT, mod=0.05)
    assert int((many_exact[3] > 0).sum()) > 5000
    _same_forward(_C, many_exact, many_auto, P, W, H)
    rep = torch.zeros(8, dtype=torch.int32).pin_memory()
    _C.reset_marks()
    _fwd_ex(_C, away, cam, bg, _C.FWD_EXACT, mod=6.0)
    _fwd_ex(_C, scene, cam, bg, _C.FWD_DEFERRED, mod=0.05, R_cap=1 << 22, R1_cap=1 << 22, report=rep)
    torch.cuda.synchronize()
    assert int(rep[5]) & 8, rep        # bit 3 of the overflow word: V > V_cap
    _C.reset_marks()
    _fwd_ex(_C, scene, cam, bg, _C.FWD_EXACT)

    # DEFERRED: no host wait; counts arrive in the pinned report
    report = torch.zeros(8, dtype=torch.int32).pin_memory()
    dfr = _fwd_ex(_C, scene, cam, bg, _C.FWD_DEFERRED, report=report)
    torch.cuda.synchronize()
    assert dfr[0] == -1 and int(report[0]) == exact[0] and int(report[5]) == 0 and int(report[4]) == int((exact[3] > 0).sum())
    _same_forward(_C, exact, (exact[0],) + tuple(dfr[1:]), P, W, H)
    # backward of a deferred state (num_rendered = -1) equals the backward of the exact one
    Wc, _ = (t.to(DEV) for t in synthetic.loss_weights(W, H))
    e = torch.Tensor([])

    def bwd(fw):
        return _C.rasterize_gaussians_backward(bg, scene.means3D, fw[3], e, scene.scales, scene.rotations, 1.0, e,
                                               cam.viewmatrix, cam.projmatrix, cam.tanfovx, cam.tanfovy, Wc, e, scene.shs,
                                               scene.sh_degree, cam.campos, fw[4], fw[0], fw[5], fw[6], False)

    for ga, gb in zip(bwd(exact), bwd(dfr)):
        assert pl.rel_l2(ga, gb) <= 1e-5
    # DEFERRED with capacities that are far too small: flagged, memory-safe, nothing hangs
    tiny = _fwd_ex(_C, scene, cam, bg, _C.FWD_DEFERRED, R_cap=64, R1_cap=32, depth_bits=8, report=report)
    torch.cuda.synchronize()
    assert int(report[5]) & 3 == 3 and int(report[0]) == exact[0]
    assert torch.isfinite(tiny[1]).all()
    _C.reset_marks()


def test_render_views_deferred_batch_recovers_from_overflow_and_replays_in_a_cuda_graph():
    """render_views issues DEFERRED forwards (one host wait per batch).  (1) With stale high-water marks most
    views overflow their capacities and must be re-rendered exactly; (2) a DEFERRED forward + backward is free of
    host synchronisation, so it can be captured in a CUDA graph and replayed with new camera contents."""
    api = pl.ours()
    _C = api._C
    scene = synthetic.make_scene(30_000, "band", "precomp", -4.4, seed=5).to(DEV)
    W, H = 256, 160
    cams = [synthetic.yaw_camera(W, H, 0.9 * k).to(DEV) for k in range(7)]
    bg = torch.tensor([0.05, 0.1, 0.2], device=DEV)
    mk = lambda mod: [synthetic.raster_settings(c, 0, bg, api.GaussianRasterizationSettings, scale_modifier=mod) for c in cams]
    kw = dict(colors_precomp=scene.colors_precomp, scales=scene.scales, rotations=scene.rotations, keep_radii=True)

    def singles(settings):
        outs = []
        with torch.no_grad():
            for rs in settings:
                outs.append(api.GaussianRasterizer(rs)(scene.means3D, torch.zeros_like(scene.means3D), scene.opacities,
                                                       colors_precomp=scene.colors_precomp, scales=scene.scales,
                                                       rotations=scene.rotations))
        return outs

    _C.reset_marks()
    small = api.render_views(mk(0.5), scene.means3D, scene.opacities, streams=3, **kw)  # seeds small marks
    _C.forward_stats(True)
    # ~36x the instances: overflows (one host thread, so that this thread's counters see every forward)
    big = api.render_views(mk(3.0), scene.means3D, scene.opacities, streams=3, host_threads=False, **kw)
    st = _C.forward_stats(False)
    assert st["deferred"] == len(cams) and st["exact"] >= 1, st
    for settings, got in ((mk(0.5), small), (mk(3.0), big)):
        for k, (c, r, d) in enumerate(singles(settings)):
            assert torch.equal(c, got[0][k]) and torch.equal(d, got[1][k]) and torch.equal(r, got[2][k]), k

    # CUDA graph: capture one deferred forward + backward on static buffers, replay it for another camera
    Wc, _ = (t.to(DEV) for t in synthetic.loss_weights(W, H))
    e = torch.Tensor([])
    view, proj, campos = (cams[0].viewmatrix.clone(), cams[0].projmatrix.clone(), cams[0].campos.clone())
    report = torch.zeros(8, dtype=torch.int32).pin_memory()
    ref_report = torch.zeros(8, dtype=torch.int32).pin_memory()
    cam0 = cams[0]

    def fwd_bwd(rep):
        fw = _C.rasterize_gaussians_ex(bg, scene.means3D, scene.colors_precomp, scene.opacities, scene.scales, scene.rotations,
                                       1.0, e, view, proj, cam0.tanfovx, cam0.tanfovy, H, W, e, 0, campos, False, False,
                                       _C.FWD_DEFERRED, 0, 0, 0, rep)
        g = _C.rasterize_gaussians_backward(bg, scene.means3D, fw[3], scene.colors_precomp, scene.scales, scene.rotations, 1.0,
                                            e, view, proj, cam0.tanfovx, cam0.tanfovy, Wc, e, e, 0, campos, fw[4], fw[0], fw[5],
                                            fw[6], False)
        return fw[1], fw[2], g[3], g[6]  # colour, depth, dL_dmeans3D, dL_dscales

    api.render_views(mk(1.0), scene.means3D, scene.opacities, streams=1, **kw)  # marks for scale modifier 1
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        fwd_bwd(report)  # warm-up outside the capture
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        static_out = fwd_bwd(report)
    for k in (3, 5):
        view.copy_(cams[k].viewmatrix)
        proj.copy_(cams[k].projmatrix)
        campos.copy_(cams[k].campos)
        graph.replay()
        torch.cuda.synchronize()
        assert int(report[5]) == 0
        got = [t.clone() for t in static_out]
        want = fwd_bwd(ref_report)
        torch.cuda.synchronize()
        assert int(report[0]) == int(ref_report[0]) > 0
        assert torch.equal(got[0], want[0]) and torch.equal(got[1], want[1])
        assert pl.rel_l2(got[2], want[2]) <= 1e-5 and pl.rel_l2(got[3], want[3]) <= 1e-5
    _C.reset_marks()


def test_graphed_step_matches_the_plain_step_and_survives_an_overflow():
    """GraphedStep (SURVEY.md 8f N1): per-view forward + loss + backward replayed from CUDA graphs must give the
    plain step's gradients; when the captured capacities become too small the step is repeated un-graphed."""
    from bloomscene_b200.multiview import GraphedStep, view_sharded_step
    from workload.params import GaussianParams

    api = pl.ours()
    _C = api._C
    _C.reset_marks()
    scene = synthetic.make_scene(8000, "object", "sh3", -3.8, seed=17).to(DEV)
    W, H = 208, 144
    cams = [synthetic.orbit_camera(W, H, 0.7 * k).to(DEV) for k in range(7)]
    Wc, Wd = [t.to(DEV) for t in synthetic.loss_weights(W, H)]
    targets = torch.rand(len(cams), 3, H, W, device=DEV)
    bg = torch.tensor([0.2, 0.1, 0.4], device=DEV)
    loss3 = lambda c, d, t: ((c - t) ** 2 * Wc).sum() + (d * Wd).sum()
    got, want = GaussianParams(scene), GaussianParams(scene)
    step = GraphedStep(got, cams, bg, api.GaussianRasterizer, loss3, streams=3, targets=targets)
    step()  # plain + capture
    for _ in range(2):
        res = step()
    assert step.replays == 2 * len(cams) and step.fallbacks == 0
    ref = view_sharded_step(want, cams, bg, api.GaussianRasterizer, lambda c, d, vi: loss3(c, d, targets[vi]), streams=1)
    assert float(res["loss"]) == pytest.approx(float(ref["loss"]), rel=1e-6)
    for name in got.names:
        assert float(want.tensors[name].grad.abs().max()) > 0, name
        assert pl.rel_l2(got.tensors[name].grad, want.tensors[name].grad) <= pl.GRAD_TOL, name
    # the Gaussians grow 3x: the captured capacities overflow -> the step is repeated un-graphed and re-captured
    with torch.no_grad():
        got.tensors["scales"].mul_(3.0)
        want.tensors["scales"].mul_(3.0)
    res = step()
    assert step.fallbacks == 1
    ref = view_sharded_step(want, cams, bg, api.GaussianRasterizer, lambda c, d, vi: loss3(c, d, targets[vi]), streams=1)
    for name in got.names:
        assert pl.rel_l2(got.tensors[name].grad, want.tensors[name].grad) <= pl.GRAD_TOL, name
    res = step()  # graphs again, with the larger capacities
    assert step.fallbacks == 1
    for name in got.names:
        assert pl.rel_l2(got.tensors[name].grad, want.tensors[name].grad) <= pl.GRAD_TOL, name
    _C.reset_marks()
