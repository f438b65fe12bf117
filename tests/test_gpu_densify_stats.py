"""GPU: densification statistics computed by the backward kernel (brs_densify_stats) against the reference's torch
statement (scene/gaussian_model.py:756-759) applied to the same call's means2D.grad and radii:

    update_filter = radii > 0
    grad_norm = torch.norm(viewspace_point_tensor.grad[update_filter, :2], dim=-1, keepdim=True)
    accum[combined_mask] += grad_norm;  denom[combined_mask] += 1
"""
import ctypes as C

import pytest
import torch

import parity_lib as pl
from test_gpu_c_abi import ALLOC, Arena, FwdState, Gaussians, Grads, View, _lib, _ptr
from workload import synthetic

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


class Stats(C.Structure):  # brs_densify_stats
    _fields_ = [("grad_norm", C.c_void_p), ("count", C.c_void_p), ("index", C.c_void_p), ("rows", C.c_int)]


def _reference(radii, m2grad, index=None, rows=None):
    """Per-slot (grad-norm sum, count) of one view from radii and means2D.grad, with the reference's torch ops."""
    P = radii.shape[0]
    vis = radii > 0
    norm = torch.zeros(P, device=radii.device)
    norm[vis] = torch.norm(m2grad[vis, :2], dim=-1)
    if index is None:
        return norm, vis.float()
    ok = vis & (index >= 0) & (index < rows)
    n = torch.zeros(rows, device=radii.device).index_add_(0, index[ok], norm[ok])
    c = torch.zeros(rows, device=radii.device).index_add_(0, index[ok], torch.ones_like(norm[ok]))
    return n, c


def _close(got, want, rtol):
    got, want = got.reshape(-1), want.reshape(-1)
    bad = (got - want).abs() > rtol * want.abs()
    assert not bad.any(), (int(bad.sum()), got[bad][:5], want[bad][:5])


def _scene_view(color, P=20000, W=256, H=192, seed=3):
    scene = synthetic.make_scene(P, "object", color, -3.6, seed=seed).to(DEV)
    cam = synthetic.orbit_camera(W, H, 0.4).to(DEV)
    Wc, Wd = [t.to(DEV) for t in synthetic.loss_weights(W, H)]
    return scene, cam, Wc, Wd


def _run(api, scene, cam, Wc, Wd, mode, stats=None):
    leaf = lambda t: None if t is None else t.detach().clone().requires_grad_(True)
    means3D, opac, scales, rots, shs, cols = map(leaf, (scene.means3D, scene.opacities, scene.scales, scene.rotations,
                                                       scene.shs, scene.colors_precomp))
    means2D = torch.zeros_like(means3D, requires_grad=True)
    kw = {} if stats is None else {"densify_stats": stats}
    inputs = {"means3D": means3D, "opacities": opac, "scales": scales, "rotations": rots, "shs": shs, "colors_precomp": cols}
    sinks = None
    if mode == "depth_gradient":
        kw["depth_gradient"] = True
    elif mode == "grad_sink":
        sinks = {n: torch.zeros_like(t) for n, t in inputs.items() if t is not None}
        kw["grad_sink"] = sinks
    settings = synthetic.raster_settings(cam, scene.sh_degree, torch.tensor([0.1, 0.2, 0.3], device=DEV),
                                         api.GaussianRasterizationSettings)
    color, radii, depth = api.GaussianRasterizer(settings, **kw)(means3D=means3D, means2D=means2D, opacities=opac, shs=shs,
                                                                colors_precomp=cols, scales=scales, rotations=rots)
    ((color * Wc).sum() + (depth * Wd).sum()).backward()
    torch.cuda.synchronize()
    grads = {n: (sinks[n] if sinks is not None else t.grad) for n, t in inputs.items() if t is not None}
    grads["means2D"] = means2D.grad
    return radii, means2D.grad, grads


@pytest.mark.parametrize("mode", ["plain", "depth_gradient", "grad_sink"])
@pytest.mark.parametrize("color", ["sh3", "precomp"])
def test_single_view_stats_match_the_torch_statement(color, mode):
    api = pl.ours()
    assert api.GaussianRasterizer.supports_densify_stats
    scene, cam, Wc, Wd = _scene_view(color)
    P = scene.P
    stats = {"grad_norm": torch.zeros(P, 1, device=DEV), "count": torch.zeros(P, 1, device=DEV)}  # [rows, 1] accumulators
    radii, m2, grads = _run(api, scene, cam, Wc, Wd, mode, stats)
    want_n, want_c = _reference(radii, m2)
    assert int(want_c.sum()) > 1000 and float(want_n.sum()) > 0
    assert torch.equal(stats["count"].reshape(-1), want_c)
    _close(stats["grad_norm"], want_n, 1e-6)
    if mode == "plain":
        # the statistics change no gradient (two runs differ only by the blend backward's float-atomic order)
        radii0, _, grads0 = _run(api, scene, cam, Wc, Wd, mode)
        assert torch.equal(radii0, radii)
        for n, g in grads0.items():
            assert pl.rel_l2(grads[n], g) <= pl.GRAD_TOL, n


def test_scaffold_slot_map_through_the_fused_epilogue():
    """Anchors -> fused.neural_gaussians -> rasterizer, statistics into per-(anchor, offset) accumulators of ALL
    anchors (rows > P), with Scaffold-GS's training_statis combined_mask written out as the reference."""
    from bloomscene_b200.fused import neural_gaussians
    from test_gpu_fused import _neural_inputs

    api = pl.ours()
    N_all, K = 5000, 10
    g = torch.Generator().manual_seed(11)
    anchor_visible_mask = (torch.rand(N_all, generator=g) < 0.6).to(DEV)
    anchor_idx = torch.nonzero(anchor_visible_mask).squeeze(1)
    N = int(anchor_idx.numel())
    anchor, gs, off, nop, col, sr = _neural_inputs(N, K, seed=5)
    xyz, color, opacity, scaling, rot, mask = neural_gaussians(anchor * 0.5, gs * 0.02, off * 0.5,
                                                               torch.sigmoid(nop) * (nop > 0), col, sr)
    j = torch.nonzero(mask).squeeze(1)
    slot = anchor_idx[j // K] * K + j % K
    P = xyz.shape[0]
    offset_gradient_accum = torch.full((N_all * K, 1), 0.25, device=DEV)  # running accumulators: added to, not overwritten
    offset_denom = torch.full((N_all * K, 1), 2.0, device=DEV)
    want_accum, want_denom = offset_gradient_accum.clone(), offset_denom.clone()
    cam = synthetic.orbit_camera(128, 96, 0.3).to(DEV)
    st = synthetic.raster_settings(cam, 0, torch.zeros(3, device=DEV), api.GaussianRasterizationSettings)
    viewspace_point_tensor = torch.zeros_like(xyz, requires_grad=True)
    rast = api.GaussianRasterizer(st, densify_stats={"grad_norm": offset_gradient_accum, "count": offset_denom, "index": slot})
    img, radii, depth = rast(means3D=xyz, means2D=viewspace_point_tensor, opacities=opacity, colors_precomp=color,
                             scales=scaling, rotations=rot)
    (img * torch.rand_like(img)).sum().backward()
    torch.cuda.synchronize()
    assert N * K > P and int((radii > 0).sum()) > 100

    # Scaffold-GS training_statis, literally
    update_filter = radii > 0
    offset_selection_mask = mask
    anchor_visible_mask_k = anchor_visible_mask.unsqueeze(dim=1).repeat([1, K]).view(-1)
    combined_mask = torch.zeros_like(want_accum, dtype=torch.bool).squeeze(dim=1)
    combined_mask[anchor_visible_mask_k] = offset_selection_mask
    temp_mask = combined_mask.clone()
    combined_mask[temp_mask] = update_filter
    grad_norm = torch.norm(viewspace_point_tensor.grad[update_filter, :2], dim=-1, keepdim=True)
    want_accum[combined_mask] += grad_norm
    want_denom[combined_mask] += 1
    assert torch.equal(offset_denom, want_denom)
    _close(offset_gradient_accum, want_accum, 1e-6)


def test_slot_map_skips_out_of_range_slots_and_adds_duplicates():
    """rows < P, slots -1 and >= rows (skipped), several Gaussians sharing a slot (float reductions add them)."""
    api = pl.ours()
    scene, cam, Wc, Wd = _scene_view("sh1", P=12000)
    P, rows = scene.P, 3000
    g = torch.Generator().manual_seed(2)
    index = torch.randint(-3, rows + 3, (P,), generator=g).to(DEV)
    index[:50] = -1
    index[50:100] = rows
    stats = {"grad_norm": torch.zeros(rows, device=DEV), "count": torch.zeros(rows, device=DEV), "index": index}
    radii, m2, _ = _run(api, scene, cam, Wc, Wd, "plain", stats)
    want_n, want_c = _reference(radii, m2, index, rows)
    assert int(want_c.max()) >= 2 and int(((radii > 0) & ((index < 0) | (index >= rows))).sum()) > 0
    assert torch.equal(stats["count"], want_c)
    _close(stats["grad_norm"], want_n, 1e-5)
    with pytest.raises(Exception, match="one entry per Gaussian"):
        _run(api, scene, cam, Wc, Wd, "plain", dict(stats, index=index[:-1]))
    with pytest.raises(Exception, match="at least P rows"):
        _run(api, scene, cam, Wc, Wd, "plain", {"grad_norm": stats["grad_norm"], "count": stats["count"]})


def _step_scene():
    scene = synthetic.make_scene(8000, "object", "sh3", -3.8, seed=17).to(DEV)
    W, H = 208, 144
    cams = [synthetic.orbit_camera(W, H, 0.7 * k).to(DEV) for k in range(7)]
    Wc, Wd = [t.to(DEV) for t in synthetic.loss_weights(W, H)]
    return scene, cams, Wc, Wd


def test_view_sharded_step_on_four_streams_matches_per_view_reference():
    from bloomscene_b200.multiview import view_sharded_step
    from workload.params import GaussianParams

    api = pl.ours()
    scene, cams, Wc, Wd = _step_scene()
    bg = torch.tensor([0.2, 0.1, 0.4], device=DEV)
    loss = lambda c, d, vi: (c * Wc).sum() * (1.0 + 0.1 * vi) + (d * Wd).sum()
    plain = GaussianParams(scene)
    ref = view_sharded_step(plain, cams, bg, api.GaussianRasterizer, loss, streams=4)
    params = GaussianParams(scene, densify_stats=True)
    res = view_sharded_step(params, cams, bg, api.GaussianRasterizer, loss, streams=4, keep_means2D_grad=True)
    torch.cuda.synchronize()
    want_n = torch.zeros(params.P, device=DEV)
    want_c = torch.zeros(params.P, device=DEV)
    m2 = dict(res["means2D_grad"])
    for vi, radii in res["radii"]:
        n, c = _reference(radii, m2[vi])
        want_n += n
        want_c += c
    assert len(res["radii"]) == len(cams) >= 6 and int(want_c.max()) >= 2
    assert torch.equal(res["densify"]["count"], want_c)
    _close(res["densify"]["grad_norm"], want_n, 1e-5)
    assert float(res["loss"]) == pytest.approx(float(ref["loss"]), rel=1e-6)
    for name in plain.names:
        assert pl.rel_l2(params.tensors[name].grad, plain.tensors[name].grad) <= pl.GRAD_TOL, name


def test_graphed_step_stats_match_the_plain_step_through_an_overflow():
    from bloomscene_b200.multiview import GraphedStep, view_sharded_step
    from workload.params import GaussianParams

    api = pl.ours()
    _C = api._C
    _C.reset_marks()
    scene, cams, Wc, Wd = _step_scene()
    targets = torch.rand(len(cams), 3, cams[0].image_height, cams[0].image_width, device=DEV)
    bg = torch.tensor([0.2, 0.1, 0.4], device=DEV)
    loss3 = lambda c, d, t: ((c - t) ** 2 * Wc).sum() + (d * Wd).sum()
    got, want = GaussianParams(scene, densify_stats=True), GaussianParams(scene, densify_stats=True)
    step = GraphedStep(got, cams, bg, api.GaussianRasterizer, loss3, streams=3, targets=targets)

    def check(res):
        ref = view_sharded_step(want, cams, bg, api.GaussianRasterizer, lambda c, d, vi: loss3(c, d, targets[vi]), streams=1)
        torch.cuda.synchronize()
        assert torch.equal(res["densify"]["count"], ref["densify"]["count"])
        assert int(ref["densify"]["count"].max()) >= 2
        _close(res["densify"]["grad_norm"], ref["densify"]["grad_norm"], 1e-5)
        for name in got.names:
            assert pl.rel_l2(got.tensors[name].grad, want.tensors[name].grad) <= pl.GRAD_TOL, name

    check(step())  # plain + capture
    first = step()
    kept = {k: v.clone() for k, v in first["densify"].items()}
    second = step()  # per step: the same numbers again, not twice them
    assert step.replays == 2 * len(cams) and step.fallbacks == 0
    assert torch.equal(second["densify"]["count"], kept["count"])
    _close(second["densify"]["grad_norm"], kept["grad_norm"], 1e-5)
    check(second)
    with torch.no_grad():
        got.tensors["scales"].mul_(3.0)
        want.tensors["scales"].mul_(3.0)
    res = step()  # captured capacities overflow: repeated un-graphed
    assert step.fallbacks == 1
    check(res)
    res = step()  # graphs again
    assert step.fallbacks == 1
    check(res)
    _C.reset_marks()


def test_deferred_forward_and_backward_with_stats_in_a_cuda_graph():
    api = pl.ours()
    _C = api._C
    _C.reset_marks()
    scene = synthetic.make_scene(20000, "object", "precomp", -3.6, seed=9).to(DEV)
    W, H = 192, 128
    cams = [synthetic.orbit_camera(W, H, 0.5 * k).to(DEV) for k in range(6)]
    bg = torch.tensor([0.3, 0.2, 0.1], device=DEV)
    Wc = synthetic.loss_weights(W, H)[0].to(DEV)
    settings = [synthetic.raster_settings(c, 0, bg, api.GaussianRasterizationSettings) for c in cams]
    api.render_views(settings, scene.means3D, scene.opacities, colors_precomp=scene.colors_precomp, scales=scene.scales,
                     rotations=scene.rotations, streams=1)  # high-water marks of this shape
    e = torch.Tensor([])
    view, proj, campos = cams[0].viewmatrix.clone(), cams[0].projmatrix.clone(), cams[0].campos.clone()
    report = torch.zeros(8, dtype=torch.int32).pin_memory()
    gn = torch.zeros(scene.P, device=DEV)
    cnt = torch.zeros(scene.P, device=DEV)

    def fwd_bwd():
        fw = _C.rasterize_gaussians_ex(bg, scene.means3D, scene.colors_precomp, scene.opacities, scene.scales, scene.rotations,
                                       1.0, e, view, proj, cams[0].tanfovx, cams[0].tanfovy, H, W, e, 0, campos, False, False,
                                       _C.FWD_DEFERRED, 0, 0, 0, report)
        g = _C.rasterize_gaussians_backward(bg, scene.means3D, fw[3], scene.colors_precomp, scene.scales, scene.rotations, 1.0,
                                            e, view, proj, cams[0].tanfovx, cams[0].tanfovy, Wc, e, e, 0, campos, fw[4],
                                            fw[0], fw[5], fw[6], False, stats_grad_norm=gn, stats_count=cnt)
        return fw[3], g[0]  # radii, dL_dmeans2D

    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        fwd_bwd()  # warm-up outside the capture
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        static_radii, static_m2 = fwd_bwd()
    for k in (2, 5):
        view.copy_(cams[k].viewmatrix)
        proj.copy_(cams[k].projmatrix)
        campos.copy_(cams[k].campos)
        gn.zero_()
        cnt.zero_()
        graph.replay()
        torch.cuda.synchronize()
        assert int(report[5]) == 0 and int(report[0]) > 0
        want_n, want_c = _reference(static_radii, static_m2)
        assert int(want_c.sum()) > 1000
        assert torch.equal(cnt, want_c)
        _close(gn, want_n, 1e-6)
    _C.reset_marks()


def test_backward_ex_through_ctypes_only():
    lib = _lib()
    lib.brs_backward_ex.argtypes = [C.POINTER(View), C.POINTER(Gaussians), C.c_void_p, C.POINTER(FwdState), C.c_void_p,
                                    C.c_void_p, C.POINTER(Grads), C.c_void_p, ALLOC, C.c_void_p, C.c_void_p]
    W, H = 150, 94
    scene = synthetic.make_scene(5000, "object", "sh2", -3.4, seed=31).to(DEV)
    cam = synthetic.orbit_camera(W, H, 0.6).to(DEV)
    bg = torch.tensor([0.2, 0.4, 0.1], device=DEV)
    M, P = scene.shs.shape[1], scene.P
    view = View(W, H, cam.tanfovx, cam.tanfovy, 1.0, scene.sh_degree, M, 0, 0, _ptr(bg), _ptr(cam.viewmatrix),
                _ptr(cam.projmatrix), _ptr(cam.campos))
    g = Gaussians(P, _ptr(scene.means3D), _ptr(scene.opacities), _ptr(scene.shs), None, _ptr(scene.scales),
                  _ptr(scene.rotations), None)
    color_img, depth_img = torch.empty(3, H, W, device=DEV), torch.empty(1, H, W, device=DEV)
    radii = torch.empty(P, dtype=torch.int32, device=DEV)
    arena, state = Arena(), FwdState()
    stream = torch.cuda.current_stream().cuda_stream
    assert lib.brs_forward(C.byref(view), C.byref(g), color_img.data_ptr(), depth_img.data_ptr(), radii.data_ptr(), arena.fn,
                           None, C.byref(state), stream) == 0
    Wc = synthetic.loss_weights(W, H)[0].to(DEV).contiguous()
    shapes = {"dL_dmeans2D": (P, 3), "dL_dcolors": (P, 3), "dL_dopacity": (P, 1), "dL_dmeans3D": (P, 3), "dL_dcov3D": (P, 6),
              "dL_dsh": (P, M, 3), "dL_dscales": (P, 3), "dL_drotations": (P, 4)}

    def backward(stats):
        out = {k: torch.full(s, float("nan"), device=DEV) for k, s in shapes.items()}
        grads = Grads(*[out[k].data_ptr() for k in shapes], 0, 0, None)
        if stats is False:
            rc = lib.brs_backward(C.byref(view), C.byref(g), radii.data_ptr(), C.byref(state), Wc.data_ptr(), None,
                                  C.byref(grads), arena.fn, None, stream)
        else:
            rc = lib.brs_backward_ex(C.byref(view), C.byref(g), radii.data_ptr(), C.byref(state), Wc.data_ptr(), None,
                                     C.byref(grads), None if stats is None else C.addressof(stats), arena.fn, None, stream)
        assert rc == 0, lib.brs_error_string(rc)
        torch.cuda.synchronize()
        return out

    base = backward(False)
    for k, v in backward(None).items():
        assert pl.rel_l2(v, base[k]) <= pl.GRAD_TOL, k
    gn, cnt = torch.zeros(P, device=DEV), torch.zeros(P, device=DEV)
    stats = Stats(gn.data_ptr(), cnt.data_ptr(), None, P)
    out = backward(stats)
    for k, v in out.items():
        assert pl.rel_l2(v, base[k]) <= pl.GRAD_TOL, k
    want_n, want_c = _reference(radii, out["dL_dmeans2D"])
    assert int(want_c.sum()) > 500
    assert torch.equal(cnt, want_c)
    _close(gn, want_n, 1e-6)


def test_full_size_one_view_config_c():
    api = pl.ours()
    scene = synthetic.config_scene("C").to(DEV)
    cam = synthetic.config_cameras("C")[0].to(DEV)
    W, H = cam.image_width, cam.image_height
    Wc, Wd = [t.to(DEV) for t in synthetic.loss_weights(W, H)]
    stats = {"grad_norm": torch.zeros(scene.P, device=DEV), "count": torch.zeros(scene.P, device=DEV)}
    radii, m2, _ = _run(api, scene, cam, Wc, Wd, "plain", stats)
    want_n, want_c = _reference(radii, m2)
    assert scene.P == 1_000_000 and int(want_c.sum()) > 100_000
    assert torch.equal(stats["count"], want_c)
    _close(stats["grad_norm"], want_n, 1e-6)
