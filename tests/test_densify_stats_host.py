"""CPU: densification statistics (brs_densify_stats) on the host side — the view-sharded step's stat slots over
gloo with the oracle-backed stand-in, the GaussianParams layout, C-ABI argument validation, and the stand-in's
refusal."""
import ctypes as C
import os
import socket

import pytest
import torch
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
N_VIEWS = 4
P = 300
W, H = 40, 24


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _setup(densify_stats):
    from workload import synthetic
    from workload.params import GaussianParams
    from bloomscene_b200.rasterizer import bind
    from oracle_backend import OracleBackend

    torch.set_num_threads(1)
    api = bind(OracleBackend(threads=1))
    scene = synthetic.make_scene(P, "object", "sh1", -2.8, seed=5)
    cams = [synthetic.orbit_camera(W, H, 2 * 3.14159265 * k / N_VIEWS) for k in range(N_VIEWS)]
    Wc, Wd = synthetic.loss_weights(W, H, seed=2)
    loss_fn = lambda color, depth, vi: (color * Wc).sum() * (1.0 + 0.1 * vi) + (depth * Wd).sum()
    return api, GaussianParams(scene, densify_stats=densify_stats), cams, loss_fn


def _worker(rank, world, port, out_dir):
    import sys

    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    sys.path.insert(0, ROOT)
    import torch.distributed as dist

    from bloomscene_b200.multiview import view_sharded_step

    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    api, params, cams, loss_fn = _setup(True)
    res = view_sharded_step(params, cams, torch.zeros(3), api.GaussianRasterizer, loss_fn, rank=rank, world=world)
    torch.save({"bucket": params.grad_bucket.clone(), "loss": res["loss"],
                "densify": {k: v.clone() for k, v in res["densify"].items()}},
               os.path.join(out_dir, f"rank{rank}.pt"))
    dist.barrier()
    dist.destroy_process_group()


def _reference_stats(api, params, cams, loss_fn):
    """The reference's torch statement (scene/gaussian_model.py:756-759), one view at a time."""
    from workload import synthetic
    from bloomscene_b200.rasterizer import GaussianRasterizationSettings

    acc = torch.zeros(params.P, 1)
    denom = torch.zeros(params.P, 1)
    for vi, cam in enumerate(cams):
        rast = api.GaussianRasterizer(synthetic.raster_settings(cam, params.sh_degree, torch.zeros(3),
                                                                GaussianRasterizationSettings))
        viewspace_point_tensor = torch.zeros(params.P, 3, requires_grad=True)
        t = {n: v.detach() for n, v in params.tensors.items()}
        color, radii, depth = rast(means3D=t["means3D"], means2D=viewspace_point_tensor, opacities=t["opacities"],
                                   shs=t["shs"], scales=t["scales"], rotations=t["rotations"])
        loss_fn(color, depth, vi).backward()
        update_filter = radii > 0
        acc[update_filter] += torch.norm(viewspace_point_tensor.grad[update_filter, :2], dim=-1, keepdim=True)
        denom[update_filter] += 1
    return acc[:, 0], denom[:, 0]


def test_stats_ride_in_the_all_reduce_and_leave_gradients_unchanged(tmp_path):
    from bloomscene_b200.multiview import view_sharded_step

    api, plain, cams, loss_fn = _setup(False)
    ref = view_sharded_step(plain, cams, torch.zeros(3), api.GaussianRasterizer, loss_fn)
    assert ref["densify"] is None
    _, params, _, _ = _setup(True)
    single = view_sharded_step(params, cams, torch.zeros(3), api.GaussianRasterizer, loss_fn)
    # the statistics change neither the gradients nor the loss
    assert torch.equal(params.grad_bucket, plain.grad_bucket) and torch.equal(single["loss"], ref["loss"])
    want_norm, want_count = _reference_stats(api, params, cams, loss_fn)
    assert torch.equal(single["densify"]["count"], want_count) and want_count.max() >= 2
    assert torch.allclose(single["densify"]["grad_norm"], want_norm, rtol=1e-6, atol=0)
    assert float(want_norm.sum()) > 0
    # per step: a second step gives the same numbers, not twice them
    again = view_sharded_step(params, cams, torch.zeros(3), api.GaussianRasterizer, loss_fn)
    assert torch.equal(again["densify"]["count"], want_count)

    port = _free_port()
    mp.spawn(_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    r0 = torch.load(tmp_path / "rank0.pt")
    r1 = torch.load(tmp_path / "rank1.pt")
    for k in ("grad_norm", "count"):
        assert torch.equal(r0["densify"][k], r1["densify"][k]), k
    assert torch.equal(r0["densify"]["count"], want_count)
    assert torch.allclose(r0["densify"]["grad_norm"], single["densify"]["grad_norm"], rtol=1e-6, atol=0)
    rel = (r0["bucket"].double() - plain.grad_bucket.double()).norm() / plain.grad_bucket.double().norm()
    assert rel <= 1e-5


def test_params_layout_is_unchanged_by_default():
    from workload import synthetic
    from workload.params import GaussianParams

    scene = synthetic.make_scene(50, "object", "sh1", -2.8, seed=1)
    G = sum(t.numel() for t in scene.tensors().values())
    p = GaussianParams(scene)
    assert p.densify is None
    assert p.grad_bucket.numel() == G and p.reduce_buffer().numel() == G + 2
    assert p.loss_slot.data_ptr() == p.reduce_buffer().data_ptr() + 4 * G
    assert p.flag_slot.data_ptr() == p.reduce_buffer().data_ptr() + 4 * (G + 1)
    q = GaussianParams(scene, densify_stats=True)
    assert q.grad_bucket.numel() == G and q.reduce_buffer().numel() == G + 2 * 50 + 2
    base = q.reduce_buffer().data_ptr()
    assert q.densify["grad_norm"].data_ptr() == base + 4 * G and q.densify["grad_norm"].numel() == 50
    assert q.densify["count"].data_ptr() == base + 4 * (G + 50) and q.densify["count"].numel() == 50
    assert q.loss_slot.data_ptr() == base + 4 * (G + 100) and q.flag_slot.data_ptr() == base + 4 * (G + 101)
    q.reduce_buffer().fill_(3.0)
    q.zero_grad()
    assert not q.reduce_buffer().any()


class _View(C.Structure):
    _fields_ = [("image_width", C.c_int), ("image_height", C.c_int), ("tanfovx", C.c_float), ("tanfovy", C.c_float),
                ("scale_modifier", C.c_float), ("sh_degree", C.c_int), ("sh_coeffs", C.c_int), ("prefiltered", C.c_int),
                ("debug", C.c_int), ("bg", C.c_void_p), ("viewmatrix", C.c_void_p), ("projmatrix", C.c_void_p),
                ("campos", C.c_void_p)]


class _Gaussians(C.Structure):
    _fields_ = [("P", C.c_int)] + [(n, C.c_void_p) for n in ("means3D", "opacities", "shs", "colors_precomp", "scales",
                                                             "rotations", "cov3D_precomp")]


class _State(C.Structure):
    _fields_ = [("geom", C.c_void_p), ("geom_bytes", C.c_size_t), ("binning", C.c_void_p), ("binning_bytes", C.c_size_t),
                ("image", C.c_void_p), ("image_bytes", C.c_size_t), ("num_rendered", C.c_int)]


class _Grads(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("dL_dmeans2D", "dL_dcolors", "dL_dopacity", "dL_dmeans3D", "dL_dcov3D", "dL_dsh",
                                          "dL_dscales", "dL_drotations")] + \
               [("accumulate", C.c_int), ("depth_gradient", C.c_int), ("out_depth", C.c_void_p)]


class _Stats(C.Structure):
    _fields_ = [("grad_norm", C.c_void_p), ("count", C.c_void_p), ("index", C.c_void_p), ("rows", C.c_int)]


def test_backward_ex_rejects_bad_statistics_without_touching_the_gpu():
    """Every bad brs_densify_stats is refused before any CUDA call (the pointers are fake).  A good one passes
    validation and reaches the allocator, which returns NULL here: BRS_ERR_ALLOC, still before any CUDA call."""
    lib = C.CDLL(os.path.join(ROOT, "bloomscene_b200", "libbloomrast.so"))
    ALLOC = C.CFUNCTYPE(C.c_void_p, C.c_void_p, C.c_int, C.c_size_t)
    alloc = ALLOC(lambda ctx, which, n: None)
    fake = 0x1000
    n = 100
    view = _View(64, 48, 0.5, 0.5, 1.0, 0, 0, 0, 0, fake, fake, fake, fake)
    g = _Gaussians(n, fake, fake, None, fake, fake, fake, None)
    state = _State(fake, 1 << 40, fake, 1 << 40, fake, 1 << 40, 10)
    grads = _Grads(*([fake] * 8), 0, 0, None)

    def call(stats):
        return lib.brs_backward_ex(C.byref(view), C.byref(g), C.c_void_p(fake), C.byref(state), C.c_void_p(fake), None,
                                   C.byref(grads), None if stats is None else C.byref(stats), alloc, None, None)

    assert call(None) == -2                                  # no statistics: brs_backward's path up to the allocator
    assert call(_Stats(fake, fake, None, n)) == -2           # identity map with rows == P: accepted
    assert call(_Stats(fake, fake, fake, 3)) == -2           # explicit index: any rows >= 0
    assert call(_Stats(None, fake, None, n)) == -1           # grad_norm NULL
    assert call(_Stats(fake, None, None, n)) == -1           # count NULL
    assert call(_Stats(fake, fake, fake, -1)) == -1          # negative rows
    assert call(_Stats(fake, fake, None, n - 1)) == -1       # identity map needs rows >= P
    assert lib.brs_backward(C.byref(view), C.byref(g), C.c_void_p(fake), C.byref(state), C.c_void_p(fake), None,
                            C.byref(grads), alloc, None, None) == -2


def test_stand_in_has_no_densification_statistics():
    from workload import synthetic
    from bloomscene_b200.rasterizer import GaussianRasterizationSettings, bind
    from oracle_backend import OracleBackend

    api = bind(OracleBackend())
    assert not api.GaussianRasterizer.supports_densify_stats
    scene = synthetic.make_scene(20, "object", "precomp", -3.0, seed=2)
    rs = synthetic.raster_settings(synthetic.orbit_camera(32, 24, 0.1), 0, torch.zeros(3), GaussianRasterizationSettings)
    stats = {"grad_norm": torch.zeros(20), "count": torch.zeros(20)}
    with pytest.raises(Exception, match="no densification statistics"):
        api.GaussianRasterizer(rs, densify_stats=stats)(scene.means3D, torch.zeros_like(scene.means3D), scene.opacities,
                                                        colors_precomp=scene.colors_precomp, scales=scene.scales,
                                                        rotations=scene.rotations)
    from bloomscene_b200.multiview import GraphedStep

    class _NoStats(api.GaussianRasterizer):  # passes GraphedStep's other checks, lacks only the statistics
        supports_deferred = True
        supports_grad_sink = True
        supports_densify_stats = False

    with pytest.raises(Exception, match="no densification statistics"):
        GraphedStep(_setup(True)[1], [synthetic.orbit_camera(32, 24, 0.1)], torch.zeros(3), _NoStats,
                    lambda c, d, t: c.sum())
