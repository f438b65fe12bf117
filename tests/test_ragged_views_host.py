"""CPU: stacks of views with their own Gaussians — brs_forward_views_ex validation through ctypes (fake pointers,
rejected before any CUDA call) and render_views(view_counts=...) on the CPU oracle against single calls."""
import ctypes as C
import os

import pytest
import torch

from test_host_api import _Gaussians, _View

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_forward_views_ex_validates_the_view_counts_without_touching_the_gpu():
    lib = C.CDLL(os.path.join(ROOT, "bloomscene_b200", "libbloomrast.so"))
    ALLOC = C.CFUNCTYPE(C.c_void_p, C.c_void_p, C.c_int, C.c_size_t)
    alloc = ALLOC(lambda ctx, which, n: None)
    fake = 0x1000

    def view(W=64, H=48, deg=0):
        return _View(W, H, 0.5, 0.5, 1.0, deg, 0, 0, 0, fake, fake, fake, fake)

    def call(views, g, counts, alloc_fn=alloc):
        arr = (_View * len(views))(*views)
        vp = None if counts is None else (C.c_int * len(counts))(*counts)
        return lib.brs_forward_views_ex(arr, len(views), C.byref(g), vp, C.c_void_p(fake), C.c_void_p(fake),
                                        C.c_void_p(fake), alloc_fn, None, None, None, None)

    g = _Gaussians(100, fake, fake, None, fake, fake, fake, None)
    three = [view(), view(), view()]
    assert call(three, g, [40, -1, 61]) == -1                 # negative count
    assert call(three, g, [40, 0, 59]) == -1                  # sum 99 != P
    assert call(three, g, [40, 0, 61]) == -1                  # sum 101 != P
    assert call(three, g, [2**30, 2**30, 0]) == -4            # 2^31 instances do not fit 32-bit ids: BRS_ERR_UNSUPPORTED
    assert call(three, g, [2**31 - 1, 2**31 - 1, 5]) == -4
    # the checks of brs_forward_views come first and stay as they are
    assert call([view(), view(W=80), view()], g, [40, 0, 60]) == -1
    assert call([view(), view(deg=1), view()], g, [40, 0, 60]) == -1
    assert call([view(H=16 * 40000), view(H=16 * 40000)], g, [50, 50]) == -4  # 80 000 stacked tile rows > 16 bits
    # valid counts reach the next check (no allocator) — still before any CUDA call
    assert call(three, g, [40, 0, 60], alloc_fn=ALLOC()) == -1
    # NULL counts: every view sees all rows, exactly brs_forward_views (3 * 2^30 instances are too many)
    big = _Gaussians(2**30, fake, fake, None, fake, fake, fake, None)
    assert call(three, big, None) == -4
    assert call(three, big, [2**30, 0, 0], alloc_fn=ALLOC()) == -1  # the same rows split over views fit
    assert lib.brs_forward_views_ex(None, 2, C.byref(g), None, None, None, None, alloc, None, None, None, None) == -1


def _ragged_scene(counts, seed):
    from workload import synthetic

    base = synthetic.make_scene(300, "object", "sh1", -3.0, seed=seed)
    g = torch.Generator(device="cpu").manual_seed(seed)
    idx = torch.cat([torch.randperm(base.P, generator=g)[:c] for c in counts])
    return {k: v.index_select(0, idx).contiguous() for k, v in base.tensors().items()}


def test_render_views_with_view_counts_equals_single_calls_with_oracle_backend():
    """Each view renders its own rows; a view with no rows gives zeros without background (reference P == 0)."""
    from workload import synthetic
    from bloomscene_b200.rasterizer import GaussianRasterizationSettings, bind
    from oracle_backend import OracleBackend

    api = bind(OracleBackend())
    counts = [120, 0, 1, 77, 300]
    t = _ragged_scene(counts, seed=4)
    bg = torch.tensor([0.2, 0.1, 0.3])
    settings = [synthetic.raster_settings(synthetic.orbit_camera(40, 24, 0.7 * k), 1, bg, GaussianRasterizationSettings)
                for k in range(len(counts))]
    kw = dict(shs=t["shs"], scales=t["scales"], rotations=t["rotations"])
    color, depth, radii = api.render_views(settings, t["means3D"], t["opacities"], keep_radii=True, view_counts=counts,
                                           stack=2, **kw)  # no stacked binding here: the per-view route
    assert color.shape == (5, 3, 24, 40) and depth.shape == (5, 1, 24, 40)
    assert [tuple(r.shape) for r in radii] == [(c,) for c in counts]
    off = 0
    for k, (rs, c) in enumerate(zip(settings, counts)):
        rows = {n: v[off:off + c].clone() for n, v in t.items()}
        off += c
        col, r, d = api.GaussianRasterizer(rs)(rows["means3D"], torch.zeros_like(rows["means3D"]), rows["opacities"],
                                               shs=rows["shs"], scales=rows["scales"], rotations=rows["rotations"])
        assert torch.equal(col, color[k]) and torch.equal(d, depth[k]) and torch.equal(r, radii[k]), k
    assert not color[1].any() and not depth[1].any()
    assert color[0].any()
    for bad in ([120, 0, 1, 77], [120, 0, 1, 77, 299], [121, -1, 1, 77, 300]):
        with pytest.raises(Exception, match="view_counts"):
            api.render_views(settings, t["means3D"], t["opacities"], view_counts=bad, **kw)
