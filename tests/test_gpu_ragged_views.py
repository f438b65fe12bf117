"""GPU: stacks of views where every view renders its own Gaussians (render_views(view_counts=...),
brs_forward_views_ex) against one GaussianRasterizer call per view on that view's rows, bit for bit."""
import pytest
import torch

import parity_lib as pl
from workload import synthetic

pytestmark = pytest.mark.gpu

DEV = torch.device("cuda:0")


def _attrs(scene, cov3D=None):
    """Keyword inputs of render_views / GaussianRasterizer for a scene (cov3D replaces scales and rotations)."""
    kw = dict(shs=scene.shs, colors_precomp=scene.colors_precomp)
    if cov3D is None:
        kw.update(scales=scene.scales, rotations=scene.rotations)
    else:
        kw.update(cov3D_precomp=cov3D)
    return kw


def _ragged(scene, counts, seed, cov3D=None):
    """View j gets its own seeded subset of `counts[j]` rows of `scene` (repeated when it asks for more rows than the
    scene has).  Returns the concatenated (means3D, opacities, kw)."""
    g = torch.Generator(device="cpu").manual_seed(seed)
    P = scene.P
    idx = torch.cat([torch.randint(0, P, (c,), generator=g) if c > P else torch.randperm(P, generator=g)[:c] for c in counts])
    idx = idx.to(scene.means3D.device)
    pick = lambda t: None if t is None else t.index_select(0, idx).contiguous()
    kw = {k: pick(v) for k, v in _attrs(scene, cov3D).items()}
    return pick(scene.means3D), pick(scene.opacities), kw


def _singles(api, settings, m3, op, kw, counts):
    """One GaussianRasterizer call per view on a fresh copy of that view's rows: [(color, radii, depth)]."""
    out, off = [], 0
    with torch.no_grad():
        for rs, c in zip(settings, counts):
            rows = lambda t: None if t is None else t[off:off + c].clone()
            vkw = {k: rows(v) for k, v in kw.items()}
            m = rows(m3)
            out.append(api.GaussianRasterizer(rs)(m, torch.zeros_like(m), rows(op), **vkw))
            off += c
    torch.cuda.synchronize()
    return out


def _assert_equal(want, color, depth, radii, tag):
    for k, (c, r, d) in enumerate(want):
        assert torch.equal(r, radii[k]), (tag, k)
        assert torch.equal(c, color[k]), (tag, k)
        assert torch.equal(d, depth[k]), (tag, k)


def _setup(color_kind, base_P, W, H, B, cov=False, seed=11, kind="band"):
    from golden.make_golden import cov3d_from_scale_rot

    api = pl.ours()
    scene = synthetic.make_scene(base_P, kind, color_kind, -4.6 if kind == "band" else -3.6, seed=seed)
    cov3D = cov3d_from_scale_rot(scene.scales, scene.rotations).to(DEV) if cov else None
    scene = scene.to(DEV)
    camera = synthetic.yaw_camera if kind == "band" else synthetic.orbit_camera
    cams = [camera(W, H, 0.35 * k).to(DEV) for k in range(B)]
    bg = torch.tensor([0.3, 0.2, 0.1], device=DEV)
    settings = [synthetic.raster_settings(c, scene.sh_degree, bg, api.GaussianRasterizationSettings) for c in cams]
    return api, scene, cov3D, settings


def _counts(B, pattern, seed):
    """`pattern` for the first views, seeded sizes below 3000 for the rest."""
    g = torch.Generator(device="cpu").manual_seed(seed)
    extra = torch.randint(0, 3000, (B,), generator=g).tolist()
    return [pattern[k] if k < len(pattern) else extra[k] for k in range(B)]


CASES = {
    # color, scene rows, W, H, views, stack, counts pattern, cov3D_precomp[, scene kind]
    "sh3m16_130x70_17views_stack17": ("sh3", 20000, 130, 70, 17, 17, [0, 1, 127, 128, 129, 20000, 3, 0, 255, 7], False),
    "sh1_200x120_5views_stack2": ("sh1", 8000, 200, 120, 5, 2, [129, 0, 8000, 1, 127], False),
    "precomp_130x70_33views_stack33": ("precomp", 30000, 130, 70, 33, 33, [30000, 0, 1, 128, 0, 0, 129, 127], False),
    "cov3d_sh3_96x64_33views_stack8": ("sh3", 6000, 96, 64, 33, 8, [1, 6000, 0, 129, 33], True),
    "sh3m16_320x192_5views_stack3": ("sh3", 60000, 320, 192, 5, 3, [60000, 17, 1, 45001, 0], False),
    # an object in front of orbiting cameras: most Gaussians are visible, so the optimistic calls request every SH
    # row up front (the EAGER bulk copies) at odd row offsets
    "sh3m16_object_160x96_17views_stack17": ("sh3", 20000, 160, 96, 17, 17, [1, 127, 0, 129, 20000, 5, 128], False, "object"),
}


@pytest.mark.parametrize("case", list(CASES.values()), ids=list(CASES))
def test_ragged_stacks_are_bit_identical_to_single_calls(case):
    """Views with their own row counts (0, 1, odd, 127/128/129 around the preprocess block, one view far larger than
    the others) as stacks of views: more than 16 views in a stack (several preprocess launches), stacks that do not
    divide the views, ragged image sizes; one stream, then two lanes, each called twice (EXACT first, optimistic
    after)."""
    color_kind, base_P, W, H, B, stack, pattern, cov, *kind = case
    api, scene, cov3D, settings = _setup(color_kind, base_P, W, H, B, cov, kind=kind[0] if kind else "band")
    counts = _counts(B, pattern, seed=B)
    m3, op, kw = _ragged(scene, counts, seed=5, cov3D=cov3D)
    want = _singles(api, settings, m3, op, kw, counts)
    api._C.reset_marks()
    for streams in (1, 2):
        for rep in range(2):
            color, depth, radii = api.render_views(settings, m3, op, keep_radii=True, stack=stack, streams=streams,
                                                   view_counts=counts, **kw)
            torch.cuda.synchronize()
            assert color.shape == (B, 3, H, W) and depth.shape == (B, 1, H, W)
            assert [tuple(r.shape) for r in radii] == [(c,) for c in counts]
            _assert_equal(want, color, depth, radii, (streams, rep))
    for k, c in enumerate(counts):
        if c == 0:  # no Gaussians: zeros, not the background (reference P == 0 forward)
            assert not color[k].any() and not depth[k].any()
    assert sum(int((r > 0).sum()) for r in radii) > 100


def test_ragged_views_per_view_route_slices_each_views_rows():
    """Without `stack`: the per-view route (four streams, host threads, deferred batch) on each view's rows."""
    api, scene, _, settings = _setup("sh3", 20000, 160, 96, 9)
    counts = _counts(9, [0, 129, 20000, 1, 128], seed=3)
    m3, op, kw = _ragged(scene, counts, seed=6)
    want = _singles(api, settings, m3, op, kw, counts)
    for host_threads in (True, False):
        for rep in range(2):
            color, depth, radii = api.render_views(settings, m3, op, keep_radii=True, streams=4, host_threads=host_threads,
                                                   view_counts=counts, **kw)
            torch.cuda.synchronize()
            _assert_equal(want, color, depth, radii, (host_threads, rep))


def test_ragged_stack_overflow_rerun_still_matches():
    """A second stack with the same total rows but far larger footprints overflows the high-water marks of the first:
    the optimistic forward is run again with exact sizes (forward_stats) and still gives each view's single call."""
    api, scene, _, settings = _setup("precomp", 20000, 256, 160, 6)
    counts = [3000, 0, 129, 20000, 1, 4870]
    m3, op, kw = _ragged(scene, counts, seed=7)
    api._C.reset_marks()
    api.render_views(settings, m3, op, stack=6, streams=1, view_counts=counts, **kw)  # EXACT: seeds the marks
    kw_big = dict(kw, scales=kw["scales"] * 6.0)
    want = _singles(api, settings, m3, op, kw_big, counts)
    before = api._C.forward_stats()
    color, depth, radii = api.render_views(settings, m3, op, keep_radii=True, stack=6, streams=1, view_counts=counts, **kw_big)
    torch.cuda.synchronize()
    after = api._C.forward_stats()
    assert after["optimistic"] == before["optimistic"] + 1
    assert after["overflow_reruns"] == before["overflow_reruns"] + 1
    _assert_equal(want, color, depth, radii, "rerun")


@pytest.mark.parametrize("color_kind", ["sh3", "precomp"])
def test_concatenated_copies_give_the_uniform_stack(color_kind):
    """B copies of one scene with view_counts=[P] * B render exactly what the stack of one shared scene renders."""
    B, P = 7, 12345
    api, scene, _, settings = _setup(color_kind, P, 200, 120, B)
    kw = _attrs(scene)
    color_u, depth_u, radii_u = api.render_views(settings, scene.means3D, scene.opacities, keep_radii=True, stack=B,
                                                 streams=1, **kw)
    rep = lambda t: None if t is None else t.repeat((B,) + (1,) * (t.dim() - 1)).contiguous()
    color_r, depth_r, radii_r = api.render_views(settings, rep(scene.means3D), rep(scene.opacities), keep_radii=True,
                                                 stack=B, streams=1, view_counts=[P] * B,
                                                 **{k: rep(v) for k, v in kw.items()})
    torch.cuda.synchronize()
    assert torch.equal(color_u, color_r) and torch.equal(depth_u, depth_r)
    for k in range(B):
        assert torch.equal(radii_u[k], radii_r[k]), k


def test_config_B_sized_ragged_stack():
    """Config B's 500 K Gaussians split unevenly over 8 views at 512 x 512, rendered as one stack of 8."""
    api = pl.ours()
    scene = synthetic.config_scene("B").to(DEV)
    cams = [c.to(DEV) for c in synthetic.config_cameras("B", 8)]
    bg = torch.tensor([0.0, 0.0, 0.0], device=DEV)
    settings = [synthetic.raster_settings(c, 0, bg, api.GaussianRasterizationSettings) for c in cams]
    g = torch.Generator(device="cpu").manual_seed(8)
    w = torch.rand(8, generator=g) + 0.2
    counts = (w / w.sum() * scene.P).long().tolist()
    counts[-1] = scene.P - sum(counts[:-1])
    perm = torch.randperm(scene.P, generator=g).to(DEV)
    m3, op = scene.means3D[perm].contiguous(), scene.opacities[perm].contiguous()
    kw = {k: v[perm].contiguous() for k, v in _attrs(scene).items() if v is not None}
    want = _singles(api, settings, m3, op, kw, counts)
    color, depth, radii = api.render_views(settings, m3, op, keep_radii=True, stack=8, streams=1, view_counts=counts, **kw)
    torch.cuda.synchronize()
    _assert_equal(want, color, depth, radii, "B")
    assert all(int((r > 0).sum()) > 1000 for r in radii)
