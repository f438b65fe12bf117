"""Python surface of the rasterizer — same names, arguments, return values and error behaviour as the
reference package `depth_diff_gaussian_rasterization` (reference:
submodules/depth-diff-gaussian-rasterization/depth_diff_gaussian_rasterization/__init__.py:17-250).

`bind(_C)` builds the public objects on top of a native module exposing the reference's four
binding functions (ext.cpp:15-20).  The product binds bloomscene_b200._C (the B200-native CUDA
library); tests bind the reference's own extension through the very same wrapper, so parity tests
exercise identical Python on both sides.
"""
from __future__ import annotations

from concurrent.futures import ThreadPoolExecutor
from functools import partial
from types import SimpleNamespace
from typing import NamedTuple

import torch
import torch.nn as nn


class GaussianRasterizationSettings(NamedTuple):
    # field order is part of the API (reference __init__.py:158-170)
    image_height: int
    image_width: int
    tanfovx: float
    tanfovy: float
    bg: torch.Tensor
    scale_modifier: float
    viewmatrix: torch.Tensor
    projmatrix: torch.Tensor
    sh_degree: int
    campos: torch.Tensor
    prefiltered: bool
    debug: bool


def cpu_deep_copy_tuple(input_tuple):
    # reference __init__.py:17-19 (debug snapshots)
    copied_tensors = [item.cpu().clone() if isinstance(item, torch.Tensor) else item for item in input_tuple]
    return tuple(copied_tensors)


def _absent() -> torch.Tensor:
    """Placeholder for an optional input that was not given: an empty CPU tensor, whose data pointer is
    NULL — the reference's own convention (reference __init__.py:198-208)."""
    return torch.Tensor([])


def _guarded(native_fn, args, debug: bool, dump_file: str, message: str):
    """Call into the native module; with `debug` set, snapshot the arguments first and write them to
    `dump_file` if the call raises (reference __init__.py:83-90 forward, :133-140 backward)."""
    if not debug:
        return native_fn(*args)
    snapshot = cpu_deep_copy_tuple(args)  # taken before the call so a crash cannot corrupt it
    try:
        return native_fn(*args)
    except Exception:
        torch.save(snapshot, dump_file)
        print(message)
        raise


_LANE_STREAMS = {}
_LANE_POOLS = {}


def lane_pool(dev: torch.device, n: int) -> ThreadPoolExecutor:
    """One long-lived pool of `n` host threads per device for driving the lane streams (a fresh executor
    per call would pay thread start-up, and the library's per-thread pinned slot, on every step)."""
    key = (dev.type, dev.index if dev.index is not None else torch.cuda.current_device(), n)
    pool = _LANE_POOLS.get(key)
    if pool is None:
        pool = _LANE_POOLS[key] = ThreadPoolExecutor(max_workers=n, thread_name_prefix="brs-lane")
    return pool


def lane_streams(dev: torch.device, n: int):
    """`n` long-lived high-priority CUDA streams of `dev` that a batch of views is dealt onto.  High
    priority makes the library move its blend kernels to a lowest-priority companion stream
    (brs_blend_companion_stream), so the small kernels of one view are dispatched underneath another
    view's blend grid."""
    key = (dev.type, dev.index if dev.index is not None else torch.cuda.current_device())
    pool = _LANE_STREAMS.setdefault(key, [])
    while len(pool) < n:
        pool.append(torch.cuda.Stream(device=dev, priority=-1))
    return pool[:n]


def bind(_C) -> SimpleNamespace:
    """Create (rasterize_gaussians, _RasterizeGaussians, GaussianRasterizer) bound to native module `_C`."""

    class _RasterizeGaussians(torch.autograd.Function):
        """Autograd node around _C.rasterize_gaussians / _C.rasterize_gaussians_backward; argument orders
        are those of the binding (reference __init__.py:53-73 forward, :108-131 backward)."""

        @staticmethod
        def forward(ctx, means3D, means2D, sh, colors_precomp, opacities, scales, rotations, cov3Ds_precomp,
                    raster_settings, grad_sink=None, depth_gradient=False, deferred_overflow=None, densify_stats=None):
            rs = raster_settings
            args = (rs.bg, means3D, colors_precomp, opacities, scales, rotations, rs.scale_modifier, cov3Ds_precomp,
                    rs.viewmatrix, rs.projmatrix, rs.tanfovx, rs.tanfovy, rs.image_height, rs.image_width, sh,
                    rs.sh_degree, rs.campos, rs.prefiltered, rs.debug)
            if deferred_overflow is not None:
                # extension: no host wait at all (brs_fwd_options DEFERRED); capacity overflows are OR-ed into the
                # caller's device word, which it checks once per batch of views (a CUDA graph can hold this call)
                out = _C.rasterize_gaussians_ex(*args, _C.FWD_DEFERRED, 0, 0, 0, None, deferred_overflow)
            else:
                out = _guarded(_C.rasterize_gaussians, args, rs.debug, "snapshot_fw.dump",
                               "\nAn error occured in forward. Please forward snapshot_fw.dump for debugging.")
            num_rendered, color, depth, radii, geom, binning, image = out
            ctx.raster_settings = rs
            ctx.grad_sink = grad_sink
            ctx.densify_stats = densify_stats
            ctx.num_rendered = num_rendered
            ctx.depth_gradient = bool(depth_gradient)
            # extension: with depth_gradient the backward also needs the depth image the forward produced
            extra = (depth,) if depth_gradient else ()
            ctx.save_for_backward(colors_precomp, means3D, scales, rotations, cov3Ds_precomp, radii, sh, geom,
                                  binning, image, *extra)
            return color, radii, depth

        @staticmethod
        def backward(ctx, grad_out_color, grad_radii, grad_depth):
            rs = ctx.raster_settings
            colors_precomp, means3D, scales, rotations, cov3Ds_precomp, radii, sh, geom, binning, image = ctx.saved_tensors[:10]
            out_depth = ctx.saved_tensors[10] if ctx.depth_gradient else None
            # extension: the kernel adds this view's densification statistics into the caller's accumulators
            ds = ctx.densify_stats
            stats = {} if ds is None else {"stats_grad_norm": ds["grad_norm"], "stats_count": ds["count"],
                                           "stats_index": ds.get("index")}
            bw = lambda fn: partial(fn, **stats) if stats else fn
            if ctx.grad_sink is not None:
                # extension: parameter gradients are added in place to the caller's sinks by the kernel
                # (brs_grads.accumulate); autograd only carries the per-view means2D gradient
                k = ctx.grad_sink
                d_means2D = _guarded(
                    bw(_C.rasterize_gaussians_backward_accumulate),
                    (rs.bg, means3D, radii, colors_precomp, scales, rotations, rs.scale_modifier, cov3Ds_precomp,
                     rs.viewmatrix, rs.projmatrix, rs.tanfovx, rs.tanfovy, grad_out_color, grad_depth, sh, rs.sh_degree,
                     rs.campos, geom, ctx.num_rendered, binning, image, rs.debug,
                     k.get("means3D"), k.get("colors_precomp"), k.get("opacities"), k.get("cov3D_precomp"), k.get("shs"),
                     k.get("scales"), k.get("rotations"), out_depth),
                    rs.debug, "snapshot_bw.dump",
                    "\nAn error occured in backward. Writing snapshot_bw.dump for debugging.\n")
                return None, d_means2D, None, None, None, None, None, None, None, None, None, None, None
            if ctx.depth_gradient:
                # extension: grad_depth is back-propagated through the depth image (default off = reference)
                g = _guarded(
                    bw(_C.rasterize_gaussians_backward_depth),
                    (rs.bg, means3D, radii, colors_precomp, scales, rotations, rs.scale_modifier, cov3Ds_precomp,
                     rs.viewmatrix, rs.projmatrix, rs.tanfovx, rs.tanfovy, grad_out_color, grad_depth, sh, rs.sh_degree,
                     rs.campos, geom, ctx.num_rendered, binning, image, rs.debug, out_depth),
                    rs.debug, "snapshot_bw.dump",
                    "\nAn error occured in backward. Writing snapshot_bw.dump for debugging.\n")
                d_means2D, d_colors, d_opacities, d_means3D, d_cov3D, d_sh, d_scales, d_rotations = g
                return d_means3D, d_means2D, d_sh, d_colors, d_opacities, d_scales, d_rotations, d_cov3D, None, None, None, None, None
            g = _guarded(
                bw(_C.rasterize_gaussians_backward),
                (rs.bg, means3D, radii, colors_precomp, scales, rotations, rs.scale_modifier, cov3Ds_precomp,
                 rs.viewmatrix, rs.projmatrix, rs.tanfovx, rs.tanfovy, grad_out_color, grad_depth, sh, rs.sh_degree,
                 rs.campos, geom, ctx.num_rendered, binning, image, rs.debug),
                rs.debug, "snapshot_bw.dump",
                "\nAn error occured in backward. Writing snapshot_bw.dump for debugging.\n")
            d_means2D, d_colors, d_opacities, d_means3D, d_cov3D, d_sh, d_scales, d_rotations = g
            # one gradient per autograd input, in input order (reference __init__.py:144-154);
            # grad_radii carries nothing and grad_depth is plumbed down but unused by the kernels
            return d_means3D, d_means2D, d_sh, d_colors, d_opacities, d_scales, d_rotations, d_cov3D, None, None, None, None, None

    has_sink = hasattr(_C, "rasterize_gaussians_backward_accumulate")
    has_depth_grad = hasattr(_C, "rasterize_gaussians_backward_depth")

    has_deferred = hasattr(_C, "rasterize_gaussians_ex")
    has_densify_stats = bool(getattr(_C, "HAS_DENSIFY_STATS", False))

    def rasterize_gaussians(means3D, means2D, sh, colors_precomp, opacities, scales, rotations, cov3Ds_precomp,
                            raster_settings, grad_sink=None, depth_gradient=False, deferred_overflow=None,
                            densify_stats=None):
        # reference __init__.py:21-42; `grad_sink`, `depth_gradient`, `deferred_overflow` and `densify_stats` are
        # extensions (see GaussianRasterizer)
        if densify_stats is not None and not has_densify_stats:
            raise Exception('this native module has no densification statistics')
        if depth_gradient and not has_depth_grad:
            raise Exception('this native module has no depth gradient (the reference comments it out)')
        if deferred_overflow is not None and not has_deferred:
            raise Exception('this native module has no deferred forward')
        if grad_sink is not None:
            if not has_sink:
                raise Exception('this native module has no in-place gradient accumulation (grad_sink)')
            given = {"means3D": means3D, "opacities": opacities, "shs": sh, "colors_precomp": colors_precomp,
                     "scales": scales, "rotations": rotations, "cov3D_precomp": cov3Ds_precomp}
            for name, t in given.items():
                if t.numel() != 0 and t.requires_grad and name not in grad_sink:
                    raise Exception(f'grad_sink has no entry for {name}, whose gradient would be dropped')
        return _RasterizeGaussians.apply(means3D, means2D, sh, colors_precomp, opacities, scales, rotations,
                                         cov3Ds_precomp, raster_settings, grad_sink, depth_gradient, deferred_overflow,
                                         densify_stats)

    class GaussianRasterizer(nn.Module):
        """reference __init__.py:172-249: forward / visible_filter / markVisible with the same signatures.

        Extension: `grad_sink` (default None = reference behaviour) maps input names ("means3D", "opacities",
        "shs" | "colors_precomp", "scales", "rotations" | "cov3D_precomp") to contiguous fp32 tensors of the
        inputs' shapes.  With it, backward ADDS those inputs' gradients to the sinks inside the kernel and
        autograd receives None for them — a multi-view step accumulates straight into its allreduce bucket
        instead of materialising (44 + 12 M) bytes per Gaussian per view and adding them afterwards.

        Extension: `depth_gradient` (default False = reference behaviour, where the depth output carries no
        gradient because every depth line of the reference's backward is commented out, backward.cu:443-554).
        With it, the gradient of the returned depth image flows back through D / acc (and its acc > 0.5
        gate, forward.cu:464-468) into opacities, means3D and scales / rotations | cov3D_precomp, so
        BloomScene's depth losses (bloomscene.py:298-325) can act on the geometry.

        Extension: `densify_stats` (default None) = {"grad_norm": t, "count": t, "index": optional int64 [P]} of
        caller-owned fp32 accumulators (any shape, same number of elements, e.g. [rows, 1]).  The backward then adds,
        for every Gaussian i with radii[i] > 0, |means2D.grad[i, :2]| to grad_norm[slot] and 1 to count[slot], with
        slot = index[i] (skipped outside [0, rows)) or i — what the densification statistics of Scaffold-GS
        (training_statis, scene/gaussian_model.py:742-759) and 3DGS (add_densification_stats) compute from
        means2D.grad and radii after every view, here without any per-view torch op, inside CUDA graphs and with
        grad_sink."""

        supports_grad_sink = has_sink
        supports_depth_gradient = has_depth_grad
        supports_deferred = has_deferred
        supports_densify_stats = has_densify_stats

        def __init__(self, raster_settings, grad_sink=None, depth_gradient=False, deferred_overflow=None,
                     densify_stats=None):
            super().__init__()
            self.raster_settings = raster_settings
            self.grad_sink = grad_sink
            self.depth_gradient = depth_gradient
            # Extension: a CUDA int32[1] tensor switches the forward to brs_fwd_options DEFERRED - no host
            # synchronisation in forward or backward, buffers sized from the high-water marks of the shape, capacity
            # overflows OR-ed into the tensor (non-zero = this forward's results are invalid, run it again without).
            self.deferred_overflow = deferred_overflow
            self.densify_stats = densify_stats

        def markVisible(self, positions):
            rs = self.raster_settings
            with torch.no_grad():
                return _C.mark_visible(positions, rs.viewmatrix, rs.projmatrix)

        def forward(self, means3D, means2D, opacities, shs=None, colors_precomp=None, scales=None, rotations=None,
                    cov3D_precomp=None):
            # same two checks and messages (typo included) as reference __init__.py:192-196
            if (shs is None) == (colors_precomp is None):
                raise Exception('Please provide excatly one of either SHs or precomputed colors!')
            has_any_sr, has_both_sr = (scales is not None or rotations is not None), (scales is not None and rotations is not None)
            if (not has_both_sr and cov3D_precomp is None) or (has_any_sr and cov3D_precomp is not None):
                raise Exception('Please provide exactly one of either scale/rotation pair or precomputed 3D covariance!')
            opt = lambda t: _absent() if t is None else t
            return rasterize_gaussians(means3D, means2D, opt(shs), opt(colors_precomp), opacities, opt(scales),
                                       opt(rotations), opt(cov3D_precomp), self.raster_settings, self.grad_sink,
                                       self.depth_gradient, self.deferred_overflow, self.densify_stats)

        def visible_filter(self, means3D, scales=None, rotations=None, cov3D_precomp=None):
            rs = self.raster_settings
            opt = lambda t: _absent() if t is None else t
            with torch.no_grad():
                return _C.rasterize_aussians_filter(means3D, opt(scales), opt(rotations), rs.scale_modifier,
                                                    opt(cov3D_precomp), rs.viewmatrix, rs.projmatrix, rs.tanfovx,
                                                    rs.tanfovy, rs.image_height, rs.image_width, rs.prefiltered, rs.debug)

        def visible_filter_indices(self, means3D, scales=None, rotations=None, cov3D_precomp=None):
            """Extension (SURVEY.md 8f N2): `visible_filter` fused with the compaction BloomScene does next.  Returns
            (radii int32 [P], visible_idx int64 [V]): visible_idx lists, ascending, the Gaussians with radii > 0 —
            what `torch.nonzero(radii > 0)` would give — written by the same kernel, so the caller gathers its
            per-anchor tensors with `t[visible_idx]` (index_select) instead of one boolean-mask nonzero each
            (reference gaussian_renderer/__init__.py:39-60 indexes five tensors with visible_mask)."""
            rs = self.raster_settings
            opt = lambda t: _absent() if t is None else t
            with torch.no_grad():
                radii, idx, count = _C.rasterize_gaussians_filter_compact(
                    means3D, opt(scales), opt(rotations), rs.scale_modifier, opt(cov3D_precomp), rs.viewmatrix, rs.projmatrix,
                    rs.tanfovx, rs.tanfovy, rs.image_height, rs.image_width, rs.prefiltered, rs.debug)
                return radii, idx[: int(count.item())]

    def render_views(raster_settings_list, means3D, opacities, shs=None, colors_precomp=None, scales=None,
                     rotations=None, cov3D_precomp=None, streams=4, keep_radii=False, host_threads=True, stack=0):
        """Forward-only render of one Gaussian set from a list of cameras (BloomScene's render_video loop,
        reference bloomscene.py:191-204, one `GaussianRasterizer` call per frame there).  Extension: no
        autograd graph, no saved state, and on a GPU the views are dealt onto `streams` CUDA streams so that
        one view's preprocess / sort / binning kernels and its host wait for the instance count run under
        another view's blend; with `host_threads` every stream is driven by its own host thread (the native
        forward releases the GIL).  Returns (color [B,3,H,W], depth [B,1,H,W], radii list or None); every view's
        result is bit-identical to a single `GaussianRasterizer` call with the same settings.  The call returns
        after ONE host synchronisation for the whole batch (the reference waits once per frame,
        rasterizer_impl.cu:282), plus one for the first frame of a (P, W, H) shape it has never seen.

        `stack` > 1: consecutive views are rendered `stack` at a time as ONE pipeline (`brs_forward_views`): one
        preprocess launch per view into a shared instance space, then one depth sort, one emission / coarse sort /
        fine binning and one blend launch for the whole stack, at most one host wait per stack; the stacks are
        dealt onto `streams` lanes (streams=1: everything on the caller's stream).  Same bits as the per-view path.  Views of a stack must share background, scale modifier and flags
        (a run of views that does not is cut into shorter stacks)."""
        views = list(raster_settings_list)
        if (shs is None) == (colors_precomp is None):
            raise Exception('Please provide excatly one of either SHs or precomputed colors!')
        has_any_sr, has_both_sr = (scales is not None or rotations is not None), (scales is not None and rotations is not None)
        if (not has_both_sr and cov3D_precomp is None) or (has_any_sr and cov3D_precomp is not None):
            raise Exception('Please provide exactly one of either scale/rotation pair or precomputed 3D covariance!')
        opt = lambda t: _absent() if t is None else t.detach()
        dev = means3D.device
        B = len(views)
        H, W = (views[0].image_height, views[0].image_width) if B else (0, 0)
        color = torch.empty((B, 3, H, W), dtype=torch.float32, device=dev)
        depth = torch.empty((B, 1, H, W), dtype=torch.float32, device=dev)
        radii = [None] * B if keep_radii else None
        m3, op = means3D.detach(), opacities.detach()
        sh_, cp_, sc_, ro_, cv_ = opt(shs), opt(colors_precomp), opt(scales), opt(rotations), opt(cov3D_precomp)

        # Native module with brs_fwd_options: every view is a DEFERRED forward (no host wait at all; buffers sized
        # from the high-water marks of this shape); the instance counts land in pinned host memory and are
        # checked ONCE for the whole batch.  A view whose capacities were too small is rendered again in EXACT
        # mode.  Any other module (the reference build): one plain call per view.
        deferred = hasattr(_C, "rasterize_gaussians_ex") and dev.type == "cuda" and B > 0
        reports = torch.zeros((B, 8), dtype=torch.int32).pin_memory() if deferred else None

        def one(j, rs, exact=False):
            if (rs.image_height, rs.image_width) != (H, W):
                raise Exception('render_views: all views of a batch must share one resolution')
            args = (rs.bg, m3, cp_, op, sc_, ro_, rs.scale_modifier, cv_, rs.viewmatrix, rs.projmatrix, rs.tanfovx,
                    rs.tanfovy, rs.image_height, rs.image_width, sh_, rs.sh_degree, rs.campos, rs.prefiltered, rs.debug)
            if deferred and not exact:
                out = _C.rasterize_gaussians_ex(*args, _C.FWD_DEFERRED, 0, 0, 0, reports[j])
            elif deferred:
                out = _C.rasterize_gaussians_ex(*args, _C.FWD_EXACT, 0, 0, 0, None)
            else:
                out = _C.rasterize_gaussians(*args)
            color[j].copy_(out[1])
            depth[j].copy_(out[2])
            if keep_radii:
                radii[j] = out[3]

        if int(stack) > 1 and hasattr(_C, "rasterize_gaussians_views") and dev.type == "cuda" and B > 0:
            same = lambda a, b: (a.bg.data_ptr() == b.bg.data_ptr() and a.scale_modifier == b.scale_modifier and
                                 a.sh_degree == b.sh_degree and a.prefiltered == b.prefiltered and a.debug == b.debug)
            groups, j = [], 0
            while j < B:
                n = 1
                while n < int(stack) and j + n < B and same(views[j], views[j + n]):
                    n += 1
                groups.append((j, n))
                j += n
            for rs in views:
                if (rs.image_height, rs.image_width) != (H, W):
                    raise Exception('render_views: all views of a batch must share one resolution')

            def one_stack(j, n):
                grp = views[j:j + n]
                rs = grp[0]
                vm = torch.stack([v.viewmatrix for v in grp])
                pm = torch.stack([v.projmatrix for v in grp])
                cps = torch.stack([v.campos for v in grp])
                _, _, _, r = _C.rasterize_gaussians_views(
                    rs.bg, m3, cp_, op, sc_, ro_, rs.scale_modifier, cv_, vm, pm, [float(v.tanfovx) for v in grp],
                    [float(v.tanfovy) for v in grp], H, W, sh_, rs.sh_degree, cps, rs.prefiltered, rs.debug,
                    color_out=color[j:j + n], depth_out=depth[j:j + n])  # written in place
                if keep_radii:
                    for q in range(n):
                        radii[j + q] = r[q]
                return r

            with torch.no_grad():
                n_lanes = max(1, min(int(streams), len(groups)))
                if n_lanes == 1:
                    for j, n in groups:
                        one_stack(j, n)
                else:
                    # stacks are dealt onto lanes: one stack's preprocess / sort / binning under another's blend
                    cur = torch.cuda.current_stream(dev)
                    lanes = lane_streams(dev, n_lanes)
                    for st in lanes:
                        st.wait_stream(cur)
                    for k, (j, n) in enumerate(groups):
                        with torch.cuda.stream(lanes[k % n_lanes]):
                            r = one_stack(j, n)
                            if keep_radii:
                                r.record_stream(cur)
                    for st in lanes:
                        cur.wait_stream(st)
            return color, depth, radii

        with torch.no_grad():
            n_lanes = max(1, min(int(streams), B)) if dev.type == "cuda" else 1
            first = 0
            if deferred and not _C.has_marks(m3.shape[0], W, H):
                one(0, views[0], exact=True)  # a shape never seen before: one EXACT forward seeds its high-water marks
                first = 1
            if n_lanes == 1:
                for j in range(first, B):
                    one(j, views[j])
            else:
                cur = torch.cuda.current_stream(dev)
                lanes = lane_streams(dev, n_lanes)
                for st in lanes:
                    st.wait_stream(cur)  # inputs and the output stacks were produced on the caller's stream

                def drive(lane):  # one host thread per stream: the native forward releases the GIL while it
                    with torch.no_grad(), torch.cuda.stream(lanes[lane]):  # launches (and, non-deferred, waits)
                        for j in range(first + lane, B, n_lanes):
                            one(j, views[j])

                if host_threads:
                    pool = lane_pool(dev, n_lanes)
                    for f in [pool.submit(drive, lane) for lane in range(n_lanes)]:
                        f.result()
                else:
                    for j in range(first, B):
                        with torch.cuda.stream(lanes[(j - first) % n_lanes]):
                            one(j, views[j])
                for st in lanes:
                    cur.wait_stream(st)
                if keep_radii:
                    for r in radii[first:]:
                        r.record_stream(cur)  # allocated on a lane stream, consumed on the caller's
            if deferred:
                # the one host wait of the batch: every report has landed once the caller's stream is drained
                torch.cuda.current_stream(dev).synchronize()
                for j in range(first, B):
                    _C.note_counts(m3.shape[0], W, H, reports[j])
                    if int(reports[j, 5]) != 0:
                        one(j, views[j], exact=True)
        return color, depth, radii

    return SimpleNamespace(
        _C=_C,
        render_views=render_views,
        _RasterizeGaussians=_RasterizeGaussians,
        rasterize_gaussians=rasterize_gaussians,
        GaussianRasterizer=GaussianRasterizer,
        GaussianRasterizationSettings=GaussianRasterizationSettings,
    )
