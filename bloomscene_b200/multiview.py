"""View-sharded training step (SURVEY.md §8e): the one place the hot path meets a collective.

Views are independent given the Gaussian set, so the path shards by camera view: every rank holds
the full (replicated) Gaussian parameters, renders views `rank, rank+N, ...` of the batch with the
rasterizer, and accumulates per-Gaussian parameter gradients locally.  The only exchange is ONE
sum-allreduce of the flat fp32 gradient bucket per step (NCCL over NVLink on GPUs, gloo in the CPU
tests).  `means2D` gradients and `radii` are per-view statistics (BloomScene's densification uses
per-view norms, reference scene/gaussian_model.py:756-759) and are not reduced; what densification derives
from them (the per-Gaussian gradient-norm sum and count) rides in the bucket when the parameters carry
slots for it (`GaussianParams(scene, densify_stats=True)`).

The reference has no such mode (single process, one view per step: bloomscene.py:237-243); this is
the data-parallel scaling axis BASELINE.json names.  The rasterizer class is injected so host-side
logic can be tested on CPU with an oracle-backed stand-in (tests only).
"""
from __future__ import annotations

from typing import Callable, Dict, List, Optional, Sequence

import torch

from .rasterizer import GaussianRasterizationSettings, lane_pool, lane_streams
from workload.params import GaussianParams, shard_views
from workload.synthetic import Camera, raster_settings


def default_loss(color: torch.Tensor, depth: torch.Tensor, Wc: torch.Tensor, Wd: torch.Tensor) -> torch.Tensor:
    return (color * Wc).sum() + (depth * Wd).sum()


def view_sharded_step(params: GaussianParams, cameras: Sequence[Camera], bg: torch.Tensor, rasterizer_cls,
                      loss_fn: Callable[[torch.Tensor, torch.Tensor, int], torch.Tensor],
                      rank: int = 0, world: int = 1, group=None, allreduce: bool = True,
                      streams: int = 4, host_threads: bool = False, keep_means2D_grad: bool = False) -> Dict[str, object]:
    """Render this rank's slice of `cameras`, backpropagate `loss_fn(color, depth, view_index)`, sum the
    parameter gradients over ranks.  Returns the step loss (summed over all views), per-view radii
    counts and the number of views rendered locally.

    When `params.densify` is set, `res["densify"]` = {"grad_norm": [P], "count": [P]}: the densification statistics
    of this step's views (of all ranks after the all-reduce), views into the bucket valid until the next step.
    The native rasterizer adds them in its backward kernel; any other rasterizer gets them from means2D.grad and
    radii with the reference's torch statement.

    With the native rasterizer on a GPU the views are dealt round-robin onto `streams` CUDA streams: a
    view's preprocess / sort / binning kernels (small grids, latency- and bandwidth-bound) then run
    under another view's blend kernels (issue-bound), and the forward's one host wait for a view falls
    while the other stream still has a backward queued.  All streams add into the one gradient bucket:
    the kernel accumulates with float reductions (brs_grads.accumulate)."""
    mine = shard_views(len(cameras), rank, world)
    dev = params.flat.device
    visible = []
    # the native rasterizer adds parameter gradients straight into the bucket slices (grad_sink);
    # any other rasterizer (the reference build, the CPU stand-in of the tests) goes through autograd
    use_sink = getattr(rasterizer_cls, "supports_grad_sink", False)
    n_lanes = max(1, min(streams, len(mine))) if (use_sink and dev.type == "cuda") else 1
    sink = params.grads() if use_sink else None
    stats = params.densify
    native_stats = stats is not None and getattr(rasterizer_cls, "supports_densify_stats", False)
    extra = {"densify_stats": stats} if native_stats else {}
    losses = [torch.zeros((), dtype=torch.float32, device=dev) for _ in range(n_lanes)]

    zeroed = None
    if n_lanes > 1:
        # the bucket is zeroed on a side stream: only the first BACKWARD of every lane has to wait for it, the
        # forwards of the first views start at once
        cur = torch.cuda.current_stream(dev)
        zs = _zero_stream(dev)
        zs.wait_stream(cur)
        with torch.cuda.stream(zs):
            params.zero_grad()
            zeroed = torch.cuda.Event()
            zeroed.record()
    else:
        params.zero_grad()
    waited = [zeroed is None] * n_lanes

    def one_view(vi: int, lane: int):
        cam = cameras[vi]
        settings = raster_settings(cam, params.sh_degree, bg, GaussianRasterizationSettings)
        rast = (rasterizer_cls(settings, grad_sink=sink, **extra) if sink is not None
                else rasterizer_cls(raster_settings=settings, **extra))
        means2D = params.zero_means2D().detach().requires_grad_(True)  # fresh leaf over a shared zero buffer
        color, radii, depth = rast(means3D=params.tensors["means3D"], means2D=means2D,
                                   opacities=params.tensors["opacities"], shs=params.get("shs"),
                                   colors_precomp=params.get("colors_precomp"), scales=params.tensors["scales"],
                                   rotations=params.tensors["rotations"], cov3D_precomp=None)
        loss = loss_fn(color, depth, vi)
        if not waited[lane]:
            torch.cuda.current_stream(dev).wait_event(zeroed)
            waited[lane] = True
        loss.backward()
        losses[lane] += loss.detach()
        if stats is not None and not native_stats:
            # reference scene/gaussian_model.py:756-759 (identity slot map)
            with torch.no_grad():
                update_filter = radii > 0
                grad_norm = torch.norm(means2D.grad[update_filter, :2], dim=-1)
                stats["grad_norm"][update_filter] += grad_norm
                stats["count"][update_filter] += 1
        # per-view statistics for the caller's densification (reference scene/gaussian_model.py:742-759 reads
        # viewspace_points.grad[:, :2] and radii > 0 after every view)
        visible.append((vi, radii, means2D.grad if keep_means2D_grad else None))

    if n_lanes == 1:
        for vi in mine:
            one_view(vi, 0)
    else:
        lanes = lane_streams(dev, n_lanes)
        for st in lanes:
            st.wait_stream(cur)  # parameters
        if host_threads:
            # one host thread per stream: the native calls release the GIL, so one view's host wait and
            # kernel launches do not hold up the other streams' launches
            def drive(lane: int):
                with torch.cuda.stream(lanes[lane]):
                    for vi in mine[lane::n_lanes]:
                        one_view(vi, lane)

            pool = lane_pool(dev, n_lanes)
            for f in [pool.submit(drive, lane) for lane in range(n_lanes)]:
                f.result()
        else:
            for j, vi in enumerate(mine):
                with torch.cuda.stream(lanes[j % n_lanes]):
                    one_view(vi, j % n_lanes)
        for st in lanes:
            cur.wait_stream(st)
        cur.wait_event(zeroed)  # (a rank without views still hands a zeroed bucket to the collective)
        for _, radii, m2 in visible:  # allocated on a lane stream, handed to the caller's stream
            radii.record_stream(cur)
            if m2 is not None:
                m2.record_stream(cur)
    loss_sum = losses[0]
    for extra in losses[1:]:
        loss_sum = loss_sum + extra
    if world > 1 and allreduce:
        import torch.distributed as dist

        # ONE collective per step: the loss rides in the word behind the gradient bucket
        params.loss_slot.copy_(loss_sum.reshape(1))
        dist.all_reduce(params.reduce_buffer(), op=dist.ReduceOp.SUM, group=group)
        loss_sum = params.loss_slot[0].clone()
    return {"loss": loss_sum, "views": mine, "radii": [(vi, r) for vi, r, _ in visible],
            "means2D_grad": [(vi, m2) for vi, _, m2 in visible] if keep_means2D_grad else None,
            "densify": stats}


class GraphedStep:
    """The view-sharded step with the per-view work captured in CUDA graphs (SURVEY.md §8f N1).

    One graph per lane stream holds a whole view: DEFERRED forward (no host wait: buffer capacities from the
    high-water marks of the shape, brs_fwd_options) -> `loss_fn(color, depth, target)` -> backward adding the
    parameter gradients into the bucket.  A step then costs the host one small copy (the view's camera into the
    lane's static camera block) and one graph launch per view instead of ~30 kernel launches and a dozen Python
    dispatches, which is what bounds the un-graphed step once the kernels are fast (profiles/).  Results are
    identical to `view_sharded_step`.

    Capacity overflows of any view are OR-ed into one device word; it rides through the step's all-reduce as a
    count, so that every rank learns whether SOME rank overflowed and all of them repeat the step un-graphed
    (exact sizes, marks raised) and re-capture.  All cameras must share resolution and field of view.

    When `params.densify` is set, every view (captured or in the un-graphed fallback) adds its densification
    statistics there, and `res["densify"]` returns them as in `view_sharded_step`."""

    def __init__(self, params: GaussianParams, cameras: Sequence[Camera], bg: torch.Tensor, rasterizer_cls,
                 loss_fn: Callable[[torch.Tensor, torch.Tensor, Optional[torch.Tensor]], torch.Tensor],
                 rank: int = 0, world: int = 1, group=None, streams: int = 4, targets: Optional[torch.Tensor] = None):
        if not getattr(rasterizer_cls, "supports_deferred", False) or not getattr(rasterizer_cls, "supports_grad_sink", False):
            raise Exception("GraphedStep needs the native rasterizer (deferred forward + in-kernel gradient accumulation)")
        if params.densify is not None and not getattr(rasterizer_cls, "supports_densify_stats", False):
            raise Exception("GraphedStep: this rasterizer has no densification statistics")
        self.params, self.bg, self.rasterizer_cls, self.loss_fn = params, bg, rasterizer_cls, loss_fn
        self.rank, self.world, self.group = rank, world, group
        self.cameras = list(cameras)
        c0 = self.cameras[0]
        for c in self.cameras:
            if (c.image_width, c.image_height, c.tanfovx, c.tanfovy) != (c0.image_width, c0.image_height, c0.tanfovx, c0.tanfovy):
                raise Exception("GraphedStep: all cameras must share resolution and field of view")
        self.mine = shard_views(len(self.cameras), rank, world)
        self.dev = params.flat.device
        self.n_lanes = max(1, min(streams, len(self.mine)))
        self.cams_dev = torch.stack([torch.cat([c.viewmatrix.flatten(), c.projmatrix.flatten(), c.campos.flatten()])
                                     for c in self.cameras]).to(self.dev).contiguous()
        self.targets = targets
        self.overflow = torch.zeros(1, dtype=torch.int32, device=self.dev)
        self.host_flag = torch.zeros(1, dtype=torch.float32).pin_memory()
        self.lanes = None
        self.replays = 0
        self.fallbacks = 0

    # -- one view on the current stream, reading the lane's static camera block ------------------------------
    def _one_view(self, lane):
        c0, p = self.cameras[0], self.params
        settings = GaussianRasterizationSettings(
            image_height=c0.image_height, image_width=c0.image_width, tanfovx=c0.tanfovx, tanfovy=c0.tanfovy, bg=self.bg,
            scale_modifier=1.0, viewmatrix=lane["cam"][0:16].view(4, 4), projmatrix=lane["cam"][16:32].view(4, 4),
            sh_degree=p.sh_degree, campos=lane["cam"][32:35], prefiltered=False, debug=False)
        extra = {} if p.densify is None else {"densify_stats": p.densify}
        rast = self.rasterizer_cls(settings, grad_sink=p.grads(), deferred_overflow=self.overflow, **extra)
        means2D = p.zero_means2D().detach().requires_grad_(True)
        color, radii, depth = rast(means3D=p.tensors["means3D"], means2D=means2D, opacities=p.tensors["opacities"],
                                   shs=p.get("shs"), colors_precomp=p.get("colors_precomp"), scales=p.tensors["scales"],
                                   rotations=p.tensors["rotations"], cov3D_precomp=None)
        loss = self.loss_fn(color, depth, lane["target"])
        loss.backward()
        lane["loss"] += loss.detach()

    def _capture(self):
        streams = lane_streams(self.dev, self.n_lanes)
        cur = torch.cuda.current_stream(self.dev)
        keep = self.params.reduce_buffer().clone()  # the warm-up views below really run and add into the bucket
        self.lanes = []
        for li, st in enumerate(streams):
            lane = {"stream": st, "cam": self.cams_dev[self.mine[li % len(self.mine)]].clone(),
                    "target": None if self.targets is None else self.targets[self.mine[0]].clone(),
                    "loss": torch.zeros((), dtype=torch.float32, device=self.dev)}
            st.wait_stream(cur)
            with torch.cuda.stream(st):
                self._one_view(lane)  # warm-up outside the capture (allocator, autograd, lazy initialisations)
            st.synchronize()
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph, stream=st, capture_error_mode="thread_local"):
                self._one_view(lane)
            lane["graph"] = graph
            self.lanes.append(lane)
        torch.cuda.synchronize(self.dev)
        self.params.reduce_buffer().copy_(keep)

    def _plain(self):
        loss3 = lambda color, depth, vi: self.loss_fn(color, depth, None if self.targets is None else self.targets[vi])
        return view_sharded_step(self.params, self.cameras, self.bg, self.rasterizer_cls, loss3, rank=self.rank,
                                 world=self.world, group=self.group, streams=self.n_lanes)

    def __call__(self) -> Dict[str, object]:
        if self.lanes is None:
            res = self._plain()  # seeds the high-water marks of this shape with every view of this rank
            self._capture()
            return res
        p, dev = self.params, self.dev
        cur = torch.cuda.current_stream(dev)
        p.zero_grad()
        self.overflow.zero_()
        for lane in self.lanes:
            lane["stream"].wait_stream(cur)
            with torch.cuda.stream(lane["stream"]):
                lane["loss"].zero_()
        for j, vi in enumerate(self.mine):
            lane = self.lanes[j % self.n_lanes]
            with torch.cuda.stream(lane["stream"]):
                lane["cam"].copy_(self.cams_dev[vi], non_blocking=True)
                if self.targets is not None:
                    lane["target"].copy_(self.targets[vi], non_blocking=True)
                lane["graph"].replay()
        self.replays += len(self.mine)
        for lane in self.lanes:
            cur.wait_stream(lane["stream"])
        loss_sum = self.lanes[0]["loss"]
        for lane in self.lanes[1:]:
            loss_sum = loss_sum + lane["loss"]
        p.loss_slot.copy_(loss_sum.reshape(1))
        p.flag_slot.copy_((self.overflow != 0).to(torch.float32))
        if self.world > 1:
            import torch.distributed as dist

            dist.all_reduce(p.reduce_buffer(), op=dist.ReduceOp.SUM, group=self.group)
        self.host_flag.copy_(p.flag_slot, non_blocking=True)
        cur.synchronize()  # the step's one host wait: did any rank overflow a captured capacity?
        if float(self.host_flag[0]) != 0.0:
            self.fallbacks += 1
            res = self._plain()
            self._capture()
            return res
        return {"loss": p.loss_slot[0].clone(), "views": self.mine, "radii": None, "means2D_grad": None,
                "densify": p.densify}


_ZERO_STREAMS = {}


def _zero_stream(dev: torch.device):
    key = dev.index if dev.index is not None else torch.cuda.current_device()
    if key not in _ZERO_STREAMS:
        _ZERO_STREAMS[key] = torch.cuda.Stream(device=dev)
    return _ZERO_STREAMS[key]


def _slice_bounds(numel: int, rank: int, world: int):
    """Contiguous 1/world slice of a flat buffer owned by `rank` (last slice takes the remainder)."""
    per = (numel + world - 1) // world
    lo = min(numel, rank * per)
    return lo, min(numel, lo + per)


def upload_params(params: GaussianParams, host_flat: torch.Tensor, rank: int = 0, world: int = 1, group=None) -> int:
    """Host -> device refresh of the replicated parameter buffer for steps whose parameters live on the
    host (e.g. a host-side optimizer).  With N ranks every rank copies only ITS 1/N slice over its own
    PCIe link and the slices are exchanged over NVLink (all-gather), so the host traffic of the whole
    job is one copy of the parameters instead of N.  Returns the bytes this rank copied from the host."""
    n = params.flat.numel()
    with torch.no_grad():
        if world == 1:
            params.flat.copy_(host_flat, non_blocking=True)
            return n * 4
        import torch.distributed as dist

        lo, hi = _slice_bounds(n, rank, world)
        params.flat[lo:hi].copy_(host_flat[lo:hi], non_blocking=True)
        if n % world == 0:
            mine = params.flat[lo:hi]  # NCCL gathers in place (input = this rank's slot of the output)
            dist.all_gather_into_tensor(params.flat, mine if mine.is_cuda else mine.clone(), group=group)
        else:
            for r in range(world):
                a, b = _slice_bounds(n, r, world)
                if b > a:
                    dist.broadcast(params.flat[a:b], src=r, group=group)
        return (hi - lo) * 4


def download_grads(params: GaussianParams, host_grads: torch.Tensor, rank: int = 0, world: int = 1) -> int:
    """Device -> host copy of the (already all-reduced) gradient bucket: rank r writes slice r of the
    host buffer, so the N ranks of a node fill one host gradient with N parallel PCIe copies.
    Returns the bytes this rank copied."""
    lo, hi = _slice_bounds(params.grad_bucket.numel(), rank, world)
    host_grads[lo:hi].copy_(params.grad_bucket[lo:hi], non_blocking=True)
    return (hi - lo) * 4

