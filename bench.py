#!/usr/bin/env python
"""Benchmark of the hot path: the view-sharded training step of BASELINE.json.

    python bench.py --gpus N --steps K --warmup W [--impl ours|reference|cpu] [--dump-outputs DIR]

A "step" = forward + loss + backward of EVERY view of a 64-view 1080p batch over 1M SH3 Gaussians
(config E of BASELINE.md; every view is config C), sharded round-robin over the N ranks, plus ONE
NCCL sum-allreduce of the flat gradient bucket when N > 1.  Total work is fixed as N grows
("scaling": "strong").  One JSON line is printed by rank 0:

  value          views/s with Gaussians, cameras and loss weights resident in HBM (CUDA events, max over ranks)
  e2e            same metric with, inside the timed region of every step, the host->device copy of the
                 step's inputs (all Gaussian parameters + cameras, from pinned host memory) and the
                 device->host read of the step's result (reduced gradient bucket + loss)
  roofline       dominant kernel (blend backward, FP32-pipe bound): algorithmic flops / CUDA-event time,
                 against a live FFMA micro-benchmark; `stages` gives every stage against its own bound
  cpu_baseline   the CPU oracle port (oracle/rasterizer_oracle.c) on a bounded sample, N=1 rank 0 only

--dump-outputs DIR writes what the last timed step returned (its loss and parameter gradients, for a fixed
sample of Gaussians) as DIR/<name>.npy; the inputs are seeded, so two builds can be compared output for output.

--impl reference runs the reference's OWN CUDA rasterizer (oracle/_ref, built unmodified from
/root/reference) through the same Python wrapper and the same step loop on one GPU: the reference has
no CPU implementation of this path, its only implementation is CUDA, and BASELINE.json asks for the
comparison "next to the reference CUDA rasterizer on one B200".  --impl cpu times the CPU port.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

METRIC = "views/sec, fwd+bwd @1M Gaussians 1080p SH3 (64-view training step)"
UNIT = "views/s"
CONFIG_NAME = "E"
N_VIEWS = 64


# DRAM traffic (dram__bytes_read.sum + dram__bytes_write.sum) per launch at config C, read from the
# `ncu --set full` captures summarised under profiles/ (refreshed whenever a blend kernel changes).
NCU_TRAFFIC = {
    "blend_bwd": {"bytes": int((112.7 + 8.306) * 1e6), "source": "profiles/r02_ncu_full.md"},
    "blend_fwd": {"bytes": int((76.57 + 23.49) * 1e6), "source": "profiles/r02_ncu_full.md"},
}


# ---- clocks --------------------------------------------------------------------------------------

class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.index)], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm = sorted(int(float(r[0])) for r in self.rows if r and r[0].replace(".", "").isdigit())
        mx = [int(float(r[1])) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 3 + i and r[3 + i].lower().startswith("active") for r in self.rows)]
        pw = [float(r[2]) for r in self.rows if len(r) > 2 and r[2].replace(".", "").isdigit()]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm), "power_w_max": max(pw) if pw else None}


# ---- helpers -------------------------------------------------------------------------------------

def bind_to_gpu_numa_node(index: int):
    """Best effort: run this rank on the CPUs of the NUMA node its GPU hangs off, BEFORE any pinned host buffer is
    allocated (first touch then places the staging buffers of the end-to-end leg next to the GPU's PCIe root)."""
    try:
        bus = subprocess.run(["nvidia-smi", "--query-gpu=pci.bus_id", "--format=csv,noheader", "-i", str(index)],
                             capture_output=True, text=True, timeout=20).stdout.strip().lower()
        bus = bus[-12:] if len(bus) > 12 else bus  # 00000000:1B:00.0 -> 0000:1b:00.0
        node = int(open(f"/sys/bus/pci/devices/{bus}/numa_node").read().strip())
        if node < 0:
            return {"numa_node": None, "note": "the platform reports no NUMA node for this GPU"}
        cpus = []
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.extend(range(int(lo), int(hi or lo) + 1))
        allowed = sorted(set(cpus) & os.sched_getaffinity(0))
        if not allowed:
            return {"numa_node": node, "note": "no allowed CPU on that node"}
        os.sched_setaffinity(0, allowed)
        return {"numa_node": node, "cpus": len(allowed)}
    except Exception as e:  # pragma: no cover
        return {"numa_node": None, "note": str(e)[:120]}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "MEASURED_PEAKS.json (driver-measured copy bandwidth)"
    return 6650.0, "fallback of B200_PROFILING.md (MEASURED_PEAKS.json absent)"


DUMP_GAUSSIANS = 65536  # Gaussians whose gradients --dump-outputs writes (15.5 MB at SH degree 3; the bucket is 236 MB)


def dump_outputs(out_dir, params, host_loss):
    """--dump-outputs: the loss of the last timed step and the gradient of every parameter tensor (the all-reduced
    bucket the step returns) for the same seeded sample of Gaussians in every run, as float32 .npy files."""
    import numpy as np

    os.makedirs(out_dir, exist_ok=True)
    idx = torch.randperm(params.P, generator=torch.Generator().manual_seed(0))[:DUMP_GAUSSIANS].sort().values
    np.save(os.path.join(out_dir, "loss.npy"), host_loss.numpy().astype(np.float32))
    np.save(os.path.join(out_dir, "gaussian_index.npy"), idx.numpy().astype(np.float64))
    rows = idx.to(params.flat.device)
    for n in params.names:
        np.save(os.path.join(out_dir, f"grad_{n}.npy"), params.tensors[n].grad.index_select(0, rows).cpu().numpy().astype(np.float32))


def get_api():
    import bloomscene_b200

    return bloomscene_b200._api


def make_config(cfg, views, world):
    """The workload description both arms print (identical for the product and the reference arm)."""
    W, H = cfg["W"], cfg["H"]
    return {"workload": f"config E of BASELINE.md: {cfg['P']} Gaussians SH degree 3 (M=16), {W}x{H}, {views}-view "
                        f"orbit batch, fwd+loss+bwd per view, view-sharded over {world} rank(s)"
                        + (" + NCCL allreduce of the 236 MB gradient bucket" if world > 1 else ""),
            "P": cfg["P"], "views": views, "resolution": [W, H], "sh_degree": 3,
            "l2": "inputs larger than L2 (236 MB of parameters re-read per view, ~0.5 GB working set vs 126 MB L2)",
            "parallelism": f"view-sharded dp{world}"}


def kernel_census(fn):
    """Names and counts of the CUDA kernels `fn()` launches (torch profiler / CUPTI, outside any timed region)."""
    try:
        from torch.profiler import ProfilerActivity, profile

        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            fn()
            torch.cuda.synchronize()
        names = {}
        for ev in prof.events():
            if getattr(ev, "device_type", None) is not None and "cuda" in str(ev.device_type).lower():
                n = ev.name.split("(")[0].split("<")[0]
                if n.lower().startswith("memcpy") or n.lower().startswith("memset"):
                    continue
                names[n] = names.get(n, 0) + 1
        return names
    except Exception as e:  # pragma: no cover
        return {"unavailable": str(e)[:200]}


def reference_arm(a):
    """bench.py --impl reference: the reference's OWN rasterizer through the reference's OWN Python
    package and stock code path — GaussianRasterizationSettings / GaussianRasterizer exactly as
    gaussian_renderer/__init__.py:211-262 uses them, one view after the other on the current stream,
    plain autograd accumulation into the parameters' .grad.  This function imports nothing of the
    product: no bloomscene_b200 module, no libbloomrast.so, no product kernel.  The reference has no
    CPU implementation of this path (its only implementation is CUDA), so the arm runs on ONE B200
    whatever --gpus says; ranks other than 0 exit without work."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import build_ref
    from workload import synthetic
    from workload.params import GaussianParams

    ref = build_ref.load_reference_package()
    if ref is None:
        print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref (reference CUDA rasterizer + its Python package) is not "
                          "built; it needs /root/reference at build time"}))
        return
    assert "bloomscene_b200" not in sys.modules, "the reference arm must not load the product"
    assert torch.cuda.is_available(), "the reference's only implementation of this path is CUDA"
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    cfg = synthetic.CONFIGS[CONFIG_NAME]
    W, H = cfg["W"], cfg["H"]
    config = make_config(cfg, a.views, 1)

    scene_cpu = synthetic.config_scene(CONFIG_NAME)
    cams_cpu = synthetic.config_cameras(CONFIG_NAME, a.views)
    Wc_cpu, Wd_cpu = synthetic.loss_weights(W, H)
    params = GaussianParams(scene_cpu.to(dev))
    cams = [c.to(dev) for c in cams_cpu]
    Wc_flat, Wd_flat = Wc_cpu.to(dev).reshape(-1), Wd_cpu.to(dev).reshape(-1)
    bg = torch.zeros(3, device=dev)
    t = params.tensors

    def one_view(cam):
        settings = synthetic.raster_settings(cam, params.sh_degree, bg, ref.GaussianRasterizationSettings)
        rast = ref.GaussianRasterizer(raster_settings=settings)
        means2D = torch.zeros_like(t["means3D"], requires_grad=True)  # gaussian_renderer/__init__.py:224-229
        color, radii, depth = rast(means3D=t["means3D"], means2D=means2D, opacities=t["opacities"], shs=t["shs"],
                                   colors_precomp=None, scales=t["scales"], rotations=t["rotations"], cov3D_precomp=None)
        loss = torch.dot(color.reshape(-1), Wc_flat) + torch.dot(depth.reshape(-1), Wd_flat)
        loss.backward()
        return loss.detach()

    def step():
        params.zero_grad()
        total = torch.zeros((), device=dev)
        for cam in cams:
            total += one_view(cam)
        return total

    host_params = torch.empty_like(params.flat, device="cpu").pin_memory()
    host_params.copy_(params.flat)
    host_grads = torch.empty_like(params.flat, device="cpu").pin_memory()
    host_loss = torch.zeros(1).pin_memory()
    cam_host = torch.stack([torch.cat([c.viewmatrix.flatten(), c.projmatrix.flatten(), c.campos]) for c in cams_cpu]).pin_memory()
    cam_dev = torch.empty_like(cam_host, device=dev)

    def step_e2e():
        with torch.no_grad():
            params.flat.copy_(host_params, non_blocking=True)
            cam_dev.copy_(cam_host, non_blocking=True)
        total = step()
        host_grads.copy_(params.grad_bucket, non_blocking=True)
        host_loss.copy_(total.reshape(1), non_blocking=True)

    def timed(fn, steps):
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / steps

    for _ in range(max(a.warmup, 3)):
        step()
    sampler = ClockSampler(local_rank)
    sampler.start()
    ms_step = timed(step, a.steps)
    step_e2e()
    ms_e2e = timed(step_e2e, a.steps)
    clocks = sampler.stop()
    census = kernel_census(lambda: one_view(cams[0]))
    per_view = sum(v for v in census.values() if isinstance(v, int))
    assert "bloomscene_b200" not in sys.modules
    out = {"impl": "reference", "metric": METRIC, "value": a.views / (ms_step * 1e-3), "unit": UNIT, "n_gpus": 1,
           "steps": a.steps, "warmup": max(a.warmup, 3), "ms_per_step": ms_step, "ms_per_view": ms_step / a.views,
           "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
           "config": config, "clocks": clocks,
           "e2e": {"value": a.views / (ms_e2e * 1e-3), "unit": UNIT, "h2d_bytes_per_step": host_params.numel() * 4 + cam_host.numel() * 4,
                   "d2h_bytes_per_step": host_grads.numel() * 4 + 4, "ms_per_step": ms_e2e},
           "loss": float(host_loss.item()),
           "reference_kind": "the reference's own CUDA rasterizer (oracle/_ref/_ref_C.so: unmodified sources built for sm_100a) "
                             "through the reference's own Python package (oracle/_ref/pkg) on one B200; the reference has no CPU "
                             "implementation of this path",
           "cpu_baseline": {"value": a.views / (ms_step * 1e-3), "unit": UNIT, "cores": os.cpu_count(), "kind": "reference",
                            "sample": f"all {a.views} views per step on one B200 (reference CUDA, not CPU)"},
           "gpu_launches": per_view * a.views * a.steps, "kernels_per_view": census,
           "product_modules_loaded": sorted(m for m in sys.modules if m.startswith("bloomscene_b200"))}
    print(json.dumps(out))


def stage_model(P, V, R, R1, M, npix, ntile, E, C, Eb):
    """Algorithmic bytes / flops per view and stage (SURVEY.md §8d; binning stages as built, DESIGN.md §3).
    R1 = (supertile, Gaussian) instances, the only thing the coarse level sorts."""
    return {
        "preprocess": ("hbm", 52 * P + (12 * M + 67) * V),
        # histogram reads P keys; pass 1 reads P keys, writes V pairs; pass 2 moves V pairs; pass 3 reads V pairs, writes V ids
        "depth_sort": ("hbm", 8 * P + (8 + 16 + 12) * V),
        "coarse_emit": ("hbm", 12 * V + 8 * R1),  # order + rect in, (supertile, id) instances out
        "coarse_sort": ("hbm", (8 + 4) * R1),  # one pass: pairs in, ids out (digit totals come from the emission's histogram)
        "fine_bin": ("hbm", 2 * (4 + 8) * R1 + 4 * R + 16 * ntile),  # count + scatter passes read id + rect; ids written once
        "blend_fwd": ("fp32", 21 * E + 16 * C),
        "blend_bwd": ("fp32", 21 * Eb + 70 * C),
        "preprocess_bwd": ("hbm", 4 * P + 48 * P + (171 + 24 * M) * V),
    }


def run_cpu_sample(scene_cpu, cams_cpu, Wc_cpu, n_views):
    """The oracle port on `n_views` views with all host threads; returns (views/s, threads)."""
    from oracle import oracle as cpu_oracle

    t0 = time.time()
    threads = 1
    for cam in cams_cpu[:n_views]:
        o = cpu_oracle.run_scene(scene_cpu, cam, torch.zeros(3), dL_dcolor=Wc_cpu)
        threads = o["oracle"].threads
    dt = time.time() - t0
    return n_views / dt, threads, dt


# ---- main ----------------------------------------------------------------------------------------

def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5, help="timed steps per leg (at least 1)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "cpu"])
    ap.add_argument("--views", type=int, default=N_VIEWS)
    ap.add_argument("--cpu-views", type=int, default=3, help="views of the bounded CPU-baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--streams", type=int, default=0, help="CUDA streams the views of a rank are dealt onto (0: 4, or one per view when a rank has at most 8)")
    ap.add_argument("--host-threads", type=int, default=0, help="1: one host thread per stream (ours only)")
    ap.add_argument("--graphs", type=int, default=-1, help="1: per-view work replayed from CUDA graphs (GraphedStep); 0: launched kernel by kernel; "
                    "-1: graphs when a rank has at most 16 views (the host's launch rate matters when a step is short)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's loss and a fixed sample of its "
                    "gradients to DIR/<name>.npy (ours only)")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    a.warmup = max(a.warmup, 3) if a.impl != "cpu" else a.warmup

    if a.impl == "reference":
        return reference_arm(a)

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    from workload import synthetic

    cfg = synthetic.CONFIGS[CONFIG_NAME]
    W, H = cfg["W"], cfg["H"]
    config = make_config(cfg, a.views, world)

    # ---- CPU port as its own arm -------------------------------------------------------------------
    if a.impl == "cpu":
        if rank != 0:
            return
        scene_cpu = synthetic.config_scene(CONFIG_NAME)
        cams_cpu = synthetic.config_cameras(CONFIG_NAME, a.views)
        Wc_cpu, _ = synthetic.loss_weights(W, H)
        n = max(1, min(a.cpu_views, a.views))
        vps, threads, dt = run_cpu_sample(scene_cpu, cams_cpu, Wc_cpu, n)
        sample = f"{n} of {a.views} views of the step (forward+backward each), {dt:.1f} s on {threads} host threads"
        print(json.dumps({"impl": "cpu", "metric": METRIC, "value": vps, "unit": UNIT, "n_gpus": 0, "steps": 1, "warmup": 0,
                          "ms_per_step": 1e3 * a.views / vps, "higher_is_better": True, "scaling": "strong",
                          "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config,
                          "cpu_baseline": {"value": vps, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
                          "e2e": {"value": vps, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                          "gpu_launches": 0}))
        return

    world_eff, rank_eff = world, rank
    views_per_rank = len(range(rank, a.views, world))
    if a.streams <= 0:
        a.streams = 4

    assert torch.cuda.is_available(), "bench.py needs a CUDA device (there is no CPU fallback for the product path)"
    numa = bind_to_gpu_numa_node(local_rank) if world > 1 else None
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world_eff > 1:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=dev)

    api = get_api()

    from bloomscene_b200.multiview import GraphedStep, download_grads, upload_params, view_sharded_step
    from workload.params import GaussianParams

    scene_cpu = synthetic.config_scene(CONFIG_NAME)
    cams_cpu = synthetic.config_cameras(CONFIG_NAME, a.views)
    Wc_cpu, Wd_cpu = synthetic.loss_weights(W, H)
    scene = scene_cpu.to(dev)
    cams = [c.to(dev) for c in cams_cpu]
    Wc, Wd = Wc_cpu.to(dev), Wd_cpu.to(dev)
    bg = torch.zeros(3, device=dev)
    params = GaussianParams(scene)
    del scene
    # loss = <color, Wc> + <depth, Wd> (SURVEY.md 8d), written as two dot products: one reduction kernel
    # forward and one scaling kernel backward per term, for both arms alike
    Wc_flat, Wd_flat = Wc.reshape(-1), Wd.reshape(-1)
    loss_fn = lambda color, depth, vi: torch.dot(color.reshape(-1), Wc_flat) + torch.dot(depth.reshape(-1), Wd_flat)

    # pinned host mirrors for the end-to-end leg
    host_params = torch.empty_like(params.flat, device="cpu").pin_memory()
    host_params.copy_(params.flat)
    host_grads = torch.empty_like(params.flat, device="cpu").pin_memory()
    host_loss = torch.zeros(1).pin_memory()
    cam_host = torch.stack([torch.cat([c.viewmatrix.flatten(), c.projmatrix.flatten(), c.campos]) for c in cams_cpu]).pin_memory()
    cam_dev = torch.empty_like(cam_host, device=dev)

    def barrier():
        if world_eff > 1:
            import torch.distributed as dist

            dist.barrier()
        torch.cuda.synchronize()

    def plain_step():
        return view_sharded_step(params, cams, bg, api.GaussianRasterizer, loss_fn, rank=rank_eff, world=world_eff,
                                 streams=a.streams, host_threads=bool(a.host_threads))

    # kernels one view launches (counted on a plain step; a graphed step replays exactly these)
    api._C.launch_count(True)
    plain_step()
    torch.cuda.synchronize()
    kernels_per_view = api._C.launch_count(False) // max(views_per_rank, 1)
    graphed = None
    if a.graphs < 0:
        a.graphs = 1 if views_per_rank <= 16 else 0
    if a.graphs:
        graphed = GraphedStep(params, cams, bg, api.GaussianRasterizer, lambda c, d, t: loss_fn(c, d, 0), rank=rank_eff,
                              world=world_eff, streams=a.streams)
        graphed()  # first call: plain step + capture
    step = graphed if graphed is not None else plain_step

    moved = {"h2d": 0, "d2h": 0}

    copy_stream = torch.cuda.Stream(device=dev)
    grads_on_host = torch.cuda.Event()
    grads_on_host.record()

    marks = {}

    def step_e2e():
        # every rank moves its 1/N slice of the parameters / gradients over its own PCIe link; the slices
        # travel between GPUs over NVLink (all-gather in upload_params, the step's allreduce before download).
        # The device->host copy of a step's gradients runs on its own stream, so the next step's host->device
        # copy of the parameters overlaps it (PCIe is full duplex); the bucket is not touched before it has left.
        main = torch.cuda.current_stream(dev)
        ev = {k: torch.cuda.Event(enable_timing=True) for k in ("t0", "up", "step", "down")}
        ev["t0"].record()
        moved["h2d"] = upload_params(params, host_params, rank_eff, world_eff) + cam_host.numel() * 4
        with torch.no_grad():
            cam_dev.copy_(cam_host, non_blocking=True)
        main.wait_event(grads_on_host)
        ev["up"].record()
        res = step()
        ev["step"].record()
        copy_stream.wait_stream(main)
        with torch.cuda.stream(copy_stream):
            moved["d2h"] = download_grads(params, host_grads, rank_eff, world_eff) + 4
            host_loss.copy_(res["loss"].reshape(1), non_blocking=True)
            grads_on_host.record()
            ev["down"].record()
        marks.update(ev)
        return res

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        torch.cuda.current_stream(dev).wait_event(grads_on_host)  # the last step's device->host copy is inside the timed region
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world_eff > 1:
            import torch.distributed as dist

            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return ms.item() / steps

    for _ in range(a.warmup):
        step()
    count_launches = True
    sampler = ClockSampler(local_rank)
    if rank_eff == 0:
        sampler.start()
    ms_step = timed(step, a.steps)
    launches = kernels_per_view * views_per_rank * a.steps
    for _ in range(1):
        step_e2e()
    ms_e2e = timed(step_e2e, a.steps)
    clocks = sampler.stop() if rank_eff == 0 else None
    loss_value = float(host_loss.item())
    torch.cuda.synchronize()
    if a.dump_outputs and rank_eff == 0:
        dump_outputs(a.dump_outputs, params, host_loss)  # before anything below reuses the gradient bucket
    e2e_breakdown = {"upload_h2d_allgather_and_wait_for_previous_d2h_ms": round(marks["t0"].elapsed_time(marks["up"]), 4),
                     "step_ms": round(marks["up"].elapsed_time(marks["step"]), 4),
                     "download_d2h_ms": round(marks["step"].elapsed_time(marks["down"]), 4),
                     "note": "rank 0, last timed step; the download of step s overlaps the upload of step s+1"}

    # ---- the step's one collective on its own (outside the timed region) -------------------------------
    collective = None
    if world_eff > 1:
        import torch.distributed as dist

        buf = params.reduce_buffer()
        for _ in range(2):
            dist.all_reduce(buf)
        barrier()
        c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        c0.record()
        for _ in range(5):
            dist.all_reduce(buf)
        c1.record()
        torch.cuda.synchronize()
        ms = torch.tensor([c0.elapsed_time(c1) / 5], device=dev)
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        nbytes = buf.numel() * 4
        collective = {"op": "ncclAllReduce sum fp32 (gradient bucket + loss word)", "bytes": nbytes, "ms": round(ms.item(), 4),
                      "busbw_GBps": round(2 * (world_eff - 1) / world_eff * nbytes / (ms.item() * 1e-3) / 1e9, 1),
                      "share_of_step": round(ms.item() / ms_step, 4)}

    # ---- gradient parity of the step (SURVEY.md 8e), outside the timed region -----------------------
    # The bucket the step produced (views dealt over ranks and streams, in-kernel accumulation, NCCL
    # allreduce when N > 1) against the same 64-view sum computed on rank 0 alone the plain way: one
    # stream, fresh gradient tensors per view, autograd's own accumulation.  Bar: relative L2 <= 1e-4.
    step()
    torch.cuda.synchronize()
    grad_parity = None
    if rank_eff == 0:
        got = params.grad_bucket.clone()

        class PlainRasterizer(api.GaussianRasterizer):
            supports_grad_sink = False

        view_sharded_step(params, cams, bg, PlainRasterizer, loss_fn, rank=0, world=1, allreduce=False, streams=1)
        torch.cuda.synchronize()
        want = params.grad_bucket
        grad_parity = {"rel_l2": float((got.double() - want.double()).norm() / want.double().norm())}
        off = 0
        for n in params.names:
            sz = params.tensors[n].numel()
            g, w = got[off:off + sz].double(), want[off:off + sz].double()
            grad_parity[n] = float((g - w).norm() / w.norm())
            off += sz
        del got
    barrier()

    if count_launches and world_eff > 1:
        import torch.distributed as dist

        t = torch.tensor([launches], device=dev, dtype=torch.int64)
        dist.all_reduce(t)
        launches = int(t.item())

    # whole-job host traffic per step = sum over ranks of what each rank copied
    h2d, d2h = moved["h2d"], moved["d2h"]
    if world_eff > 1:
        import torch.distributed as dist

        t = torch.tensor([h2d, d2h], device=dev, dtype=torch.int64)
        dist.all_reduce(t)
        h2d, d2h = int(t[0].item()), int(t[1].item())
    out = {
        "metric": METRIC, "value": a.views / (ms_step * 1e-3), "unit": UNIT, "n_gpus": world_eff, "steps": a.steps,
        "warmup": a.warmup, "ms_per_step": ms_step, "ms_per_view": ms_step / a.views,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": config, "clocks": clocks,
        "e2e": {"value": a.views / (ms_e2e * 1e-3), "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "ms_per_step": ms_e2e, "breakdown": e2e_breakdown,
                "what": "per step: all Gaussian parameters + cameras pinned host->device, then the view loop through "
                        "GaussianRasterizer / autograd, then gradient bucket + loss device->pinned host; with N ranks "
                        "each rank copies its 1/N slice of the parameters / the reduced gradients over its own PCIe "
                        "link (slices exchanged over NVLink), bytes are whole-job totals; a step's device->host copy runs on a "
                        "copy stream and overlaps the next step's host->device copy (both inside the timed region)"},
        "loss": loss_value,
        "grad_parity_rel_l2": None if grad_parity is None else grad_parity["rel_l2"],
        "grad_parity": {"bar": 1e-4, "per_parameter": grad_parity,
                        "what": "the step's (all-reduced) gradient bucket vs the same 64-view sum on rank 0 alone: one stream, "
                                "fresh per-view gradient tensors, autograd accumulation"},
    }
    out["gpu_launches"] = launches
    out["streams_per_rank"] = a.streams
    out["cuda_graphs"] = None if graphed is None else {"views_replayed": graphed.replays, "steps_repeated_ungraphed": graphed.fallbacks}
    out["kernels_per_view"] = kernels_per_view
    out["views_per_rank"] = views_per_rank
    out["collective"] = collective
    out["numa_binding"] = numa

    # ---- stage profile + roofline (ours, rank 0, outside the timed region) --------------------------
    if rank_eff == 0:
        from bloomscene_b200.profiling import profile_views

        prof = profile_views(api, params, cams, bg, Wc, rank_eff, world_eff, max_views=8)
        hbm_peak, hbm_src = measured_peaks()
        fp32_peak = api._C.probe_fp32_tflops()
        st = prof["stats"]
        model = stage_model(cfg["P"], st["V"], st["R"], st["R1"], 16, W * H, ((W + 15) // 16) * ((H + 15) // 16), st["E"], st["C"], st["Eb"])
        stages = {}
        t_roof = 0.0
        for name, (bound, work) in model.items():
            ms = prof["ms"][name]
            if bound == "hbm":
                ach, peak, unit = work / (ms * 1e-3) / 1e9, hbm_peak, "GB/s"
            else:
                ach, peak, unit = work / (ms * 1e-3) / 1e12, fp32_peak, "TFLOP/s"
            stages[name] = {"bound": bound, "ms": round(ms, 4), "work": int(work), "achieved": round(ach, 2),
                            "peak": round(peak, 2), "unit": unit, "frac": round(ach / peak, 4)}
            t_roof += (work / (peak * (1e9 if bound == "hbm" else 1e12))) * 1e3
        dom = max(stages, key=lambda k: stages[k]["ms"])
        d = stages[dom]
        # DRAM bytes of the dominant kernel per launch, from the committed `ncu --set full` capture
        traffic = NCU_TRAFFIC.get(dom, {}).get("bytes")
        # the same kernel against the HBM roof: algorithmic floor bytes of SURVEY.md 8(d) / measured time
        hbm_floor = {"blend_bwd": 4 * st["R"] + 72 * st["V"] + 20 * W * H, "blend_fwd": 4 * st["R"] + 40 * st["V"] + 24 * W * H}.get(dom)
        hbm_view = None
        if hbm_floor is not None:
            gbs = hbm_floor / (d["ms"] * 1e-3) / 1e9
            hbm_view = {"algorithmic_bytes": int(hbm_floor), "achieved": round(gbs, 1), "peak": hbm_peak, "unit": "GB/s",
                        "frac": round(gbs / hbm_peak, 4),
                        "note": "far below the HBM roof: the kernel is bound by FP32/ALU issue slots, not by memory"}
        out["roofline"] = {"kernel": dom, "bound": d["bound"], "achieved": d["achieved"], "peak": d["peak"], "unit": d["unit"],
                           "frac": d["frac"], "traffic": traffic, "traffic_source": NCU_TRAFFIC.get(dom, {}).get("source"),
                           "hbm_view": hbm_view,
                           "peak_source": ("live dependent-FFMA micro-benchmark brs_probe_fp32_tflops()" if d["bound"] == "fp32" else hbm_src),
                           "note": "the dominant kernel is FP32-pipe bound (no dense contraction on this path, tensor cores "
                                   "not applicable); algorithmic flops = 21*E_b + 70*C with E_b, C counted by brs_count_pairs",
                           "hbm_peak_GBps": hbm_peak, "hbm_peak_source": hbm_src, "fp32_peak_TFLOPs": round(fp32_peak, 2),
                           "pipeline_frac": round(t_roof / sum(s["ms"] for s in stages.values()), 4),
                           "pipeline_frac_serial": round(t_roof / sum(s["ms"] for s in stages.values()), 4),
                           "pipeline_frac_overlapped": round(t_roof / (ms_step / len(range(rank_eff, a.views, world_eff))), 4),
                           "pipeline_note": "stage times are measured with the views on ONE stream (serial sum); the step itself deals "
                                            "the views of a rank onto several streams, so its ms per view is below that sum "
                                            "(pipeline_frac_overlapped = roofline time / measured ms per view of this rank)",
                           "stages": stages, "per_view": st}

    # ---- CPU baseline (oracle port), N == 1 rank 0 only ----------------------------------------------
    if world_eff == 1 and rank_eff == 0 and not a.no_cpu_baseline:
        n = max(1, min(a.cpu_views, a.views))
        vps, threads, dt = run_cpu_sample(scene_cpu, cams_cpu, Wc_cpu, n)
        out["cpu_baseline"] = {"value": vps, "unit": UNIT, "cores": threads, "kind": "port",
                               "sample": f"{n} of the {a.views} views of one step (forward+backward each) in {dt:.1f} s, "
                                         f"oracle/rasterizer_oracle.c with OpenMP on {threads} host threads"}
    else:
        out["cpu_baseline"] = None

    if rank_eff == 0:
        print(json.dumps(out))
    if world_eff > 1:
        import torch.distributed as dist

        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
