"""Cost of the densification statistics in the training step (config E: 1 M Gaussians, SH3, 1920x1080, 64 views).

Three arms in one process, alternated for --rounds rounds (median reported), each timed over --steps steps:
  off    GraphedStep on GaussianParams(scene)                       (what bench.py's step computes)
  on     GraphedStep on GaussianParams(scene, densify_stats=True)   (statistics from the backward kernel),
         plus the caller adding the step's result into its own accumulators (two adds)
  torch  view_sharded_step(keep_means2D_grad=True) plus the reference's per-view torch statement
         (scene/gaussian_model.py:756-759): the only route to these numbers without the feature
The GPU's name, power limit and clocks are read in the same run.  Writes one JSON file (--out).

    python tools/bench_densify_stats.py --out profiles/densify_stats.json
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm,clocks.mem"
    try:
        out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"], capture_output=True,
                             text=True, timeout=30).stdout.strip()
        return dict(zip(q.split(","), [v.strip() for v in out.split(",")]))
    except Exception as e:  # noqa: BLE001
        return {"error": str(e)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--views", type=int, default=64)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--streams", type=int, default=4)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "densify_stats.json"))
    a = ap.parse_args()
    assert torch.cuda.is_available(), "this measurement needs a CUDA device"

    import bloomscene_b200
    from bloomscene_b200.multiview import GraphedStep, view_sharded_step
    from workload import synthetic
    from workload.params import GaussianParams

    api = bloomscene_b200._api
    dev = torch.device("cuda", 0)
    cfg = synthetic.CONFIGS["E"]
    W, H = cfg["W"], cfg["H"]
    scene = synthetic.config_scene("E").to(dev)
    cams = [c.to(dev) for c in synthetic.config_cameras("E", a.views)]
    Wc, Wd = [t.to(dev).reshape(-1) for t in synthetic.loss_weights(W, H)]
    bg = torch.zeros(3, device=dev)
    loss_fn = lambda color, depth, vi: torch.dot(color.reshape(-1), Wc) + torch.dot(depth.reshape(-1), Wd)
    loss3 = lambda c, d, t: loss_fn(c, d, 0)
    P = scene.P

    p_off = GaussianParams(scene)
    p_on = GaussianParams(scene, densify_stats=True)
    p_torch = GaussianParams(scene)
    del scene
    accum = {k: torch.zeros(P, device=dev) for k in ("on", "torch")}
    denom = {k: torch.zeros(P, device=dev) for k in ("on", "torch")}
    g_off = GraphedStep(p_off, cams, bg, api.GaussianRasterizer, loss3, streams=a.streams)
    g_on = GraphedStep(p_on, cams, bg, api.GaussianRasterizer, loss3, streams=a.streams)

    def step_on():
        res = g_on()
        accum["on"] += res["densify"]["grad_norm"]
        denom["on"] += res["densify"]["count"]

    def step_torch():
        res = view_sharded_step(p_torch, cams, bg, api.GaussianRasterizer, loss_fn, streams=a.streams,
                                keep_means2D_grad=True)
        m2 = dict(res["means2D_grad"])
        for vi, radii in res["radii"]:
            update_filter = radii > 0
            grad_norm = torch.norm(m2[vi][update_filter, :2], dim=-1)
            accum["torch"][update_filter] += grad_norm
            denom["torch"][update_filter] += 1

    arms = {"off": g_off, "on": step_on, "torch": step_torch}
    for fn in arms.values():  # warm-up: first GraphedStep call captures, every arm runs twice
        fn()
        fn()
    torch.cuda.synchronize()

    def timed(fn):
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(a.steps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / a.steps

    info_before = gpu_info()
    ms = {k: [] for k in arms}
    for _ in range(a.rounds):
        for k, fn in arms.items():
            ms[k].append(timed(fn))
    info_after = gpu_info()

    # the two routes compute the same statistics (same views, same number of calls each)
    for k in ("on", "torch"):
        accum[k].zero_()
        denom[k].zero_()
    step_on()
    step_torch()
    torch.cuda.synchronize()
    count_equal = bool(torch.equal(denom["on"], denom["torch"]))
    rel = float((accum["on"] - accum["torch"]).norm() / accum["torch"].norm())

    med = {k: statistics.median(v) for k, v in ms.items()}
    out = {
        "what": "config E training step (1 M Gaussians, SH3, 1920x1080, one process), densification statistics off / on "
                "(GraphedStep) / torch route (view_sharded_step keep_means2D_grad + per-view torch ops)",
        "views": a.views, "steps_per_round": a.steps, "rounds": a.rounds, "streams": a.streams,
        "gpu_before": info_before, "gpu_after": info_after,
        "ms_per_step": ms, "ms_per_step_median": med,
        "views_per_s_median": {k: a.views / (v * 1e-3) for k, v in med.items()},
        "ms_per_view_median": {k: v / a.views for k, v in med.items()},
        "on_vs_off_overhead_pct": 100.0 * (med["on"] / med["off"] - 1.0),
        "torch_vs_off_overhead_pct": 100.0 * (med["torch"] / med["off"] - 1.0),
        "fallbacks": {"off": g_off.fallbacks, "on": g_on.fallbacks},
        "stats_agree": {"count_equal": count_equal, "grad_norm_rel_l2": rel},
    }
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
