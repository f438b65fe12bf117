#!/usr/bin/env python
"""Forward-only render of views that each have their OWN Gaussians (BloomScene's render_video / render_set: every
frame culls anchors and generates its own neural Gaussians, reference bloomscene.py:174-219), in a config-B shape:

  * config B's 500 K band scene and its 120 rotate360 yaws at 512 x 512;
  * view j keeps a seeded subset of the rows (keep rate uniform in [0.6, 0.9]) with its own colors_precomp, and the
    views' rows are concatenated (about 45 M rows, 2.5 GB: larger than L2, so no view reads another's rows from L2,
    unlike config B where all views share one set);
  * routes: a loop of GaussianRasterizer calls on each view's rows; render_views(view_counts, streams=4); stacks of
    8 and 16 views (render_views(view_counts, stack=k), brs_forward_views_ex) on 1 and 2 lanes.

Each route: one warm-up pass (it seeds the high-water marks of every shape), then the median ms/view over --passes
passes, each device-synchronised on both sides.  Every route's images are compared bit for bit with the loop's.
One JSON line per route, then one summary line, each with the GPU's name, power limit and SM clock.

    python tools/bench_ragged_views.py > profiles/r04_ragged_views.jsonl"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from workload import synthetic  # noqa: E402


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip().split(", ")
        return {"gpu": out[0], "power_limit_w": float(out[1]), "sm_mhz": int(out[2]), "sm_max_mhz": int(out[3])}
    except Exception as e:  # the numbers stand without it, but say so
        return {"gpu": torch.cuda.get_device_name(0), "nvidia_smi": f"unavailable: {e}"}


def ragged_inputs(scene, n_views, seed, dev):
    """Per view a seeded subset of the scene's rows and its own colours, concatenated in view order."""
    g = torch.Generator(device="cpu").manual_seed(seed)
    gc = torch.Generator(device=dev).manual_seed(seed)
    idx, counts = [], []
    for _ in range(n_views):
        keep = 0.6 + 0.3 * float(torch.rand(1, generator=g))
        rows = torch.nonzero(torch.rand(scene.P, generator=g) < keep).squeeze(1)
        idx.append(rows)
        counts.append(int(rows.numel()))
    idx = torch.cat(idx).to(dev)
    pick = lambda t: t.index_select(0, idx).contiguous()
    colors = torch.rand((idx.numel(), 3), generator=gc, device=dev)
    return counts, dict(means3D=pick(scene.means3D), opacities=pick(scene.opacities), scales=pick(scene.scales),
                        rotations=pick(scene.rotations), colors_precomp=colors)


def median_ms_per_view(fn, passes, n_views):
    fn()  # warm-up pass
    times, out = [], None
    for _ in range(passes):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        out = fn()
        torch.cuda.synchronize()
        times.append((time.perf_counter() - t0) / n_views * 1e3)
    return sorted(times)[len(times) // 2], times, out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--views", type=int, default=120)
    ap.add_argument("--passes", type=int, default=7)
    ap.add_argument("--stacks", default="8,16")
    ap.add_argument("--seed", type=int, default=4)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_ragged_views.py needs a CUDA device")
    import bloomscene_b200

    api = bloomscene_b200._api
    dev = torch.device("cuda:0")
    scene = synthetic.config_scene("B").to(dev)
    cams = [c.to(dev) for c in synthetic.config_cameras("B", a.views)]
    bg = torch.zeros(3, device=dev)
    settings = [synthetic.raster_settings(c, 0, bg, api.GaussianRasterizationSettings) for c in cams]
    counts, t = ragged_inputs(scene, a.views, a.seed, dev)
    offs = [0]
    for c in counts:
        offs.append(offs[-1] + c)
    info = gpu_info()
    base = {"workload": f"config B scene (500 K band, precomp colours), {a.views} rotate360 yaws at 512x512, per-view "
                        "seeded subsets (keep rate 0.6-0.9) with their own colours, rows concatenated",
            "rows_total": offs[-1], "rows_min": min(counts), "rows_max": max(counts), "passes": a.passes, **info}

    def loop():
        color = torch.empty((a.views, 3, 512, 512), device=dev)
        depth = torch.empty((a.views, 1, 512, 512), device=dev)
        with torch.no_grad():
            for j, rs in enumerate(settings):
                rows = {k: v[offs[j]:offs[j + 1]] for k, v in t.items()}
                m3 = rows.pop("means3D")
                c, _, d = api.GaussianRasterizer(rs)(m3, torch.zeros_like(m3), rows.pop("opacities"), **rows)
                color[j].copy_(c)
                depth[j].copy_(d)
        return color, depth

    kw = {k: v for k, v in t.items() if k not in ("means3D", "opacities")}
    routes = [("loop_GaussianRasterizer", loop),
              ("render_views_4_streams",
               lambda: api.render_views(settings, t["means3D"], t["opacities"], streams=4, view_counts=counts, **kw)[:2])]
    for k in [int(x) for x in a.stacks.split(",") if x]:
        for lanes in (1, 2):
            routes.append((f"stack{k}_{lanes}_lane{'s' if lanes > 1 else ''}",
                           lambda k=k, lanes=lanes: api.render_views(settings, t["means3D"], t["opacities"], streams=lanes,
                                                                     stack=k, view_counts=counts, **kw)[:2]))
    ref, summary = None, {}
    for name, fn in routes:
        ms, times, out = median_ms_per_view(fn, a.passes, a.views)
        if ref is None:
            ref = out
        equal = bool(torch.equal(out[0], ref[0]) and torch.equal(out[1], ref[1]))
        summary[name] = {"ms_per_view": round(ms, 4), "equal_to_loop": equal}
        print(json.dumps({"route": name, "ms_per_view": round(ms, 4), "views_per_s": round(1e3 / ms, 1),
                          "pass_ms_per_view": [round(x, 4) for x in times], "bit_equal_to_loop": equal, **base}), flush=True)
    loop_ms = summary["loop_GaussianRasterizer"]["ms_per_view"]
    print(json.dumps({"summary": {k: dict(v, speedup_vs_loop=round(loop_ms / v["ms_per_view"], 2)) for k, v in summary.items()},
                      "all_routes_bit_equal": all(v["equal_to_loop"] for v in summary.values()), **gpu_info()}), flush=True)


if __name__ == "__main__":
    main()
