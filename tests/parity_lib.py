"""Shared helpers for GPU parity tests: run an implementation (ours or the reference's own CUDA
extension from oracle/_ref) on a synthetic scene and compare every stage.

Parity levels (BASELINE.json north_star):
  bit-exact : radii, num_rendered, tile keys (tile id + depth bits), sorted point list, tile ranges,
              n_contrib, final_T
  <= 1e-5   : colour, depth (max abs)
  <= 1e-4   : every gradient tensor (relative L2)

The parity tests of tests/test_gpu_parity.py compare against stored records (`Recorded`,
tests/golden/parity/*.npz) instead of a live build of the reference, so that they run from the
repository alone.  A record keeps, per compared call, a SHA-256 digest of every bit-exact array and,
for every array compared with a tolerance, the array itself when it is small, otherwise a fixed
sample of it (`sample_index`) and its L2 norm.
"""
from __future__ import annotations

import hashlib
import os
import re
import sys
from typing import Dict, Optional

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from workload import synthetic  # noqa: E402
from bloomscene_b200.rasterizer import GaussianRasterizationSettings, bind  # noqa: E402

COLOR_TOL = 1e-5
GRAD_TOL = 1e-4

_ref_api = None


def ours():
    import bloomscene_b200

    return bloomscene_b200._api


def reference():
    """The reference's own CUDA extension (oracle/_ref/_ref_C.so) under the same Python wrapper; None if absent."""
    global _ref_api
    if _ref_api is None:
        from oracle import build_ref

        mod = build_ref.load()
        if mod is None:
            return None
        _ref_api = bind(mod)
    return _ref_api


def forward_args(scene: synthetic.Scene, cam: synthetic.Camera, bg: torch.Tensor, scale_modifier=1.0, cov3D=None,
                 debug=False, prefiltered=False):
    e = torch.Tensor([])
    return (
        bg, scene.means3D,
        scene.colors_precomp if scene.colors_precomp is not None else e,
        scene.opacities,
        scene.scales if cov3D is None else e,
        scene.rotations if cov3D is None else e,
        scale_modifier,
        cov3D if cov3D is not None else e,
        cam.viewmatrix, cam.projmatrix, cam.tanfovx, cam.tanfovy, cam.image_height, cam.image_width,
        scene.shs if scene.shs is not None else e,
        scene.sh_degree, cam.campos, prefiltered, debug,
    )


def run_autograd(api, scene: synthetic.Scene, cam: synthetic.Camera, bg, Wc, Wd, scale_modifier=1.0, cov3D=None):
    """Forward + backward through the public Python API; returns outputs and gradients."""
    leaf = lambda t: None if t is None else t.detach().clone().requires_grad_(True)
    means3D, opac = leaf(scene.means3D), leaf(scene.opacities)
    scales, rots = (leaf(scene.scales), leaf(scene.rotations)) if cov3D is None else (None, None)
    cov = leaf(cov3D)
    shs, cols = leaf(scene.shs), leaf(scene.colors_precomp)
    means2D = torch.zeros_like(means3D, requires_grad=True)
    settings = synthetic.raster_settings(cam, scene.sh_degree, bg, GaussianRasterizationSettings,
                                         scale_modifier=scale_modifier)
    rast = api.GaussianRasterizer(raster_settings=settings)
    color, radii, depth = rast(means3D=means3D, means2D=means2D, opacities=opac, shs=shs, colors_precomp=cols,
                               scales=scales, rotations=rots, cov3D_precomp=cov)
    loss = (color * Wc).sum() + (depth * Wd).sum()
    loss.backward()
    out = {"color": color.detach(), "depth": depth.detach(), "radii": radii.detach()}
    grads = {"means3D": means3D.grad, "means2D": means2D.grad, "opacities": opac.grad}
    if scales is not None:
        grads["scales"], grads["rotations"] = scales.grad, rots.grad
    if cov is not None:
        grads["cov3D_precomp"] = cov.grad
    if shs is not None:
        grads["shs"] = shs.grad
    if cols is not None:
        grads["colors_precomp"] = cols.grad
    out["grads"] = grads
    return out


def rel_l2(a: torch.Tensor, b: torch.Tensor) -> float:
    a, b = a.double(), b.double()
    denom = b.norm().item()
    if denom == 0.0:
        return a.norm().item()
    return (a - b).norm().item() / denom


def compare_stages(scene, cam, bg, scale_modifier=1.0, cov3D=None) -> Dict[str, object]:
    """Raw-binding forward on both implementations and a stage-by-stage comparison (bit level)."""
    from bloomscene_b200.debug import state_views
    from oracle import ref_state

    mine, ref = ours(), reference()
    args = forward_args(scene, cam, bg, scale_modifier, cov3D)
    R0, col0, dep0, rad0, g0, b0, i0 = mine._C.rasterize_gaussians(*args)
    R1, col1, dep1, rad1, g1, b1, i1 = ref._C.rasterize_gaussians(*args)
    P, W, H = scene.P, cam.image_width, cam.image_height
    rep: Dict[str, object] = {"P": P, "R_ours": R0, "R_ref": R1}
    rep["radii_mismatch"] = int((rad0 != rad1).sum().item())
    rep["visible"] = int((rad1 > 0).sum().item())
    if P == 0:
        rep["color_maxabs"] = float((col0 - col1).abs().max().item()) if col0.numel() else 0.0
        return rep
    sv = state_views(mine._C, g0, b0, i0, P, R0, W, H)
    rg, ri = ref_state.geom_views(g1, P), ref_state.image_views(i1, W, H)
    vis = rad1 > 0
    # per-Gaussian intermediates (bitwise on visible Gaussians; -0.0 == 0.0 tolerated through float ==)
    rep["depth_bits_mismatch"] = int((sv["depth_key"][vis] != rg["depths"].view(torch.int32)[vis]).sum().item())
    rep["means2D_mismatch"] = int((sv["means2D"][vis] != rg["means2D"][vis]).any(dim=1).sum().item())
    rep["conic_opacity_mismatch"] = int((sv["conic_opacity"][vis] != rg["conic_opacity"][vis]).any(dim=1).sum().item())
    if scene.shs is not None:
        rep["rgb_maxabs"] = float((sv["rgb"][vis] - rg["rgb"][vis]).abs().max().item()) if vis.any() else 0.0
        rep["rgb_mismatch"] = int((sv["rgb"][vis] != rg["rgb"][vis]).any(dim=1).sum().item())
    rect = sv["rect"]
    tiles = ((rect[:, 0] >> 16) - (rect[:, 0] & 0xFFFF)) * ((rect[:, 1] >> 16) - (rect[:, 1] & 0xFFFF))
    rep["tiles_touched_mismatch"] = int((tiles != rg["tiles_touched"]).sum().item())
    if R0 == R1 and R1 > 0:
        rb = ref_state.binning_views(b1, R1)
        rep["point_list_mismatch"] = int((sv["point_list"] != rb["point_list"]).sum().item())
        # sorted 64-bit keys, reconstructed on our side from (tile of the range, depth bits of the id)
        ntiles = sv["ranges"].shape[0]
        rep["ranges_mismatch"] = int((sv["ranges"] != ri["ranges"][:ntiles]).any(dim=1).sum().item())
        starts = sv["ranges"][:, 0].long()
        ends = sv["ranges"][:, 1].long()
        tile_of = torch.repeat_interleave(torch.arange(ntiles, device=starts.device), (ends - starts).clamp(min=0))
        if tile_of.numel() == R1:
            dk = sv["depth_key"].long() & 0xFFFFFFFF
            keys = (tile_of << 32) | dk[sv["point_list"].long()]
            rep["sorted_keys_mismatch"] = int((keys != rb["keys"]).sum().item())
        else:
            rep["sorted_keys_mismatch"] = -1
    rep["n_contrib_mismatch"] = int((sv["n_contrib"] != ri["n_contrib"]).sum().item())
    rep["final_T_mismatch"] = int((sv["final_T"] != ri["accum_alpha"]).sum().item())
    rep["color_maxabs"] = float((col0 - col1).abs().max().item())
    rep["depth_maxabs"] = float((dep0 - dep1).abs().max().item())
    return rep


def compare_autograd(scene, cam, bg, Wc, Wd, scale_modifier=1.0, cov3D=None) -> Dict[str, float]:
    mine, ref = ours(), reference()
    a = run_autograd(mine, scene, cam, bg, Wc, Wd, scale_modifier, cov3D)
    b = run_autograd(ref, scene, cam, bg, Wc, Wd, scale_modifier, cov3D)
    b2 = run_autograd(ref, scene, cam, bg, Wc, Wd, scale_modifier, cov3D)  # reference run-to-run spread (float atomics)
    rep = {"color_maxabs": float((a["color"] - b["color"]).abs().max().item()) if a["color"].numel() else 0.0,
           "depth_maxabs": float((a["depth"] - b["depth"]).abs().max().item()) if a["depth"].numel() else 0.0,
           "radii_mismatch": int((a["radii"] != b["radii"]).sum().item())}
    for k in b["grads"]:
        ga, gb = a["grads"][k], b["grads"][k]
        if gb is None:
            rep["grad_" + k] = 0.0 if ga is None else float("nan")
            continue
        rep["grad_" + k] = rel_l2(ga, gb)
        rep["refspread_" + k] = rel_l2(b2["grads"][k], gb)
    return rep


# ---- stored records ----------------------------------------------------------------------------------

GOLDEN_DIR = os.path.join(ROOT, "tests", "golden", "parity")
RECORD_ENV = "BRS_RECORD_PARITY"  # a directory: write new records there instead of comparing
FULL = 256  # tolerance-compared arrays up to this many elements are stored whole
SAMPLE = 4096  # larger ones as this many elements at sample_index(n, SAMPLE)


def sample_index(n: int, k: int) -> np.ndarray:
    """k element indices spread over [0, n) by the golden-ratio sequence.  The first j indices of a sample
    of k are the sample of j, so a stored sample can be shortened without being recorded again."""
    j = np.arange(1, k + 1, dtype=np.float64)
    return np.floor((j * 0.6180339887498949) % 1.0 * n).astype(np.int64)


def digest(t: torch.Tensor) -> str:
    """SHA-256 of dtype, shape and bytes (float -0.0 counted as 0.0, as `==` does)."""
    t = t.detach()
    if t.is_floating_point():
        t = t + 0.0
    a = t.contiguous().cpu().numpy()
    h = hashlib.sha256(f"{a.dtype.str}{a.shape}".encode())
    h.update(a.tobytes())
    return h.hexdigest()


def floats(name: str, t: torch.Tensor) -> Dict[str, np.ndarray]:
    """An array compared with a tolerance: whole when small, else its sample; and its L2 norm."""
    a = t.detach().reshape(-1).float()
    if a.numel() > FULL:
        a = a[torch.from_numpy(sample_index(a.numel(), SAMPLE)).to(a.device)]
    return {name: a.cpu().numpy(), name + ".norm": np.float64(t.detach().double().norm().item())}


def rec_maxabs(mine, want, k, finite_only=False) -> float:
    b = want[k].astype(np.float64)
    a = mine[k][:b.size].astype(np.float64)
    if finite_only:
        ok = np.isfinite(b)
        a, b = a[ok], b[ok]
    return float(np.abs(a - b).max()) if b.size else 0.0


def rec_rel_l2(mine, want, k) -> float:
    """Relative L2 distance on the stored elements; never below the relative distance of the norms of the
    whole arrays (|‖a‖ - ‖b‖| <= ‖a - b‖, so this adds no condition the full comparison would not)."""
    b = want[k].astype(np.float64)
    a = mine[k][:b.size].astype(np.float64)
    nb = np.linalg.norm(b)
    e = float(np.linalg.norm(a - b) / nb) if nb > 0 else float(np.linalg.norm(a))
    n_want = float(want[k + ".norm"])
    if n_want > 0:
        e = max(e, abs(float(mine[k + ".norm"]) - n_want) / n_want)
    return e


def rec_mismatch(mine, want, k) -> int:
    return int(str(want[k]) != str(mine[k]))


class Recorded:
    """The stored results of one test: `take(mine, reference)` returns the record of the test's next compared call.

    With the environment variable BRS_RECORD_PARITY=<dir> the records are taken instead: `take` calls
    `reference()`, which runs the reference's own CUDA build (oracle/_ref) on the same inputs, keeps and returns
    its record, so that the test compares this library with the reference live; `finish` writes
    <dir>/<test>.npz only when the test passed (tests/golden/make_golden_parity.py)."""

    def __init__(self, test_name: str):
        self.name = re.sub(r"[^A-Za-z0-9_.-]+", "-", test_name).strip("-")
        self.out = os.environ.get(RECORD_ENV)
        self.calls = []
        self.pos = 0
        if self.out:
            assert reference() is not None, "recording needs the reference's own CUDA build (oracle/_ref/_ref_C.so)"
        else:
            path = os.path.join(GOLDEN_DIR, self.name + ".npz")
            with np.load(path) as z:
                data = {k: z[k] for k in z.files}
            for i in range(int(data["calls"])):
                p = f"c{i}."
                self.calls.append({k[len(p):]: v for k, v in data.items() if k.startswith(p)})

    def take(self, mine: Dict[str, object], reference_record) -> Dict[str, object]:
        if self.out:
            want = reference_record()
            self.calls.append(want)
        else:
            assert self.pos < len(self.calls), f"{self.name}: more compared calls than stored records ({len(self.calls)})"
            want = self.calls[self.pos]
            self.pos += 1
        assert set(want) == set(mine), (self.name, len(self.calls) - 1, sorted(set(want) ^ set(mine)))
        return want

    def finish(self, passed: bool):
        if not passed:
            return
        if self.out:
            os.makedirs(self.out, exist_ok=True)
            d = {"calls": np.int64(len(self.calls))}
            for i, rec in enumerate(self.calls):
                d.update({f"c{i}.{k}": np.asarray(v) for k, v in rec.items()})
            np.savez_compressed(os.path.join(self.out, self.name + ".npz"), **d)
        else:
            assert self.pos == len(self.calls), f"{self.name}: {len(self.calls) - self.pos} stored records were not compared"


def _stage_record(R, color, depth, radii, P, views) -> Dict[str, object]:
    """A forward reduced to what the stage comparison needs; `views()` gives its per-Gaussian, binning and
    per-pixel arrays under common names (depth_bits, means2D, conic_opacity, tiles_touched, n_contrib, final_T,
    point_list, ranges, sorted_keys)."""
    rec = {"R": R, "radii": digest(radii), "visible": int((radii > 0).sum().item()), **floats("color", color)}
    if P == 0:
        return rec
    rec.update(floats("depth", depth))
    v = views()
    vis = radii > 0
    for k in ("depth_bits", "means2D", "conic_opacity"):
        rec[k] = digest(v[k][vis])
    for k in ("tiles_touched", "n_contrib", "final_T"):
        rec[k] = digest(v[k])
    if R > 0:
        for k in ("point_list", "ranges", "sorted_keys"):
            rec[k] = digest(v[k]) if isinstance(v[k], torch.Tensor) else v[k]
    return rec


def stage_record(scene, cam, bg, scale_modifier=1.0, cov3D=None) -> Dict[str, object]:
    """This library's forward through the raw binding, reduced to what the stage comparison needs."""
    from bloomscene_b200.debug import state_views

    mine = ours()
    R, color, depth, radii, geom, binning, img = mine._C.rasterize_gaussians(*forward_args(scene, cam, bg, scale_modifier, cov3D))
    P, W, H = scene.P, cam.image_width, cam.image_height

    def views():
        sv = state_views(mine._C, geom, binning, img, P, R, W, H)
        rect = sv["rect"]
        v = {"depth_bits": sv["depth_key"], "means2D": sv["means2D"], "conic_opacity": sv["conic_opacity"],
             "tiles_touched": ((rect[:, 0] >> 16) - (rect[:, 0] & 0xFFFF)) * ((rect[:, 1] >> 16) - (rect[:, 1] & 0xFFFF)),
             "n_contrib": sv["n_contrib"], "final_T": sv["final_T"], "point_list": sv["point_list"], "ranges": sv["ranges"]}
        # sorted 64-bit keys, reconstructed from (tile of the range, depth bits of the id)
        starts, ends = sv["ranges"][:, 0].long(), sv["ranges"][:, 1].long()
        tile_of = torch.repeat_interleave(torch.arange(starts.numel(), device=starts.device), (ends - starts).clamp(min=0))
        v["sorted_keys"] = ((tile_of << 32) | (sv["depth_key"].long() & 0xFFFFFFFF)[sv["point_list"].long()]
                            if tile_of.numel() == R else "ranges do not cover the point list")
        return v

    return _stage_record(R, color, depth, radii, P, views)


def reference_stage_record(scene, cam, bg, scale_modifier=1.0, cov3D=None) -> Dict[str, object]:
    """The same record of the reference's own CUDA build (its private buffers read through oracle/ref_state)."""
    from oracle import ref_state

    ref = reference()
    R, color, depth, radii, geom, binning, img = ref._C.rasterize_gaussians(*forward_args(scene, cam, bg, scale_modifier, cov3D))
    P, W, H = scene.P, cam.image_width, cam.image_height
    ntiles = ((W + 15) // 16) * ((H + 15) // 16)

    def views():
        rg, ri = ref_state.geom_views(geom, P), ref_state.image_views(img, W, H)
        v = {"depth_bits": rg["depths"].view(torch.int32), "means2D": rg["means2D"], "conic_opacity": rg["conic_opacity"],
             "tiles_touched": rg["tiles_touched"], "n_contrib": ri["n_contrib"], "final_T": ri["accum_alpha"],
             "ranges": ri["ranges"][:ntiles]}
        if R > 0:
            rb = ref_state.binning_views(binning, R)
            v["point_list"], v["sorted_keys"] = rb["point_list"], rb["keys"]
        return v

    return _stage_record(R, color, depth, radii, P, views)


def stages_vs_record(ref: Recorded, scene, cam, bg, scale_modifier=1.0, cov3D=None) -> Dict[str, object]:
    """compare_stages against a stored record: a mismatch entry is 1 when the array differs anywhere."""
    mine = stage_record(scene, cam, bg, scale_modifier, cov3D)
    want = ref.take(mine, lambda: reference_stage_record(scene, cam, bg, scale_modifier, cov3D))
    rep: Dict[str, object] = {"P": scene.P, "R_ours": mine["R"], "R_ref": int(want["R"]), "visible": int(want["visible"]),
                              "radii_mismatch": rec_mismatch(mine, want, "radii"), "color_maxabs": rec_maxabs(mine, want, "color")}
    if scene.P == 0:
        return rep
    for k in ("depth_bits", "means2D", "conic_opacity", "tiles_touched", "n_contrib", "final_T", "point_list", "ranges",
              "sorted_keys"):
        if k in want:
            rep[k + "_mismatch"] = rec_mismatch(mine, want, k)
    rep["depth_maxabs"] = rec_maxabs(mine, want, "depth")
    return rep


def autograd_record(api, scene, cam, bg, Wc, Wd, scale_modifier=1.0, cov3D=None) -> Dict[str, object]:
    a = run_autograd(api, scene, cam, bg, Wc, Wd, scale_modifier, cov3D)
    rec = {"radii": digest(a["radii"]), **floats("color", a["color"]), **floats("depth", a["depth"])}
    for k, g in a["grads"].items():
        if g is not None:
            rec.update(floats("grad_" + k, g))
    return rec


def autograd_vs_record(ref: Recorded, scene, cam, bg, Wc, Wd, scale_modifier=1.0, cov3D=None) -> Dict[str, float]:
    """compare_autograd against a stored record (gradients: relative L2 on the stored elements)."""
    mine = autograd_record(ours(), scene, cam, bg, Wc, Wd, scale_modifier, cov3D)
    want = ref.take(mine, lambda: autograd_record(reference(), scene, cam, bg, Wc, Wd, scale_modifier, cov3D))
    rep = {"color_maxabs": rec_maxabs(mine, want, "color"), "depth_maxabs": rec_maxabs(mine, want, "depth"),
           "radii_mismatch": rec_mismatch(mine, want, "radii")}
    for k in want:
        if k.startswith("grad_") and not k.endswith(".norm"):
            rep[k] = rec_rel_l2(mine, want, k)
    return rep


def time_fwd_bwd(api, scene, cam, bg, Wc, iters=20, warmup=5):
    """Median CUDA-event times (ms) of the raw forward and backward bindings."""
    args = forward_args(scene, cam, bg)
    e = torch.Tensor([])
    fw, bw = [], []
    for it in range(warmup + iters):
        s0, s1, s2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
        s0.record()
        R, color, depth, radii, geom, binning, img = api._C.rasterize_gaussians(*args)
        s1.record()
        api._C.rasterize_gaussians_backward(
            bg, scene.means3D, radii, scene.colors_precomp if scene.colors_precomp is not None else e,
            scene.scales, scene.rotations, 1.0, e, cam.viewmatrix, cam.projmatrix, cam.tanfovx, cam.tanfovy,
            Wc, e, scene.shs if scene.shs is not None else e, scene.sh_degree, cam.campos, geom, R, binning, img, False)
        s2.record()
        torch.cuda.synchronize()
        if it >= warmup:
            fw.append(s0.elapsed_time(s1))
            bw.append(s1.elapsed_time(s2))
    fw.sort()
    bw.sort()
    return {"fwd_ms": fw[len(fw) // 2], "bwd_ms": bw[len(bw) // 2], "R": int(R)}
