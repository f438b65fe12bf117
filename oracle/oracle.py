"""ctypes front end of the CPU oracle (oracle/rasterizer_oracle.c).

TEST INFRASTRUCTURE ONLY — see the header of rasterizer_oracle.c.  Only tests/,
__graft_entry__.smoke() and bench.py's cpu_baseline / reference legs may import this module; the
product path never does.

`Oracle.forward(...)` / `.backward(...)` take and return numpy arrays (fp32 / int32) and restate
CudaRasterizer::Rasterizer::{forward, backward} of the reference (rasterizer_impl.cu:198-339,
403-504); `.state()` exposes the intermediate arrays the reference keeps in its geometry / binning /
image buffers so every stage can be compared.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from pathlib import Path
from typing import Dict, Optional

import numpy as np

HERE = Path(__file__).resolve().parent
LIB = HERE / "_build" / "liboracle.so"
SRC = HERE / "rasterizer_oracle.c"

_BASE = ["-O2", "-fPIC", "-std=c99", "-ffp-contract=off", "-fno-math-errno", "-shared"]


def build(force: bool = False) -> Path:
    """Compile the oracle with gcc (OpenMP if the toolchain has it)."""
    if LIB.exists() and not force and LIB.stat().st_mtime >= SRC.stat().st_mtime:
        return LIB
    LIB.parent.mkdir(exist_ok=True)
    attempts = [
        ["gcc", *_BASE, "-fopenmp", str(SRC), "-o", str(LIB), "-lm"],
        ["gcc", *_BASE, "-fopenmp", "-B/usr/lib/gcc/x86_64-linux-gnu/13/", str(SRC), "-o", str(LIB), "-lm"],
        ["gcc", *_BASE, "-Wno-unknown-pragmas", str(SRC), "-o", str(LIB), "-lm"],
    ]
    err = ""
    for cmd in attempts:
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode == 0:
            return LIB
        err = r.stderr
    raise RuntimeError("could not build the CPU oracle:\n" + err)


class _Inputs(C.Structure):
    _fields_ = [("P", C.c_int), ("D", C.c_int), ("M", C.c_int), ("W", C.c_int), ("H", C.c_int),
                ("tanfovx", C.c_float), ("tanfovy", C.c_float), ("scale_modifier", C.c_float),
                ("bg", C.c_void_p), ("viewmatrix", C.c_void_p), ("projmatrix", C.c_void_p), ("campos", C.c_void_p),
                ("means3D", C.c_void_p), ("opacities", C.c_void_p), ("shs", C.c_void_p), ("colors_precomp", C.c_void_p),
                ("scales", C.c_void_p), ("rotations", C.c_void_p), ("cov3D_precomp", C.c_void_p)]


class _Grads(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("dL_dmeans2D", "dL_dcolors", "dL_dopacity", "dL_dmeans3D", "dL_dcov3D",
                                           "dL_dsh", "dL_dscales", "dL_drotations")]


_lib = None


def lib():
    global _lib
    if _lib is None:
        build()
        L = C.CDLL(str(LIB))
        L.orc_create.restype = C.c_void_p
        L.orc_destroy.argtypes = [C.c_void_p]
        L.orc_forward.argtypes = [C.c_void_p, C.POINTER(_Inputs), C.c_void_p, C.c_void_p, C.c_void_p]
        L.orc_forward.restype = C.c_int
        L.orc_backward.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(_Grads)]
        L.orc_backward.restype = C.c_int
        L.orc_backward_ex.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(_Grads)]
        L.orc_backward_ex.restype = C.c_int
        L.orc_preprocess_backward.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(_Grads)]
        L.orc_preprocess_backward.restype = C.c_int
        L.orc_set_f64_sums.argtypes = [C.c_int]
        L.orc_visible_filter.argtypes = [C.POINTER(_Inputs), C.c_int, C.c_void_p]
        L.orc_mark_visible.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
        L.orc_set_threads.argtypes = [C.c_int]
        L.orc_max_threads.restype = C.c_int
        L.orc_num_rendered.argtypes = [C.c_void_p]
        L.orc_num_rendered.restype = C.c_int
        for name in ("orc_pairs_evaluated", "orc_pairs_contributing"):
            getattr(L, name).argtypes = [C.c_void_p]
            getattr(L, name).restype = C.c_longlong
        for name in ("orc_depths", "orc_means2D", "orc_cov3D", "orc_conic_opacity", "orc_rgb", "orc_clamped",
                     "orc_tiles_touched", "orc_point_offsets", "orc_keys_unsorted", "orc_keys", "orc_point_list",
                     "orc_ranges", "orc_final_T", "orc_n_contrib"):
            getattr(L, name).argtypes = [C.c_void_p]
            getattr(L, name).restype = C.c_void_p
        _lib = L
    return _lib


def _f32(a) -> Optional[np.ndarray]:
    if a is None:
        return None
    if hasattr(a, "detach"):
        a = a.detach().cpu().numpy()
    a = np.ascontiguousarray(a, dtype=np.float32)
    return a if a.size else None


def _ptr(a: Optional[np.ndarray]):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


class Oracle:
    """One forward (+ optional backward) of the reference algorithm on the CPU."""

    def __init__(self, threads: int = 0):
        self.L = lib()
        if threads:
            self.L.orc_set_threads(threads)
        self.ctx = self.L.orc_create()
        self._keep = []
        self.P = self.W = self.H = self.M = 0

    def __del__(self):
        try:
            self.L.orc_destroy(self.ctx)
        except Exception:
            pass

    @property
    def threads(self) -> int:
        return self.L.orc_max_threads()

    def _inputs(self, W, H, tanfovx, tanfovy, bg, viewmatrix, projmatrix, campos, sh_degree, means3D, opacities,
                shs=None, colors_precomp=None, scales=None, rotations=None, cov3D_precomp=None, scale_modifier=1.0):
        arrs = dict(bg=_f32(bg), viewmatrix=_f32(viewmatrix), projmatrix=_f32(projmatrix), campos=_f32(campos),
                    means3D=_f32(means3D), opacities=_f32(opacities), shs=_f32(shs),
                    colors_precomp=_f32(colors_precomp), scales=_f32(scales), rotations=_f32(rotations),
                    cov3D_precomp=_f32(cov3D_precomp))
        self._keep = list(arrs.values())
        P = 0 if arrs["means3D"] is None else arrs["means3D"].shape[0]
        M = 0 if arrs["shs"] is None else arrs["shs"].shape[1]
        inp = _Inputs(P, int(sh_degree), M, int(W), int(H), float(tanfovx), float(tanfovy), float(scale_modifier),
                      *[_ptr(arrs[k]) for k in ("bg", "viewmatrix", "projmatrix", "campos", "means3D", "opacities",
                                                "shs", "colors_precomp", "scales", "rotations", "cov3D_precomp")])
        self.P, self.W, self.H, self.M = P, int(W), int(H), M
        return inp

    def forward(self, **kw):
        """Returns (num_rendered, color[3,H,W], depth[1,H,W], radii[P])."""
        inp = self._inputs(**kw)
        color = np.zeros((3, self.H, self.W), np.float32)
        depth = np.zeros((1, self.H, self.W), np.float32)
        radii = np.zeros((self.P,), np.int32)
        R = self.L.orc_forward(self.ctx, C.byref(inp), _ptr(color), _ptr(depth), _ptr(radii))
        return R, color, depth, radii

    def backward(self, dL_dcolor, dL_ddepth=None, f64_sums: bool = False) -> Dict[str, np.ndarray]:
        """Gradients in the reference's shapes (rasterize_points.cu:154-162). Call after forward().
        `dL_ddepth` (default None = the reference: depth carries no gradient) switches on the opt-in
        depth-gradient extension."""
        P, M = self.P, self.M
        d = _f32(dL_dcolor)
        dd = _f32(dL_ddepth) if dL_ddepth is not None else None
        g = {"dL_dmeans2D": np.zeros((P, 3), np.float32), "dL_dcolors": np.zeros((P, 3), np.float32),
             "dL_dopacity": np.zeros((P, 1), np.float32), "dL_dmeans3D": np.zeros((P, 3), np.float32),
             "dL_dcov3D": np.zeros((P, 6), np.float32), "dL_dsh": np.zeros((P, M, 3), np.float32),
             "dL_dscales": np.zeros((P, 3), np.float32), "dL_drotations": np.zeros((P, 4), np.float32)}
        gs = _Grads(*[_ptr(g[n]) if g[n].size else None for n, _ in _Grads._fields_])
        # f64_sums (diagnostic): the per-Gaussian sums of the blend backward are accumulated in double and rounded
        # once, which separates summation error from arithmetic differences
        self.L.orc_set_f64_sums(1 if f64_sums else 0)
        try:
            if P:
                self.L.orc_backward_ex(self.ctx, _ptr(d), _ptr(dd), C.byref(gs))
        finally:
            self.L.orc_set_f64_sums(0)
        return g

    def preprocess_backward(self, dL_dmeans2D, dL_dconic, dL_dcolors, dL_dz=None) -> Dict[str, np.ndarray]:
        """The per-Gaussian stage of backward() alone, fed with arbitrary blend sums: dL_dmeans2D [P,3],
        dL_dconic [P,4] (x, y, -, w; the reference's per-pair -0.5 included), dL_dcolors [P,3], dL_dz [P] or None (no
        depth term).  Returns dL_dmeans3D, dL_dcov3D, dL_dsh, dL_dscales, dL_drotations (zeros where radii <= 0).
        Call after forward()."""
        P, M = self.P, self.M
        ins = [_f32(np.asarray(a).reshape(P, k)) for a, k in ((dL_dmeans2D, 3), (dL_dconic, 4), (dL_dcolors, 3))]
        dz = None if dL_dz is None else _f32(np.asarray(dL_dz).reshape(P))
        g = {"dL_dmeans3D": np.zeros((P, 3), np.float32), "dL_dcov3D": np.zeros((P, 6), np.float32),
             "dL_dsh": np.zeros((P, M, 3), np.float32), "dL_dscales": np.zeros((P, 3), np.float32),
             "dL_drotations": np.zeros((P, 4), np.float32)}
        gs = _Grads(*[_ptr(g[n]) if n in g and g[n].size else None for n, _ in _Grads._fields_])
        if P:
            self.L.orc_preprocess_backward(self.ctx, *[_ptr(a) for a in ins], _ptr(dz), C.byref(gs))
        return g

    def visible_filter(self, scales_stride: int = 3, **kw) -> np.ndarray:
        inp = self._inputs(bg=None, campos=None, sh_degree=0, opacities=None, **kw)
        radii = np.zeros((self.P,), np.int32)
        if self.P:
            self.L.orc_visible_filter(C.byref(inp), scales_stride, _ptr(radii))
        return radii

    def mark_visible(self, means3D, viewmatrix) -> np.ndarray:
        m, v = _f32(means3D), _f32(viewmatrix)
        P = 0 if m is None else m.shape[0]
        out = np.zeros((P,), np.uint8)
        if P:
            self.L.orc_mark_visible(P, _ptr(m), _ptr(v), _ptr(out))
        return out.astype(bool)

    def _arr(self, name, dtype, shape):
        n = int(np.prod(shape))
        if n == 0:
            return np.zeros(shape, dtype)
        p = getattr(self.L, "orc_" + name)(self.ctx)
        buf = (C.c_char * (n * np.dtype(dtype).itemsize)).from_address(p)
        return np.frombuffer(buf, dtype=dtype).reshape(shape).copy()

    def state(self) -> Dict[str, np.ndarray]:
        P, W, H = self.P, self.W, self.H
        R = self.L.orc_num_rendered(self.ctx)
        ntiles = ((W + 15) // 16) * ((H + 15) // 16)
        if P == 0:
            return {"num_rendered": 0}
        return {
            "num_rendered": R,
            "pairs_evaluated": self.L.orc_pairs_evaluated(self.ctx),
            "pairs_contributing": self.L.orc_pairs_contributing(self.ctx),
            "depths": self._arr("depths", np.float32, (P,)),
            "means2D": self._arr("means2D", np.float32, (P, 2)),
            "cov3D": self._arr("cov3D", np.float32, (P, 6)),
            "conic_opacity": self._arr("conic_opacity", np.float32, (P, 4)),
            "rgb": self._arr("rgb", np.float32, (P, 3)),
            "clamped": self._arr("clamped", np.uint8, (P, 3)),
            "tiles_touched": self._arr("tiles_touched", np.uint32, (P,)),
            "point_offsets": self._arr("point_offsets", np.uint32, (P,)),
            "keys_unsorted": self._arr("keys_unsorted", np.uint64, (R,)),
            "keys": self._arr("keys", np.uint64, (R,)),
            "point_list": self._arr("point_list", np.uint32, (R,)),
            "ranges": self._arr("ranges", np.uint32, (ntiles, 2)),
            "final_T": self._arr("final_T", np.float32, (H * W,)),
            "n_contrib": self._arr("n_contrib", np.uint32, (H * W,)),
        }


def run_scene(scene, cam, bg, threads: int = 0, dL_dcolor=None, scale_modifier: float = 1.0, cov3D_precomp=None):
    """Convenience: forward (+ backward) on a bloomscene_b200.synthetic Scene / Camera."""
    o = Oracle(threads)
    R, color, depth, radii = o.forward(
        W=cam.image_width, H=cam.image_height, tanfovx=cam.tanfovx, tanfovy=cam.tanfovy, bg=bg,
        viewmatrix=cam.viewmatrix, projmatrix=cam.projmatrix, campos=cam.campos, sh_degree=scene.sh_degree,
        means3D=scene.means3D, opacities=scene.opacities, shs=scene.shs, colors_precomp=scene.colors_precomp,
        scales=None if cov3D_precomp is not None else scene.scales,
        rotations=None if cov3D_precomp is not None else scene.rotations, cov3D_precomp=cov3D_precomp,
        scale_modifier=scale_modifier)
    out = {"num_rendered": R, "color": color, "depth": depth, "radii": radii, "oracle": o}
    if dL_dcolor is not None:
        out["grads"] = o.backward(dL_dcolor)
    return out
