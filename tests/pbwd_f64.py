"""Double-precision referee for the preprocess backward: a ctypes front end of tests/native/pbwd_f64.cpp.

`Problem(...)` holds one backward's per-Gaussian inputs exactly as the kernel sees them (Gaussians, camera, radii, the
blend accumulator [P, 12]).  `evaluate` runs the referee's statements in double, in float or with error bounds;
`check` compares an implementation's outputs, packed per Gaussian as
    dL_dmeans3D 3 | dL_dcov3D 6 (off-diagonals doubled) | dL_dscales 3 | dL_drotations 4 | dL_dsh 3 M
(`pack`), with the bounds: |got - ref| <= K e + u |ref| for every element of every rendered Gaussian.

K = 4 on the GPU: e bounds an fp32 evaluation of the REFERENCE's statements, and the kernel computes the same
intermediates — t, J, T, the entries of the 2D covariance, det, the conic gradient, Sigma — in another order
(preprocess_bwd_math.h: matrix form, SH coefficients contracted with dL_dRGB before the basis gradients) and with
fused multiply-adds.  Each reordered sum or product of the same terms has a first-order error bounded by a small
multiple of the same sum of term magnitudes, and an FMA only removes a rounding, so a factor of a few covers the
difference; 4 leaves room for a chain of two reordered stages.  The CPU tests show that K = 1 bounds the float
evaluation of the reference's own statements, so the model, not K, carries the error estimate."""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "native", "pbwd_f64.cpp")
EPS = 2.0 ** -24
K_GPU = 4.0
ST_CHECKED, ST_RESOLVED, ST_EXCLUDED, ST_INVISIBLE = 0, 1, 2, 3

_lib = None


class _Scene(C.Structure):
    _fields_ = [(n, C.c_int) for n in ("P", "D", "M", "W", "H", "depth_gradient")] + [
        (n, C.c_float) for n in ("tanfovx", "tanfovy", "scale_modifier")] + [
        (n, C.c_void_p) for n in ("view", "proj", "campos", "means3D", "scales", "rotations", "cov3D_precomp", "shs",
                                  "radii", "accum", "color_hint")]


def _build_dir():
    d = os.path.join(HERE, "native", "_build")
    try:
        os.makedirs(d, exist_ok=True)
        if os.access(d, os.W_OK):
            return d
    except OSError:
        pass
    d = os.path.join(tempfile.gettempdir(), "pbwd_f64_build_%d" % os.getuid())
    os.makedirs(d, exist_ok=True)
    return d


def lib():
    global _lib
    if _lib is None:
        out = os.path.join(_build_dir(), "libpbwdf64.so")
        if not os.path.exists(out) or os.path.getmtime(out) < os.path.getmtime(SRC):
            tmp = out + ".%d.tmp" % os.getpid()
            subprocess.run(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off", SRC, "-o", tmp],
                           check=True)
            os.replace(tmp, out)
        L = C.CDLL(out)
        L.pbwd_nout.argtypes = [C.POINTER(_Scene)]
        L.pbwd_nout.restype = C.c_int
        L.pbwd_eval.argtypes = [C.POINTER(_Scene), C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
        L.pbwd_check.argtypes = [C.POINTER(_Scene), C.c_void_p, C.c_void_p, C.c_double, C.c_void_p, C.c_void_p,
                                 C.c_void_p]
        _lib = L
    return _lib


def _np(a, dtype=np.float32):
    if a is None:
        return None
    if hasattr(a, "detach"):
        a = a.detach().cpu().numpy()
    return np.ascontiguousarray(a, dtype=dtype)


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


class Problem:
    """One preprocess backward's inputs.  shs None: precomputed colours.  color_hint: the forward's (clamped) colours
    [P, 3], which are exactly 0 where a channel was clamped; it decides a colour clamp whose value lies in its band."""

    def __init__(self, W, H, tanfovx, tanfovy, viewmatrix, projmatrix, campos, means3D, radii, accum, sh_degree=0,
                 shs=None, scales=None, rotations=None, cov3D_precomp=None, scale_modifier=1.0, depth_gradient=False,
                 color_hint=None):
        self.a = {"view": _np(viewmatrix).reshape(16), "proj": _np(projmatrix).reshape(16),
                  "campos": _np(campos if campos is not None else np.zeros(3)).reshape(3), "means3D": _np(means3D),
                  "scales": None if cov3D_precomp is not None else _np(scales),
                  "rotations": None if cov3D_precomp is not None else _np(rotations),
                  "cov3D_precomp": _np(cov3D_precomp), "shs": _np(shs), "radii": _np(radii, np.int32),
                  "accum": _np(accum).reshape(-1, 12), "color_hint": _np(color_hint)}
        self.P = self.a["means3D"].shape[0]
        self.M = 0 if shs is None else self.a["shs"].shape[1]
        self.W, self.H = int(W), int(H)
        self.depth_gradient = bool(depth_gradient)
        self.s = _Scene(self.P, int(sh_degree), self.M, self.W, self.H, int(self.depth_gradient), float(tanfovx),
                        float(tanfovy), float(scale_modifier), *[_p(self.a[k]) for k in (
                            "view", "proj", "campos", "means3D", "scales", "rotations", "cov3D_precomp", "shs", "radii",
                            "accum", "color_hint")])
        self.n = lib().pbwd_nout(C.byref(self.s))

    @property
    def visible(self):
        return self.a["radii"] > 0


def evaluate(pb: Problem, kind: str = "bound"):
    """kind "double" | "float" | "bound".  Returns (values [P, n], bounds [P, n] or None, flags [P]); flags bit 0
    invisible, bit 1 excluded by the division rule, bit 2 a threshold decision inside its band."""
    k = {"double": 0, "float": 1, "bound": 2}[kind]
    v = np.zeros((pb.P, pb.n), np.float64)
    e = np.zeros((pb.P, pb.n), np.float64) if k == 2 else None
    flags = np.zeros(pb.P, np.int32)
    lib().pbwd_eval(C.byref(pb.s), k, _p(v), _p(e), _p(flags))
    return v, e, flags


def pack(pb: Problem, dL_dmeans3D, dL_dcov3D, dL_dscales=None, dL_drotations=None, dL_dsh=None):
    """An implementation's gradients as the referee's rows [P, n] (float32).  Absent gradients are taken as zero (for
    scales and rotations of a cov3D_precomp problem that is what the referee computes)."""
    P = pb.P
    z = lambda k: np.zeros((P, k), np.float32)
    cols = [_np(dL_dmeans3D).reshape(P, 3), _np(dL_dcov3D).reshape(P, 6),
            z(3) if dL_dscales is None else _np(dL_dscales).reshape(P, 3),
            z(4) if dL_drotations is None else _np(dL_drotations).reshape(P, 4)]
    if pb.M:
        cols.append(z(3 * pb.M) if dL_dsh is None else _np(dL_dsh).reshape(P, 3 * pb.M))
    return np.ascontiguousarray(np.concatenate(cols, axis=1), dtype=np.float32)


def check(pb: Problem, got, K: float = K_GPU, slack=None):
    """Every rendered Gaussian against its bound (plus `slack` [P, n], an error the comparison itself adds).  Returns a
    report: worst ratio (<= 1 passes), the number of failing Gaussians, the resolved and excluded counts, and
    per-Gaussian ratio / element / status."""
    got = np.ascontiguousarray(got, dtype=np.float32).reshape(pb.P, pb.n)
    ratio = np.zeros(pb.P, np.float64)
    elem = np.zeros(pb.P, np.int32)
    status = np.zeros(pb.P, np.int32)
    sl = None if slack is None else np.ascontiguousarray(slack, dtype=np.float64).reshape(pb.P, pb.n)
    lib().pbwd_check(C.byref(pb.s), _p(got), _p(sl), float(K), _p(ratio), _p(elem), _p(status))
    live = (status == ST_CHECKED) | (status == ST_RESOLVED)
    worst = float(ratio[live].max(initial=0.0))
    bad = np.flatnonzero(live & ~(ratio <= 1.0))
    return {"worst": worst, "fail": int(bad.size), "first_fail": int(bad[0]) if bad.size else -1,
            "fail_elem": int(elem[bad[0]]) if bad.size else -1, "resolved": int((status == ST_RESOLVED).sum()),
            "excluded": int((status == ST_EXCLUDED).sum()), "checked": int(live.sum()), "ratio": ratio,
            "status": status}


def describe(rep) -> str:
    return "worst %.3g, checked %d, resolved %d, excluded %d, failing %d" % (
        rep["worst"], rep["checked"], rep["resolved"], rep["excluded"], rep["fail"])


ELEMENTS = (["mean.%s" % c for c in "xyz"] + ["cov.%d" % i for i in range(6)] + ["scale.%s" % c for c in "xyz"] +
            ["rot.%s" % c for c in "rxyz"])


def element_name(k: int) -> str:
    return ELEMENTS[k] if k < len(ELEMENTS) else "sh[%d].%s" % ((k - 16) // 3, "rgb"[(k - 16) % 3])


# ---- constructed inputs ----------------------------------------------------------------------------------------------

def view_to_world(cam, t_view):
    """World positions whose view-space coordinates are t_view [n, 3] (camera of workload.synthetic)."""
    V = np.asarray(cam.viewmatrix, np.float64).reshape(4, 4)  # row-vector convention: t = [p, 1] @ V
    return ((np.asarray(t_view, np.float64) - V[3, :3]) @ np.linalg.inv(V[:3, :3])).astype(np.float32)


def random_quaternions(rng, n, lo=0.5, hi=2.0):
    q = rng.standard_normal((n, 4))
    q /= np.linalg.norm(q, axis=1, keepdims=True)
    return (q * rng.uniform(lo, hi, (n, 1))).astype(np.float32)


def random_accum(rng, n, scale=1.0):
    """Blend sums of plausible relative magnitudes (the means2D sums are in NDC units, the conic sums larger)."""
    acc = np.zeros((n, 12), np.float32)
    acc[:, 0:2] = rng.standard_normal((n, 2)) * 1e-3
    acc[:, 2:5] = rng.standard_normal((n, 3)) * 1e-2
    acc[:, 5:10] = rng.standard_normal((n, 5)) * 1e-2
    return (acc * scale).astype(np.float32)
