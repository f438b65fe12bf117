"""CPU: the preprocess-backward referee (tests/pbwd_f64.py) against itself and against the fp32 oracle.

- The float evaluation of the referee's statements lies within the bound (K = 1) on >= 10^5 random Gaussians, edge
  cases included: the error model bounds an fp32 evaluation of the reference's statements.
- The oracle's orc_preprocess_backward (pinned to the reference's CUDA outputs by test_oracle_golden.py) lies within
  the bound (K = 1) on every golden scene, fed with random blend sums, with and without the depth term: the referee
  has the reference's semantics.
- The same comparison flags each mutation of the oracle's outputs or inputs that a kernel bug could produce."""
import os

import numpy as np
import pytest

import pbwd_f64 as pf
from oracle import oracle as orc
from test_oracle_golden import oracle_kwargs
from workload import synthetic

GOLDEN = ["sh3_ragged", "precomp_bg_mod", "cov3d_sh0", "band_culled", "sh1_m16", "depth_ties", "saturating"]
f32 = np.float32


def sh_basis(D, d):
    """Real SH basis [n, 16] of directions d [n, 3], the reference's ordering and signs (forward.cu:20-71)."""
    x, y, z = d[:, 0], d[:, 1], d[:, 2]
    b = np.zeros((d.shape[0], 16))
    b[:, 0] = 0.28209479177387814
    if D > 0:
        c1 = 0.4886025119029199
        b[:, 1], b[:, 2], b[:, 3] = -c1 * y, c1 * z, -c1 * x
    if D > 1:
        xx, yy, zz = x * x, y * y, z * z
        b[:, 4], b[:, 5] = 1.0925484305920792 * x * y, -1.0925484305920792 * y * z
        b[:, 6], b[:, 7] = 0.31539156525252005 * (2 * zz - xx - yy), -1.0925484305920792 * x * z
        b[:, 8] = 0.5462742152960396 * (xx - yy)
    if D > 2:
        b[:, 9] = -0.5900435899266435 * y * (3 * xx - yy)
        b[:, 10] = 2.890611442640554 * x * y * z
        b[:, 11] = -0.4570457994644658 * y * (4 * zz - xx - yy)
        b[:, 12] = 0.3731763325901154 * z * (2 * zz - 3 * xx - 3 * yy)
        b[:, 13] = -0.4570457994644658 * x * (4 * zz - xx - yy)
        b[:, 14] = 1.445305721320277 * z * (xx - yy)
        b[:, 15] = -0.5900435899266435 * x * (xx - 3 * yy)
    return b


def covariance(scales, q):
    """3D covariances [n, 6] (xx xy xz yy yz zz) of scales and normalised quaternions, float64 then rounded."""
    qn = q.astype(np.float64) / np.linalg.norm(q, axis=1, keepdims=True)
    rr, x, y, z = qn.T
    R = np.stack([1 - 2 * (y * y + z * z), 2 * (x * y - rr * z), 2 * (x * z + rr * y),
                  2 * (x * y + rr * z), 1 - 2 * (x * x + z * z), 2 * (y * z - rr * x),
                  2 * (x * z - rr * y), 2 * (y * z + rr * x), 1 - 2 * (x * x + y * y)], axis=1).reshape(-1, 3, 3)
    S = np.einsum("nij,nj,nkj->nik", R, np.asarray(scales, np.float64) ** 2, R)
    return S[:, [0, 0, 0, 1, 1, 2], [0, 1, 2, 1, 2, 2]].astype(f32)


def edge_gaussians(rng, n, cam, D, M, cov_precomp=False):
    """n Gaussians mixing ordinary ones with the edges of the preprocess backward: |t/t_z| just inside and outside
    1.3 tan fov on both axes, depth just above the 0.2 near plane, needles up to 1:300, sub-pixel Gaussians (det of
    the 2D covariance near 0.09, where the 1e-7 added to det^2 matters), |q| from 0.5 to 2, and colour channels
    negative, near zero and positive.  Returns a dict of float32 arrays."""
    tz = rng.uniform(0.5, 20.0, n)
    near = rng.random(n) < 0.1
    tz[near] = 0.2 * (1 + 10.0 ** rng.uniform(-6, -2, near.sum()))
    lims = (1.3 * cam.tanfovx, 1.3 * cam.tanfovy)
    r = np.stack([rng.uniform(-1.0, 1.0, n) * lims[0], rng.uniform(-1.0, 1.0, n) * lims[1]], axis=1)
    for ax in range(2):
        edge = rng.random(n) < 0.15
        k = edge.sum()
        r[edge, ax] = rng.choice([-1, 1], k) * lims[ax] * (1 + rng.choice([-1, 1], k) * 10.0 ** rng.uniform(-7, -2, k))
        far = rng.random(n) < 0.05
        r[far, ax] = rng.uniform(-3, 3, far.sum()) * lims[ax]
    t_view = np.stack([r[:, 0] * tz, r[:, 1] * tz, tz], axis=1)
    means = pf.view_to_world(cam, t_view)
    scales = np.exp(rng.normal(-4.0, 1.0, (n, 3))) * (tz[:, None] / 5)  # projected sizes independent of depth
    needle = (rng.random(n) < 0.15) & ~near  # a needle spanning hundreds of pixels at z = 0.2: det cancels entirely
    scales[needle, 1:] = scales[needle, :1] / rng.uniform(30, 300, (needle.sum(), 2))
    sub = rng.random(n) < 0.15
    scales[sub] = 10.0 ** rng.uniform(-7, -5, (sub.sum(), 3)) * tz[sub, None]
    q = pf.random_quaternions(rng, n)
    out = {"means3D": means, "scales": scales.astype(f32), "rotations": q}
    if cov_precomp:
        out["cov3D_precomp"] = covariance(scales, q)
    if M:
        shs = rng.standard_normal((n, M, 3)) * 0.3
        d = means.astype(np.float64) - np.asarray(cam.campos, np.float64)
        b = sh_basis(D, d / np.linalg.norm(d, axis=1, keepdims=True))
        kmax = (D + 1) ** 2
        rest = np.einsum("nk,nkc->nc", b[:, 1:kmax], shs[:, 1:kmax])
        target = rng.uniform(-1.0, 1.0, (n, 3))
        tiny = rng.random((n, 3)) < 0.2
        target[tiny] = rng.choice([-1, 1], tiny.sum()) * 10.0 ** rng.uniform(-7, -3, tiny.sum())
        shs[:, 0] = (target - 0.5 - rest) / 0.28209479177387814
        out["shs"] = shs.astype(f32)
    return out


def edge_problem(seed, n, D, M, cov_precomp=False, scale_modifier=1.0, depth=False, W=640, H=480):
    rng = np.random.default_rng(seed)
    cam = synthetic.make_camera(W, H, synthetic._rot_y(rng.uniform(-3, 3)), rng.uniform(-2, 2, 3))
    gs = edge_gaussians(rng, n, cam, D, M, cov_precomp)
    pb = pf.Problem(W, H, cam.tanfovx, cam.tanfovy, cam.viewmatrix, cam.projmatrix, cam.campos, gs["means3D"],
                    np.ones(n, np.int32), pf.random_accum(rng, n), sh_degree=D, shs=gs.get("shs"), scales=gs["scales"],
                    rotations=gs["rotations"], cov3D_precomp=gs.get("cov3D_precomp"), scale_modifier=scale_modifier,
                    depth_gradient=depth)
    return pb


# D = 0..3 with M in {1, 4, 9, 16} and M larger than (D + 1)^2; precomputed colours; cov3D_precomp; scale_modifier
EDGE_CASES = [(0, 1, False, 1.0, False), (0, 4, False, 0.7, True), (1, 4, False, 1.0, False), (1, 16, True, 1.0, True),
              (2, 9, False, 1.6, True), (2, 16, False, 1.0, False), (3, 16, False, 1.0, True), (3, 16, True, 0.5, False),
              (0, 0, False, 1.3, True), (0, 0, True, 1.0, False)]


@pytest.mark.parametrize("case", range(len(EDGE_CASES)))
def test_float_evaluation_within_bound(case):
    """10 cases x 12 000 Gaussians: the float instantiation of the referee's statements is within K = 1 of the bound
    on every Gaussian the division rule keeps."""
    D, M, cov_pre, mod, depth = EDGE_CASES[case]
    pb = edge_problem(100 + case, 12000, D, M, cov_pre, mod, depth)
    vf, _, _ = pf.evaluate(pb, "float")
    rep = pf.check(pb, vf.astype(f32), K=1.0)
    print("float vs bound, D=%d M=%d cov3D_precomp=%s mod=%g depth=%s: %s" % (D, M, cov_pre, mod, depth,
                                                                              pf.describe(rep)))
    assert rep["fail"] == 0, (rep["first_fail"], pf.element_name(rep["fail_elem"]), rep["worst"])
    # the rare exclusion is a needle seen obliquely, whose det = a c - b^2 cancels to a relative error above 1/2 in fp32
    assert rep["excluded"] <= 2
    assert rep["resolved"] > 0  # the edge populations do put decisions inside their bands
    # the bound is not vacuous: the float evaluation differs from the double one, and the bound is far below |ref|
    vd, e, _ = pf.evaluate(pb, "bound")
    assert (vf != vd).any()
    big = np.abs(vd) > 1e-20
    assert np.median(e[big] / np.abs(vd[big])) < 1e-3


def golden_problem(name, seed, depth):
    """The oracle's forward of a golden scene, random blend sums, the oracle's per-Gaussian backward and the referee's
    Problem for the same inputs."""
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", name + ".npz"))
    kw = oracle_kwargs(g)
    o = orc.Oracle()
    _, _, _, radii = o.forward(**kw)
    st = o.state()
    P, W, H = radii.shape[0], kw["W"], kw["H"]
    acc = pf.random_accum(np.random.default_rng(seed), P)
    dm2 = np.zeros((P, 3), f32)
    dm2[:, 0] = acc[:, 0] * f32(0.5 * W)
    dm2[:, 1] = acc[:, 1] * f32(0.5 * H)
    dcon = np.zeros((P, 4), f32)
    dcon[:, 0], dcon[:, 1], dcon[:, 3] = f32(-0.5) * acc[:, 2], f32(-0.5) * acc[:, 3], f32(-0.5) * acc[:, 4]
    out = o.preprocess_backward(dm2, dcon, acc[:, 6:9], acc[:, 9] if depth else None)
    pb = pf.Problem(W, H, kw["tanfovx"], kw["tanfovy"], kw["viewmatrix"], kw["projmatrix"], kw["campos"],
                    kw["means3D"], radii, acc, sh_degree=kw["sh_degree"], shs=kw["shs"], scales=kw["scales"],
                    rotations=kw["rotations"], cov3D_precomp=kw["cov3D_precomp"], scale_modifier=kw["scale_modifier"],
                    depth_gradient=depth, color_hint=st["rgb"] if kw["shs"] is not None else None)
    return o, pb, out, (dm2, dcon, acc)


def pack_oracle(pb, out):
    return pf.pack(pb, out["dL_dmeans3D"], out["dL_dcov3D"], out["dL_dscales"], out["dL_drotations"], out["dL_dsh"])


@pytest.mark.parametrize("depth", [False, True])
@pytest.mark.parametrize("name", GOLDEN)
def test_oracle_within_bound_on_golden_scenes(name, depth):
    _, pb, out, _ = golden_problem(name, 7, depth)
    rep = pf.check(pb, pack_oracle(pb, out), K=1.0)
    print("oracle %s depth=%s: %s" % (name, depth, pf.describe(rep)))
    assert rep["checked"] > 0
    assert rep["fail"] == 0, (rep["first_fail"], pf.element_name(rep["fail_elem"]), rep["worst"])
    assert rep["excluded"] == 0


def _flagged(pb, got):
    rep = pf.check(pb, got, K=1.0)
    return rep["fail"] > 0


def test_mutations_are_flagged():
    """Each mutation of the oracle's output (or its inputs) fails the comparison that the unmutated output passes."""
    _, pb, out, _ = golden_problem("sh3_ragged", 3, True)
    got = pack_oracle(pb, out)
    assert not _flagged(pb, got)
    vis = np.flatnonzero(pb.visible)
    sh0 = 16
    # two neighbours' SH rows swapped
    i, j = vis[10], vis[11]
    m = got.copy()
    m[[i, j], sh0:] = m[[j, i], sh0:]
    assert _flagged(pb, m)
    # a dL_dsh chunk (4 coefficients x 3 channels) shifted by one coefficient
    m = got.copy()
    m[i, sh0 + 12 + 3:sh0 + 24 + 3] = got[i, sh0 + 12:sh0 + 24]
    assert _flagged(pb, m)
    # r and g swapped in one row
    m = got.copy()
    m[i, sh0::3], m[i, sh0 + 1::3] = got[i, sh0 + 1::3], got[i, sh0::3]
    assert _flagged(pb, m)
    # the depth term dropped
    o, pb_d, _, (dm2, dcon, acc) = golden_problem("sh3_ragged", 3, True)
    no_depth = o.preprocess_backward(dm2, dcon, acc[:, 6:9], None)
    assert _flagged(pb_d, pack_oracle(pb_d, no_depth))
    # dL_dcov3D off-diagonals not doubled (the cov3D_precomp scene: the cov3D gradient is a final output there)
    _, pb_c, out_c, _ = golden_problem("cov3d_sh0", 3, False)
    m = pack_oracle(pb_c, out_c)
    assert not _flagged(pb_c, m)
    m[:, [4, 5, 7]] *= 0.5
    assert _flagged(pb_c, m)
    # the quaternion gradient taken for the normalised quaternion: (I - n n^T) g / |q|
    q = pb.a["rotations"].astype(np.float64)
    nq = q / np.linalg.norm(q, axis=1, keepdims=True)
    gq = got[:, 12:16].astype(np.float64)
    m = got.copy()
    m[:, 12:16] = (gq - nq * (nq * gq).sum(1, keepdims=True)) / np.linalg.norm(q, axis=1, keepdims=True)
    assert _flagged(pb, m)


def test_mutation_colour_clamp_ignored():
    """The oracle with its clamp flags cleared (every channel passes its gradient) is flagged; the scene has clamped
    channels with non-zero upstream colour gradients."""
    import ctypes as C

    o, pb, out, (dm2, dcon, acc) = golden_problem("sh3_ragged", 5, False)
    assert not _flagged(pb, pack_oracle(pb, out))
    clamped = o.state()["clamped"]
    assert clamped[pb.visible].any()
    p = o.L.orc_clamped(o.ctx)
    C.memset(p, 0, clamped.size)
    m = o.preprocess_backward(dm2, dcon, acc[:, 6:9], None)
    assert _flagged(pb, pack_oracle(pb, m))


def subpixel_problem(seed=21, n=2000):
    """Sub-pixel Gaussians facing the camera: the 2D covariance is ~0.3 I, det ~0.09, det^2 ~0.0081, and the
    reference's 1e-7 regulariser changes the conic gradient by ~1.2e-5 relative."""
    rng = np.random.default_rng(seed)
    W, H = 320, 240
    cam = synthetic.make_camera(W, H, np.eye(3), np.zeros(3))
    tz = rng.uniform(1.0, 4.0, n)
    t_view = np.stack([rng.uniform(-0.8, 0.8, n) * cam.tanfovx * tz, rng.uniform(-0.8, 0.8, n) * cam.tanfovy * tz, tz], 1)
    means = pf.view_to_world(cam, t_view)
    scales = (10.0 ** rng.uniform(-6, -5, (n, 3)) * tz[:, None]).astype(f32)
    q = pf.random_quaternions(rng, n)
    acc = pf.random_accum(rng, n)
    acc[:, 0:2] = 0  # only the conic path: its gradient is what the regulariser scales
    acc[:, 6:10] = 0
    return pf.Problem(W, H, cam.tanfovx, cam.tanfovy, cam.viewmatrix, cam.projmatrix, cam.campos, means,
                      np.ones(n, np.int32), acc, scales=scales, rotations=q)


def test_mutation_regulariser_dropped():
    """Scaling the conic-path gradients by det^2 / (det^2 + 1e-7) (the 1e-7 dropped) is flagged on sub-pixel
    Gaussians: the bound resolves effects near 1e-5 relative."""
    pb = subpixel_problem()
    vd, e, _ = pf.evaluate(pb, "bound")
    vf, _, _ = pf.evaluate(pb, "float")
    assert pf.check(pb, vf.astype(f32), K=1.0)["fail"] == 0
    det2 = 0.09 ** 2
    # without the regulariser every conic-path output grows by (det^2 + 1e-7) / det^2 - 1 ~ 1.2e-5 (relative)
    m = (vd * (1 + 1e-7 / det2)).astype(f32)
    rep = pf.check(pb, m, K=1.0)
    assert rep["fail"] > 0.5 * pb.P, pf.describe(rep)
    rel = np.median(e[:, :16][np.abs(vd[:, :16]) > 0] / np.abs(vd[:, :16][np.abs(vd[:, :16]) > 0]))
    assert rel < 1e-5, rel


def test_threshold_cases_are_resolved_not_excluded():
    """Gaussians placed exactly on the clamp threshold and with colours at 0 are resolved by trying both branches:
    both branch results pass, none is excluded."""
    pb = edge_problem(77, 3000, 3, 16, depth=True)
    vf, _, flags = pf.evaluate(pb, "bound")
    rep = pf.check(pb, pf.evaluate(pb, "float")[0].astype(f32), K=1.0)
    assert rep["resolved"] == int(((flags & 4) != 0).sum()) > 0
    assert rep["excluded"] == 0 and rep["fail"] == 0
