"""CPU: the double-precision blend referee (tests/blend_f64.py, tests/native/blend_f64.c) against the fp32 CPU oracle,
element by element, and proof that its bounds catch the bugs it is meant to catch.

The oracle runs with f64_sums=True (its per-pair fp32 terms summed in double), so what remains between the two is the
fp32 arithmetic of the pixel chains, which the referee's error model bounds.  Each mutation test perturbs the referee
the way a blend-kernel bug would perturb the kernel, and the unchanged comparison must flag it."""
import os

import numpy as np
import pytest

import blend_f64 as bf
from oracle import oracle as orc
from test_oracle_golden import oracle_kwargs

GOLDEN = ["sh3_ragged", "precomp_bg_mod", "cov3d_sh0", "band_culled", "sh1_m16", "depth_ties", "saturating"]
BW_SLOTS = [0, 1, 5, 6, 7, 8]  # what the oracle exposes: dL_dmeans2D x, y, dL_dopacity, dL_dcolors


def _compare(ref, out, W, H):
    fw = bf.check_forward(ref, out["final_T"], out["n_contrib"], out["color"], out["depth"])
    g = out["grads"]
    impl = np.concatenate([g["dL_dmeans2D"][:, :2], g["dL_dopacity"], g["dL_dcolors"]], 1)
    # the oracle multiplies every pair by ddelx_dx = (float)(0.5 W) (backward.cu:473-474)
    bw = bf.check_backward(ref, impl, BW_SLOTS, scale=[np.float32(0.5 * W), np.float32(0.5 * H), 1, 1, 1, 1])
    return fw, bw


def _assert_agree(fw, bw, ref, what):
    print(what, "forward worst %.3g" % fw["worst"], "backward worst %.3g" % bw["worst"], ref["stats"])
    assert fw["n_contrib_mismatch"] == 0 and fw["fail"] == 0 and fw["worst"] <= 1.0, (what, fw)
    assert bw["fail"] == 0 and bw["worst"] <= 1.0, (what, bw)


@pytest.mark.parametrize("depth_grad", [False, True])
@pytest.mark.parametrize("name", GOLDEN)
def test_reference_matches_oracle_on_golden_scenes(name, depth_grad):
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", name + ".npz"))
    kw = oracle_kwargs(g)
    W, H = kw["W"], kw["H"]
    o = orc.Oracle()
    _, color, depth, radii = o.forward(**kw)
    dd = g["Wd"] if depth_grad else None
    state, out = bf.oracle_outputs(o, color, depth, radii, kw["colors_precomp"], g["Wc"], dd)
    ref = bf.reference(state, W, H, kw["bg"], g["Wc"], dd, impl_T=out["final_T"], impl_n=out["n_contrib"])
    fw, bw = _compare(ref, out, W, H)
    _assert_agree(fw, bw, ref, name)
    # golden scenes are random: undecided threshold decisions may exclude a few pixels, never more than 0.1 %
    assert ref["stats"]["pixels_excluded"] <= 1e-3 * W * H
    assert ref["excluded"].sum() <= 1e-3 * ref["excluded"].size


def _synthetic(seed, W, H, n, opacity_hi):
    rng = np.random.default_rng(seed)
    theta = rng.uniform(0, np.pi, n)
    cov = np.stack([bf.needle_cov(a, b, t) for a, b, t in
                    zip(rng.uniform(0.6, 9.0, n), rng.uniform(0.56, 3.0, n), theta)])
    u, v = rng.uniform(-4, W + 4, n), rng.uniform(-4, H + 4, n)
    z = 1.0 + rng.permutation(n) * 0.01
    return bf.pixel_scene(W, H, u, v, cov, rng.uniform(0.02, opacity_hi, n), rng.uniform(-0.2, 1.2, (n, 3)), z)


@pytest.mark.parametrize("seed,W,H,n,opacity_hi", [(1, 45, 37, 300, 0.99), (2, 64, 33, 900, 1.7), (3, 17, 70, 150, 0.3)])
def test_reference_matches_oracle_on_synthetic_scenes(seed, W, H, n, opacity_hi):
    scene, cam = _synthetic(seed, W, H, n, opacity_hi)
    rng = np.random.default_rng(seed + 100)
    bg = np.array([0.3, -0.2, 0.8], np.float32)
    dpix = rng.standard_normal((3, H, W)).astype(np.float32)
    ddep = rng.standard_normal((1, H, W)).astype(np.float32)
    state, out = bf.oracle_state(scene, cam, bg, dpix, ddep)
    ref = bf.reference(state, W, H, bg, dpix, ddep, impl_T=out["final_T"], impl_n=out["n_contrib"])
    assert ref["stats"]["pairs_contributing"] > 10 * n
    fw, bw = _compare(ref, out, W, H)
    _assert_agree(fw, bw, ref, "synthetic-%d" % seed)
    assert ref["stats"]["pixels_excluded"] <= 1e-3 * W * H


# ---- mutations --------------------------------------------------------------------------------------------------

def _mutation_scene():
    """32 x 32 (4 tiles, 16 blocks), 29 Gaussians of moderate opacity: Gaussian 0 is centred on pixel (5, 5) and spans
    several blocks; the rest overlap so that blocks stage between 9 and 29 records (never a multiple of 8 everywhere)."""
    rng = np.random.default_rng(7)
    n = 29
    u = np.concatenate([[5.0], rng.uniform(0, 32, n - 1)])
    v = np.concatenate([[5.0], rng.uniform(0, 32, n - 1)])
    cov = np.stack([bf.needle_cov(a, b, t) for a, b, t in
                    zip(rng.uniform(3.0, 8.0, n), rng.uniform(2.0, 5.0, n), rng.uniform(0, np.pi, n))])
    cov[0] = bf.needle_cov(6.0, 6.0, 0.0)
    z = 1.0 + np.arange(n) * 0.05  # Gaussian 0 in front
    opacity = rng.uniform(0.1, 0.4, n)
    opacity[0] = 0.5
    return bf.pixel_scene(32, 32, u, v, cov, opacity, rng.uniform(0, 1, (n, 3)), z)


@pytest.fixture(scope="module")
def mutation_case():
    scene, cam = _mutation_scene()
    W, H = 32, 32
    rng = np.random.default_rng(8)
    bg = np.array([0.1, 0.5, 0.9], np.float32)
    dpix = rng.standard_normal((3, H, W)).astype(np.float32)
    state, out = bf.oracle_state(scene, cam, bg, dpix)
    run = lambda **m: bf.reference(state, W, H, bg, dpix, impl_T=out["final_T"], impl_n=out["n_contrib"], **m)
    return run, out


def test_mutation_scene_agrees_unmutated(mutation_case):
    run, out = mutation_case
    ref = run()
    fw, bw = _compare(ref, out, 32, 32)
    _assert_agree(fw, bw, ref, "mutation scene")
    assert ref["stats"]["pixels_excluded"] == 0 and not ref["excluded"].any()
    assert (out["n_contrib"] > 0).all()


@pytest.mark.parametrize("mutation,a,b", [
    ("drop_pair", 5 * 32 + 5, 0),       # Gaussian 0 at pixel (5, 5)
    ("drop_block", 0, 0),               # Gaussian 0 in block (0, 0)
    ("row_shift", -1, -1),              # second pixel of a lane at y + 3
    ("row_shift", 1, -1),               # ... at y + 5
    ("double_record", 0, 0),            # Gaussian 0 flushed twice in block (0, 0)
    ("drop_partial_group", -1, -1),     # the last partial group of every batch
    ("skip_first_live", -1, -1),        # the record at warp_first_live + 1 of every block
])
def test_mutation_is_flagged(mutation_case, mutation, a, b):
    run, out = mutation_case
    ref = run(mutation=mutation, mut_a=a, mut_b=b)
    fw, bw = _compare(ref, out, 32, 32)
    print(mutation, a, "forward", fw, "backward", bw)
    assert fw["fail"] > 0 or fw["n_contrib_mismatch"] > 0 or bw["fail"] > 0, (mutation, fw, bw)


def test_partial_group_mutation_drops_only_remainders():
    """The batch / group simulation itself: one tile, n records all blended by every pixel -> each block stages n
    records per batch of 128; the dropped ones are the last n mod 8 of each batch."""
    n = 141  # batches of 128 and 13 -> remainders 0 and 5
    u = np.full(n, 7.5)
    v = np.full(n, 7.5)
    cov = np.tile([400.0, 0.0, 400.0], (n, 1))
    scene, cam = bf.pixel_scene(16, 16, u, v, cov, np.full(n, 0.006), np.ones((n, 3)), 1.0 + np.arange(n) * 0.01)
    dpix = np.ones((3, 16, 16), np.float32)
    state, out = bf.oracle_state(scene, cam, np.zeros(3, np.float32), dpix)
    assert (out["n_contrib"] == n).all()
    full = bf.reference(state, 16, 16, np.zeros(3), dpix)
    cut = bf.reference(state, 16, 16, np.zeros(3), dpix, mutation="drop_partial_group")
    changed = np.flatnonzero(np.abs(cut["g"] - full["g"]).max(axis=1) > 0)
    pos = {int(i): k for k, i in enumerate(state["point_list"])}
    # walked back to front, batch 0 = positions 140..13, batch 1 = positions 12..0: 128 % 8 == 0, 13 % 8 == 5 -> the
    # five records at positions 4..0 are dropped
    assert sorted(pos[int(i)] for i in changed) == [0, 1, 2, 3, 4]
    assert np.all(cut["g"][changed] == 0)
