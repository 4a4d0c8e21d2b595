"""The rotation and xyztheta motion models without a GPU: the numpy warps' Jacobians, the CPU oracle against the
reference's own pipeline (tests/golden/cmax_models.npz, tests/golden/make_cmax_models.py), the oracle's analytic
gradient against finite differences of its objective, and xyztheta reducing to linvel."""
import os

import numpy as np
import pytest

import cmax_model_scenes as S
from event_utils_b200.contrast_max.warps import linvel_warp, pure_rotation_warp, xyztheta_warp
from oracle import evk_oracle as O
from oracle import evk_oracle_models as M

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "cmax_models.npz")


@pytest.mark.parametrize("warp,params", [(pure_rotation_warp(), (120.0, 90.0, 1.5)), (pure_rotation_warp(), (-30.0, 400.0, -7.0)),
                                         (xyztheta_warp(), (40.0, -25.0, 1.2, 0.4)), (xyztheta_warp(), (-80.0, 10.0, -3.0, 2.5))])
def test_warp_jacobians_match_finite_differences(warp, params):
    rng = np.random.default_rng(1)
    n = 500
    xs, ys, ts = rng.random(n) * 240, rng.random(n) * 180, np.sort(rng.random(n)) * 0.3
    ps = np.ones(n)
    xw, yw, jx, jy = warp.warp(xs, ys, ts, ps, ts[-1], np.array(params), compute_grad=True)
    assert jx.shape == jy.shape == (warp.dims, n) and len(params) == warp.dims
    x2, y2, _, _ = warp.warp(xs, ys, ts, ps, ts[-1], np.array(params), compute_grad=False)
    assert np.array_equal(xw, x2) and np.array_equal(yw, y2)
    h = 1e-5
    for k in range(warp.dims):
        up, dn = np.array(params, dtype=np.float64), np.array(params, dtype=np.float64)
        up[k] += h
        dn[k] -= h
        xu, yu, _, _ = warp.warp(xs, ys, ts, ps, ts[-1], up)
        xd, yd, _, _ = warp.warp(xs, ys, ts, ps, ts[-1], dn)
        # central differences of a smooth function: O(h^2) truncation, O(eps |x| / h) ~ 1e-9 rounding
        np.testing.assert_allclose((xu - xd) / (2 * h), jx[k], rtol=1e-6, atol=1e-7)
        np.testing.assert_allclose((yu - yd) / (2 * h), jy[k], rtol=1e-6, atol=1e-7)


def test_model_parameter_counts():
    assert pure_rotation_warp().dims == 3 and xyztheta_warp().dims == 4
    assert pure_rotation_warp().fused_kind == "rotation" and xyztheta_warp().fused_kind == "xyztheta"


def test_oracle_matches_the_reference_pipeline():
    g = np.load(GOLDEN)
    scenes = [str(s) for s in g["scenes"]]
    names = [str(s) for s in g["objectives"]]
    events = {tag: S.scene(g, tag) for tag in scenes}
    kinds = {"rot": "rotation", "rot_real": "rotation", "xyz": "xyztheta"}
    checked = 0
    for row in g["evals"]:
        tag, name, sigma = scenes[int(row[0])], names[int(row[1])], float(row[2])
        dims = M.MODELS[kinds[tag]][1]
        prm, f_ref, g_ref = row[3:3 + dims], row[7], row[8:8 + dims]
        f, gr = M.cmax_model(name, kinds[tag], prm, *events[tag], blur_sigma=sigma)
        assert abs(f - f_ref) <= 1e-5 * abs(f_ref), (tag, name, sigma, prm, f, f_ref)
        if not np.isnan(g_ref).any():
            assert np.abs(gr - g_ref).max() <= 1e-5 * np.abs(g_ref).max(), (tag, name, sigma, prm, gr, g_ref)
        checked += 1
    assert checked == len(g["evals"]) >= 60
    # the images behind them: per-channel sums of get_iwe at the first point of each scene
    for tag in scenes:
        row = next(r for r in g["evals"] if scenes[int(r[0])] == tag)
        iwe, d = M.iwe_model(kinds[tag], row[3:3 + M.MODELS[kinds[tag]][1]], *events[tag], compute_gradient=True)
        sums = np.array([iwe.astype(np.float64).sum()] + [c.astype(np.float64).sum() for c in d])
        np.testing.assert_allclose(sums, g[tag + "_iwe_sum"], rtol=0, atol=1e-5 * g[tag + "_iwe_absum"].max())


def _big_scene(kind, n=1_000_000):
    return S.rotating(seed=7, n=n) if kind == "rotation" else S.moving(seed=8, n=n)


@pytest.mark.parametrize("kind,params,steps", [
    ("rotation", (118.0, 93.0, 1.3), (0.5, 0.5, 0.01)),
    ("xyztheta", (37.0, -22.0, 1.0, 0.3), (0.5, 0.5, 0.005, 0.005)),
])
def test_oracle_gradient_is_the_derivative_without_blur(kind, params, steps):
    """At blur_sigma = 0 the variance gradient is exactly df/dparams: the IWE is a bilinear splat, piecewise smooth
    in the warped positions.  f has kinks where events cross pixel boundaries, so the difference quotient over a
    step that moves events by ~0.01-0.1 pixel is smooth only on average: with 1 M events crossing at independent
    places the kinks average out to a relative deviation of the order of 1e-3 (measured 9e-4 for rotation, 1.3e-3 for xyztheta on these scenes).
    The bound 2e-2 of the largest entry leaves margin and still catches a wrong sign, a wrong channel or a missing
    factor."""
    ev = _big_scene(kind)
    f0, g0 = M.cmax_model("variance", kind, params, *ev, blur_sigma=0.0)
    fd = []
    for k, h in enumerate(steps):
        up, dn = np.array(params), np.array(params)
        up[k] += h
        dn[k] -= h
        fu, _ = M.cmax_model("variance", kind, up, *ev, blur_sigma=0.0, want_grad=False)
        fl, _ = M.cmax_model("variance", kind, dn, *ev, blur_sigma=0.0, want_grad=False)
        fd.append((fu - fl) / (2 * h))
    fd = np.array(fd)
    assert np.abs(fd - g0).max() <= 2e-2 * np.abs(g0).max(), (fd, g0)


def test_xyztheta_without_expansion_and_rotation_is_linvel():
    g = np.load(os.path.join(os.path.dirname(GOLDEN), "cmax.npz"))
    import cmax_scenes
    ev = cmax_scenes.events(g, "lat")
    for v in [(45.0, -20.0), (60.0, -35.0), (0.0, 0.0)]:
        iwe_l, d_l = O.iwe_linvel(v, *ev, (180, 240), compute_gradient=True)
        iwe_x, d_x = M.iwe_model("xyztheta", (v[0], v[1], 0.0, 0.0), *ev, compute_gradient=True)
        assert np.array_equal(iwe_l, iwe_x) and np.array_equal(d_l, d_x[:2])
        for sigma in (1.0, 0.0):
            fl, gl = O.cmax_variance(v, *ev, blur_sigma=sigma)
            fx, gx = M.cmax_model("variance", "xyztheta", (v[0], v[1], 0.0, 0.0), *ev, blur_sigma=sigma)
            assert fx == fl
            if sigma == 0.0:     # with blur, scipy's 3-D blur mixes all four channels, so only the unblurred g agrees
                np.testing.assert_allclose(gx[:2], gl, rtol=1e-12, atol=0)


def test_linvel_warp_is_unchanged():
    rng = np.random.default_rng(3)
    xs, ys, ts = rng.random(100) * 240, rng.random(100) * 180, np.sort(rng.random(100))
    xw, yw, jx, jy = linvel_warp().warp(xs, ys, ts, None, ts[-1], (3.0, -2.0), compute_grad=True)
    assert jx.shape == (2, 100) and np.array_equal(xw, xs - (ts - ts[-1]) * 3.0)
