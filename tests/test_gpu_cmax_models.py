"""The rotation and xyztheta motion models on the GPU: fused f / g against the reference's own pipeline
(tests/golden/cmax_models.npz) and against the CPU oracle, in both precisions and both event-pass back ends; get_iwe
images; the K-channel precomputed-image form; user-defined warps; 50 M events; BFGS on synthetic scenes."""
import functools
import os

import numpy as np
import pytest
import scipy.optimize as opt

import cmax_model_scenes as S
from event_utils_b200.contrast_max import events_cmax, objectives as OB
from event_utils_b200.contrast_max.warps import linvel_warp, pure_rotation_warp, warp_function, xyztheta_warp
from oracle import evk_oracle as O
from oracle import evk_oracle_models as M

pytestmark = pytest.mark.gpu

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "cmax_models.npz")
WARPS = {"rotation": pure_rotation_warp, "xyztheta": xyztheta_warp}
CLASSES = {"variance": OB.variance_objective, "sos": OB.sos_objective, "soe": OB.soe_objective, "isoa": OB.isoa_objective,
           "sosa": OB.sosa_objective}


@pytest.fixture
def mode():
    """restores the module-level precision / event_pass switches after a test"""
    saved = (OB.precision, OB.event_pass)
    yield
    OB.precision, OB.event_pass = saved
    OB.clear_cache()


def grad_scale(name, kind, params, ev, sigma, p_scale=1.0):
    """|g_k| <= c sum |W D_k| <= c P sqrt(mean(W^2) mean(D_k^2)) (Cauchy-Schwarz) with W the objective's weight image
    (objectives.py:251-523; SURVEY 8d's scale-normalised gradient tolerance)"""
    use_pol = O.OBJECTIVE_DEFAULTS[name][0]
    iwe, d = M.iwe_model(kind, params, ev[0], ev[1], ev[2], np.asarray(ev[3]) * p_scale, compute_gradient=True,
                         use_polarity=use_pol)
    return image_grad_scale(name, iwe, d, sigma)


def image_grad_scale(name, iwe, d, sigma):
    """the bound above for given images"""
    _, default_blur, prm = O.OBJECTIVE_DEFAULTS[name]
    sigma = default_blur if sigma is None else sigma
    I = iwe.astype(np.float64)
    G = O.gaussian_filter_f32(iwe, sigma).astype(np.float64) if sigma > 0 else I
    P = I.size
    if name == "variance":
        w, c = 2 * (I - I.mean()), 1.0 / P
    elif name == "sos":
        w, c = 2 * I, 1.0 / P
    elif name == "soe":
        w, c = np.exp(G), 1.0 / P
    elif name == "isoa":
        w, c = (G > prm).astype(np.float64), 1.0
    else:
        w, c = prm * np.exp(-prm * G), 1.0
    return c * P * np.sqrt(np.mean(w * w) * np.mean(d.astype(np.float64) ** 2))


def check(name, kind, params, ev, sigma, f, g, tol, p_scale=1.0):
    fo, go = M.cmax_model(name, kind, params, ev[0], ev[1], ev[2], ev[3], blur_sigma=sigma, p_scale=p_scale)
    assert abs(f - fo) <= tol * abs(fo) + 1e-12, (name, kind, params, sigma, f, fo)
    assert g.shape == go.shape
    assert np.abs(g - go).max() <= tol * grad_scale(name, kind, params, ev, sigma, p_scale), (name, kind, params, sigma, g, go)


@pytest.mark.parametrize("event_pass", ["onchip", "l2"])
def test_fused_models_match_the_reference_goldens(mode, event_pass):
    OB.event_pass = event_pass
    g = np.load(GOLDEN)
    scenes, names = [str(s) for s in g["scenes"]], [str(s) for s in g["objectives"]]
    kinds = {"rot": "rotation", "rot_real": "rotation", "xyz": "xyztheta"}
    for row in g["evals"]:
        tag, name, sigma = scenes[int(row[0])], names[int(row[1])], float(row[2])
        kind = kinds[tag]
        dims = WARPS[kind]().dims
        prm, f_ref, g_ref = row[3:3 + dims], row[7], row[8:8 + dims]
        ev = S.scene(g, tag)
        obj = CLASSES[name]()
        f = obj.evaluate_function(prm, *ev, WARPS[kind](), (180, 240), sigma)
        gr = obj.evaluate_gradient(prm, *ev, WARPS[kind](), (180, 240), sigma)
        assert abs(f - f_ref) <= 1e-5 * abs(f_ref), (tag, name, sigma, prm, f, f_ref)
        assert gr.shape == (dims,)
        if not np.isnan(g_ref).any():
            assert np.abs(gr - g_ref).max() <= 1e-5 * grad_scale(name, kind, prm, ev, sigma), (tag, name, sigma, prm, gr, g_ref)


def _random_scene(seed, n, pol):
    rng = np.random.default_rng(seed)
    xs, ys = rng.random(n) * 239, rng.random(n) * 179
    ts = np.sort(rng.random(n)) * 0.1
    ps = rng.integers(0, 2, n) * 2.0 - 1 if pol == "pm1" else rng.standard_normal(n)
    return xs, ys, ts, ps


@pytest.mark.parametrize("precision,tol", [("f64", 1e-5), ("f32", 1e-4)])
@pytest.mark.parametrize("event_pass", ["onchip", "l2"])
@pytest.mark.parametrize("pol", ["pm1", "real"])
def test_fused_models_match_the_oracle(mode, precision, tol, event_pass, pol):
    OB.precision, OB.event_pass = precision, event_pass
    ev = _random_scene(5, 300000, pol)
    for kind, params in (("rotation", (100.0, 80.0, 3.0)), ("xyztheta", (30.0, -20.0, 2.0, -1.5))):
        for name in ("variance", "sos", "soe", "isoa", "sosa"):
            for sigma in (None, 0.0):
                obj = CLASSES[name]()
                f = obj.evaluate_function(params, *ev, WARPS[kind](), (180, 240), sigma)
                g = obj.evaluate_gradient(params, *ev, WARPS[kind](), (180, 240), sigma)
                check(name, kind, params, ev, sigma, f, g, tol)


def test_get_iwe_images(mode):
    ev = _random_scene(6, 200000, "real")
    for kind, params in (("rotation", (100.0, 80.0, 3.0)), ("xyztheta", (30.0, -20.0, 2.0, -1.5))):
        for use_pol, size in ((True, (180, 240)), (False, (120, 200))):
            iwe, d = OB.get_iwe(params, *ev, WARPS[kind](), size, compute_gradient=True, use_polarity=use_pol)
            io, do = M.iwe_model(kind, params, *ev, size, compute_gradient=True, use_polarity=use_pol)
            assert d.shape == do.shape == (WARPS[kind]().dims, 181, 241)
            assert np.abs(iwe - io).max() <= 1e-5 * np.abs(io).max()
            assert np.abs(d - do).max() <= 1e-5 * np.abs(do).max()
            i2, d2 = OB.get_iwe(params, *ev, WARPS[kind](), size, compute_gradient=False, use_polarity=use_pol)
            assert d2 is None and np.abs(i2 - io).max() <= 1e-5 * np.abs(io).max()   # float atomics: order differs
        OB.precision = "f32"     # the images are f64-warped in either precision
        i3, _ = OB.get_iwe(params, *ev, WARPS[kind](), (180, 240), compute_gradient=True)
        OB.precision = "f64"
        io, _ = M.iwe_model(kind, params, *ev, (180, 240))
        assert np.abs(i3 - io).max() <= 1e-5 * np.abs(io).max()


def test_precomputed_images_with_three_and_four_channels():
    ev = _random_scene(7, 200000, "pm1")
    for kind, params in (("rotation", (100.0, 80.0, 3.0)), ("xyztheta", (30.0, -20.0, 2.0, -1.5))):
        iwe, d = M.iwe_model(kind, params, *ev, compute_gradient=True)
        for name in ("variance", "sos", "soe", "isoa", "sosa"):
            for sigma in (1.0, 0.0, 2.3):
                obj = CLASSES[name]()
                f = obj.evaluate_function(iwe=iwe, blur_sigma=sigma)
                g = obj.evaluate_gradient(iwe=iwe, d_iwe=d, blur_sigma=sigma)
                fo, go = M.objective_of_images_k(name, iwe, d, sigma)
                assert abs(f - fo) <= 1e-5 * abs(fo) + 1e-12, (kind, name, sigma)
                assert g.shape == (d.shape[0],)
                assert np.abs(g - go).max() <= 1e-5 * image_grad_scale(name, iwe, d, sigma), (kind, name, sigma, g, go)


class my_rotation(warp_function):
    """a user-defined 3-DoF warp: the generic (host warp) path"""
    fused_kind = None

    def __init__(self):
        super().__init__("my_rotation", 3)

    def warp(self, xs, ys, ts, ps, t0, params, compute_grad=False):
        return pure_rotation_warp().warp(xs, ys, ts, ps, t0, params, compute_grad)


def test_user_defined_three_parameter_warp_gets_three_gradient_entries():
    ev = _random_scene(8, 100000, "pm1")
    params = (100.0, 80.0, 3.0)
    for name in ("variance", "soe", "isoa"):
        obj = CLASSES[name]()
        g = obj.evaluate_gradient(params, *ev, my_rotation(), (180, 240), None)
        f = obj.evaluate_function(params, *ev, my_rotation(), (180, 240), None)
        assert g.shape == (3,)
        check(name, "rotation", params, ev, None, f, g, 1e-5)
    r = events_cmax.optimize_contrast(*ev, my_rotation(), OB.variance_objective(), x0=np.array(params),
                                      optimizer=functools.partial(opt.fmin_bfgs, maxiter=2))
    assert r.shape == (3,)


def test_xyztheta_without_expansion_and_rotation_is_linvel():
    ev = _random_scene(9, 300000, "pm1")
    obj = OB.variance_objective()
    for v in ((45.0, -20.0), (0.0, 0.0)):
        for sigma in (1.0, 0.0):
            fl = obj.evaluate_function(v, *ev, linvel_warp(), (180, 240), sigma)
            gl = obj.evaluate_gradient(v, *ev, linvel_warp(), (180, 240), sigma)
            fx = obj.evaluate_function((v[0], v[1], 0.0, 0.0), *ev, xyztheta_warp(), (180, 240), sigma)
            gx = obj.evaluate_gradient((v[0], v[1], 0.0, 0.0), *ev, xyztheta_warp(), (180, 240), sigma)
            assert abs(fx - fl) <= 1e-6 * abs(fl)            # the same IWE; float atomics may reorder the sums
            if sigma == 0.0:   # with blur the 3-D blur mixes four channels instead of two (objectives.py:253)
                assert np.abs(gx[:2] - gl).max() <= 1e-5 * grad_scale("variance", "xyztheta", (v[0], v[1], 0.0, 0.0), ev, 0.0)


def test_adaptive_lifespan_slices_and_scales_like_the_reference(mode):
    ev = S.rotating(seed=21, n=60000)
    obj = OB.variance_objective(adaptive_lifespan=True, minimum_events=20000)
    prm = (118.0, 92.0, 1.4)
    obj.iter_update(prm)
    f = obj.evaluate_function(prm, *ev, pure_rotation_warp(), (180, 240), 1.0)
    g = obj.evaluate_gradient(prm, *ev, pure_rotation_warp(), (180, 240), 1.0)
    s = int(obj.s_idx)
    assert 0 < s <= 40000              # objectives.py:137-139: at most len - minimum_events
    sl = tuple(np.asarray(a)[s:-1] for a in ev)        # objectives.py:224-225: xs[s_idx:-1], ps*100
    check("variance", "rotation", prm, sl, 1.0, f, g, 1e-5, p_scale=100.0)


@pytest.mark.parametrize("kind,params", [("rotation", (118.0, 92.0, 1.4)), ("xyztheta", (37.0, -22.0, 1.0, 0.3))])
def test_fifty_million_events(mode, kind, params):
    n = 50_000_000
    ev = S.rotating(seed=31, n=n) if kind == "rotation" else S.moving(seed=32, n=n)
    obj = OB.variance_objective()
    f = obj.evaluate_function(params, *ev, WARPS[kind](), (180, 240), 1.0)
    g = obj.evaluate_gradient(params, *ev, WARPS[kind](), (180, 240), 1.0)
    check("variance", kind, params, ev, 1.0, f, g, 1e-5)


@pytest.mark.parametrize("kind,truth,x0,seed", [
    ("rotation", S.ROTATION_TRUE, (115.0, 95.0, 1.2), 11),
    ("xyztheta", S.XYZTHETA_TRUE, (30.0, -15.0, 0.5, 0.2), 12),
])
def test_bfgs_recovers_the_motion(kind, truth, x0, seed):
    """Start points and bounds chosen by running scipy's fmin_bfgs on the CPU oracle over the same scenes:
    rotation ended at (118.2, 94.3, 1.559) for the truth (120, 90, 1.5); xyztheta at (30.2, -14.4, 1.181, 0.295) for
    (40, -25, 1.2, 0.4).  Over a 0.1-0.2 s window the rotation centre trades against omega, and the translation
    against the expansion about the origin, so the angular velocity and the expansion are what the scenes pin down."""
    ev = S.rotating(seed=seed, n=200000) if kind == "rotation" else S.moving(seed=seed, n=200000)
    obj = OB.variance_objective()
    r = events_cmax.optimize_contrast(*ev, WARPS[kind](), obj, x0=np.array(x0), blur_sigma=1.0)
    f0 = obj.evaluate_function(np.array(x0), *ev, WARPS[kind](), (180, 240), 1.0)
    fr = obj.evaluate_function(r, *ev, WARPS[kind](), (180, 240), 1.0)
    assert fr < f0
    if kind == "rotation":
        assert abs(r[2] - truth[2]) <= 0.1 and np.hypot(r[0] - truth[0], r[1] - truth[1]) <= 8.0, r
    else:
        assert abs(r[2] - truth[2]) <= 0.1 and abs(r[3] - truth[3]) <= 0.15, r


def test_default_start_point_has_the_model_dimension():
    ev = _random_scene(10, 50000, "pm1")
    calls = []

    def fake(fun, x0, **kw):
        calls.append(np.array(x0))
        return x0
    for warp in (linvel_warp(), pure_rotation_warp(), xyztheta_warp()):
        events_cmax.optimize_contrast(*ev, warp, OB.variance_objective(), optimizer=fake)
    assert [c.shape for c in calls] == [(2,), (3,), (4,)] and not any(c.any() for c in calls)
