"""ctypes front-end to oracle/evk_oracle_models.c and the objectives of K-channel derivative images --
TEST INFRASTRUCTURE ONLY, the oracle of the rotation and xyztheta models (same rules as evk_oracle.py).

The image-space part restates evk_oracle.objective_of_images for `dims` derivative channels: scipy's
gaussian_filter blurs the (dims, H, W) stack along all three axes (objectives.py:253), and the gradient has one
entry per channel (objectives.py:258-263 loops over d_iwe.shape[0])."""
import ctypes
import os
import subprocess

import numpy as np

from . import evk_oracle as O

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "evk_oracle_models.c")
_SO = os.path.join(_HERE, "libevk_oracle_models.so")
MODELS = {"rotation": (1, 3), "xyztheta": (2, 4)}   # kind: (oracle model id, dims)
_lib = None


def build(force=False):
    """gcc with the flags of oracle/Makefile -> oracle/libevk_oracle_models.so"""
    if force or not os.path.exists(_SO) or os.path.getmtime(_SO) < os.path.getmtime(_SRC):
        subprocess.check_call(["gcc", "-O2", "-fPIC", "-ffp-contract=off", "-fno-fast-math", "-fvisibility=hidden", "-Wall",
                               "-Wextra", "-std=c11", "-shared", "-o", _SO, _SRC, "-lm"])
    return _SO


def lib():
    global _lib
    if _lib is None:
        build()
        L = ctypes.CDLL(_SO)
        vp, i64, f64, ci = ctypes.c_void_p, ctypes.c_int64, ctypes.c_double, ctypes.c_int
        L.evo_iwe_model.restype = i64
        L.evo_iwe_model.argtypes = [ci, vp, vp, vp, vp, vp, i64, f64, ci, ci, ci, ci, ci, vp, vp]
        _lib = L
    return _lib


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def iwe_model(kind, params, xs, ys, ts, ps, img_size=(180, 240), compute_gradient=False, use_polarity=True,
              sensor_size=(180, 240), t_ref=None):
    """get_iwe (objectives.py:184-192) with the rotation / xyztheta model -> (iwe, d_iwe [dims] or None)."""
    model, dims = MODELS[kind]
    prm = np.ascontiguousarray(np.asarray(params, dtype=np.float64).reshape(-1))
    assert prm.shape[0] == dims
    x, y, t, p = (np.ascontiguousarray(a, dtype=np.float64) for a in (xs, ys, ts, ps))
    Hs, Ws = int(sensor_size[0]), int(sensor_size[1])
    iwe = np.zeros((Hs + 1, Ws + 1), np.float32)
    d = np.zeros((dims, Hs + 1, Ws + 1), np.float32) if compute_gradient else None
    oob = lib().evo_iwe_model(model, _p(prm), _p(x), _p(y), _p(t), _p(p), x.shape[0], float(t[-1] if t_ref is None else t_ref),
                              int(img_size[0]), int(img_size[1]), Hs, Ws, int(bool(use_polarity)), _p(iwe),
                              _p(d) if d is not None else None)
    if oob:
        raise O.OracleIndexError("%d warped events index outside the IWE canvas" % oob)
    return iwe, d


def objective_of_images_k(name, iwe, d_iwe=None, blur_sigma=None, param=None):
    """f (and the K-entry g) of any objective of evk_oracle.OBJECTIVE_DEFAULTS on a precomputed IWE and a
    (K, H, W) derivative stack.  variance: objectives.py:231-264 (evo_variance_f / evo_variance_g for K channels);
    the others: evk_oracle.objective_of_images with range(K).  Returns (f, g or None)."""
    _, default_blur, default_param = O.OBJECTIVE_DEFAULTS[name]
    sigma = default_blur if blur_sigma is None else blur_sigma
    prm = default_param if param is None else param
    img = np.asarray(iwe, dtype=np.float32)
    f = O.variance_f(img, sigma) if name == "variance" else O.objective_of_images(name, img, None, sigma, prm)[0]
    if d_iwe is None or name in ("moa", "r1"):
        return float(f), None
    stack = np.asarray(d_iwe, dtype=np.float32)
    stack = O.gaussian_filter_f32(stack, sigma) if sigma > 0 else stack
    blurred = O.gaussian_filter_f32(img, sigma) if sigma > 0 else img
    K = stack.shape[0]
    if name == "variance":
        mu = np.float32(img.astype(np.float64).mean())
        comp = np.float32(2.0) * (img - mu)
        g = [-((comp * stack[k]).astype(np.float64).sum() / img.size) for k in range(K)]
    elif name == "rms":
        g = [-2.0 * np.mean(img * stack[k]) for k in range(K)]
    elif name == "sos":
        g = [-np.mean(stack[k] * (img * 2.0)) for k in range(K)]
    elif name == "soe":
        g = [-np.mean(np.exp(blurred.astype(np.float64)) * stack[k]) for k in range(K)]
    elif name == "isoa":
        g = [-np.sum(stack[k] * (blurred > prm).astype(np.float32)) for k in range(K)]
    else:  # sosa
        g = [-np.sum(stack[k] * (-prm * np.exp((-prm * blurred).astype(np.float64)))) for k in range(K)]
    return float(f), np.array(g, dtype=np.float64)


def cmax_model(name, kind, params, xs, ys, ts, ps, img_size=(180, 240), blur_sigma=None, param=None, want_grad=True,
               p_scale=1.0):
    """objective `name` with motion model `kind` on raw events -> (f, g[dims] or None)."""
    use_polarity = O.OBJECTIVE_DEFAULTS[name][0]
    iwe, d = iwe_model(kind, params, xs, ys, ts, np.asarray(ps, dtype=np.float64) * p_scale, img_size,
                       compute_gradient=want_grad, use_polarity=use_polarity)
    return objective_of_images_k(name, iwe, d, blur_sigma, param)
