"""Seeded event scenes for the rotation and xyztheta motion models (tests/golden/cmax_models.npz and the tests that
use it).  A scene is a lattice of line segments at the reference time t0 = ts[-1], transported back to every
event's timestamp by the inverse of the model's warp, plus uniformly scattered noise events; warping with the true
parameters therefore re-aligns the lattice.  Regenerated from the seed, checked against a stored SHA-256."""
import hashlib

import numpy as np

ROTATION_TRUE = (120.0, 90.0, 1.5)            # (cx, cy, omega): a 0.3 rad turn over the 0.2 s window
XYZTHETA_TRUE = (40.0, -25.0, 1.2, 0.4)       # (vx, vy, vz, omega)


def _lattice(rng, n):
    k = rng.integers(1, 8, n) * 25.0 + 10.0
    along = rng.random(n)
    vertical = rng.random(n) < 0.5
    xr = np.where(vertical, k, 20.0 + along * 200.0)
    yr = np.where(vertical, 20.0 + along * 140.0, np.minimum(k, 160.0))
    return xr, yr


def _finish(rng, xs, ys, ts, noise, pol):
    n = xs.shape[0]
    ps = np.ones(n) if pol == "pm1" else rng.standard_normal(n)
    m = rng.random(n) < noise
    xs[m], ys[m] = rng.random(m.sum()) * 239, rng.random(m.sum()) * 179
    if pol == "pm1":
        ps[m] = rng.integers(0, 2, m.sum()) * 2.0 - 1
    return xs, ys, ts, ps


def rotating(seed=101, n=20000, truth=ROTATION_TRUE, T=0.2, noise=0.2, pol="pm1"):
    """Lattice rotating by omega about (cx, cy): x = c + R(omega d) (x0 - c) with d = t - t0."""
    rng = np.random.default_rng(seed)
    ts = np.sort(rng.random(n)) * T
    cx, cy, om = truth
    xr, yr = _lattice(rng, n)
    a = om * (ts - ts[-1])
    xs = cx + np.cos(a) * (xr - cx) - np.sin(a) * (yr - cy)
    ys = cy + np.sin(a) * (xr - cx) + np.cos(a) * (yr - cy)
    return _finish(rng, xs, ys, ts, noise, pol)


def moving(seed=202, n=20000, truth=XYZTHETA_TRUE, T=0.1, noise=0.2, pol="pm1"):
    """Lattice translating, expanding and turning: the exact inverse of the first-order xyztheta warp."""
    rng = np.random.default_rng(seed)
    ts = np.sort(rng.random(n)) * T
    vx, vy, vz, om = truth
    xr, yr = _lattice(rng, n)
    d = ts - ts[-1]
    # x' = x (1 - d vz) + d om y - d vx,  y' = y (1 - d vz) - d om x - d vy  ->  solve for (x, y)
    a, b = 1 - d * vz, d * om
    rx, ry = xr + d * vx, yr + d * vy
    det = a * a + b * b
    xs = (a * rx - b * ry) / det
    ys = (b * rx + a * ry) / det
    return _finish(rng, xs, ys, ts, noise, pol)


SCENES = {
    "rot": lambda: rotating(),
    "rot_real": lambda: rotating(seed=103, n=12000, pol="real"),
    "xyz": lambda: moving(),
}


def sha256(ev):
    return hashlib.sha256(b"".join(np.ascontiguousarray(a, dtype=np.float64).tobytes() for a in ev)).hexdigest()


def scene(g, tag):
    """(xs, ys, ts, ps) of scene `tag`, checked against the SHA-256 stored in the loaded golden file `g`."""
    ev = SCENES[tag]()
    assert sha256(ev) == str(g[tag + "_sha256"]), "scene %s no longer regenerates bit for bit" % tag
    return ev
