"""Motion models for contrast maximisation -- drop-in for the reference's lib/contrast_max/warps.py
(`warp_function` ABC :6-42, `linvel_warp` :44-61, the two empty stubs :63-83).

An objective from `event_utils_b200.contrast_max.objectives` that is handed one of the three models here
never calls `warp()`: it recognises the model through `fused_kind` and evaluates warp, bounds mask, image
formation, objective and gradient on the GPU over the device-resident events (csrc/evk_cmax.cu): one pass
for linvel, two (image, then the gradient in gather form) for the rotation and xyztheta models.  `warp()` is still provided, with the reference's semantics, for user code that
calls it directly and for the generic (non-fused) path taken by other `warp_function` subclasses.
"""
from abc import ABC, abstractmethod

import numpy as np


class warp_function(ABC):
    """A parametrised, differentiable motion model that transports events to a reference time.
    `name` identifies the model, `dims` is its number of degrees of freedom (used by the grid
    search drivers, events_cmax.py:282)."""

    fused_kind = None   # set by models the fused kernels implement natively

    def __init__(self, name, dims):
        self.name, self.dims = name, dims
        super().__init__()

    @abstractmethod
    def warp(self, xs, ys, ts, ps, t0, params, compute_grad=False):
        """Transport the events (xs, ys, ts, ps) to time t0 under `params`.
        Returns (xs_warped, ys_warped, jacobian_x, jacobian_y); the Jacobians have shape
        (dims, N) -- d x'/d params and d y'/d params per event -- or are None without
        compute_grad."""


class linvel_warp(warp_function):
    """Global optic flow: every event moves with one image-plane velocity (vx, vy) = params,
        x' = x - (t - t0) vx,      y' = y - (t - t0) vy,
    so d x'/d vx = d y'/d vy = -(t - t0) and the cross terms vanish (reference warps.py:51-61)."""

    fused_kind = "linvel"

    def __init__(self):
        super().__init__('linvel_warp', 2)

    def warp(self, xs, ys, ts, ps, t0, params, compute_grad=False):
        lag = ts - t0
        moved = (xs - lag * params[0], ys - lag * params[1])
        if not compute_grad:
            return moved[0], moved[1], None, None
        nothing = np.zeros_like(lag, dtype=np.float64)
        return moved[0], moved[1], np.stack((-lag, nothing)), np.stack((nothing, -lag))


class pure_rotation_warp(warp_function):
    """Rotation of the image plane about a centre (cx, cy) with angular velocity omega; params = (cx, cy, omega),
    dims = 3.  With d = t - t0, th = -omega d, c = cos th, s = sin th:
        x' = cx + c (x - cx) - s (y - cy),       y' = cy + s (x - cx) + c (y - cy)
        dx'/d(cx, cy, omega) = (1 - c,  s,  d (y' - cy))
        dy'/d(cx, cy, omega) = (-s, 1 - c, -d (x' - cx))
    The reference declares this model with an empty warp (warps.py:74-83); its README and docstring list three
    parameters, its constructor registers dims=4, which is a slip: dims is 3 here."""

    fused_kind = "rotation"

    def __init__(self):
        super().__init__('pure_rotation_warp', 3)

    def warp(self, xs, ys, ts, ps, t0, params, compute_grad=False):
        cx, cy, omega = float(params[0]), float(params[1]), float(params[2])
        lag = ts - t0
        theta = -(omega * lag)
        c, s = np.cos(theta), np.sin(theta)
        X, Y = xs - cx, ys - cy
        xw = cx + c * X - s * Y
        yw = cy + s * X + c * Y
        if not compute_grad:
            return xw, yw, None, None
        return xw, yw, np.stack((1 - c, s, lag * (yw - cy))), np.stack((-s, 1 - c, -(lag * (xw - cx))))


class xyztheta_warp(warp_function):
    """First-order 4-DoF motion (Mitrokhin et al.): image-plane translation (vx, vy), expansion vz and in-plane
    rotation omega about the pixel-grid origin; params = (vx, vy, vz, omega), dims = 4.  With d = t - t0:
        x' = x - d (vx + vz x - omega y),        y' = y - d (vy + vz y + omega x)
        dx'/d(vx, vy, vz, omega) = (-d, 0, -d x,  d y)
        dy'/d(vx, vy, vz, omega) = (0, -d, -d y, -d x)
    With vz = omega = 0 this is linvel_warp bit for bit.  An empty stub in the reference (warps.py:63-72)."""

    fused_kind = "xyztheta"

    def __init__(self):
        super().__init__('xyztheta_warp', 4)

    def warp(self, xs, ys, ts, ps, t0, params, compute_grad=False):
        vx, vy, vz, omega = (float(v) for v in params[:4])
        lag = ts - t0
        xw = xs - lag * (vx + vz * xs - omega * ys)
        yw = ys - lag * (vy + vz * ys + omega * xs)
        if not compute_grad:
            return xw, yw, None, None
        nothing = np.zeros_like(lag, dtype=np.float64)
        return xw, yw, np.stack((-lag, nothing, -(lag * xs), lag * ys)), np.stack((nothing, -lag, -(lag * ys), -(lag * xs)))
