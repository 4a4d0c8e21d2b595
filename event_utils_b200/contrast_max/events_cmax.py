"""Optimiser drivers around the fused objective -- the callers of the hot path in the reference's
lib/contrast_max/events_cmax.py (`grid_cmax` :28-76, the sampling half of `draw_objective_function`
:100-158, `find_new_range` :160-182, `grid_search_optimisation` :184-239, `grid_search_initial`
:241-311, `optimize_contrast` :313-346, `optimize` :348-368, `optimize_r2` :370-389).  They are thin: scipy's BFGS stays on the host and calls the fused GPU
evaluation; the grid search evaluates ALL its sample points with one pass over the events per 32
candidates (objectives.evaluate_candidates) instead of one full evaluation per point.
"""
import contextlib
import copy

import numpy as np
import scipy.optimize as opt

from ..util.event_util import infer_resolution
from .objectives import _fused_kind, evaluate_candidates, get_iwe, pinned_events, soe_objective, variance_objective
from .warps import linvel_warp


def grid_search_initial(xs, ys, ts, ps, warp_function, objective_function, img_size, param_ranges=None,
        log_scale=True, num_samples_per_param=5):
    """
    Sample the objective on a (log- or linearly spaced) grid over the warp parameters; same inputs
    and returned dict as events_cmax.py:241-311: 'params', 'eval', 'search_axes', 'min_params',
    'min_func_eval'.  (As in the reference the blur is fixed at 1.0 and a point only becomes the
    optimum if its value is below 0.)
    """
    assert num_samples_per_param % 2 == 1
    half = int(num_samples_per_param / 2.0) + 1
    if log_scale:
        scale = np.logspace(0, 2.0, half)[1:]
        scale /= scale[-1]
    else:
        scale = np.linspace(0, 1.0, half)[1:]
    if param_ranges is None:
        param_ranges = [[-150, 150] for _ in range(warp_function.dims)]
    axes = []
    for lo, hi in param_ranges:
        span = hi - lo
        mid = lo + span / 2.0
        axes.append(np.concatenate((np.array(mid - scale * (span / 2.0))[::-1], np.array([mid]), np.array(mid + scale * (span / 2.0)))))
    coords = np.vstack([np.ravel(g) for g in np.meshgrid(*axes)])
    points = list(zip(*coords))
    evals, _ = evaluate_candidates(objective_function, points, xs, ys, ts, ps, warp_function, img_size, blur_sigma=1.0)
    output = {"params": [], "eval": [], "search_axes": axes}
    best_eval, best_params = 0, None
    for params, f_eval in zip(points, evals):
        output["params"].append(params)
        output["eval"].append(float(f_eval))
        if f_eval < best_eval:
            best_eval, best_params = float(f_eval), params
    output["min_params"] = best_params
    output["min_func_eval"] = best_eval
    return output


def optimize_contrast(xs, ys, ts, ps, warp_function, objective, optimizer=opt.fmin_bfgs, x0=None,
        numeric_grads=False, blur_sigma=None, img_size=(180, 240), grid_search_init=False, minimum_events=200):
    """
    Gradient-based contrast maximisation; same signature as events_cmax.py:313-346.  With
    grid_search_init the start point comes from grid_search_initial (the reference calls an
    undefined `recursive_search` there, events_cmax.py:336).  The default start point is zeros(warp_function.dims)
    (the reference's [0, 0] only fits 2-parameter models).
    @returns the maximising warp parameters
    """
    # nothing between here and the return modifies the event arrays (scipy hands the same `args` objects to
    # every f / f' call), so the event set is uploaded and hashed ONCE for the whole optimisation
    fused = _fused_kind(warp_function) is not None
    with (pinned_events(xs, ys, ts, ps) if fused else contextlib.nullcontext()):
        if grid_search_init and x0 is None:
            init_obj = copy.deepcopy(objective)
            init_obj.adaptive_lifespan = False
            x0 = grid_search_initial(xs, ys, ts, ps, warp_function, init_obj, img_size, log_scale=False)["min_params"]
            x0 = np.zeros(warp_function.dims) if x0 is None else np.array(x0)
        elif x0 is None:
            x0 = np.zeros(warp_function.dims)
        objective.iter_update(x0)
        args = (xs, ys, ts, ps, warp_function, img_size, blur_sigma)
        if numeric_grads:
            return optimizer(objective.evaluate_function, x0, args=args, epsilon=1, disp=False, callback=objective.iter_update)
        return optimizer(objective.evaluate_function, x0, fprime=objective.evaluate_gradient, args=args, disp=False,
                         callback=objective.iter_update)


def optimize(xs, ys, ts, ps, warp, obj, numeric_grads=True, img_size=(180, 240)):
    """events_cmax.py:348-368: optimize_contrast with blur 1.0, numeric gradients unless the objective has analytic ones."""
    numeric_grads = numeric_grads if obj.has_derivative else True
    return optimize_contrast(xs, ys, ts, ps, warp, obj, numeric_grads=numeric_grads, blur_sigma=1.0, img_size=img_size)


def optimize_r2(xs, ys, ts, ps, warp, obj, numeric_grads=True, img_size=(180, 240)):
    """events_cmax.py:370-389: optimise `obj` at its default blur, then refine from that optimum with the
    sum-of-exponentials objective at blur 1.0.  As in the reference `img_size` is accepted but NOT forwarded
    (both stages run at optimize_contrast's default (180, 240))."""
    soe_obj = soe_objective()
    numeric_grads = numeric_grads if obj.has_derivative else True
    argmax_an = optimize_contrast(xs, ys, ts, ps, warp, obj, numeric_grads=numeric_grads, blur_sigma=None)
    return optimize_contrast(xs, ys, ts, ps, warp, soe_obj, x0=argmax_an, numeric_grads=numeric_grads, blur_sigma=1.0)


def find_new_range(search_axes, param):
    """
    The next, narrower search interval of one parameter axis once `param` was the best sample:
    it reaches from the neighbouring sample below to the one above, so the whole unsearched
    neighbourhood is covered (events_cmax.py:160-182; at the ends of the axis the outermost
    spacing is reused, at index 0 -- as in the reference -- the distance to the LAST sample).
    """
    k = int(np.searchsorted(search_axes, param))
    last = len(search_axes) - 1
    if k >= last:
        below = above = abs(search_axes[-1] - search_axes[-2])
    elif k == 0:
        below, above = abs(search_axes[0] - search_axes[-1]), abs(search_axes[0] - search_axes[1])
    else:
        below, above = abs(search_axes[k] - search_axes[k - 1]), abs(search_axes[k] - search_axes[k + 1])
    return [param - below, param + above]


def grid_search_optimisation(xs, ys, ts, ps, warp_function, objective_function, img_size, param_ranges=None,
        log_scale=True, num_samples_per_param=5, depth=0, th0=1, max_iters=20):
    """
    Coarse-to-fine grid search (SOFAS): sample the parameter grid, re-centre a narrower grid on
    the best sample, stop when the widest interval is below th0 or after max_iters levels.
    Signature and returned dict as events_cmax.py:184-239.  Every level is one batched pass over
    the events per 32 sample points.  (The reference recurses through an undefined name,
    `recursive_search`, :235; the recursion here is the one its docstring describes.)
    """
    assert num_samples_per_param % 2 == 1 and num_samples_per_param >= 5
    level = grid_search_initial(xs, ys, ts, ps, warp_function, copy.deepcopy(objective_function), img_size,
                                param_ranges=param_ranges, log_scale=log_scale, num_samples_per_param=num_samples_per_param)
    if level["min_params"] is None:
        return level
    ranges = [find_new_range(axis, value) for axis, value in zip(level["search_axes"], level["min_params"])]
    widest = max(abs(hi - lo) for lo, hi in ranges)
    if widest < th0 or depth >= max_iters:
        return level
    return grid_search_optimisation(xs, ys, ts, ps, warp_function, objective_function, img_size, param_ranges=ranges,
                                    log_scale=log_scale, num_samples_per_param=num_samples_per_param, depth=depth + 1,
                                    th0=th0, max_iters=max_iters)


def sample_objective_function(xs, ys, ts, ps, objective=None, warpfunc=None, x_range=(-200, 200), y_range=(-200, 200),
        resolution=20, img_size=(180, 240), norm_min=None, norm_max=None):
    """
    The image draw_objective_function plots (events_cmax.py:119-130): pixel (row, col) is the negated
    objective at params = (col*resolution + x_range[0], row*resolution + y_range[0]) with
    blur_sigma=0, min-max normalised with a 1e-6 guard.  All sample points go through the batched
    evaluation (32 parameter points per pass over the events).
    """
    objective = variance_objective(minimum_events=1) if objective is None else objective
    warpfunc = linvel_warp() if warpfunc is None else warpfunc
    rows = int((y_range[1] - y_range[0]) / resolution + 0.5)
    cols = int((x_range[1] - x_range[0]) / resolution + 0.5)
    points = [(c * resolution + x_range[0], r * resolution + y_range[0]) for r in range(rows) for c in range(cols)]
    f, _ = evaluate_candidates(objective, points, xs, ys, ts, ps, warpfunc, img_size, blur_sigma=0)
    img = -np.asarray(f, dtype=np.float64).reshape(rows, cols)
    lo = np.min(img) if norm_min is None else norm_min
    hi = np.max(img) if norm_max is None else norm_max
    return (img - lo) / ((hi - lo) + 1e-6)


def draw_objective_function(xs, ys, ts, ps, objective=None, warpfunc=None, x_range=(-200, 200), y_range=(-200, 200),
        gt=(0, 0), show_gt=True, resolution=20, img_size=(180, 240), show_axes=True, norm_min=None, norm_max=None,
        show=True):
    """events_cmax.py:100-158: sample the objective over a parameter window and plot it.  The sampling is
    `sample_objective_function`; plotting needs matplotlib (an ImportError says so if it is absent)."""
    img = sample_objective_function(xs, ys, ts, ps, objective, warpfunc, x_range, y_range, resolution, img_size,
                                    norm_min, norm_max)
    import matplotlib.pyplot as plt
    plt.imshow(img, interpolation='bilinear', cmap='viridis')
    if show_axes:
        plt.xlabel("$v_x$")
        plt.ylabel("$v_y$")
    else:
        plt.xticks([])
        plt.yticks([])
    if show_gt:
        plt.axhline(y=(gt[1] - y_range[0]) / (y_range[1] - y_range[0]) * img.shape[0], color='r', linestyle='--')
        plt.axvline(x=(gt[0] - x_range[0]) / (x_range[1] - x_range[0]) * img.shape[1], color='r', linestyle='--')
    if show:
        plt.show()
    return img


def grid_cmax(xs, ys, ts, ps, roi_size=(20, 20), step=None, warp=None, obj=None, min_events=10):
    """
    Contrast maximisation per tile of the sensor: the events of every roi (step[0] rows x step[1]
    columns, stepping by `step`, `roi_size` when step is None) are optimised on their own -- a grid-search
    start at blur 2.0, then a refinement at blur 1.0 from that point -- and the optimum is scored by the
    objective of the image of ALL events warped with it.  Signature and return (parameters, rois
    [y, x, step_y, step_x], scores) as events_cmax.py:28-76; like the reference a fresh
    variance_objective(adaptive_lifespan=True, minimum_events=105) is used for every roi whatever `obj`
    is, and a roi needs MORE than min_events events.
    """
    step = roi_size if step is None else step
    warp = linvel_warp() if warp is None else warp
    xs, ys, ts, ps = (np.asarray(a) for a in (xs, ys, ts, ps))
    resolution = infer_resolution(xs, ys)
    found, rois, scores = [], [], []
    for x_lo in range(0, int(resolution[1]), step[1]):
        in_cols = np.flatnonzero((xs >= x_lo) & (xs < x_lo + step[1]))
        ys_cols = ys[in_cols]
        for y_lo in range(0, int(resolution[0]), step[0]):
            sel = in_cols[(ys_cols >= y_lo) & (ys_cols < y_lo + step[0])]
            if len(sel) <= min_events:
                continue
            ex, ey, et, ep = xs[sel], ys[sel], ts[sel], ps[sel]
            roi_obj = variance_objective(adaptive_lifespan=True, minimum_events=105)
            start = optimize_contrast(ex, ey, et, ep, warp, roi_obj, numeric_grads=False, blur_sigma=2.0,
                                      img_size=resolution, grid_search_init=True)
            best = optimize_contrast(ex, ey, et, ep, warp, roi_obj, numeric_grads=False, blur_sigma=1.0,
                                     img_size=resolution, x0=start)
            iwe, _ = get_iwe(best, xs, ys, ts, ps, warp, resolution, use_polarity=True, compute_gradient=False)
            found.append(best)
            rois.append([y_lo, x_lo, step[0], step[1]])
            scores.append(roi_obj.evaluate_function(iwe=iwe))
    return found, rois, scores
