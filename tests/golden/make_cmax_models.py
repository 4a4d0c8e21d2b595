"""Generate tests/golden/cmax_models.npz by running the reference's OWN contrast-maximisation pipeline on CPU
(loaded through oracle/ref_loader.py) with the rotation and xyztheta motion models:

    EVK_REFERENCE_ROOT=<checkout of TimoStoff/event_utils> python tests/golden/make_cmax_models.py

get_iwe, events_to_image_drv, interpolate_to_image, interpolate_to_derivative_img and the objectives'
evaluate_function / evaluate_gradient are the reference's code.  Two things are not:
  * the warp object is this repository's numpy model (event_utils_b200/contrast_max/warps.py) -- the
    reference's two classes are empty stubs (warps.py:63-83);
  * image.py:210 allocates 2 derivative channels whatever the Jacobians hold; that one line is patched in
    memory to jacobian_x.shape[0] (interpolate_to_derivative_img, image.py:131-135, already loops over all
    channels).
The scenes are regenerated from their seeds (tests/cmax_model_scenes.py); only their SHA-256 is stored.
"""
import contextlib
import io
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import cmax_model_scenes as S  # noqa: E402
from event_utils_b200.contrast_max.warps import pure_rotation_warp, xyztheta_warp  # noqa: E402
from oracle import ref_loader  # noqa: E402

OUT = os.path.dirname(os.path.abspath(__file__))
ref = ref_loader.load()

# image.py:210, in memory only: one derivative channel per Jacobian row
_src = open(os.path.join(ref_loader.REF_ROOT, "lib", "representations", "image.py")).read()
_fn = _src[_src.index("def events_to_image_drv("):]
_fn = _fn[:_fn.index("\ndef ", 1)]
assert _fn.count("d_img = torch.zeros((2, *img_size))") == 1
_ns = dict(ref.image.__dict__)
exec(compile(_fn.replace("d_img = torch.zeros((2, *img_size))", "d_img = torch.zeros((jacobian_x.shape[0], *img_size))"),
             "image.py (patched line 210)", "exec"), _ns)
ref.image.events_to_image_drv = _ns["events_to_image_drv"]
ref.objectives.events_to_image_drv = _ns["events_to_image_drv"]

O = ref.objectives
OBJS = {"variance": O.variance_objective, "sos": O.sos_objective, "soe": O.soe_objective, "isoa": O.isoa_objective,
        "sosa": O.sosa_objective}
cases = {}
rows = []   # [scene, objective, sigma, params[4], f, g[4]]
points = {
    "rot": (pure_rotation_warp(), [S.ROTATION_TRUE, (110.0, 100.0, 1.0), (130.0, 80.0, -0.5)]),
    "rot_real": (pure_rotation_warp(), [(125.0, 85.0, 1.2)]),
    "xyz": (xyztheta_warp(), [S.XYZTHETA_TRUE, (30.0, -15.0, 0.5, -0.3), (45.0, -20.0, 0.0, 0.0)]),
}
for si, (tag, (warp, prms)) in enumerate(points.items()):
    xs, ys, ts, ps = S.SCENES[tag]()
    cases[tag + "_sha256"] = np.array(S.sha256((xs, ys, ts, ps)))
    for oi, (name, cls) in enumerate(OBJS.items()):
        for prm in prms:
            for sigma in (None, 0.0):
                o = cls()
                with contextlib.redirect_stdout(io.StringIO()):
                    f = o.evaluate_function(prm, xs, ys, ts, ps, warp, (180, 240), sigma)
                    try:
                        g = list(o.evaluate_gradient(prm, xs, ys, ts, ps, warp, (180, 240), sigma))
                    except NameError:          # sos: undefined find_lifespan (objectives.py:345)
                        g = [np.nan] * warp.dims
                s = o.default_blur if sigma is None else sigma
                rows.append([si, oi, s] + list(prm) + [np.nan] * (4 - len(prm)) + [f] + g + [np.nan] * (4 - len(g)))
    # the images of one point (get_iwe, objectives.py:165-199): stored as their sums per channel
    iwe, d = O.get_iwe(prms[0], xs, ys, ts, ps, warp, (180, 240), compute_gradient=True)
    cases[tag + "_iwe_sum"] = np.array([iwe.astype(np.float64).sum()] + [c.astype(np.float64).sum() for c in d])
    cases[tag + "_iwe_absum"] = np.array([np.abs(iwe).astype(np.float64).sum()] + [np.abs(c).astype(np.float64).sum() for c in d])
cases["scenes"] = np.array(list(points))
cases["objectives"] = np.array(list(OBJS))
cases["evals"] = np.array(rows, dtype=np.float64)
path = os.path.join(OUT, "cmax_models.npz")
np.savez_compressed(path, **cases)
print("cmax_models.npz %.1f KB, %d evaluations" % (os.path.getsize(path) / 1024, len(rows)))
