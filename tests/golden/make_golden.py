"""Generate the golden vectors in tests/golden/ by running the UNMODIFIED reference
(loaded through oracle/ref_loader.py):

    EVK_REFERENCE_ROOT=<checkout of TimoStoff/event_utils> python tests/golden/make_golden.py

The .npz files are committed; the tests only read them.
Every case stores its inputs and the reference's outputs.
"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import cmax_scenes  # noqa: E402
from oracle import ref_loader  # noqa: E402

OUT = os.path.dirname(os.path.abspath(__file__))
ref = ref_loader.load()
T = torch.tensor


def events(seed, n, H, W, frac=True, tscale=0.1, t_offset=0.0, pol="pm1"):
    rng = np.random.default_rng(seed)
    xs = rng.random(n) * (W - 1) if frac else rng.integers(0, W, n).astype(np.float64)
    ys = rng.random(n) * (H - 1) if frac else rng.integers(0, H, n).astype(np.float64)
    ts = np.sort(rng.random(n)) * tscale + t_offset
    if pol == "pm1":
        ps = rng.integers(0, 2, n) * 2.0 - 1.0
    elif pol == "ones":
        ps = np.ones(n)
    else:
        ps = rng.standard_normal(n)
    return xs, ys, ts, ps


def f32(*a):
    return [T(v, dtype=torch.float32) for v in a]


def save(name, **kw):
    path = os.path.join(OUT, name + ".npz")
    np.savez_compressed(path, **kw)
    print("%-28s %8.1f KB" % (name, os.path.getsize(path) / 1024))


# ---- voxel, torch f32 (voxel_grid.py:114-153) -------------------------------------------------
cases = {}
for tag, (seed, n, B, H, W, frac, pol) in {
    "a": (1, 6000, 5, 48, 64, True, "pm1"),
    "b": (2, 4000, 3, 30, 40, False, "ones"),
    "c": (3, 3000, 1, 20, 24, True, "real"),
    "d": (4, 5000, 9, 36, 52, True, "pm1"),
    "e": (5, 2, 5, 8, 8, True, "pm1"),
}.items():
    xs, ys, ts, ps = events(seed, n, H, W, frac=frac, pol=pol)
    xt, yt, tt, pt = f32(xs, ys, ts, ps)
    v = ref.voxel_grid.events_to_voxel_torch(xt, yt, tt, pt, B, sensor_size=(H, W)).numpy()
    cases.update({tag + "_x": xt.numpy(), tag + "_y": yt.numpy(), tag + "_t": tt.numpy(), tag + "_p": pt.numpy(),
                  tag + "_B": B, tag + "_HW": np.array([H, W]), tag + "_out": v})
# negative coordinates wrap (quirk B6), single timestamp -> NaN (A1)
xt, yt, tt, pt = f32([-0.5, -1.0, -1.5, 2.0], [0.0, 0.0, -2.0, 1.0], [0.0, 0.1, 0.2, 0.3], [1, 10, 100, 1000])
cases.update(dict(neg_x=xt.numpy(), neg_y=yt.numpy(), neg_t=tt.numpy(), neg_p=pt.numpy(), neg_B=3,
                  neg_HW=np.array([4, 6]),
                  neg_out=ref.voxel_grid.events_to_voxel_torch(xt, yt, tt, pt, 3, sensor_size=(4, 6)).numpy()))
xt, yt, tt, pt = f32([1.0, 2.0], [1.0, 3.0], [0.5, 0.5], [1, 1])
cases.update(dict(nan_x=xt.numpy(), nan_y=yt.numpy(), nan_t=tt.numpy(), nan_p=pt.numpy(), nan_B=3,
                  nan_HW=np.array([4, 6]),
                  nan_out=ref.voxel_grid.events_to_voxel_torch(xt, yt, tt, pt, 3, sensor_size=(4, 6)).numpy()))
# neg/pos split (voxel_grid.py:155-182)
xs, ys, ts, ps = events(6, 3000, 24, 32)
xt, yt, tt, pt = f32(xs, ys, ts, ps)
vp, vn = ref.voxel_grid.events_to_neg_pos_voxel_torch(xt, yt, tt, pt, 4, sensor_size=(24, 32))
cases.update(dict(np_x=xt.numpy(), np_y=yt.numpy(), np_t=tt.numpy(), np_p=pt.numpy(), np_B=4,
                  np_HW=np.array([24, 32]), np_pos=vp.numpy(), np_neg=vn.numpy()))
save("voxel_torch", **cases)

# ---- voxel, numpy f64 (voxel_grid.py:184-217) --------------------------------------------------
cases = {}
for tag, (seed, n, B, H, W, toff) in {"a": (11, 5000, 5, 40, 56, 0.0), "b": (12, 3000, 4, 26, 34, 1.6e9)}.items():
    rng = np.random.default_rng(seed)
    xs = rng.integers(0, W + 1, n)   # includes x == W: dropped by the canvas crop
    ys = rng.integers(0, H + 1, n)
    ts = np.sort(rng.random(n)) * 0.05 + toff
    ps = rng.integers(0, 2, n) * 2.0 - 1.0
    v = ref.voxel_grid.events_to_voxel(xs, ys, ts, ps, B, sensor_size=(H, W))
    cases.update({tag + "_x": xs, tag + "_y": ys, tag + "_t": ts, tag + "_p": ps, tag + "_B": B,
                  tag + "_HW": np.array([H, W]), tag + "_out": v})
save("voxel_numpy", **cases)

# ---- event images (image.py:5-115) ----------------------------------------------------------
cases = {}
xs, ys, ts, ps = events(21, 5000, 40, 56, pol="real")
# push some events beyond the clip thresholds
xs[::17] += 3.0
ys[::23] += 2.5
xt, yt, pt = f32(xs, ys, ps)
cases.update(dict(ev_x=xt.numpy(), ev_y=yt.numpy(), ev_p=pt.numpy(), ev_HW=np.array([40, 56])))
variants = {
    "nearest_default": dict(),
    "nearest_nopad": dict(padding=False),
    "nearest_fill": dict(padding=False, default=7),
    "bilinear_default": dict(interpolation='bilinear'),
    "bilinear_nopad": dict(interpolation='bilinear', padding=False),
    "bilinear_fill": dict(interpolation='bilinear', default=2.5),
}
for tag, kw in variants.items():
    cases["img_" + tag] = ref.image.events_to_image_torch(xt, yt, pt, sensor_size=(40, 56), **kw).numpy()
# in-range stream without clipping
xs2, ys2, _, ps2 = events(22, 4000, 40, 56, pol="pm1")
xt2, yt2, pt2 = f32(xs2, ys2, ps2)
cases.update(dict(in_x=xt2.numpy(), in_y=yt2.numpy(), in_p=pt2.numpy()))
cases["img_noclip_nearest"] = ref.image.events_to_image_torch(xt2, yt2, pt2, sensor_size=(40, 56), clip_out_of_range=False).numpy()
cases["img_noclip_bilinear"] = ref.image.events_to_image_torch(xt2, yt2, pt2, sensor_size=(40, 56), clip_out_of_range=False, interpolation='bilinear').numpy()
# Appendix C known answers (SURVEY.md)
kx, ky, kp = f32([1, 5, 2, 1.9], [1, 1, 3, 2.9], [1, 10, 100, 1000])
cases.update(dict(k1_x=kx.numpy(), k1_y=ky.numpy(), k1_p=kp.numpy()))
cases["k1_default"] = ref.image.events_to_image_torch(kx, ky, kp, sensor_size=(4, 6)).numpy()
cases["k1_nopad"] = ref.image.events_to_image_torch(kx, ky, kp, sensor_size=(4, 6), padding=False).numpy()
cases["k1_noclip"] = ref.image.events_to_image_torch(kx, ky, kp, sensor_size=(4, 6), clip_out_of_range=False).numpy()
kx, ky, kp = f32([-0.5, -1.0, -1.5], [0, 0, 0], [1, 10, 100])
cases.update(dict(k2_x=kx.numpy(), k2_y=ky.numpy(), k2_p=kp.numpy()))
cases["k2_noclip"] = ref.image.events_to_image_torch(kx, ky, kp, sensor_size=(4, 6), clip_out_of_range=False).numpy()
kx, ky, kp = f32([1.25, 5.5, 5.999, 6.0, -0.25], [1.5, 3.5, 0, 0, 0], [1, 10, 100, 1000, 10000])
cases.update(dict(k4_x=kx.numpy(), k4_y=ky.numpy(), k4_p=kp.numpy()))
cases["k4_bilinear"] = ref.image.events_to_image_torch(kx, ky, kp, sensor_size=(4, 6), interpolation='bilinear').numpy()
# numpy flavour (image.py:5-44)
rng = np.random.default_rng(23)
xi, yi = rng.integers(0, 57, 3000), rng.integers(0, 41, 3000)
pi = rng.standard_normal(3000)
cases.update(dict(np_x=xi, np_y=yi, np_p=pi))
cases["np_nearest"] = ref.image.events_to_image(xi, yi, pi, sensor_size=(40, 56))
cases["np_meanval"] = ref.image.events_to_image(xi, yi, pi, sensor_size=(40, 56), meanval=True, default=-1)
save("image", **cases)

# ---- timestamp images (image.py:219-353) ------------------------------------------------------
cases = {}
rng = np.random.default_rng(51)
n = 6000
xs = (rng.random(n) * 60 - 1).astype(np.float32)      # a few negative coordinates (wrap)
ys = (rng.random(n) * 44).astype(np.float32)
xs[::19] += 3                                          # and some beyond the clip threshold
ts = (np.sort(rng.random(n)) * 0.3 + 2).astype(np.float32)
ps = (rng.integers(0, 2, n) * 2 - 1).astype(np.float32)
cases.update(dict(x=xs, y=ys, t=ts, p=ps))
for tag, kw in {"default": dict(), "reverse": dict(timestamp_reverse=True), "nopad": dict(padding=False)}.items():
    a, b = ref.image.events_to_timestamp_image_torch(T(xs), T(ys), T(ts), T(ps), sensor_size=(40, 56), **kw)
    cases[tag + "_pos"], cases[tag + "_neg"] = a.numpy(), b.numpy()
t64 = ts.astype(np.float64) + 1.6e9
a, b = ref.image.events_to_timestamp_image(xs.astype(np.float64), ys.astype(np.float64), t64, ps.astype(np.float64), sensor_size=(40, 56))
cases.update(dict(np_t=t64, np_pos=a, np_neg=b))
# normalize_timestamps=False (image.py:261): the weights are the stamps relative to ts[0], not divided by the span
a, b = ref.image.events_to_timestamp_image(xs.astype(np.float64), ys.astype(np.float64), t64, ps.astype(np.float64), sensor_size=(40, 56),
                                           normalize_timestamps=False)
cases.update(dict(np_raw_pos=a, np_raw_neg=b))
save("tsimg", **cases)

# ---- lower-level helpers (image.py:102-160) and the bounds mask -------------------------------
cases = {}
rng = np.random.default_rng(31)
n = 2000
px, py = rng.integers(-3, 20, n), rng.integers(-2, 14, n)   # negatives wrap
dx, dy = rng.random(n).astype(np.float32), rng.random(n).astype(np.float32)
w = rng.standard_normal(n).astype(np.float32)
img = torch.zeros(16, 22)
ref.image.interpolate_to_image(T(px), T(py), T(dx), T(dy), T(w), img)
w1, w2 = rng.standard_normal((2, n)).astype(np.float32), rng.standard_normal((2, n)).astype(np.float32)
dimg = torch.zeros(2, 16, 22)
ref.image.interpolate_to_derivative_img(T(px), T(py), T(dx), T(dy), dimg, T(w1), T(w2))
cases.update(dict(px=px, py=py, dx=dx, dy=dy, w=w, w1=w1, w2=w2, img=img.numpy(), dimg=dimg.numpy()))
xe, ye = rng.random(n) * 23 - 0.5, rng.random(n) * 16 - 0.5
src = rng.standard_normal((16, 22)).astype(np.float32)
cases.update(dict(g_x=xe, g_y=ye, g_img=src, g_out=ref.image.image_to_event_weights(xe, ye, src)))
mx, my = np.array([0, 1e-9, 240, 240.1, 5, 5]), np.array([5, 5, 5, 5, 0, 180.0])
cases.update(dict(m_x=mx, m_y=my, m_out=ref.event_util.events_bounds_mask(mx, my, 0, 240, 0, 180)))
# events_to_image_drv with general Jacobians
xs, ys, ts, ps = events(32, 3000, 180, 240, pol="real")
xs[::11] += 5
jx, jy = rng.standard_normal((2, 3000)), rng.standard_normal((2, 3000))
i0, d0 = ref.image.events_to_image_drv(xs, ys, ps, jx, jy, compute_gradient=True)
cases.update(dict(drv_x=xs, drv_y=ys, drv_p=ps, drv_jx=jx, drv_jy=jy, drv_img=i0, drv_dimg=d0))
save("taps", **cases)

# ---- dense-flow warp (optic_flow.py:5-46) ------------------------------------------------------
cases = {}
xs, ys, ts, ps = events(41, 4000, 30, 44)
xs[::9] -= 1.0  # some events left of the field
ys[::13] += 1.5
xt, yt, tt, pt = f32(xs, ys, ts, ps)
flow = torch.randn(2, 30, 44, generator=torch.Generator().manual_seed(5)) * 40
xw, yw = ref.optic_flow.warp_events_flow_torch(xt, yt, tt, pt, flow)
xw2, yw2 = ref.optic_flow.warp_events_flow_torch(xt.unsqueeze(1), yt.unsqueeze(1), tt.unsqueeze(1), pt.unsqueeze(1),
                                                 flow.unsqueeze(0), t0=0.02)
cases.update(dict(x=xt.numpy(), y=yt.numpy(), t=tt.numpy(), p=pt.numpy(), flow=flow.numpy(), xw=xw.numpy(),
                  yw=yw.numpy(), xw_t0=xw2.numpy(), yw_t0=yw2.numpy()))
fl = torch.zeros(2, 4, 6)
fl[0] = 10 * torch.arange(6.0)[None, :]
fl[1] = 100 * torch.arange(4.0)[:, None]
kx, ky, kt, kp = f32([2.5, 5, 5.5, -0.5], [1.5, 3, 3, 0], [0.0, 0.1, 0.2, 1.0], [1, 1, 1, 1])
a, b = ref.optic_flow.warp_events_flow_torch(kx, ky, kt, kp, fl)
cases.update(dict(k_x=kx.numpy(), k_y=ky.numpy(), k_t=kt.numpy(), k_flow=fl.numpy(), k_xw=a.numpy(), k_yw=b.numpy()))
save("flow", **cases)

# ---- contrast maximisation (objectives.py:165-264) --------------------------------------------
cases = {}
obj, warp = ref.objectives.variance_objective(), ref.warps.linvel_warp()


def lattice(seed, n, v=(60.0, -35.0), T_=0.05, noise=0.2):
    rng = np.random.default_rng(seed)
    ts = np.sort(rng.random(n)) * T_
    k = rng.integers(1, 11, n) * 20.0
    along = rng.random(n)
    vertical = rng.random(n) < 0.5
    xr = np.where(vertical, k, along * 239)
    yr = np.where(vertical, along * 179, np.minimum(k, 170.0))
    xs = xr + (ts - ts[-1]) * v[0]
    ys = yr + (ts - ts[-1]) * v[1]
    ps = np.ones(n)
    m = rng.random(n) < noise
    xs[m], ys[m] = rng.random(m.sum()) * 239, rng.random(m.sum()) * 179
    ps[m] = rng.integers(0, 2, m.sum()) * 2.0 - 1
    return xs, ys, ts, ps


scenes = {
    "c9": events(0, 20000, 180, 240),  # SURVEY Appendix C9 draw order is reproduced below
    "lat": lattice(7, 30000),
}
scenes["c9"] = cmax_scenes.c9_events()
cases["c9_sha256"] = np.array(cmax_scenes.c9_sha256(scenes["c9"]))     # regenerated by the tests, not stored
cases.update({"lat" + k: a for k, a in zip(("_x", "_y", "_t", "_p"), scenes["lat"])})
evals = []
for sname, (xs, ys, ts, ps) in scenes.items():
    for params in [(30.0, -20.0), (60.0, -35.0), (45.0, -20.0), (0.0, 0.0)]:
        for sigma in (1.0, 0.0, 2.3):
            f = obj.evaluate_function(params, xs, ys, ts, ps, warp, (180, 240), sigma)
            g = obj.evaluate_gradient(params, xs, ys, ts, ps, warp, (180, 240), sigma)
            evals.append([{"c9": 0, "lat": 1}[sname], params[0], params[1], sigma, f, g[0], g[1]])
cases["evals"] = np.array(evals)
xs, ys, ts, ps = scenes["lat"]
iwe, diwe = ref.objectives.get_iwe((45.0, -20.0), xs, ys, ts, ps, warp, (180, 240), compute_gradient=True)
cases.update(dict(lat_iwe=iwe, lat_diwe=diwe))
iwe2, _ = ref.objectives.get_iwe((45.0, -20.0), xs, ys, ts, ps, warp, (120, 200), use_polarity=False)
cases["lat_iwe_abs_small"] = iwe2
# img_size larger than the fixed sensor: events beyond (180,240) get zero weight (quirk B7)
f_big = obj.evaluate_function((30.0, -20.0), scenes["c9"][0] * 2, scenes["c9"][1] * 2, scenes["c9"][2], scenes["c9"][3],
                              warp, (480, 640), 1.0)
cases["c9_f_big"] = f_big
# precomputed-image form
cases["pre_f"] = obj.evaluate_function(iwe=iwe, blur_sigma=1.0)
cases["pre_g"] = obj.evaluate_gradient(iwe=iwe, d_iwe=diwe, blur_sigma=1.0)
# adaptive lifespan branch (objectives.py:217-225, 244-249)
o2 = ref.objectives.variance_objective(adaptive_lifespan=True, minimum_events=5000)
o2.iter_update((60.0, -35.0))
import io, contextlib
with contextlib.redirect_stdout(io.StringIO()):
    fa = o2.evaluate_function((50.0, -30.0), xs, ys, ts, ps, warp, (180, 240), 1.0)
    ga = o2.evaluate_gradient((50.0, -30.0), xs, ys, ts, ps, warp, (180, 240), 1.0)
cases.update(dict(adapt_f=fa, adapt_g=ga, adapt_sidx=o2.s_idx))
save("cmax", **cases)

# ---- the other objective functions (objectives.py:266-596) on the lattice scene --------------------
cases = {}
O = ref.objectives
objs = {"rms": O.rms_objective(), "sos": O.sos_objective(), "soe": O.soe_objective(), "moa": O.moa_objective(),
        "isoa": O.isoa_objective(), "sosa": O.sosa_objective(), "r1": O.r1_objective()}
xs, ys, ts, ps = scenes["lat"]
for name, o in objs.items():
    for prm in [(45.0, -20.0), (60.0, -35.0)]:
        for tag, sigma in (("d", None), ("0", 0.0)):      # default blur of the objective, and no blur
            f = o.evaluate_function(prm, xs, ys, ts, ps, warp, (180, 240), sigma)
            try:
                gr = o.evaluate_gradient(prm, xs, ys, ts, ps, warp, (180, 240), sigma)
            except (NameError, TypeError):                # sos: undefined find_lifespan; moa: other signature
                gr = None
            gr = [np.nan, np.nan] if gr is None else list(gr)
            cases["%s_%g_%g_%s" % (name, prm[0], prm[1], tag)] = np.array([f] + gr, dtype=np.float64)
save("objectives", **cases)

# ---- zhu_timestamp_objective (objectives.py:524-558) ------------------------------------------------
# As shipped it raises NameError: it calls `events_to_zhu_timestamp_image`, which exists nowhere in the
# reference.  The golden is the reference's own code with that one name bound to the function it evidently
# means, events_to_timestamp_image (image.py:219-284), through an adapter that drops the two keyword
# arguments that function does not take.
def _zhu_images(xs, ys, ts, ps, compute_gradient=False, showimg=False):
    return ref.image.events_to_timestamp_image(xs, ys, ts, ps)


O.events_to_zhu_timestamp_image = _zhu_images
cases = {}
xs, ys, ts, ps = scenes["lat"]
for prm in [(45.0, -20.0), (60.0, -35.0), (0.0, 0.0)]:
    for tag, sigma in (("d", None), ("0", 0.0), ("1", 1.0)):
        cases["zhu_%g_%g_%s" % (prm[0], prm[1], tag)] = np.array(
            O.zhu_timestamp_objective().evaluate_function(prm, xs, ys, ts, ps, warp, (180, 240), sigma), dtype=np.float64)
save("zhu", **cases)

# ---- RobustNorm (data_augmentation.py:75-136) ----------------------------------------------------
import importlib.util
spec = importlib.util.spec_from_file_location("ref_data_augmentation", os.path.join(ref_loader.REF_ROOT, "lib/data_loaders/data_augmentation.py"))
da = importlib.util.module_from_spec(spec)
spec.loader.exec_module(da)
cases = {}
rng = np.random.default_rng(61)
v1 = torch.from_numpy(ref.voxel_grid.events_to_voxel_torch(*f32(*events(62, 30000, 60, 80)), 5, sensor_size=(60, 80)).numpy())
v2 = torch.from_numpy(rng.standard_normal((3, 17, 23)).astype(np.float32))
v3 = torch.zeros(2, 8, 8); v3[0, 1, 1] = 5.0          # 95th percentile and minimum are both 0 -> returned unchanged
for tag, v, kw in (("voxel", v1, {}), ("normal", v2, dict(low_perc=10, top_perc=90)), ("sparse", v3, {})):
    cases[tag + "_in"] = v.numpy()
    cases[tag + "_out"] = da.RobustNorm(**kw)(v).numpy()
    cases[tag + "_p"] = np.array([da.RobustNorm.percentile(v, q) for q in (0, 5, 50, 95, 100)])
save("robust_norm", **cases)

