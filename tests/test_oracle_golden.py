"""The CPU oracle (oracle/evk_oracle.c) against the golden vectors generated from the REAL
reference (tests/golden/make_golden.py).  Runs without a GPU.  This is the oracle's pin."""
import numpy as np
import pytest

import cmax_scenes
from conftest import assert_close_to_max, golden


def test_voxel_torch_cases(oracle):
    g = golden("voxel_torch")
    for tag in "abcde":
        H, W = g[tag + "_HW"]
        out = oracle.voxel_f32(g[tag + "_x"], g[tag + "_y"], g[tag + "_t"], g[tag + "_p"], int(g[tag + "_B"]), (H, W))
        # sequential f32 accumulation in event order == torch CPU index_put_ order: bit exact
        assert np.array_equal(out, g[tag + "_out"]), tag


def test_voxel_negative_wrap_and_nan(oracle):
    g = golden("voxel_torch")
    out = oracle.voxel_f32(g["neg_x"], g["neg_y"], g["neg_t"], g["neg_p"], 3, tuple(g["neg_HW"]))
    assert np.array_equal(out, g["neg_out"])
    out = oracle.voxel_f32(g["nan_x"], g["nan_y"], g["nan_t"], g["nan_p"], 3, tuple(g["nan_HW"]))
    assert np.array_equal(np.isnan(out), np.isnan(g["nan_out"]))
    assert np.isnan(out).sum() == 6  # V[:, y, x] of both events


def test_voxel_oob_is_index_error(oracle):
    with pytest.raises(IndexError):
        oracle.voxel_f32([6.0], [0.0], [0.0], [1.0], 2, (4, 6))
    with pytest.raises(IndexError):
        oracle.voxel_f32([0.0, 1.0], [0.0, -5.0], [0.0, 1.0], [1.0, 1.0], 2, (4, 6))


def test_voxel_numpy_cases(oracle):
    g = golden("voxel_numpy")
    for tag in "ab":
        out = oracle.voxel_f64(g[tag + "_x"], g[tag + "_y"], g[tag + "_t"], g[tag + "_p"], int(g[tag + "_B"]),
                               tuple(g[tag + "_HW"]))
        assert_close_to_max(out, g[tag + "_out"], 1e-12, tag)
    with pytest.raises(IndexError):
        oracle.voxel_f64([-1], [0], [0.0], [1.0], 2, (4, 6))


IMG_VARIANTS = {
    "nearest_default": dict(),
    "nearest_nopad": dict(padding=False),
    "nearest_fill": dict(padding=False, default=7),
    "bilinear_default": dict(interpolation='bilinear'),
    "bilinear_nopad": dict(interpolation='bilinear', padding=False),
    "bilinear_fill": dict(interpolation='bilinear', default=2.5),
}


def test_image_variants(oracle):
    g = golden("image")
    hw = tuple(g["ev_HW"])
    for tag, kw in IMG_VARIANTS.items():
        out = oracle.image_torch_f32(g["ev_x"], g["ev_y"], g["ev_p"], sensor_size=hw, **kw)
        assert_close_to_max(out, g["img_" + tag], 2e-6, tag)
    out = oracle.image_torch_f32(g["in_x"], g["in_y"], g["in_p"], sensor_size=hw, clip_out_of_range=False)
    assert np.array_equal(out, g["img_noclip_nearest"])
    out = oracle.image_torch_f32(g["in_x"], g["in_y"], g["in_p"], sensor_size=hw, clip_out_of_range=False,
                                 interpolation='bilinear')
    assert_close_to_max(out, g["img_noclip_bilinear"], 2e-6)


def test_image_known_answers(oracle):
    g = golden("image")
    # SURVEY Appendix C1: clipped events dump their full weight at pixel (0,0)
    out = oracle.image_torch_f32(g["k1_x"], g["k1_y"], g["k1_p"], sensor_size=(4, 6))
    assert np.array_equal(out, g["k1_default"]) and out[0, 0] == 110 and out[1, 1] == 1 and out[2, 1] == 1000
    assert np.array_equal(oracle.image_torch_f32(g["k1_x"], g["k1_y"], g["k1_p"], sensor_size=(4, 6), padding=False), g["k1_nopad"])
    assert np.array_equal(oracle.image_torch_f32(g["k1_x"], g["k1_y"], g["k1_p"], sensor_size=(4, 6), clip_out_of_range=False), g["k1_noclip"])
    # C2: negative indices wrap, (-1,0) truncates to 0
    out = oracle.image_torch_f32(g["k2_x"], g["k2_y"], g["k2_p"], sensor_size=(4, 6), clip_out_of_range=False)
    assert np.array_equal(out, g["k2_noclip"]) and out[0, 0] == 1 and out[0, 5] == 110
    # C3: x == W without clipping -> IndexError
    with pytest.raises(IndexError):
        oracle.image_torch_f32([6.0], [0.0], [1.0], sensor_size=(4, 6), clip_out_of_range=False)
    # C4 bilinear incl. wrap of x = -0.25
    out = oracle.image_torch_f32(g["k4_x"], g["k4_y"], g["k4_p"], sensor_size=(4, 6), interpolation='bilinear')
    assert_close_to_max(out, g["k4_bilinear"], 1e-7)
    assert out.shape == (5, 7) and out[0, 0] == 7500 and out[0, 6] >= 2500


def test_timestamp_images(oracle):
    g = golden("tsimg")
    ev = [g[k] for k in "xytp"]
    for tag, kw in {"default": dict(), "reverse": dict(timestamp_reverse=True), "nopad": dict(padding=False)}.items():
        pos, neg = oracle.timestamp_image_f32(*ev, sensor_size=(40, 56), **kw)
        assert_close_to_max(pos, g[tag + "_pos"], 2e-6, tag)
        assert_close_to_max(neg, g[tag + "_neg"], 2e-6, tag)
    rel = (g["np_t"] - g["np_t"][0]).astype(np.float32)
    pos, neg = oracle.timestamp_image_f32(g["x"], g["y"], rel, g["p"], sensor_size=(40, 56))
    assert_close_to_max(pos, g["np_pos"], 2e-6)
    assert_close_to_max(neg, g["np_neg"], 2e-6)
    pos, neg = oracle.timestamp_image_f32(g["x"], g["y"], rel, g["p"], sensor_size=(40, 56), normalize_timestamps=False)
    assert_close_to_max(pos, g["np_raw_pos"], 2e-6)
    assert_close_to_max(neg, g["np_raw_neg"], 2e-6)


def test_flow_warp(oracle):
    g = golden("flow")
    xw, yw = oracle.warp_flow_f32(g["x"], g["y"], g["t"], g["flow"])
    assert_close_to_max(xw, g["xw"], 1e-6)
    assert_close_to_max(yw, g["yw"], 1e-6)
    xw, yw = oracle.warp_flow_f32(g["x"], g["y"], g["t"], g["flow"], t0=0.02)
    assert_close_to_max(xw, g["xw_t0"], 1e-6)
    assert_close_to_max(yw, g["yw_t0"], 1e-6)
    xw, yw = oracle.warp_flow_f32(g["k_x"], g["k_y"], g["k_t"], g["k_flow"])
    assert_close_to_max(xw, g["k_xw"], 1e-6)
    assert_close_to_max(yw, g["k_yw"], 1e-6)


def test_bounds_mask(oracle):
    g = golden("taps")
    assert np.array_equal(oracle.bounds_mask(g["m_x"], g["m_y"], 0, 240, 0, 180), g["m_out"])


def test_cmax_f_and_g(oracle):
    g = golden("cmax")
    scenes = {0: "c9", 1: "lat"}
    for row in g["evals"]:
        s, vx, vy, sigma, f_ref, g0, g1 = row
        tag = scenes[int(s)]
        f, grad = oracle.cmax_variance((vx, vy), *cmax_scenes.events(g, tag), blur_sigma=sigma)
        assert abs(f - f_ref) <= 1e-6 * abs(f_ref) + 1e-12, (tag, vx, vy, sigma, f, f_ref)
        gref = np.array([g0, g1])
        assert np.abs(grad - gref).max() <= 2e-5 * np.abs(gref).max() + 1e-9, (tag, vx, vy, sigma, grad, gref)


def test_cmax_images(oracle):
    g = golden("cmax")
    iwe, d = oracle.iwe_linvel((45.0, -20.0), g["lat_x"], g["lat_y"], g["lat_t"], g["lat_p"], (180, 240), True)
    assert iwe.shape == (181, 241) and d.shape == (2, 181, 241)
    assert_close_to_max(iwe, g["lat_iwe"], 2e-6)
    assert_close_to_max(d, g["lat_diwe"], 2e-6)
    iwe2, _ = oracle.iwe_linvel((45.0, -20.0), g["lat_x"], g["lat_y"], g["lat_t"], g["lat_p"], (120, 200), False,
                                use_polarity=False)
    assert_close_to_max(iwe2, g["lat_iwe_abs_small"], 2e-6)
    assert abs(oracle.variance_f(g["lat_iwe"], 1.0) - g["pre_f"]) <= 1e-6 * abs(g["pre_f"])
    gg = oracle.variance_g(g["lat_iwe"], g["lat_diwe"], 1.0)
    assert np.abs(gg - g["pre_g"]).max() <= 1e-5 * np.abs(g["pre_g"]).max()


def test_gaussian_matches_scipy(oracle):
    from scipy.ndimage import gaussian_filter
    rng = np.random.default_rng(3)
    for shape in [(181, 241), (2, 181, 241), (7, 5), (3,)]:
        a = rng.standard_normal(shape).astype(np.float32)
        for sigma in (0.5, 1.0, 2.3):
            assert_close_to_max(oracle.gaussian_filter_f32(a, sigma), gaussian_filter(a, sigma), 1e-6, str(shape))


def test_robust_norm(oracle):
    g = golden("robust_norm")
    for tag, kw in (("voxel", {}), ("normal", dict(low_perc=10, top_perc=90)), ("sparse", {})):
        out = oracle.robust_norm_f32(g[tag + "_in"], **kw)
        assert_close_to_max(out, g[tag + "_out"], 1e-7, tag)
    assert np.array_equal(oracle.robust_norm_f32(g["sparse_in"]), g["sparse_in"])



def test_zhu_objective_composition(oracle):
    """warp -> bounds mask -> timestamp images -> blur -> sum of squares (objectives.py:536-550) restated
    from the oracle's pieces against the golden of the reference's code"""
    c, z = golden("cmax"), golden("zhu")
    xs, ys, ts, ps = (c["lat" + k] for k in ("_x", "_y", "_t", "_p"))
    for key in z.files:
        _, vx, vy, tag = key.split("_")
        sigma = {"d": 2.0, "0": 0.0, "1": 1.0}[tag]
        lag = ts - ts[-1]
        xw, yw = xs - lag * float(vx), ys - lag * float(vy)
        m = oracle.bounds_mask(xw, yw, 0, 240, 0, 180)
        tm = ts * m
        pos, neg = oracle.timestamp_image_f32(xw * m, yw * m, tm - tm[0], ps * m)
        if sigma > 0:
            pos, neg = oracle.gaussian_filter_f32(pos, sigma), oracle.gaussian_filter_f32(neg, sigma)
        f = -(np.sum(pos * pos) + np.sum(neg * neg))
        assert abs(f - float(z[key])) <= 1e-5 * abs(float(z[key])), (key, f, float(z[key]))


def test_other_objectives(oracle):
    """rms / sos / soe / moa / isoa / sosa / r1 restated in the oracle against the reference's goldens"""
    g, c = golden("objectives"), golden("cmax")
    ev = [c["lat" + k] for k in ("_x", "_y", "_t", "_p")]
    for key in g.files:
        name, vx, vy, tag = key.split("_")
        ref = g[key]
        f, gr = oracle.cmax_objective(name, (float(vx), float(vy)), *ev, blur_sigma=None if tag == "d" else 0.0)
        assert abs(f - ref[0]) <= 1e-6 * abs(ref[0]), (key, f, ref[0])
        if name == "sos":
            assert gr is not None                       # the reference raises NameError; formula as written there
        elif np.isnan(ref[1]):
            assert gr is None
        else:
            assert np.abs(gr - ref[1:]).max() <= 1e-5 * np.abs(ref[1:]).max(), (key, gr, ref[1:])
