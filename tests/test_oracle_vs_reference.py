"""The oracle against what the UNMODIFIED reference returned for the same seeded inputs (stored in
tests/golden/vs_reference.npz by tests/golden/make_reference_checks.py).  Larger, randomised companions
of the other golden vectors; outputs too large to store whole are compared in the sampled form of
tests/sampled.py."""
import numpy as np
import pytest
import torch

import sampled
from conftest import golden, make_events

K, NBLOCKS = 1024, 128
VOXEL_CASES = [(1, 200000, 5, 260, 346), (2, 50000, 7, 180, 240), (3, 1000, 2, 10, 12)]
IMAGE_KW = [dict(), dict(interpolation='bilinear'), dict(padding=False),
            dict(interpolation='bilinear', padding=False), dict(clip_out_of_range=False)]
CMAX_SIGMAS = [1.0, 0.0, 3.0]
CMAX_PARAMS = [(30.0, -20.0), (-400.0, 900.0)]
OTHER_OBJECTIVES = ["rms", "sos", "soe", "moa", "isoa", "sosa", "r1"]
WITH_GRADIENT = ("rms", "soe", "isoa", "sosa")
OTHER_PARAMS = [(25.0, -40.0), (-300.0, 120.0)]
OTHER_SIGMAS = (None, 0.0, 1.7)


def voxel_numpy_events():
    rng = np.random.default_rng(1234)
    n = 100000
    xs, ys = rng.integers(0, 346, n), rng.integers(0, 260, n)
    ts = np.sort(rng.random(n))
    ps = rng.integers(0, 2, n) * 2 - 1.0
    return xs, ys, ts, ps


def image_events(kw):
    x, y, t, p = make_events(5, 100000, 180, 240, pol="real")
    if kw.get("clip_out_of_range", True):
        x[::7] += 4
    return x, y, p


def flow_field():
    return (torch.randn(2, 180, 240, generator=torch.Generator().manual_seed(6)) * 30).numpy()


def find_new_range_inputs():
    rng = np.random.default_rng(0)
    for _ in range(500):
        axis = np.sort(rng.uniform(-200, 200, rng.integers(3, 9)))
        value = rng.choice(axis) if rng.random() < 0.7 else rng.uniform(-250, 250)
        yield axis, value


def window_inputs():
    rng = np.random.default_rng(3)
    ts = np.sort(rng.uniform(5.0, 7.5, 20000))
    ts[100:110] = ts[100]                                   # repeated stamps
    frame_ts = np.concatenate((np.sort(rng.uniform(5.0, 7.5, 30)), [9.0]))
    return ts, frame_ts


def window_methods():
    for k, w in ((1000, 0), (1500, 500), (333, 33)):
        yield "k_%d_%d" % (k, w), {"method": "k_events", "k": k, "sliding_window_w": w}
    for t, w in ((0.1, 0.0), (0.25, 0.05), (0.013, 0.0)):
        yield "t_%g_%g" % (t, w), {"method": "t_seconds", "t": t, "sliding_window_t": w}
    for nf in (1, 7, 40):
        yield "frames_%d" % nf, {"method": "fixed_frames", "num_frames": nf}
    yield "between_frames", {"method": "between_frames"}


@pytest.fixture(scope="module")
def ref():
    return golden("vs_reference")


def check(a, g, name, rel):
    assert tuple(np.shape(a)) == tuple(g[name + "_shape"]), (name, np.shape(a), g[name + "_shape"])
    sampled.check(a, g[name + "_val"], g[name + "_bsum"], g[name + "_max"], g[name + "_nan"], K, NBLOCKS, rel, name)


@pytest.mark.parametrize("seed,n,B,H,W", VOXEL_CASES)
def test_voxel_torch_bit_exact(ref, oracle, seed, n, B, H, W):
    x, y, t, p = make_events(seed, n, H, W)
    check(oracle.voxel_f32(x, y, t, p, B, (H, W)), ref, "voxel_torch_%d" % seed, 1e-6)


def test_voxel_numpy(ref, oracle):
    xs, ys, ts, ps = voxel_numpy_events()
    check(oracle.voxel_f64(xs, ys, ts, ps, 5, (260, 346)), ref, "voxel_numpy", 1e-12)


@pytest.mark.parametrize("kw", IMAGE_KW)
def test_image_torch(ref, oracle, kw):
    x, y, p = image_events(kw)
    check(oracle.image_torch_f32(x, y, p, **kw), ref, "image_%d" % IMAGE_KW.index(kw), 2e-6)


def test_flow(ref, oracle):
    x, y, t, p = make_events(6, 50000, 180, 240)
    xo, yo = oracle.warp_flow_f32(x, y, t, flow_field())
    check(xo, ref, "flow_x", 1e-6)
    check(yo, ref, "flow_y", 1e-6)


@pytest.mark.parametrize("sigma", CMAX_SIGMAS)
def test_cmax(ref, oracle, sigma):
    x, y, t, p = make_events(7, 100000, 180, 240, dtype=np.float64)
    for params, (f, g0, g1, scale) in zip(CMAX_PARAMS, ref["cmax_sigma_%g" % sigma]):
        fo, go = oracle.cmax_variance(params, x, y, t, p, blur_sigma=sigma)
        assert abs(fo - f) <= 1e-6 * abs(f)
        assert np.abs(go - np.array([g0, g1])).max() <= 1e-5 * scale


def test_find_new_range_matches_reference(ref):
    """the grid-search driver's interval update (events_cmax.py:160-182), host logic only"""
    from event_utils_b200.contrast_max.events_cmax import find_new_range
    expected = ref["find_new_range"]
    for i, (axis, value) in enumerate(find_new_range_inputs()):
        assert np.array_equal(expected[i], np.asarray(find_new_range(axis, value))), (axis, value)
    assert i + 1 == len(expected)


def test_window_tables_match_reference_loader(ref):
    """k_events / t_seconds / fixed_frames / between_frames tables of BaseVoxelDataset
    (base_dataset.py:322-417), built here vectorised"""
    from event_utils_b200.data_loaders import windows as Wn
    ts, frame_ts = window_inputs()
    for key, m in window_methods():
        if m["method"] == "k_events":
            got = Wn.k_event_indices(len(ts), m["k"], m["sliding_window_w"])
        elif m["method"] == "t_seconds":
            got = Wn.timeblock_indices(ts, m["t"], m["sliding_window_t"])
        elif m["method"] == "fixed_frames":
            got = Wn.fixed_frames_indices(ts, m["num_frames"])
        else:
            got = Wn.between_frame_indices(ts, frame_ts)
        assert np.array_equal(ref["windows_" + key], np.asarray(got)), key
    with pytest.raises(Exception):
        Wn.check_event_indices(Wn.k_event_indices(1000, 300, 0).tolist() + [[900, 1200]], 1000)


@pytest.mark.parametrize("name", OTHER_OBJECTIVES)
def test_other_objectives_random_scene(ref, oracle, name):
    x, y, t, p = make_events(17, 60000, 180, 240, dtype=np.float64)
    rows = iter(ref["objective_" + name])
    for params in OTHER_PARAMS:
        for sigma in OTHER_SIGMAS:
            f, g0, g1 = next(rows)
            fo, go = oracle.cmax_objective(name, params, x, y, t, p, blur_sigma=sigma)
            assert abs(fo - f) <= 1e-6 * max(abs(f), 1e-12), (name, params, sigma)
            if name in WITH_GRADIENT:
                g = np.array([g0, g1])
                assert np.abs(go - g).max() <= 1e-5 * max(np.abs(g).max(), 1e-9), (name, params, sigma)
