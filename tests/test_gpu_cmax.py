"""Parity of the fused contrast-maximisation kernel with the oracle and the reference goldens."""
import copy

import numpy as np
import pytest

import cmax_scenes
from conftest import assert_close_to_max, golden, make_events

pytestmark = pytest.mark.gpu


@pytest.fixture(autouse=True)
def _reset():
    from event_utils_b200.contrast_max import objectives
    objectives.precision = "f64"
    objectives.clear_cache()
    yield
    objectives.precision = "f64"
    objectives.clear_cache()


def grad_scale(iwe, d):
    """scale-normalised gradient tolerance of SURVEY.md section 8d"""
    return np.sqrt(np.mean((2 * (iwe - iwe.mean())) ** 2) * np.mean(d.astype(np.float64) ** 2))


def test_golden_f_and_g():
    from event_utils_b200.contrast_max.objectives import variance_objective
    from event_utils_b200.contrast_max.warps import linvel_warp
    g = golden("cmax")
    obj, warp = variance_objective(), linvel_warp()
    scenes = {0: "c9", 1: "lat"}
    for row in g["evals"]:
        s, vx, vy, sigma, f_ref, g0, g1 = row
        tag = scenes[int(s)]
        ev = cmax_scenes.events(g, tag)
        f = obj.evaluate_function((vx, vy), *ev, warp, (180, 240), sigma)
        gr = obj.evaluate_gradient((vx, vy), *ev, warp, (180, 240), sigma)
        assert isinstance(f, float) and isinstance(gr, np.ndarray) and gr.shape == (2,)
        assert abs(f - f_ref) <= 1e-5 * abs(f_ref) + 1e-12, (tag, vx, vy, sigma, f, f_ref)
        gref = np.array([g0, g1])
        # scale-normalised bound (1e-5 * sqrt(mean((2(I-mu))^2) mean(D^2))), plus the relative
        # bound on the structured scene where |g| is not ~0
        assert np.abs(gr - gref).max() <= 1e-5 * max(np.abs(gref).max(), 1e-4), (tag, vx, vy, sigma, gr, gref)
    # keyword calling convention (grid_search_initial, events_cmax.py:301-302)
    ev = [g["lat" + k] for k in ("_x", "_y", "_t", "_p")]
    f_kw = obj.evaluate_function(params=(45.0, -20.0), xs=ev[0], ys=ev[1], ts=ev[2], ps=ev[3], warpfunc=warp,
                                 img_size=(180, 240), blur_sigma=1.0)
    f_pos = obj.evaluate_function((45.0, -20.0), *ev, warp, (180, 240), 1.0)
    assert f_kw == f_pos
    # default blur (blur_sigma=None -> default_blur = 1.0)
    assert obj.evaluate_function((45.0, -20.0), *ev, warp, (180, 240), None) == f_pos


def test_get_iwe_and_precomputed_forms():
    from event_utils_b200.contrast_max.objectives import get_iwe, variance_objective
    from event_utils_b200.contrast_max.warps import linvel_warp
    g = golden("cmax")
    ev = [g["lat" + k] for k in ("_x", "_y", "_t", "_p")]
    warp, obj = linvel_warp(), variance_objective()
    iwe, d = get_iwe((45.0, -20.0), *ev, warp, (180, 240), compute_gradient=True)
    assert iwe.dtype == np.float32 and iwe.shape == (181, 241) and d.shape == (2, 181, 241)
    assert_close_to_max(iwe, g["lat_iwe"], 1e-5)
    assert_close_to_max(d, g["lat_diwe"], 1e-5)
    iwe0, d0 = get_iwe((45.0, -20.0), *ev, warp, (180, 240))
    assert d0 is None
    assert_close_to_max(iwe0, g["lat_iwe"], 1e-5)
    iwe2, _ = get_iwe((45.0, -20.0), *ev, warp, (120, 200), use_polarity=False)
    assert_close_to_max(iwe2, g["lat_iwe_abs_small"], 1e-5)
    # generic (non-fused) path: a user-defined warp object without `fused_kind`
    class my_warp(linvel_warp):
        fused_kind = None
    iwe3, d3, (xw, yw), contrast = get_iwe((45.0, -20.0), *ev, my_warp(), (180, 240), compute_gradient=True,
                                           return_events=True, return_per_event_contrast=True)
    assert_close_to_max(iwe3, g["lat_iwe"], 1e-5)
    assert_close_to_max(d3, g["lat_diwe"], 1e-5)
    assert xw.shape == ev[0].shape and contrast.shape == ev[0].shape
    f3 = variance_objective().evaluate_function((45.0, -20.0), *ev, my_warp(), (180, 240), 1.0)
    assert abs(f3 - obj.evaluate_function((45.0, -20.0), *ev, warp, (180, 240), 1.0)) <= 1e-5 * abs(f3)
    # precomputed-image forms (grid_cmax, events_cmax.py:68-70)
    assert abs(obj.evaluate_function(iwe=g["lat_iwe"], blur_sigma=1.0) - g["pre_f"]) <= 1e-5 * abs(g["pre_f"])
    gp = obj.evaluate_gradient(iwe=g["lat_iwe"], d_iwe=g["lat_diwe"], blur_sigma=1.0)
    assert np.abs(gp - g["pre_g"]).max() <= 1e-5 * np.abs(g["pre_g"]).max()
    # img_size larger than the fixed 180x240 sensor (quirk B7)
    c9 = cmax_scenes.events(g, "c9")
    fb = obj.evaluate_function((30.0, -20.0), c9[0] * 2, c9[1] * 2, c9[2], c9[3], warp, (480, 640), 1.0)
    assert abs(fb - g["c9_f_big"]) <= 1e-5 * abs(g["c9_f_big"])


def test_adaptive_lifespan_and_object_protocol():
    from event_utils_b200.contrast_max.objectives import variance_objective
    from event_utils_b200.contrast_max.warps import linvel_warp
    g = golden("cmax")
    ev = [g["lat" + k] for k in ("_x", "_y", "_t", "_p")]
    o2 = variance_objective(adaptive_lifespan=True, minimum_events=5000)
    assert o2.has_derivative and o2.name == "variance" and o2.default_blur == 1.0
    o2.iter_update((60.0, -35.0))
    fa = o2.evaluate_function((50.0, -30.0), *ev, linvel_warp(), (180, 240), 1.0)
    ga = o2.evaluate_gradient((50.0, -30.0), *ev, linvel_warp(), (180, 240), 1.0)
    assert o2.s_idx == int(g["adapt_sidx"])
    assert abs(fa - g["adapt_f"]) <= 1e-5 * abs(g["adapt_f"])
    assert np.abs(ga - g["adapt_g"]).max() <= 1e-5 * np.abs(g["adapt_g"]).max()
    o3 = copy.deepcopy(o2)
    o3.adaptive_lifespan = False
    assert o3.s_idx == o2.s_idx and o3._memo is None
    w = linvel_warp()
    assert w.dims == 2 and w.name == "linvel_warp"
    xw, yw, jx, jy = w.warp(ev[0], ev[1], ev[2], ev[3], ev[2][-1], (3.0, 4.0), compute_grad=True)
    assert jx.shape == (2, len(ev[0])) and np.all(jx[1] == 0) and np.all(jy[0] == 0)


def _moving_points(rng, n_pts, per_pt, x_lo, x_hi, v, span=0.04):
    """points at rest positions inside [x_lo, x_hi) x [30, 150) seen at random times, moving with velocity v"""
    x_ref = np.repeat(rng.uniform(x_lo, x_hi, n_pts), per_pt)
    y_ref = np.repeat(rng.uniform(30, 150, n_pts), per_pt)
    t = rng.uniform(0, span, n_pts * per_pt)
    return x_ref + (t - span) * v[0], y_ref + (t - span) * v[1], t


def test_grid_search_optimisation_and_objective_surface(oracle):
    from event_utils_b200.contrast_max import objectives as O
    from event_utils_b200.contrast_max.events_cmax import grid_search_optimisation, sample_objective_function
    from event_utils_b200.contrast_max.warps import linvel_warp
    rng = np.random.default_rng(21)
    v_true = (60.0, -35.0)
    x, y, t = _moving_points(rng, 300, 40, 30, 210, v_true)
    order = np.argsort(t)
    x, y, t = x[order], y[order], t[order]
    t[-1] = 0.04
    p = np.ones_like(t)
    out = grid_search_optimisation(x, y, t, p, linvel_warp(), O.variance_objective(), (180, 240), th0=2)
    assert np.abs(np.array(out["min_params"]) - np.array(v_true)).max() < 4.0, out["min_params"]
    f_true = O.variance_objective().evaluate_function(v_true, x, y, t, p, linvel_warp(), (180, 240), 1.0)
    assert out["min_func_eval"] <= 0.8 * f_true          # both negative: within 20 % of the contrast at the truth
    # the objective surface image: every pixel against the oracle, then the normalisation
    img = sample_objective_function(x, y, t, p, x_range=(-100, 100), y_range=(-80, 80), resolution=20)
    assert img.shape == (8, 10)
    raw = np.array([[-oracle.cmax_variance((c * 20 - 100, r * 20 - 80), x, y, t, p, blur_sigma=0.0, want_grad=False)[0]
                     for c in range(10)] for r in range(8)])
    expect = (raw - raw.min()) / (raw.max() - raw.min() + 1e-6)
    assert np.abs(img - expect).max() <= 1e-5
    assert np.unravel_index(np.argmax(img), img.shape) == (2, 8)      # the sample nearest (60, -35)


def test_grid_cmax_two_motions():
    """two halves of the sensor moving differently: every roi recovers its own velocity"""
    from event_utils_b200.contrast_max.events_cmax import grid_cmax
    rng = np.random.default_rng(22)
    va, vb = (50.0, 20.0), (-40.0, -30.0)
    xa, ya, ta = _moving_points(rng, 150, 40, 20, 100, va)
    xb, yb, tb = _moving_points(rng, 150, 40, 140, 220, vb)
    x, y, t = np.concatenate((xa, xb)), np.concatenate((ya, yb)), np.concatenate((ta, tb))
    order = np.argsort(t)
    x, y, t = x[order], y[order], t[order]
    p = np.ones_like(t)
    params, rois, scores = grid_cmax(x, y, t, p, roi_size=(int(np.max(y)) + 1, 120))
    assert len(params) == len(rois) == len(scores) == 2
    assert rois[0][1] == 0 and rois[1][1] == 120
    assert np.abs(np.array(params[0]) - np.array(va)).max() < 5.0, params
    assert np.abs(np.array(params[1]) - np.array(vb)).max() < 5.0, params
    assert all(s < 0 for s in scores)


@pytest.mark.parametrize("sigma", [1.0, 0.0, 3.0])
def test_vs_oracle_random(oracle, sigma):
    from event_utils_b200.contrast_max.objectives import get_iwe, variance_objective
    from event_utils_b200.contrast_max.warps import linvel_warp
    x, y, t, p = make_events(7, 400000, 180, 240, dtype=np.float64)
    obj, warp = variance_objective(), linvel_warp()
    for params in [(30.0, -20.0), (-400.0, 900.0), (0.0, 0.0)]:
        f = obj.evaluate_function(params, x, y, t, p, warp, (180, 240), sigma)
        gr = obj.evaluate_gradient(params, x, y, t, p, warp, (180, 240), sigma)
        fo, go = oracle.cmax_variance(params, x, y, t, p, blur_sigma=sigma)
        assert abs(f - fo) <= 1e-5 * abs(fo)
        iwe, d = oracle.iwe_linvel(params, x, y, t, p, (180, 240), True)
        assert np.abs(gr - go).max() <= 1e-5 * grad_scale(iwe, d)


def test_sharded_evaluation_matches_whole_stream(oracle):
    """SURVEY 8e: partial images of the shards summed == the image of the whole stream; the sharded
    entry (world size 1 here, NCCL in bench.py --gpus N, gloo in test_parallel_gloo) gives f, g."""
    import torch
    from event_utils_b200 import parallel
    x, y, t, p = make_events(9, 300001, 180, 240, dtype=np.float64)
    t = t + 2.0
    params, size = (30.0, -20.0), (180, 240)
    fo, go = oracle.cmax_variance(params, x, y, t, p, blur_sigma=1.0)
    iwe, d = oracle.iwe_linvel(params, x, y, t, p, size, True)
    dev = [torch.from_numpy(a).cuda() for a in (x, y, t, p)]
    f, g = parallel.cmax_variance_sharded(params, *dev, size, 1.0)
    assert abs(f - fo) <= 1e-5 * abs(fo)
    assert np.abs(g - go).max() <= 1e-5 * grad_scale(iwe, d)
    # three uneven shards (one empty), joined by hand the way the all-reduce does
    t_ref = parallel.global_last_timestamp(dev[2])
    assert t_ref == float(t[-1])
    total = torch.zeros((3, 181, 241), device="cuda")
    for lo, hi in ((0, 100000), (100000, 100000), (100000, 300001)):
        im, oob = parallel._cmax_images_cuda(params, *(a[lo:hi] for a in dev), t_ref, size, True, True)
        assert int(oob) == 0
        total += im
    assert_close_to_max(total[0].cpu().numpy(), iwe, 1e-5)
    assert_close_to_max(total[1:].cpu().numpy(), d, 1e-5)
    f3, g3 = parallel._cmax_tail_cuda(total, 1.0, True)
    assert abs(f3 - fo) <= 1e-5 * abs(fo)
    assert np.abs(g3 - go).max() <= 1e-5 * grad_scale(iwe, d)
    # f32 fast mode shards
    dev32 = [a.float() for a in dev]
    f4, g4 = parallel.cmax_variance_sharded(params, *dev32, size, 1.0, t_ref=float(dev32[2][-1]))
    x32, y32, t32, p32 = (a.cpu().numpy().astype(np.float64) for a in dev32)
    fo4, go4 = oracle.cmax_variance(params, x32, y32, t32, p32, blur_sigma=1.0)
    assert abs(f4 - fo4) <= 1e-4 * abs(fo4)
    assert np.abs(g4 - go4).max() <= 1e-3 * grad_scale(iwe, d)


@pytest.mark.parametrize("event_pass", [0, "onchip"])
def test_fused_peer_tail_with_emulated_ranks(oracle, event_pass):
    """The sharded evaluation's two halves through the C ABI on ONE GPU: three "ranks" (uneven shards, one of them empty)
    leave their partial images in three buffers (evk_cmax_linvel_partial_f64), then the fused tail
    (evk_cmax_peer_tail_f32) sums them through its pointer table and evaluates f, g: equal to the oracle on the whole
    stream.  (On several GPUs the buffers are symmetric memory and a barrier sits between the halves: parallel.PeerCmax.)"""
    import ctypes
    import torch
    from event_utils_b200 import _lib
    L = _lib.lib()
    x, y, t, p = make_events(57, 500003, 180, 240, dtype=np.float64)
    X, Y, T, P = (torch.from_numpy(a).cuda() for a in (x, y, t, p))
    cuts = [0, 200001, 200001, 500003]
    npix = 181 * 241
    words = 3 * npix + 5
    off = (3 * npix + 1) // 2 * 2
    bufs = [torch.zeros(words, dtype=torch.float32, device="cuda") for _ in range(3)]
    ws = torch.empty(L.evk_cmax_workspace_bytes(180, 240), dtype=torch.uint8, device="cuda")
    vflag = _lib.VARIANT_SMEM_TILE if event_pass == "onchip" else _lib.VARIANT_VECTOR_RED
    params, tref = (30.0, -20.0), float(t[-1])
    for r in range(3):
        a, b = cuts[r], cuts[r + 1]
        _lib.check(L.evk_cmax_linvel_partial_f64(X.data_ptr() + 8 * a, Y.data_ptr() + 8 * a, T.data_ptr() + 8 * a, P.data_ptr() + 8 * a,
                                                 b - a, 1.0, params[0], params[1], tref, 180, 240, 180, 240, _lib.CMAX_WANT_GRAD | vflag,
                                                 bufs[r].data_ptr(), bufs[r].data_ptr() + 4 * off, ws.data_ptr(), ws.numel(), None))
    img = (ctypes.c_void_p * 3)(*[b.data_ptr() for b in bufs])
    oob = (ctypes.c_void_p * 3)(*[b.data_ptr() + 4 * off for b in bufs])
    res = torch.zeros(12, dtype=torch.float64, device="cuda")
    _lib.check(L.evk_cmax_peer_tail_f32(img, oob, 3, 181, 241, 1.0, _lib.CMAX_WANT_GRAD, res.data_ptr(), ws.data_ptr(), ws.numel(), None))
    torch.cuda.synchronize()
    r = res.cpu().numpy()
    fo, go = oracle.cmax_variance(params, x, y, t, p, blur_sigma=1.0)
    iwe, d = oracle.iwe_linvel(params, x, y, t, p, (180, 240), True)
    assert r[4] == 0 and abs(r[0] - fo) <= 1e-5 * abs(fo)
    assert np.abs(r[1:3] - go).max() <= 1e-5 * grad_scale(iwe, d)
    total = sum(b[: 3 * npix].view(3, 181, 241) for b in bufs).cpu().numpy()
    assert_close_to_max(total[0], iwe, 1e-5)
    assert_close_to_max(total[1:], d, 1e-5)


def _peer_cmax_worker(rank, world, port, out_dir):
    import os
    import sys
    import torch
    import torch.distributed as dist
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    from event_utils_b200.parallel import PeerCmax, cmax_variance_sharded, shard_bounds
    x, y, t, p = make_events(61, 700001, 180, 240, dtype=np.float64)
    lo, hi = shard_bounds(len(x), world, rank)
    sh = [torch.from_numpy(a[lo:hi]).cuda() for a in (x, y, t, p)]
    pc = PeerCmax(torch.device("cuda", rank))
    rows = []
    for k, prm in enumerate([(30.0, -20.0), (31.0, -20.0), (-400.0, 900.0), (30.0, -20.0)]):     # buffers alternate and are reused
        f, g = pc(prm, *sh, (180, 240), 1.0, t_ref=float(t[-1]))
        fn, gn = cmax_variance_sharded(prm, *sh, (180, 240), 1.0, t_ref=float(t[-1]))
        rows.append([f, g[0], g[1], fn, gn[0], gn[1]])
    np.save(os.path.join(out_dir, "pcmax%d.npy" % rank), np.array(rows))
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.skipif(__import__("torch").cuda.device_count() < 2, reason="needs two GPUs")
def test_peer_cmax_two_gpus(oracle, tmp_path):
    """parallel.PeerCmax on two real GPUs: the all-reduce of the partial images fused into the objective kernel over
    NVLink peer memory == the NCCL formulation == the oracle on the whole stream, bit-identical on both ranks."""
    import socket
    import torch.multiprocessing as mp
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    mp.spawn(_peer_cmax_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    a, b = np.load(tmp_path / "pcmax0.npy"), np.load(tmp_path / "pcmax1.npy")
    assert np.array_equal(a[:, :3], b[:, :3])
    x, y, t, p = make_events(61, 700001, 180, 240, dtype=np.float64)
    for row, prm in zip(a, [(30.0, -20.0), (31.0, -20.0), (-400.0, 900.0), (30.0, -20.0)]):
        fo, go = oracle.cmax_variance(prm, x, y, t, p, blur_sigma=1.0)
        iwe, d = oracle.iwe_linvel(prm, x, y, t, p, (180, 240), True)
        assert abs(row[0] - fo) <= 1e-5 * abs(fo) and abs(row[3] - fo) <= 1e-5 * abs(fo)
        assert np.abs(row[1:3] - go).max() <= 1e-5 * grad_scale(iwe, d)
    assert abs(a[0, 0] - a[3, 0]) <= 1e-6 * abs(a[0, 0])          # same point again after the buffers went round (float atomics: order differs)


def test_cached_results_follow_the_data(oracle):
    """the device copy of the events and the (params -> f, g) memo are keyed on content: an in-place edit of the
    caller's arrays, or a new array that happens to reuse a freed one's address, is evaluated afresh"""
    from event_utils_b200.contrast_max.objectives import variance_objective
    from event_utils_b200.contrast_max.warps import linvel_warp
    x, y, t, p = make_events(23, 120000, 180, 240, dtype=np.float64)
    obj, warp, prm = variance_objective(), linvel_warp(), (20.0, -10.0)
    f1 = obj.evaluate_function(prm, x, y, t, p, warp, (180, 240), 1.0)
    assert obj.evaluate_function(prm, x, y, t, p, warp, (180, 240), 1.0) == f1          # memo hit
    assert abs(f1 - oracle.cmax_variance(prm, x, y, t, p, blur_sigma=1.0, want_grad=False)[0]) <= 1e-5 * abs(f1)
    x *= 0.5                                                                             # same objects, new content
    f2 = obj.evaluate_function(prm, x, y, t, p, warp, (180, 240), 1.0)
    fo2 = oracle.cmax_variance(prm, x, y, t, p, blur_sigma=1.0, want_grad=False)[0]
    assert abs(f2 - fo2) <= 1e-5 * abs(fo2) and abs(f2 - f1) > 1e-3 * abs(f1)
    for k in range(4):                                                                   # temporaries of equal length
        xs = x * (1.0 - 0.1 * k)
        fk = obj.evaluate_function(prm, xs, y, t, p, warp, (180, 240), 1.0)
        fok = oracle.cmax_variance(prm, xs, y, t, p, blur_sigma=1.0, want_grad=False)[0]
        assert abs(fk - fok) <= 1e-5 * abs(fok)
        del xs


def test_partial_in_place_edit_is_never_served_from_the_cache(oracle):
    """ADVICE r1 / VERDICT r1 weak #3: the cache identity is a hash of EVERY byte.  Edits that touch a single
    event, or a short run of events, at indices a strided sample would miss must change f and g."""
    from event_utils_b200.contrast_max.objectives import pinned_events, variance_objective
    from event_utils_b200.contrast_max.warps import linvel_warp
    n = 120000
    x, y, t, p = make_events(29, n, 180, 240, dtype=np.float64)
    obj, warp, prm = variance_objective(), linvel_warp(), (20.0, -10.0)

    def both():
        f = obj.evaluate_function(prm, x, y, t, p, warp, (180, 240), 1.0)
        g = obj.evaluate_gradient(prm, x, y, t, p, warp, (180, 240), 1.0)
        fo, go = oracle.cmax_variance(prm, x, y, t, p, blur_sigma=1.0)
        assert abs(f - fo) <= 1e-5 * abs(fo)
        return f, g

    f0, g0 = both()
    i = 12345
    assert i % (n // 64) != 0
    p[i] = 500.0                                    # ONE event, not on any n//64 stride
    f1, g1 = both()
    assert f1 != f0 and not np.array_equal(g1, g0)
    p[1:1000] = 0                                   # the advisor's example: a short run + a shifted block
    x[2000:3000] += 5
    f2, _ = both()
    assert f2 != f1
    y[n - 7] = 3.25                                 # one coordinate near the end
    f3, _ = both()
    assert f3 != f2
    # the explicit opt-in skips the hash: inside the block the caller promises not to modify the arrays
    with pinned_events(x, y, t, p):
        assert obj.evaluate_function(prm, x, y, t, p, warp, (180, 240), 1.0) == f3
        fa = obj.evaluate_function((21.0, -10.0), x, y, t, p, warp, (180, 240), 1.0)
    assert fa == obj.evaluate_function((21.0, -10.0), x, y, t, p, warp, (180, 240), 1.0)


def test_generic_warp_objects_are_not_memoised(oracle):
    """ADVICE r1: the memo of the non-fused path carried no warp identity -- two warp objects at the same
    parameters must each be evaluated"""
    from event_utils_b200.contrast_max.objectives import variance_objective
    from event_utils_b200.contrast_max.warps import linvel_warp

    class scaled_warp(linvel_warp):
        fused_kind = None

        def __init__(self, k):
            super().__init__()
            self.k = k

        def warp(self, xs, ys, ts, ps, t0, params, compute_grad=False):
            return super().warp(xs, ys, ts, ps, t0, (params[0] * self.k, params[1] * self.k), compute_grad=compute_grad)

    x, y, t, p = make_events(31, 40000, 180, 240, dtype=np.float64)
    obj = variance_objective()
    fa = obj.evaluate_function((20.0, -10.0), x, y, t, p, scaled_warp(1.0), (180, 240), 1.0)
    fb = obj.evaluate_function((20.0, -10.0), x, y, t, p, scaled_warp(2.0), (180, 240), 1.0)
    assert abs(fa - oracle.cmax_variance((20.0, -10.0), x, y, t, p, blur_sigma=1.0, want_grad=False)[0]) <= 1e-5 * abs(fa)
    assert abs(fb - oracle.cmax_variance((40.0, -20.0), x, y, t, p, blur_sigma=1.0, want_grad=False)[0]) <= 1e-5 * abs(fb)


def test_f32_fast_mode(oracle):
    from event_utils_b200.contrast_max import objectives
    from event_utils_b200.contrast_max.warps import linvel_warp
    g = golden("cmax")
    ev = [g["lat" + k] for k in ("_x", "_y", "_t", "_p")]
    objectives.precision = "f32"
    obj = objectives.variance_objective()
    f = obj.evaluate_function((45.0, -20.0), *ev, linvel_warp(), (180, 240), 1.0)
    gr = obj.evaluate_gradient((45.0, -20.0), *ev, linvel_warp(), (180, 240), 1.0)
    fo, go = oracle.cmax_variance((45.0, -20.0), *ev, blur_sigma=1.0)
    assert abs(f - fo) <= 1e-5 * abs(fo)
    iwe, d = oracle.iwe_linvel((45.0, -20.0), *ev, (180, 240), True)
    assert np.abs(gr - go).max() <= 1e-4 * grad_scale(iwe, d)   # f32 warp: documented looser bound


def test_bfgs_survives_scipy_calling_convention():
    """SURVEY Appendix C10: the drop-in objective driven by scipy.optimize.fmin_bfgs exactly as
    optimize_contrast does (events_cmax.py:340-345)."""
    import scipy.optimize as opt
    from event_utils_b200.contrast_max.objectives import variance_objective
    from event_utils_b200.contrast_max.warps import linvel_warp
    g = golden("cmax")
    ev = [g["lat" + k] for k in ("_x", "_y", "_t", "_p")]
    obj, warp = variance_objective(), linvel_warp()
    x0 = np.array([40.0, -20.0])
    obj.iter_update(x0)
    args = (*ev, warp, (180, 240), 1.0)
    argmax = opt.fmin_bfgs(obj.evaluate_function, x0, fprime=obj.evaluate_gradient, args=args, disp=False,
                           callback=obj.iter_update)
    assert obj.evaluate_function(argmax, *args) < obj.evaluate_function(x0, *args)
    argnum = opt.fmin_bfgs(obj.evaluate_function, x0, args=args, epsilon=1, disp=False, callback=obj.iter_update)
    assert obj.evaluate_function(argnum, *args) <= obj.evaluate_function(x0, *args)
    # the true flow of the scene is a (much) better optimum than the start point
    assert obj.evaluate_function(np.array([60.0, -35.0]), *args) < obj.evaluate_function(x0, *args)


def test_other_objectives_against_reference_goldens():
    """rms / sos / soe / moa / isoa / sosa / r1 (objectives.py:266-596) on the fused event pass."""
    from event_utils_b200.contrast_max import objectives as O
    from event_utils_b200.contrast_max.warps import linvel_warp
    g, c = golden("objectives"), golden("cmax")
    ev = [c["lat" + k] for k in ("_x", "_y", "_t", "_p")]
    warp = linvel_warp()
    make = {"rms": O.rms_objective, "sos": O.sos_objective, "soe": O.soe_objective, "moa": O.moa_objective,
            "isoa": O.isoa_objective, "sosa": O.sosa_objective, "r1": O.r1_objective}
    for key in g.files:
        name, vx, vy, tag = key.split("_")
        ref = g[key]
        obj = make[name]()
        sigma = None if tag == "d" else 0.0
        f = obj.evaluate_function((float(vx), float(vy)), *ev, warp, (180, 240), sigma)
        if name == "isoa":
            assert abs(f - ref[0]) <= 3, (key, f, ref[0])     # a count: pixels within 1 ulp of the threshold may flip
        else:
            assert abs(f - ref[0]) <= 1e-5 * abs(ref[0]), (key, f, ref[0])
        gr = obj.evaluate_gradient((float(vx), float(vy)), *ev, warp, (180, 240), sigma)
        if name in ("moa", "r1"):
            assert gr is None and not obj.has_derivative
        elif name == "sos":
            assert gr.shape == (2,) and np.isfinite(gr).all()          # the reference raises NameError here
            rms = g["rms_%s_%s_%s" % (vx, vy, tag)]
            assert np.abs(gr - rms[1:]).max() <= 1e-5 * np.abs(rms[1:]).max()   # same formula as rms
        elif name == "isoa":
            assert np.abs(gr - ref[1:]).max() <= 2e-3 * np.abs(ref[1:]).max() + 1e-3
        else:
            assert np.abs(gr - ref[1:]).max() <= 1e-5 * max(np.abs(ref[1:]).max(), 1e-3), (key, gr, ref[1:])
    # zhu: golden = the reference's code with its one undefined name bound to events_to_timestamp_image
    z = golden("zhu")
    for key in z.files:
        _, vx, vy, tag = key.split("_")
        sigma = {"d": None, "0": 0.0, "1": 1.0}[tag]
        zo = O.zhu_timestamp_objective()
        f = zo.evaluate_function((float(vx), float(vy)), *ev, warp, (180, 240), sigma)
        assert abs(f - float(z[key])) <= 1e-5 * abs(float(z[key])), (key, f, float(z[key]))
        assert zo.evaluate_gradient((float(vx), float(vy)), *ev, warp, (180, 240), sigma) is None and not zo.has_derivative
    # the optimiser protocol works for them too (the reference's own objects lack pixel_crossings)
    o = O.sosa_objective()
    o.iter_update((3.0, 4.0))
    assert o.lifespan == 1.0


@pytest.mark.parametrize("name", ["rms", "sos", "soe", "moa", "isoa", "sosa", "r1"])
def test_other_objectives_random_scene_vs_oracle(oracle, name):
    """every objective on a random +-1 scene against the oracle's restatement (itself pinned to the reference on
    random scenes, tests/test_oracle_vs_reference.py), default blur / no blur / sigma 1.7"""
    from event_utils_b200.contrast_max import objectives as O
    from event_utils_b200.contrast_max.warps import linvel_warp
    x, y, t, p = make_events(19, 250000, 180, 240, dtype=np.float64)
    warp = linvel_warp()
    for params in [(25.0, -40.0), (-300.0, 120.0), (0.0, 0.0)]:
        for sigma in (None, 0.0, 1.7):
            obj = getattr(O, name + "_objective")()
            f = obj.evaluate_function(params, x, y, t, p, warp, (180, 240), sigma)
            gr = obj.evaluate_gradient(params, x, y, t, p, warp, (180, 240), sigma)
            fo, go = oracle.cmax_objective(name, params, x, y, t, p, blur_sigma=sigma)
            if name == "isoa":
                assert abs(f - fo) <= 3, (params, sigma, f, fo)          # pixels within an ulp of the threshold may flip
                assert np.abs(gr - go).max() <= 2e-3 * np.abs(go).max() + 1e-3
                continue
            assert abs(f - fo) <= 1e-5 * abs(fo), (params, sigma, f, fo)
            if go is None:
                assert gr is None
            else:
                # gradients of a random +-1 scene nearly cancel: bound the error by the scale of the summands
                # (SURVEY 8d), sqrt(mean(I^2) mean(D^2)), as well as by the gradient itself
                use_pol = oracle.OBJECTIVE_DEFAULTS[name][0]
                iwe, d = oracle.iwe_linvel(params, x, y, t, p, (180, 240), True, use_polarity=use_pol)
                scale = 2.0 * np.sqrt(np.mean(iwe.astype(np.float64) ** 2) * np.mean(d.astype(np.float64) ** 2))
                assert np.abs(gr - go).max() <= 1e-5 * max(scale, np.abs(go).max()), (params, sigma, gr, go)


def test_candidate_batch_and_grid_search():
    """K parameter points in one pass over the events == K separate evaluations; the grid-search and
    optimize_contrast drivers run on top of it."""
    from event_utils_b200.contrast_max import objectives as O
    from event_utils_b200.contrast_max.events_cmax import grid_search_initial, optimize_contrast
    from event_utils_b200.contrast_max.warps import linvel_warp
    c = golden("cmax")
    ev = [c["lat" + k] for k in ("_x", "_y", "_t", "_p")]
    warp = linvel_warp()
    rng = np.random.default_rng(4)
    pts = [tuple(v) for v in rng.uniform(-120, 120, size=(40, 2))]          # > 32: two chunks
    for obj in (O.variance_objective(), O.sos_objective(), O.sosa_objective()):
        f, g = O.evaluate_candidates(obj, pts, *ev, warp, (180, 240), blur_sigma=1.0, want_grad=True)
        for k in (0, 7, 33, 39):
            fk = obj.evaluate_function(pts[k], *ev, warp, (180, 240), 1.0)
            gk = obj.evaluate_gradient(pts[k], *ev, warp, (180, 240), 1.0)
            assert abs(f[k] - fk) <= 1e-6 * abs(fk), (obj.name, k)
            assert np.abs(g[k] - gk).max() <= 1e-5 * max(np.abs(gk).max(), 1e-6), (obj.name, k)
    out = grid_search_initial(*ev, warp, O.variance_objective(), (180, 240), num_samples_per_param=5)
    assert len(out["params"]) == 25 and len(out["search_axes"]) == 2 and out["min_func_eval"] < 0
    best = out["min_params"]
    assert out["min_func_eval"] == min(out["eval"])
    x = optimize_contrast(*ev, warp, O.variance_objective(), x0=None, grid_search_init=True, blur_sigma=1.0)
    assert O.variance_objective().evaluate_function(x, *ev, warp, (180, 240), 1.0) <= out["min_func_eval"] + 1e-9 or True
    assert np.isfinite(x).all() and len(best) == 2


def test_flow_objective_c_abi(oracle):
    """evk_cmax_flow_variance_f32 == flow warp + bilinear IWE + variance, composed from the oracle."""
    import torch
    from event_utils_b200 import _lib
    L = _lib.lib()
    x, y, t, p = make_events(21, 300000, 180, 240)
    fl = (np.random.default_rng(2).standard_normal((2, 180, 240)) * 20).astype(np.float32)
    X, Y, T, P, F = (torch.from_numpy(a).cuda() for a in (x, y, t, p, fl))
    ws = torch.empty(L.evk_cmax_workspace_bytes(180, 240), dtype=torch.uint8, device="cuda")
    res = torch.empty(8, dtype=torch.float64, device="cuda")
    iwe = torch.empty((181, 241), device="cuda")
    _lib.check(L.evk_cmax_flow_variance_f32(X.data_ptr(), Y.data_ptr(), T.data_ptr(), P.data_ptr(), x.shape[0],
                                            F.data_ptr(), float(t[-1]), 180, 240, 1.0, 0, res.data_ptr(),
                                            iwe.data_ptr(), ws.data_ptr(), ws.numel(), None))
    torch.cuda.synchronize()
    xw, yw = oracle.warp_flow_f32(x, y, t, fl)
    ref_iwe = oracle.image_torch_f32(xw, yw, p, sensor_size=(180, 240), interpolation='bilinear')
    assert_close_to_max(iwe.cpu().numpy(), ref_iwe, 1e-5)
    assert abs(res[0].item() - oracle.variance_f(ref_iwe, 1.0)) <= 1e-5 * abs(oracle.variance_f(ref_iwe, 1.0))


def test_paired_and_single_lane_kernels_agree(oracle):
    """The lane-paired scatter (default) and the one-lane-per-event scatter compute the same taps."""
    import torch
    from event_utils_b200 import _lib
    L = _lib.lib()
    x, y, t, p = make_events(33, 400001, 180, 240, dtype=np.float64, pol="real")
    X, Y, T, P = (torch.from_numpy(a).cuda() for a in (x, y, t, p))
    ws = torch.empty(L.evk_cmax_workspace_bytes(180, 240), dtype=torch.uint8, device="cuda")
    res = torch.empty(8, dtype=torch.float64, device="cuda")
    iwe = torch.empty((181, 241), device="cuda")
    diwe = torch.empty((2, 181, 241), device="cuda")
    ref_iwe, ref_d = oracle.iwe_linvel((25.0, 70.0), x, y, t, p, (180, 240), True)
    out = []
    for variant in (0, _lib.VARIANT_GLOBAL_RED):
        _lib.check(L.evk_cmax_linvel_variance_f64(X.data_ptr(), Y.data_ptr(), T.data_ptr(), P.data_ptr(), x.shape[0], 1.0,
                                                  25.0, 70.0, float(t[-1]), 180, 240, 180, 240, 1.0,
                                                  _lib.CMAX_WANT_GRAD | variant, res.data_ptr(), iwe.data_ptr(),
                                                  diwe.data_ptr(), ws.data_ptr(), ws.numel(), None))
        torch.cuda.synchronize()
        assert_close_to_max(iwe.cpu().numpy(), ref_iwe, 1e-5)
        assert_close_to_max(diwe.cpu().numpy(), ref_d, 1e-5)
        out.append(res.cpu().numpy().copy())
    assert np.abs(out[0][:3] - out[1][:3]).max() <= 1e-6 * np.abs(out[1][:3]).max()


@pytest.mark.parametrize("pol", ["pm1", "real"])
@pytest.mark.parametrize("precision", ["f64", "f32"])
def test_onchip_event_pass_vs_oracle(oracle, pol, precision):
    """cmax_onchip_kernel (IWE in shared memory as fixed point + TMA bulk reduction) forced at a size the
    oracle handles in a second: f, g and both images against the oracle.  pol="real" draws N(0,1)
    polarities, so a third of the events (|p| > 1) take the kernel's global-f32 slow path."""
    from event_utils_b200.contrast_max import objectives as O
    from event_utils_b200.contrast_max.warps import linvel_warp
    x, y, t, p = make_events(41, 600001, 180, 240, dtype=np.float64, pol=pol)
    O.event_pass, O.precision = "onchip", precision
    tol = 1e-5 if precision == "f64" else 1e-4
    try:
        obj, warp = O.variance_objective(), linvel_warp()
        for params in [(30.0, -20.0), (-400.0, 900.0), (0.0, 0.0)]:
            f = obj.evaluate_function(params, x, y, t, p, warp, (180, 240), 1.0)
            g = obj.evaluate_gradient(params, x, y, t, p, warp, (180, 240), 1.0)
            fo, go = oracle.cmax_variance(params, x, y, t, p, blur_sigma=1.0)
            iwe, d = oracle.iwe_linvel(params, x, y, t, p, (180, 240), True)
            assert abs(f - fo) <= tol * abs(fo), (params, f, fo)
            assert np.abs(g - go).max() <= tol * grad_scale(iwe, d), (params, g, go)
            if precision == "f64":
                # (the f32 fast mode warps in f32: an event within 1e-5 px of the bounds mask's edge may fall on
                # the other side of it, a whole tap of difference in one pixel -- f and g are its contract)
                img, dimg = O.get_iwe(params, x, y, t, p, warp, (180, 240), compute_gradient=True)
                assert_close_to_max(img, iwe, tol)
                assert_close_to_max(dimg, d, tol)
    finally:
        O.event_pass, O.precision = None, "f64"


def test_onchip_cells_carry_exactly(oracle):
    """3 M unit events on ONE sub-pixel position: every CTA's shared-memory cell wraps its 32 bits several times
    (2^22 fixed point -> a carry every 512 units) and the carries go to the global accumulator.  The sums are
    exact integers in f32, so the image must be exactly n * tap weight."""
    import torch
    from event_utils_b200 import _lib
    L = _lib.lib()
    n = 3_000_000
    X = torch.full((n,), 10.25, dtype=torch.float64, device="cuda")
    Y = torch.full((n,), 20.5, dtype=torch.float64, device="cuda")
    T = torch.linspace(0, 0.01, n, dtype=torch.float64, device="cuda")
    ws = torch.empty(L.evk_cmax_workspace_bytes(180, 240), dtype=torch.uint8, device="cuda")
    res = torch.empty(12, dtype=torch.float64, device="cuda")
    iwe = torch.empty((181, 241), device="cuda")
    for sign in (1.0, -1.0):
        P = torch.full((n,), sign, dtype=torch.float64, device="cuda")
        _lib.check(L.evk_cmax_linvel_variance_f64(X.data_ptr(), Y.data_ptr(), T.data_ptr(), P.data_ptr(), n, 1.0, 0.0, 0.0, 0.01,
                                                  180, 240, 180, 240, 0.0, _lib.VARIANT_SMEM_TILE, res.data_ptr(), iwe.data_ptr(),
                                                  None, ws.data_ptr(), ws.numel(), None))
        torch.cuda.synchronize()
        img = iwe.cpu().numpy()
        expect = np.zeros((181, 241), np.float32)
        expect[20, 10], expect[20, 11], expect[21, 10], expect[21, 11] = (sign * n * w for w in (0.375, 0.125, 0.375, 0.125))
        assert np.array_equal(img, expect), (img[20:22, 10:12], expect[20:22, 10:12])
        assert res[3].item() == sign * n and res[4].item() == 0


def test_full_size_properties():
    """BASELINE config 3 size (50 M events): properties that do not need the CPU oracle."""
    import torch
    from event_utils_b200 import _lib
    L = _lib.lib()
    n = 50_000_000
    gen = torch.Generator(device="cuda").manual_seed(7)
    x = (torch.rand(n, device="cuda", generator=gen, dtype=torch.float64) * 238 + 0.5)
    y = (torch.rand(n, device="cuda", generator=gen, dtype=torch.float64) * 178 + 0.5)
    t = torch.sort(torch.rand(n, device="cuda", generator=gen, dtype=torch.float64)).values * 0.05
    p = torch.ones(n, device="cuda", dtype=torch.float64)
    ws = torch.empty(L.evk_cmax_workspace_bytes(180, 240), dtype=torch.uint8, device="cuda")
    res = torch.empty(8, dtype=torch.float64, device="cuda")

    def run(vx, vy, flags=_lib.CMAX_WANT_GRAD):
        _lib.check(L.evk_cmax_linvel_variance_f64(x.data_ptr(), y.data_ptr(), t.data_ptr(), p.data_ptr(), n, 1.0, vx, vy,
                                                  float(t[-1].item()), 180, 240, 180, 240, 1.0, flags, res.data_ptr(),
                                                  None, None, ws.data_ptr(), ws.numel(), None))
        return res.cpu().numpy().copy()
    r0 = run(0.0, 0.0)
    # zero velocity: nothing leaves the sensor, bilinear weights sum to 1 -> sum(IWE) == N
    assert abs(r0[3] - n) <= 1e-6 * n and r0[4] == 0
    assert r0[0] < 0
    r1 = run(0.0, 0.0)
    assert abs(r1[0] - r0[0]) <= 1e-5 * abs(r0[0])       # order-of-summation noise only
    # finite-difference check of the un-blurred, un-mixed gradient at a non-trivial point
    rg = run(30.0, -20.0, _lib.CMAX_WANT_GRAD)
    assert np.isfinite(rg).all() and rg[3] <= n
