"""Timing of one contrast-maximisation evaluation (variance objective) per motion model -- linvel, rotation,
xyztheta -- at 1 M and 50 M events, f64 parity mode and f32 fast mode: f alone and f + g through the fused library
entry (evk_cmax_model_objective_*, CUDA events around many back-to-back evaluations on device-resident events), and
the same evaluation through the generic path a warp object without `fused_kind` takes (host warp in numpy, upload,
image on the GPU, K-channel objective; host clock around the synchronised call).  Prints one JSON line per
measurement plus the card's name and power limit, read in the same run.

    python tools/bench_cmax_models.py [--sizes 1000000,50000000] [--out bench_cmax_models.json]
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from event_utils_b200 import _lib  # noqa: E402
from event_utils_b200.contrast_max import objectives as OB  # noqa: E402
from event_utils_b200.contrast_max.warps import linvel_warp, pure_rotation_warp, warp_function, xyztheta_warp  # noqa: E402

MODELS = {"linvel": (linvel_warp, (45.0, -20.0)), "rotation": (pure_rotation_warp, (118.0, 92.0, 1.4)),
          "xyztheta": (xyztheta_warp, (37.0, -22.0, 1.0, 0.3))}


class generic(warp_function):
    """the same model without fused_kind: the generic host-warp path"""
    fused_kind = None

    def __init__(self, inner):
        super().__init__("generic_" + inner.name, inner.dims)
        self.inner = inner

    def warp(self, *a, **k):
        return self.inner.warp(*a, **k)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else "unknown"


def scene(n, seed=1):
    rng = np.random.default_rng(seed)
    return (rng.random(n) * 239, rng.random(n) * 179, np.sort(rng.random(n)) * 0.1, rng.integers(0, 2, n) * 2.0 - 1)


def device_time(fn, iters, warm=3):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="1000000,50000000")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    L = _lib.lib()
    dev = torch.device("cuda")
    info = card()
    rows = []
    print(json.dumps({"card": info}), flush=True)
    for n in (int(s) for s in args.sizes.split(",")):
        host = scene(n)
        t_last = float(host[2][-1])
        ev64 = [torch.from_numpy(a).to(dev) for a in host]
        ev32 = [torch.from_numpy(a).to(dev).float() for a in (host[0], host[1], host[2] - t_last, host[3])]
        ws = torch.empty(L.evk_cmax_workspace_bytes(180, 240), dtype=torch.uint8, device=dev)
        res = torch.zeros(20, dtype=torch.float64, device=dev)
        iters = 200 if n <= 2_000_000 else 50
        for kind, (cls, prm) in MODELS.items():
            p = np.array(prm, dtype=np.float64)
            for prec, ev in (("f64", ev64), ("f32", ev32)):
                for want_g in (False, True):
                    flags = _lib.CMAX_WANT_GRAD if want_g else 0
                    if prec == "f64":
                        fn = lambda: _lib.check(L.evk_cmax_model_objective_f64(  # noqa: E731
                            _lib.WARP_MODELS[kind], p.ctypes.data, len(p), *(e.data_ptr() for e in ev), n, 1.0, t_last, 180, 240,
                            180, 240, 1.0, flags, 0, 0.0, res.data_ptr(), res.data_ptr() + 96, ws.data_ptr(), ws.numel(),
                            _lib.stream()))
                    else:
                        fn = lambda: _lib.check(L.evk_cmax_model_objective_f32(  # noqa: E731
                            _lib.WARP_MODELS[kind], p.ctypes.data, len(p), *(e.data_ptr() for e in ev), n, 1.0, 180, 240,
                            180, 240, 1.0, flags, 0, 0.0, res.data_ptr(), res.data_ptr() + 96, ws.data_ptr(), ws.numel(),
                            _lib.stream()))
                    ms = device_time(fn, iters)
                    row = {"n": n, "model": kind, "precision": prec, "eval": "f+g" if want_g else "f", "path": "fused",
                           "ms": round(ms, 4), "GB_per_s_one_read": round(n * (32 if prec == "f64" else 16) / ms / 1e6, 1)}
                    rows.append(row)
                    print(json.dumps(row), flush=True)
            # the generic path: one f + g evaluation, host clock around the synchronised call
            obj, w = OB.variance_objective(), generic(cls())
            reps = 3 if n <= 2_000_000 else 1
            obj.evaluate_gradient(p, *host, w, (180, 240), 1.0)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(reps):
                obj.evaluate_gradient(p, *host, w, (180, 240), 1.0)
            torch.cuda.synchronize()
            row = {"n": n, "model": kind, "precision": "f64", "eval": "f+g", "path": "generic host warp",
                   "ms": round((time.perf_counter() - t0) / reps * 1e3, 2)}
            rows.append(row)
            print(json.dumps(row), flush=True)
        del ev64, ev32
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(os.path.dirname(args.out) or ".", exist_ok=True)
        with open(args.out, "w") as f:
            json.dump({"card": info, "rows": rows}, f, indent=1)


if __name__ == "__main__":
    main()
