"""Record what the UNMODIFIED reference returns for the inputs of tests/test_oracle_vs_reference.py,
tests/test_edge_cases_cpu.py and tests/test_citations.py, so that those tests run without it:

    EVK_REFERENCE_ROOT=<checkout of TimoStoff/event_utils> python tests/golden/make_reference_checks.py

Inputs are not stored: the tests regenerate them from the same seeds.  Outputs of more than a few
thousand cells are stored in the sampled form of tests/sampled.py.
"""
import importlib
import json
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
TESTS = os.path.dirname(HERE)
ROOT = os.path.dirname(TESTS)
sys.path[:0] = [ROOT, TESTS]
from conftest import make_events  # noqa: E402
from edge_cases import cases  # noqa: E402
from oracle import ref_loader  # noqa: E402
import sampled  # noqa: E402
import test_edge_cases_cpu as EC  # noqa: E402
import test_oracle_vs_reference as VR  # noqa: E402

ref = ref_loader.load()
torch.set_num_threads(1)


def put(d, name, a, k, nblocks):
    vals, bsums, maxabs, nnan = sampled.digest(a, k, nblocks)
    d.update({name + "_shape": np.array(np.shape(a)), name + "_val": vals, name + "_bsum": bsums,
              name + "_max": np.float64(maxabs), name + "_nan": np.int64(nnan)})


# ---- tests/test_oracle_vs_reference.py ----------------------------------------------------------
out = {}
for seed, n, B, H, W in VR.VOXEL_CASES:
    x, y, t, p = make_events(seed, n, H, W)
    v = ref.voxel_grid.events_to_voxel_torch(*(torch.from_numpy(a) for a in (x, y, t, p)), B, sensor_size=(H, W)).numpy()
    put(out, "voxel_torch_%d" % seed, v, VR.K, VR.NBLOCKS)

put(out, "voxel_numpy", ref.voxel_grid.events_to_voxel(*VR.voxel_numpy_events(), 5, sensor_size=(260, 346)), VR.K, VR.NBLOCKS)

for i, kw in enumerate(VR.IMAGE_KW):
    x, y, p = VR.image_events(kw)
    a = ref.image.events_to_image_torch(torch.from_numpy(x), torch.from_numpy(y), torch.from_numpy(p), **kw).numpy()
    put(out, "image_%d" % i, a, VR.K, VR.NBLOCKS)

x, y, t, p = make_events(6, 50000, 180, 240)
flow = VR.flow_field()
xw, yw = ref.optic_flow.warp_events_flow_torch(*(torch.from_numpy(a) for a in (x, y, t, p)), torch.from_numpy(flow))
put(out, "flow_x", xw.numpy(), VR.K, VR.NBLOCKS)
put(out, "flow_y", yw.numpy(), VR.K, VR.NBLOCKS)

x, y, t, p = make_events(7, 100000, 180, 240, dtype=np.float64)
obj, warp = ref.objectives.variance_objective(), ref.warps.linvel_warp()
for sigma in VR.CMAX_SIGMAS:
    rows = []
    for params in VR.CMAX_PARAMS:
        f = obj.evaluate_function(params, x, y, t, p, warp, (180, 240), sigma)
        g = obj.evaluate_gradient(params, x, y, t, p, warp, (180, 240), sigma)
        iwe, d = ref.objectives.get_iwe(params, x, y, t, p, warp, (180, 240), compute_gradient=True)
        scale = np.sqrt(np.mean((2 * (iwe - iwe.mean())) ** 2) * np.mean(d ** 2))
        rows.append([f, g[0], g[1], scale])
    out["cmax_sigma_%g" % sigma] = np.array(rows, dtype=np.float64)

ref_cmax = importlib.import_module("lib.contrast_max.events_cmax")
out["find_new_range"] = np.array([np.asarray(ref_cmax.find_new_range(axis, value), dtype=np.float64)
                                  for axis, value in VR.find_new_range_inputs()])

bd = importlib.import_module("lib.data_loaders.base_dataset")
ts, frame_ts = VR.window_inputs()


class Probe(bd.BaseVoxelDataset):                       # the table code only, no recording behind it
    def __init__(self):
        self.num_events, self.t0, self.tk = len(ts), ts[0], ts[-1]
        self.duration = self.tk - self.t0
        self.has_frames = False

    def find_ts_index(self, timestamp):
        return np.searchsorted(ts, timestamp)           # memmap_dataset.py:81-83


dset = Probe()
for key, method in VR.window_methods():
    if method["method"] == "between_frames":
        dset.frame_ts, dset.num_frames = frame_ts, len(frame_ts)
    dset.set_voxel_method(method)
    out["windows_" + key] = np.asarray(dset.event_indices, dtype=np.int64)

x, y, t, p = make_events(17, 60000, 180, 240, dtype=np.float64)
for name in VR.OTHER_OBJECTIVES:
    o = getattr(ref.objectives, name + "_objective")()
    rows = []
    for params in VR.OTHER_PARAMS:
        for sigma in VR.OTHER_SIGMAS:
            f = o.evaluate_function(params, x, y, t, p, warp, (180, 240), sigma)
            g = (o.evaluate_gradient(params, x, y, t, p, warp, (180, 240), sigma) if name in VR.WITH_GRADIENT
                 else (np.nan, np.nan))
            rows.append([f, g[0], g[1]])
    out["objective_" + name] = np.array(rows, dtype=np.float64)
np.savez_compressed(os.path.join(HERE, "vs_reference.npz"), **out)

# ---- tests/test_edge_cases_cpu.py --------------------------------------------------------------
rec = {kind: dict(err=[], shape=[], val=[], bsum=[], max=[], nan=[]) for kind in EC.KINDS}
for c in cases(*EC.CASES):
    T = [torch.from_numpy(c[k]) for k in "xytp"]
    hw = (c["H"], c["W"])
    for kind in EC.KINDS:
        if kind == "voxel":
            r, e = EC.run(lambda: ref.voxel_grid.events_to_voxel_torch(*T, c["B"], sensor_size=hw).numpy())
        else:
            kw = EC.image_kw(c, kind)
            r, e = EC.run(lambda: ref.image.events_to_image_torch(T[0], T[1], T[3], **kw).numpy())
        R = rec[kind]
        R["err"].append(EC.ERRORS.index(e))
        shape = np.shape(r) if r is not None else ()
        R["shape"].append(list(shape) + [0] * (3 - len(shape)))
        if r is not None:
            vals, bsums, maxabs, nnan = sampled.digest(r, EC.K, EC.NBLOCKS)
            R["val"].append(vals)
            R["bsum"].append(bsums)
            R["max"].append(maxabs)
            R["nan"].append(nnan)
        else:
            R["max"].append(0.0)
            R["nan"].append(0)
out = {}
for kind, R in rec.items():
    out[kind + "_err"] = np.array(R["err"], dtype=np.int8)
    out[kind + "_shape"] = np.array(R["shape"], dtype=np.int16)
    out[kind + "_val"] = np.concatenate(R["val"]).astype(np.float32)
    out[kind + "_bsum"] = np.concatenate(R["bsum"])
    out[kind + "_max"] = np.array(R["max"], dtype=np.float64)
    out[kind + "_nan"] = np.array(R["nan"], dtype=np.int32)
np.savez_compressed(os.path.join(HERE, "edge_cases.npz"), **out)

# ---- tests/test_citations.py: every .py file of the reference tree and its line count -------------
files = {}
for dp, _, names in os.walk(ref_loader.REF_ROOT):
    for f in names:
        if f.endswith(".py"):
            path = os.path.join(dp, f)
            with open(path, errors="replace") as fh:
                files[os.path.relpath(path, ref_loader.REF_ROOT)] = sum(1 for _ in fh)
with open(os.path.join(HERE, "reference_files.json"), "w") as fh:
    json.dump(dict(sorted(files.items())), fh, indent=0)
    fh.write("\n")
print("wrote vs_reference.npz, edge_cases.npz, reference_files.json")
