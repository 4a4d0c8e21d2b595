"""Adversarial small cases: the oracle must agree with the real reference on results AND on error
behaviour.  What the reference returned (or raised) for each case is stored in tests/golden/edge_cases.npz
by tests/golden/make_reference_checks.py; outputs of more than K cells are compared in the sampled form of
tests/sampled.py."""
import numpy as np

import sampled
from conftest import golden
from edge_cases import cases

CASES = (2024, 300)
KINDS = ("voxel", "nearest", "bilinear")
ERRORS = (None, "IndexError", "ValueError", "RuntimeError")
K, NBLOCKS = 96, 8


def run(fn):
    try:
        return fn(), None
    except (IndexError, ValueError, RuntimeError) as e:
        return None, type(e).__name__


def image_kw(c, kind):
    return dict(sensor_size=(c["H"], c["W"]), clip_out_of_range=c["clip"],
                interpolation=None if kind == "nearest" else kind, padding=c["padding"])


def test_oracle_matches_reference_on_edge_cases(oracle, capsys):
    g = golden("edge_cases")
    at = {kind: [0, 0] for kind in KINDS}                  # offsets into the concatenated values / block sums
    checked = errors = 0
    for i, c in enumerate(cases(*CASES)):
        for kind in KINDS:
            if kind == "voxel":
                o, oe = run(lambda: oracle.voxel_f32(c["x"], c["y"], c["t"], c["p"], c["B"], (c["H"], c["W"])))
                rel = 1e-6
            else:
                o, oe = run(lambda: oracle.image_torch_f32(c["x"], c["y"], c["p"], **image_kw(c, kind)))
                rel = 2e-6
            re = ERRORS[g[kind + "_err"][i]]
            assert (re is None) == (oe is None), ("%s error behaviour" % kind, c["k"], re, oe)
            if re is not None:
                errors += 1
                continue
            shape = tuple(int(s) for s in g[kind + "_shape"][i][:np.ndim(o)])
            assert np.shape(o) == shape and not g[kind + "_shape"][i][np.ndim(o):].any(), (kind, c["k"], np.shape(o))
            nv, nb = len(sampled.sample_index(o.size, K)), min(NBLOCKS, o.size)
            v0, b0 = at[kind]
            sampled.check(o, g[kind + "_val"][v0:v0 + nv], g[kind + "_bsum"][b0:b0 + nb], g[kind + "_max"][i],
                          g[kind + "_nan"][i], K, NBLOCKS, rel, "%s case %d" % (kind, c["k"]))
            at[kind] = [v0 + nv, b0 + nb]
            checked += 1
    for kind in KINDS:
        assert at[kind] == [len(g[kind + "_val"]), len(g[kind + "_bsum"])], kind
    capsys.readouterr()
    assert checked > 300 and errors > 50     # both regimes are exercised
