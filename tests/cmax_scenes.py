"""The two event scenes of tests/golden/cmax.npz.  The lattice scene is stored; the uniform "c9" scene
(SURVEY Appendix C9 draw order) is regenerated from its seed, which keeps the file under 1 MB, and checked
against the SHA-256 of the arrays the golden values were computed from."""
import hashlib

import numpy as np


def c9_events():
    rng = np.random.default_rng(0)
    n = 20000
    return rng.random(n) * 239, rng.random(n) * 179, np.sort(rng.random(n)) * 0.1, rng.integers(0, 2, n) * 2.0 - 1


def c9_sha256(ev):
    return hashlib.sha256(b"".join(np.ascontiguousarray(a, dtype=np.float64).tobytes() for a in ev)).hexdigest()


def events(g, tag):
    """(xs, ys, ts, ps) of scene `tag` ("c9" or "lat") of the loaded cmax golden file `g`."""
    if tag == "lat":
        return tuple(g["lat" + k] for k in ("_x", "_y", "_t", "_p"))
    ev = c9_events()
    assert c9_sha256(ev) == str(g["c9_sha256"]), "the c9 scene no longer regenerates bit for bit"
    return ev
