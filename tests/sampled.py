"""Compact stored form of a large reference output, and the check of a computed array against it.

An output too large to store whole is kept as the values at a fixed set of cells, sums over contiguous
blocks, its largest magnitude and its NaN count.  `check` asserts only what `max|a-b| <= rel * max|b|`
over the whole array implies for those quantities, so an array that passes the full comparison passes
this one; for arrays of at most `k` cells the stored values are the whole array."""
import numpy as np

GOLDEN_RATIO = 0.6180339887498949


def sample_index(size, k):
    """Sorted, distinct flat indices: all of them for size <= k, else a low-discrepancy spread of about k."""
    if size <= k:
        return np.arange(size)
    return np.unique(np.floor((np.arange(k) * GOLDEN_RATIO) % 1.0 * size).astype(np.int64))


def _blocks(flat, nblocks):
    return np.array_split(flat, min(nblocks, flat.size)) if flat.size else []


def digest(a, k, nblocks):
    """(sampled values, block sums in f64, max |a| over the non-NaN cells, NaN count)."""
    flat = np.asarray(a).ravel()
    finite = flat[~np.isnan(flat)]
    return (flat[sample_index(flat.size, k)],
            np.array([np.nansum(b, dtype=np.float64) for b in _blocks(flat, nblocks)], dtype=np.float64),
            float(np.abs(finite).max()) if finite.size else 0.0,
            int(np.isnan(flat).sum()))


def check(a, vals, bsums, maxabs, nnan, k, nblocks, rel, what=""):
    flat = np.asarray(a).ravel()
    tol = rel * max(float(maxabs), 1e-30)
    got = flat[sample_index(flat.size, k)]
    assert got.shape == np.shape(vals), (what, got.shape, np.shape(vals))
    assert (np.isnan(got) == np.isnan(vals)).all(), what + ": NaN pattern differs"
    assert int(np.isnan(flat).sum()) == int(nnan), what + ": NaN count differs"
    ok = ~np.isnan(vals)
    err = np.abs(got[ok].astype(np.float64) - np.asarray(vals)[ok]).max() if ok.any() else 0.0
    assert err <= tol, "%s: max err %.3e at sampled cells vs scale %.3e (rel %.1e)" % (what, err, maxabs, rel)
    finite = flat[~np.isnan(flat)]
    assert abs((float(np.abs(finite).max()) if finite.size else 0.0) - float(maxabs)) <= tol, what + ": max |value| differs"
    blocks = _blocks(flat, nblocks)
    assert len(blocks) == len(bsums), what
    for i, (b, s) in enumerate(zip(blocks, bsums)):
        d = abs(float(np.nansum(b, dtype=np.float64)) - float(s))
        assert d <= tol * b.size * (1 + 1e-9), "%s: block %d sum off by %.3e (bound %.3e)" % (what, i, d, tol * b.size)
