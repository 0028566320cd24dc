"""Shared helpers for the tests: synthetic calibration, an oracle-built quantised cache, and the stored results of
the reference's own CUDA kernels and cache managers (tests/golden/refgpu_*.npz) with the comparisons against them."""
import functools
import hashlib
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from kvquant_b200 import synth  # noqa: E402
from oracle import kvq_oracle as O  # noqa: E402

GOLDEN = os.path.join(ROOT, "tests", "golden")


@functools.lru_cache(maxsize=None)
def spec(H=32, seed=0):
    return synth.SynthSpec(H, 128, seed=seed)


@functools.lru_cache(maxsize=None)
def quantizer(bits, H=32, seed=0):
    sp = spec(H, seed)
    cal = synth.calibrate(sp, bits, calib_tokens=512, seed=7)
    up, lo, kc = cal["k"]
    klut = O.build_k_lut(up, lo, kc[0])
    vcent = np.sort(cal["v"][2][0].ravel().astype(np.float32))
    return klut, vcent


@functools.lru_cache(maxsize=None)
def oracle_cache(bits, L, H=32, sparse=True, Lmax=None, seed=0):
    """Token-by-token oracle cache (reference decode semantics) of L tokens."""
    sp = spec(H, seed)
    klut, vcent = quantizer(bits, H, seed)
    Lmax = Lmax or ((L + 63) // 64 * 64 + 64)
    c = O.OracleCache(bits, H, Lmax, klut, vcent, include_sparse=sparse)
    k = sp.k_tokens(L, seed=11)
    v = sp.v_tokens(L, seed=12)
    for t in range(L):
        c.append(k[t], v[t])
    return c, k, v


def rel_err(a, b):
    """max |a-b| / max |b|  (norm-wise relative error) and rel-L2."""
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    d = np.abs(a - b)
    return float(d.max() / max(np.abs(b).max(), 1e-30)), float(np.linalg.norm(d) / max(np.linalg.norm(b), 1e-30))


# ---------------------------------------------------------------------------------------------------------------
# stored reference results.  A result that must match bit for bit is kept as the SHA-256 of its bytes.  A result
# compared to a tolerance is kept whole up to FULL elements; only the score arrays over 4K..128K tokens are larger,
# and of those a fixed sample of SAMPLE elements is kept together with, per row (last axis), the sum, the sum of
# magnitudes and the L2 norm over ALL elements, so that an error anywhere in a row still shows.  Every result keeps
# the largest magnitude of each row, the scale of the norm-wise and per-row errors.
# ---------------------------------------------------------------------------------------------------------------
FULL, SAMPLE = 65536, 16384


def _host(t):
    return t.detach().cpu().numpy() if hasattr(t, "detach") else np.asarray(t)


def digest(t):
    a = np.ascontiguousarray(_host(t))
    if a.dtype.kind == "f":
        a = a + a.dtype.type(0)          # -0.0 -> +0.0: equal as torch.equal sees them
    return "%s%s:%s" % (a.dtype.str, a.shape, hashlib.sha256(a.tobytes()).hexdigest())


def sample_index(n):
    if n <= FULL:
        return np.arange(n)
    return np.sort(np.random.default_rng(n).choice(n, SAMPLE, replace=False))


def _row_sums(a):
    """per row: (sum, sum of magnitudes, L2 norm), in float64."""
    r = a.astype(np.float64).reshape(-1, a.shape[-1])
    return r.sum(axis=1), np.abs(r).sum(axis=1), np.sqrt((r * r).sum(axis=1))


def golden_record(prefix, exact=None, close=None):
    """npz entries under `prefix` for the bit-exact results `exact` and the tolerance-compared results `close`."""
    rec = {}
    for k, t in (exact or {}).items():
        rec["%s.%s.sha" % (prefix, k)] = np.array(digest(t))
    for k, t in (close or {}).items():
        key = "%s.%s" % (prefix, k)
        a = _host(t)
        a = a.astype(np.float16 if a.dtype == np.float16 else np.float32)
        rec[key + ".shape"] = np.array(a.shape)
        rec[key + ".val"] = a.ravel()[sample_index(a.size)]
        rec[key + ".rowmax"] = np.abs(a.astype(np.float32)).reshape(-1, a.shape[-1]).max(axis=1)
        if a.size > FULL:
            rec[key + ".rowsum"], rec[key + ".rowabs"], rec[key + ".rownorm"] = _row_sums(a)
    return rec


@functools.lru_cache(maxsize=None)
def load_golden(name):
    with np.load(os.path.join(GOLDEN, name)) as z:
        return {k: z[k] for k in z.files}


def assert_bit_exact(g, prefix, exact):
    for k, t in exact.items():
        key = "%s.%s.sha" % (prefix, k)
        assert key in g, key + " is missing from the stored reference results"
        assert digest(t) == str(g[key]), "%s.%s differs from the reference's result" % (prefix, k)


def golden_pair(g, prefix, key, t):
    """(ours, reference, row scale of each element, scale of the whole result) over the stored elements."""
    a = _host(t)
    key = "%s.%s" % (prefix, key)
    assert tuple(a.shape) == tuple(g[key + ".shape"]), (key, a.shape)
    idx = sample_index(a.size)
    rowmax = g[key + ".rowmax"].astype(np.float64)
    return (a.ravel()[idx].astype(np.float64), g[key + ".val"].astype(np.float64),
            rowmax[idx // a.shape[-1]], float(rowmax.max()))


def golden_rel_err(g, prefix, key, t):
    """Relative errors against a stored reference result: (norm-wise, per-row, row sums).  Norm-wise / per-row:
    max |ours - ref| over the stored elements over the largest |ref| of the whole result / of that element's row.
    Row sums (0 for a result stored whole): over every row, the largest of |sum ours - sum ref| / sum |ref| and
    |norm ours - norm ref| / norm ref, with all elements of the row."""
    a, b, row, full = golden_pair(g, prefix, key, t)
    d = np.abs(a - b)
    e_sums = 0.0
    if "%s.%s.rowsum" % (prefix, key) in g:
        k = "%s.%s." % (prefix, key)
        s, sa, n = _row_sums(_host(t))
        e_sums = float(max((np.abs(s - g[k + "rowsum"]) / np.maximum(g[k + "rowabs"], 1e-30)).max(),
                           (np.abs(n - g[k + "rownorm"]) / np.maximum(g[k + "rownorm"], 1e-30)).max()))
    return float(d.max() / max(full, 1e-30)), float((d / np.maximum(row, 1e-30)).max()), e_sums
