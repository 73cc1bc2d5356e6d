"""Comparisons with the reference's own CUDA kernels (oracle/ref_gpu.py) that also run where those kernels are not built.

Where oracle/_ref/libpsdf_ref_gpu.so exists, `equal` / `close` run the reference kernel and compare with it directly. Elsewhere they
compare with what the reference kernels produced on the same inputs, stored in tests/golden:
  kernel_parity_checks.json   per check: shape, dtype and, for bit-exact checks, the SHA-256 of the reference's output
  kernel_parity_samples.npz   for checks within a tolerance: a fixed seeded sample of at most SAMPLE elements of the reference's output
Regenerate both on a B200 with the reference kernels built:
  PSDF_REF_GOLDEN_OUT=<dir> python -m pytest -m gpu tests/test_rayops_gpu.py tests/test_volrender_gpu.py tests/test_benchsize_parity_gpu.py
and copy the two files from <dir> into tests/golden/."""
import atexit
import hashlib
import json
import os
import zlib

import numpy as np

from oracle import ref_gpu

HERE = os.path.dirname(os.path.abspath(__file__))
CHECKS = os.path.join(HERE, "golden", "kernel_parity_checks.json")
SAMPLES = os.path.join(HERE, "golden", "kernel_parity_samples.npz")
SAMPLE = 512

_stored = None
_recorded = {"checks": {}, "samples": {}}


def _np(x):
    if hasattr(x, "detach"):
        x = x.detach().cpu().numpy()
    return np.ascontiguousarray(np.asarray(x))


def _digest(a):
    if a.dtype.kind == "f":
        a = a + a.dtype.type(0)             # -0.0 -> +0.0: the direct comparison counts them equal too
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def _sample_index(n, key):
    rng = np.random.RandomState(zlib.crc32(key.encode()))
    return np.sort(rng.choice(n, min(n, SAMPLE), replace=False))


def _golden(key):
    global _stored
    if _stored is None:
        _stored = (json.load(open(CHECKS)), dict(np.load(SAMPLES)))
    checks, samples = _stored
    assert key in checks, "%s: no stored reference output (see tests/ref_golden.py to regenerate)" % key
    return checks[key], samples.get(key)


def _record(key, b, sample=None):
    out = os.environ.get("PSDF_REF_GOLDEN_OUT")
    if not out:
        return
    assert key not in _recorded["checks"], "duplicate reference check key " + key
    entry = {"shape": list(b.shape), "dtype": b.dtype.str}
    if sample is None:
        entry["sha256"] = _digest(b)
    else:
        _recorded["samples"][key] = sample
    _recorded["checks"][key] = entry


def _write():
    out = os.environ.get("PSDF_REF_GOLDEN_OUT")
    if out and _recorded["checks"]:
        os.makedirs(out, exist_ok=True)
        checks = _recorded["checks"]
        with open(os.path.join(out, "kernel_parity_checks.json"), "w") as f:
            f.write("{\n" + ",\n".join("%s: %s" % (json.dumps(k), json.dumps(checks[k], sort_keys=True)) for k in sorted(checks)) + "\n}\n")
        np.savez_compressed(os.path.join(out, "kernel_parity_samples.npz"), **_recorded["samples"])


atexit.register(_write)


def equal(key, ours, theirs):
    """ours must be bit-identical to the reference's output. theirs: callable -> the reference's output (only called where the
    reference kernels are built)"""
    a = _np(ours)
    if ref_gpu.available():
        b = _np(theirs())
        assert a.shape == b.shape, (key, a.shape, b.shape)
        assert np.array_equal(a, b), key + ": not bit-identical to the reference kernel"
        _record(key, b)
        return
    g, _ = _golden(key)
    assert list(a.shape) == g["shape"], (key, a.shape, g["shape"])
    assert _digest(a.astype(np.dtype(g["dtype"]))) == g["sha256"], key + ": not bit-identical to the stored reference output"


def close(key, ours, theirs, atol, rtol=0.0):
    """|ours - theirs| <= atol + rtol * |theirs| elementwise; without the reference kernels on a fixed sample of the elements"""
    a = _np(ours)
    if ref_gpu.available():
        b = _np(theirs())
        assert a.shape == b.shape, (key, a.shape, b.shape)
        idx = None
        _record(key, b, b.reshape(-1)[_sample_index(b.size, key)])
    else:
        g, b = _golden(key)
        assert list(a.shape) == g["shape"], (key, a.shape, g["shape"])
        idx = _sample_index(a.size, key)
    a = a.reshape(-1).astype(np.float64) if idx is None else a.reshape(-1)[idx].astype(np.float64)
    b = b.reshape(-1).astype(np.float64)
    err = np.abs(a - b) - rtol * np.abs(b)
    assert err.size == 0 or err.max() <= atol, "%s: max err %g above the tolerance (atol %g, rtol %g)" % (key, err.max(), atol, rtol)


def once(fn):
    """fn() evaluated at most once: several checks of the outputs of one reference call"""
    memo = []

    def get():
        if not memo:
            memo.append(fn())
        return memo[0]
    return get


def fresh_generators():
    """pytest fixture body: the class-static pcg32 generators start from their initial state (the stored outputs of jittered
    reference calls were made from it, whatever ran before), and the previous generators are put back afterwards"""
    from permuto_sdf import OccupancyGrid, RaySampler, VolumeRendering
    from permuto_sdf_b200.permuto_sdf import _Pcg32Host
    classes = (OccupancyGrid, RaySampler, VolumeRendering)
    saved = [c.m_rng for c in classes]
    for c in classes:
        c.m_rng = _Pcg32Host()
    yield
    for c, r in zip(classes, saved):
        c.m_rng = r


def per_ray(start_end, *arrays):
    """packed per-sample arrays in ray order (slot order differs between implementations): one array per input"""
    se = _np(start_end)
    return [np.concatenate([a[s:e] for s, e in se] + [a[:0]], 0) for a in map(_np, arrays)]


def counts(start_end):
    se = _np(start_end)
    return se[:, 1] - se[:, 0]
