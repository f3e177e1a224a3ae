"""Helpers shared by the oracle (CPU) and CUDA (GPU) parity tests over tests/golden/*.npz."""
import glob
import hashlib
import json
import os

import numpy as np

from rl4rs_b200 import synth
from rl4rs_b200.utils.datautil import FeatureUtil

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def golden_names():
    return sorted(os.path.basename(p)[:-4] for p in glob.glob(os.path.join(GOLDEN_DIR, "*.npz")))


class Golden(object):
    def __init__(self, name):
        z = np.load(os.path.join(GOLDEN_DIR, name + ".npz"))
        self.name = name
        self.meta = json.loads(bytes(z["meta"]).decode())
        self.arr = {k: z[k] for k in z.files if k != "meta"}
        self.config = self.meta["config"]
        self.seq = self.meta["seq"]
        self.catalog = synth.Catalog.from_text(self.meta["catalog_text"])
        self.log = FeatureUtil.parse_log(self.meta["records"], self.config.get("maxlen", 64))
        self._weights = None

    @property
    def weights(self):
        if self._weights is None:
            self._weights = synth.make_weights(self.config, **self.meta["weights"])
        return self._weights

    @property
    def n_episodes(self):
        return self.arr["reward"].shape[0] // self.config["max_steps"]


# tolerance of the floating-point half (north_star: 1e-4 relative on rewards / observations).
# Observations are 256 ELU outputs of one 3456-long dot product each, some of them ~0, so the
# relative bound is taken against max(|ref|, rms(ref row)) -- an element-wise relative test on a
# value that happens to be 1e-7 would test nothing but cancellation.
RTOL = 1e-4

# Every comparison is recorded: worst error/bound under the rms-floored rule the assertion uses, and next to it the
# PLAIN element-wise worst relative error |got-ref|/|ref| (over elements with ref != 0) with the |ref| it occurred
# at, so a reader can see what the floor forgives.  conftest.py prints the table and writes
# gpurun_out/parity_margins.json at the end of a GPU session.
MARGINS = {}


def _record(what, err, bound, ref):
    key = what.split(" step ")[0]
    key = "".join(c for c in key if not c.isdigit()).strip() or "?"
    nz = np.abs(ref) > 0
    plain = np.zeros_like(err)
    plain[nz] = err[nz] / np.abs(ref[nz])
    i = int(np.argmax(plain)) if plain.size else 0
    m = MARGINS.setdefault(key, {"n": 0, "floored_err_over_bound": 0.0, "plain_rel_max": 0.0, "plain_rel_at_abs_ref": 0.0,
                                 "row_rms_there": 0.0})
    m["n"] += int(err.size)
    if err.size:
        m["floored_err_over_bound"] = max(m["floored_err_over_bound"], float((err / bound).max()))
        if float(plain.flat[i]) > m["plain_rel_max"]:
            m["plain_rel_max"] = float(plain.flat[i])
            m["plain_rel_at_abs_ref"] = float(np.abs(ref).flat[i])
            if ref.ndim >= 2:
                row = np.unravel_index(i, ref.shape)[:-1]
                m["row_rms_there"] = float(np.sqrt((ref[row] ** 2).mean()))


def assert_close_rel(got, ref, rtol=RTOL, what=""):
    got = np.asarray(got, dtype=np.float64)
    ref = np.asarray(ref, dtype=np.float64)
    assert got.shape == ref.shape, (what, got.shape, ref.shape)
    if ref.ndim >= 2:
        scale = np.sqrt((ref ** 2).mean(axis=-1, keepdims=True))
    else:
        scale = np.abs(ref)
    bound = rtol * np.maximum(np.abs(ref), scale) + 1e-12
    err = np.abs(got - ref)
    _record(what, err, bound, ref)
    bad = err > bound
    assert not bad.any(), "%s: %d/%d outside rtol=%g (worst err/bound %.3g)" % (
        what, int(bad.sum()), bad.size, rtol, float((err / bound).max()))


# ---- compact records of what the reference computed (tests/golden/reference/, made by make_reference_golden.py) -------
# A full per-step record of a reference rollout is megabytes; what is stored instead keeps every comparison: arrays that
# are compared exactly become a digest of their shape and values, observations (compared at a relative tolerance) keep a
# seeded sample of columns with each row's rms (the floor of the tolerance, and itself compared), and rewards are kept
# whole.
REFERENCE_DIR = os.path.join(GOLDEN_DIR, "reference")
SAMPLED_KEYS = ("reset_obs", "step_obs")
FULL_KEYS = {"reward": None, "click_p": None, "offline_reward": 1e-12}      # key -> rtol (None: the caller's)


def digest(a):
    """Shape and values of an array as 16 hex digits; integers, booleans and floats that are equal give equal digests."""
    a = np.ascontiguousarray(np.asarray(a, dtype=np.float64)) + 0.0          # + 0.0: -0.0 hashes like 0.0
    h = hashlib.blake2b(digest_size=8)
    h.update(repr(a.shape).encode())
    h.update(a.tobytes())
    return h.hexdigest()


def fingerprint(rec, n_cols=4, seed=0):
    """(meta, arrays) standing for the record `rec` (key -> array stacked over steps or episodes)."""
    rs = np.random.RandomState(seed)
    meta, arrays = {"digests": {}, "shapes": {}}, {}
    for key in sorted(rec):
        v = np.asarray(rec[key])
        if key in FULL_KEYS:
            arrays[key] = v
        elif key in SAMPLED_KEYS:
            cols = np.sort(rs.choice(v.shape[-1], min(n_cols, v.shape[-1]), replace=False))
            arrays[key + ".cols"], arrays[key + ".vals"] = cols, v[..., cols]
            arrays[key + ".rms"] = np.sqrt((v.astype(np.float64) ** 2).mean(axis=-1)).astype(np.float32)
            meta["shapes"][key] = list(v.shape)
        else:
            meta["digests"][key] = digest(v)
    return meta, arrays


def save_fingerprints(path, fps):
    """fps: name -> (meta, arrays); one compressed .npz."""
    out = {"meta": np.frombuffer(json.dumps({n: m for n, (m, _) in fps.items()}, sort_keys=True).encode(), np.uint8)}
    for name, (_, arrays) in fps.items():
        out.update({name + "/" + k: v for k, v in arrays.items()})
    np.savez_compressed(path, **out)


def load_fingerprint(path, name):
    z = np.load(path)
    meta = json.loads(bytes(z["meta"]).decode())[name]
    arrays = {k[len(name) + 1:]: z[k] for k in z.files if k.startswith(name + "/")}
    return meta, arrays


def check_fingerprint(rec, fp, rtol=RTOL, what=""):
    """Hold the record `rec` to the stored fingerprint of the reference's record: same keys, exact keys equal, sampled
    observations and their row rms within rtol (the rms at 2 x rtol: what rtol per element allows it), rewards within
    rtol."""
    meta, arrays = fp
    keys = set(meta["digests"]) | set(meta["shapes"]) | {k for k in arrays if "." not in k}
    assert set(rec) == keys, (what, sorted(set(rec) ^ keys))
    for key, d in sorted(meta["digests"].items()):
        assert digest(rec[key]) == d, "%s: %s differs from the reference's" % (what, key)
    for key, shape in sorted(meta["shapes"].items()):
        got = np.asarray(rec[key], dtype=np.float64)
        assert list(got.shape) == shape, (what, key, got.shape, shape)
        ref = arrays[key + ".vals"].astype(np.float64)
        rms = arrays[key + ".rms"].astype(np.float64)
        bound = rtol * np.maximum(np.abs(ref), rms[..., None]) + 1e-12
        err = np.abs(got[..., arrays[key + ".cols"]] - ref)
        _record("%s %s" % (what, key), err, bound, ref)
        assert not (err > bound).any(), "%s %s: %d/%d sampled values outside rtol=%g (worst err/bound %.3g)" % (
            what, key, int((err > bound).sum()), err.size, rtol, float((err / bound).max()))
        got_rms = np.sqrt((got ** 2).mean(axis=-1))
        assert (np.abs(got_rms - rms) <= 2 * rtol * rms + 1e-6).all(), "%s %s: row rms" % (what, key)
    for key in sorted(k for k in arrays if "." not in k):
        assert_close_rel(rec[key], arrays[key], rtol=FULL_KEYS[key] or rtol, what="%s %s" % (what, key))
