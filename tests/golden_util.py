"""Loader / replayer of the committed fixtures under tests/golden/ -- vectors produced by the reference itself
(oracle/_ref, see tests/golden/make_golden.py and tests/golden/make_reference_records.py)."""
import glob
import hashlib
import os

import numpy as np

from groundgrid_b200 import synth

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
CLOUD_FIELDS = ("x", "y", "z", "intensity", "ring")
SAMPLE = 16


def cloud_values(pts):
    """The value fields of PointXYZIR records as an (n, 5) array (the padding bytes are not part of the value)."""
    return np.stack([pts[f].astype(np.float64) for f in CLOUD_FIELDS], axis=-1)


def _canonical(value):
    """float64 (NaN canonical, -0 -> +0) or int64 copy: equal canonical bytes <=> np.array_equal(..., equal_nan=True)."""
    a = np.asarray(value)
    if a.dtype.kind == "f":
        return np.ascontiguousarray(np.where(np.isnan(a), np.nan, a.astype(np.float64)) + 0.0)
    return np.ascontiguousarray(a.astype(np.int64))


class ReferenceRecord:
    """What the reference computed in one scenario, stored in tests/golden/ref_<name>.npz as a sequence of checks:
    per check its key, the sha256 of the shape and values, and a seeded sample of the values for the failure message.
    The reference's outputs at full size do not fit the repository; their digests do, and they keep every comparison
    bit for bit.  record=True (tests/golden/make_reference_records.py, with oracle/_ref built) runs the scenario on the
    reference and stores the sequence; otherwise every check compares against it, in the same order."""

    def __init__(self, name, record=False):
        self.name = name
        self.path = os.path.join(GOLDEN_DIR, f"ref_{name}.npz")
        self.record = record
        self.pos = 0
        if record:
            self.keys, self.digests, self.samples, self.given_values = [], [], [], {}
        else:
            z = np.load(self.path)
            self.keys, self.digests = [str(k) for k in z["keys"]], [str(d) for d in z["digests"]]
            self.samples = [s[:n] for s, n in zip(z["samples"], z["sample_len"])]
            self.given_values = dict(zip((str(k) for k in z["given_keys"]), z["given_values"].tolist()))

    def check(self, key, value):
        a = _canonical(value)
        h = hashlib.sha256(repr(a.shape).encode())
        h.update(a.tobytes())
        flat = a.reshape(-1)
        idx = np.sort(np.random.default_rng(flat.size).choice(flat.size, min(SAMPLE, flat.size), replace=False))
        sample = flat[idx].astype(np.float64)
        if self.record:
            self.keys.append(key)
            self.digests.append(h.hexdigest())
            self.samples.append(sample)
            return
        assert self.pos < len(self.keys) and self.keys[self.pos] == key, \
            f"{self.name}: check {key!r} where the record has {self.keys[self.pos] if self.pos < len(self.keys) else 'nothing'}"
        want, want_sample = self.digests[self.pos], self.samples[self.pos]
        self.pos += 1
        assert h.hexdigest() == want, (f"{self.name}: {key} differs from the reference (shape {a.shape}); sampled elements "
                                       f"{idx.tolist()}: here {sample.tolist()}, reference {want_sample.tolist()}")

    def given(self, key, compute):
        """A number only the reference can decide (e.g. which geometries it accepts): compute() when recording,
        the recorded value otherwise."""
        if self.record:
            self.given_values[key] = compute()
        return self.given_values[key]

    def finish(self):
        if not self.record:
            assert self.pos == len(self.keys), f"{self.name}: {len(self.keys) - self.pos} recorded checks were not made"
            return
        samples = np.full((len(self.keys), SAMPLE), np.nan)
        for k, s in enumerate(self.samples):
            samples[k, :len(s)] = s
        np.savez_compressed(self.path, keys=np.array(self.keys), digests=np.array(self.digests), samples=samples,
                            sample_len=np.array([len(s) for s in self.samples], np.int32),
                            given_keys=np.array(list(self.given_values), dtype="U64"),
                            given_values=np.array(list(self.given_values.values()), np.float64))
LAYER_NAMES = ("points", "ground", "groundpatch", "minGroundHeight", "maxGroundHeight", "groundCandidates", "planeDist",
               "m2", "meanVariance", "pointsRaw", "variance")


def case_files():
    return sorted(glob.glob(os.path.join(GOLDEN_DIR, "case_*.npz")))


def load_case(path):
    z = np.load(path)
    case = {"name": os.path.basename(path), "dimension": float(z["dimension"]), "resolution": float(z["resolution"]),
            "cells": int(z["cells"]), "expected": z["expected"],
            "config": {str(k): float(v) for k, v in zip(z["config_keys"], z["config_values"])},
            "ground_0": z["ground_0"], "groundpatch_0": z["groundpatch_0"], "scans": [],
            "final": {name: z["layer_" + name] for name in LAYER_NAMES}}
    for k in range(int(z["n_scans"])):
        pts = z[f"points_{k}"].view(synth.POINT_DTYPE)
        case["scans"].append({"points": pts, "origin": z[f"origin_{k}"], "base_z": float(z[f"base_z_{k}"]),
                              "labels": z[f"labels_{k}"], "order": z[f"order_{k}"], "pose": z[f"pose_{k}"], "q": z[f"q_{k}"],
                              "t": z[f"t_{k}"], "T": z[f"T_{k}"], "moved": int(z[f"moved_{k}"]), "position": z[f"position_{k}"],
                              "prior_ground": z[f"prior_ground_{k}"], "prior_groundpatch": z[f"prior_groundpatch_{k}"]})
    return case


def int_config(cfg):
    """Integer-typed configuration fields come back from the fixture as floats."""
    ints = {"point_count_cell_variance_threshold", "max_ring", "thread_count"}
    return {k: (int(v) if k in ints else v) for k, v in cfg.items()}


def same(a, b):
    return np.array_equal(a, b, equal_nan=True)


def replay(case, impl, update, filter_cloud, layers=LAYER_NAMES):
    """Runs one fixture through an implementation and asserts every recorded number bit for bit.
    impl: object with set_config / init_map / position / layer;  update(impl, x, y, T) -> moved;
    filter_cloud(impl, points, origin, base_z) -> (labels, order)."""
    name = case["name"]
    if case["config"]:
        impl.set_config(**int_config(case["config"]))
    impl.init_map(0.0, 0.0, 0.0)
    assert impl.n == case["cells"], name
    assert same(impl.layer("ground"), case["ground_0"]) and same(impl.layer("groundpatch"), case["groundpatch_0"]), name
    for k, s in enumerate(case["scans"]):
        if k:
            moved = update(impl, float(s["pose"][0]), float(s["pose"][1]), s["T"])
            assert int(bool(moved)) == s["moved"], (name, k)
        assert np.array_equal(np.asarray(impl.position()), s["position"]), (name, k, impl.position(), s["position"])
        assert same(impl.layer("ground"), s["prior_ground"]), (name, k, "rolled ground")
        assert same(impl.layer("groundpatch"), s["prior_groundpatch"]), (name, k, "rolled groundpatch")
        labels, order = filter_cloud(impl, s["points"], s["origin"], s["base_z"])
        assert np.array_equal(labels, s["labels"]), (name, k, int((labels != s["labels"]).sum()))
        assert np.array_equal(order, s["order"]), (name, k)
    for lname in layers:
        assert same(impl.layer(lname), case["final"][lname]), (name, lname)
