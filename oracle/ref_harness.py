"""TEST INFRASTRUCTURE ONLY -- harness around the UNMODIFIED reference.

Imports ``/root/reference/Code/variationalRegionGrowing.py`` as it lies (read
only, never copied), neutralises its nondeterministic 120 s exit (VRG:38,97),
and wraps ``update`` (VRG:124) to record, per iteration, what the parity tests
compare against:

* ``n_flips``                      len(flipedPoints)               (VRG:88,91)
* ``n_in``, ``n_out``              region sizes after the update   (VRG:113-116)
* ``band`` samples                 innerProb/innerSize, outerProb/outerSize at
                                   every band voxel                (VRG:79-82)
* quirk counters Q2, Q3 and the incremental-vs-full drift (SURVEY.md section 8(a)):
  bit-identity to the reference is only well-defined when they are zero.

``/root/reference`` exists only in the build container, so nothing in the
``-m gpu`` tests, ``smoke()`` or ``bench.py`` may import this module.  It is
used by ``tests/golden/make_golden.py``, which writes the committed fixtures.
"""
from __future__ import annotations

import contextlib
import io
import os
import re
import sys
import types

import numpy as np

REFERENCE_DIR = os.environ.get("VRG_REFERENCE_DIR", "/root/reference/Code")


def reference_available() -> bool:
    return os.path.isfile(os.path.join(REFERENCE_DIR, "variationalRegionGrowing.py"))


_ref_module = None


def load_reference():
    """Import the reference module unmodified (SURVEY.md appendix A recipe)."""
    global _ref_module
    if _ref_module is not None:
        return _ref_module
    if not reference_available():
        raise RuntimeError("reference not present at %s" % REFERENCE_DIR)
    sys.dont_write_bytecode = True  # the reference dir is read-only
    for name in ("nibabel", "nrrd"):  # imported at VRG:3-4, never used
        sys.modules.setdefault(name, types.ModuleType(name))
    import importlib.util

    spec = importlib.util.spec_from_file_location(
        "_reference_vrg", os.path.join(REFERENCE_DIR, "variationalRegionGrowing.py")
    )
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)

    class _FrozenTimer:  # VRG:38,97 -- the 120 s exit must never fire
        default_timer = staticmethod(lambda: 0.0)

    mod.timeit = _FrozenTimer
    _ref_module = mod
    return mod


def canonical_labels(seg: np.ndarray, excl: np.ndarray) -> np.ndarray:
    """Order-free classification of (seg, excl) into the label alphabet (VRG:21)."""
    from .vrg_oracle import canonical_labels as _c

    return _c(seg.astype(bool), excl.astype(bool))


def run_reference(data, value_map, H=2.25, max_segment_size=None, record_band=True,
                  check_drift=True):
    """Run the reference; return a dict with outputs, stdout, trace and quirk counters.

    ``value_map`` is copied (the reference mutates it in place, VRG:137-228).
    """
    ref = load_reference()
    data = np.asarray(data)
    vm = np.array(value_map, copy=True)
    if max_segment_size is None:
        max_segment_size = int(data.size) + 1
    trace = []
    band_samples = []
    quirks = {"Q2_iters": 0, "Q2_voxels": 0, "Q3_dropped": 0, "max_drift": 0.0}
    orig_update = ref.update
    A = ref.A

    def full_probs(dataArray, valueMap, pts, H):
        inner = dataArray[(valueMap == 0) | (valueMap == 1)]
        outer = dataArray[(valueMap == 2) | (valueMap == 3)]
        out = np.empty((len(pts), 2))
        for i, p in enumerate(pts):
            v = dataArray[tuple(p)]
            out[i, 0] = np.sum(A * np.exp(-0.5 * H * (inner - v) ** 2))
            out[i, 1] = np.sum(A * np.exp(-0.5 * H * (outer - v) ** 2))
        return out

    def wrapped(dataArray, segmented, segmentedMap, valueMap, H_, flipedPoints=None,
                innerBnd=None, outerBnd=None, innerProb=None, outerProb=None):
        res = orig_update(dataArray, segmented, segmentedMap, valueMap, H_, flipedPoints,
                          innerBnd, outerBnd, innerProb, outerProb)
        segmented2, segMap2, vm2, iB, oB, iP, oP = res
        n_in = int(np.count_nonzero((vm2 == 0) | (vm2 == 1)))
        n_out = int(np.count_nonzero((vm2 == 2) | (vm2 == 3)))
        n_flips = -1 if flipedPoints is None else int(len(flipedPoints))
        trace.append((n_flips, n_in, n_out))
        canon = canonical_labels(segMap2 == 1, vm2 == 4)
        q2 = int(np.count_nonzero(canon != vm2))
        if q2:
            quirks["Q2_iters"] += 1
            quirks["Q2_voxels"] += q2
        if flipedPoints is not None and len(flipedPoints):
            post = vm2[tuple(np.asarray(flipedPoints).T)]
            quirks["Q3_dropped"] += int(np.count_nonzero((post != 1) & (post != 2)))
        band = np.concatenate([np.asarray(iB).reshape(-1, 3), np.asarray(oB).reshape(-1, 3)])
        band = band.astype(np.int64)
        if record_band and len(band):
            idx = tuple(band.T)
            band_samples.append({
                "coords": band.copy(),
                "p_in": (iP[idx] / n_in).copy(),
                "p_out": (oP[idx] / n_out).copy(),
            })
        if check_drift and len(band) and dataArray.size <= 64 ** 3:
            full = full_probs(dataArray, vm2, band, H_)
            idx = tuple(band.T)
            got = np.stack([iP[idx], oP[idx]], axis=1)
            den = np.maximum(np.abs(full), 1e-300)
            quirks["max_drift"] = max(quirks["max_drift"], float(np.max(np.abs(got - full) / den)))
        return res

    ref.update = wrapped
    buf = io.StringIO()
    try:
        with contextlib.redirect_stdout(buf), np.errstate(all="ignore"):
            segmented, segmented_map, vm_out = ref.variationalRegionGrowing(
                data, vm, H=H, maxSegmentSize=max_segment_size)
    finally:
        ref.update = orig_update
    out = buf.getvalue()
    m = re.search(r"Finished at iteration (\d+)", out)
    iters = int(m.group(1)) if m else None
    return {
        "segmented": np.asarray(segmented),
        "segmented_map": np.asarray(segmented_map),
        "value_map": np.asarray(vm_out),
        "stdout": out,
        "iterations": iters,
        "trace": np.asarray(trace, dtype=np.int64),  # row 0 = init (n_flips = -1)
        "band_samples": band_samples,
        "quirks": quirks,
    }
