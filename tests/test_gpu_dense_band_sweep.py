"""The f64_dense mode's sweeps between two refreshes run on k_sweep_band, with the decision bits from the bit-plane (B200 only).

A refresh sweep (the first of a run, and the one behind every change of the decision table) evaluates every decision bit
from the fp64 intensities and keeps it in the bit-plane.  The sweeps after it are the band / index modes' sweep kernel with
D read from that plane: on one volume, only the rows next to the last front are evaluated again.  That incremental pass
assumes the refresh left the flip words, row flags and front list as a full band pass would.  These runs check that the
dense mode takes this path, and that its results equal the index mode's and the oracle's."""
import re

import numpy as np
import pytest

from golden_util import load_golden

pytestmark = pytest.mark.gpu

COUNTERS = ("iterations", "exit_reason", "n_in", "n_out", "n_excluded", "sweeps", "q_cancelled", "q_add_to_inside",
            "q_remove_to_outside", "q_cancel_repromoted")
DENSE_BAND = re.compile(r"\bk_sweep_band<0, false>")


def run(data, vm, H, max_seg, mode, monkeypatch, env=(), profile=False):
    """One run on a fresh handle with the environment switches `env` set while the handle is created; with `profile`, also
    the names of the kernels it launched (torch.profiler), one entry per launch."""
    from arterynetwork_b200.engine import VRGEngine
    for k in env:
        monkeypatch.setenv(k, "1")
    try:
        eng = VRGEngine(data.shape, H=H, max_segment_size=max_seg, intensity=mode)
    finally:
        for k in env:
            monkeypatch.delenv(k)
    names = None
    with eng:
        eng.upload(np.asarray(data, dtype=np.float64), np.asarray(vm, dtype=np.uint8))
        if profile:
            from torch.profiler import ProfilerActivity, profile as prof_ctx
            with prof_ctx(activities=[ProfilerActivity.CUDA]) as prof:
                eng.init()
                out = dict(eng.run())
            names = [e.name for e in prof.events()]
        else:
            eng.init()
            out = dict(eng.run())
        out["labels"] = eng.labels()
        out["trace"] = eng.trace()
    out["kernels"] = names
    return out


def assert_same_result(a, b, what):
    for k in COUNTERS:
        assert a[k] == b[k], (what, k)
    assert np.array_equal(a["labels"], b["labels"]) and np.array_equal(a["trace"], b["trace"]), what


def assert_dense_band_path(o):
    """Every sweep enqueues the refresh kernel and the band kernel (one of them returns at once), and nothing else sweeps."""
    names = o["kernels"]
    assert not any("k_sweep_dense_cached" in n for n in names)
    assert sum(1 for n in names if DENSE_BAND.search(n)) >= o["sweeps"]
    assert 1 <= o["dense_refresh_sweeps"] < o["sweeps"]


def test_c1_dense_run_sweeps_on_the_band_kernel(monkeypatch):
    """The 128^3 fixture (config C1): the dense run launches k_sweep_band<F64_DENSE> and no cached sweep, refreshes once
    (its table never changes), and equals the index mode's run and the fixture."""
    g = load_golden("c1_128")
    args = (g["data"], g["value_map_in"], g["H"], g["max_segment_size"])
    dense = run(*args, "f64_dense", monkeypatch, profile=True)
    index = run(*args, "index", monkeypatch)
    assert_dense_band_path(dense)
    assert dense["dense_refresh_sweeps"] == 1
    assert_same_result(dense, index, "dense vs index")
    assert dense["iterations"] == g["iterations"] and np.array_equal(dense["trace"], g["trace"])
    assert np.array_equal(dense["labels"], g["labels"])


@pytest.mark.parametrize("env", [(), ("VRG_PIPELINE",), ("VRG_NO_FUSED_TAIL",)])
def test_refresh_to_incremental_hand_off_behind_every_table_change(env, monkeypatch):
    """tests/random_cases.table_shift_case: the decision table changes twice in the middle of the run, so a refresh is
    followed by incremental band sweeps three times.  In order, pipelined and with the separate kernels behind the sweep, the
    dense run equals the index mode's run and the C oracle, with one refresh per table change."""
    from random_cases import table_shift_case
    from oracle.c_oracle import vrg_oracle_c
    data, vm = table_shift_case()
    ref = vrg_oracle_c(data, vm, H=2.25, max_segment_size=10 ** 9, record_tables=True)
    changes = sum(not np.array_equal(pa >= qa, pb >= qb)
                  for (pa, qa), (pb, qb) in zip(ref["tables"][:-1], ref["tables"][1:]))
    assert changes >= 2
    dense = run(data, vm, 2.25, 10 ** 9, "f64_dense", monkeypatch, env=env, profile=True)
    index = run(data, vm, 2.25, 10 ** 9, "index", monkeypatch, env=env)
    assert_dense_band_path(dense)
    assert dense["dense_refresh_sweeps"] == 1 + changes
    assert_same_result(dense, index, "dense vs index")
    assert dense["iterations"] == ref["iterations"] and dense["exit_reason"] == ref["exit"]
    assert np.array_equal(dense["trace"], ref["trace"]) and np.array_equal(dense["labels"], ref["labels"])
