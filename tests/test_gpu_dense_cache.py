"""The f64_dense mode's decision bit-plane (B200 only).

A dense sweep is a REFRESH (every voxel's decision bit from its fp64 intensity, kept in a bit-plane) at the start of a run and
behind every change of the decision table or caller-chosen flips; every other sweep is CACHED and takes the bits from the
plane.  VRG_NO_DCACHE=1 makes every sweep a refresh: it is the reference these tests compare against, bit for bit, besides
the golden fixtures and the oracles."""
import os

import numpy as np
import pytest

from golden_util import golden_names, load_golden

pytestmark = pytest.mark.gpu

TABLE_NAMES = [n for n in golden_names() if not n.endswith("_cont")]
UPDATE_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "update")
COUNTERS = ("iterations", "exit_reason", "n_in", "n_out", "n_excluded", "sweeps", "q_cancelled", "q_add_to_inside",
            "q_remove_to_outside", "q_cancel_repromoted")


def run_dense(data, vm, H, max_seg, monkeypatch, env=(), iter_max=200, unaligned=False):
    """One f64_dense run on a fresh handle with the environment switches `env` set while the handle is created.
    `unaligned`: attach the intensities zero-copy from a CUDA buffer that is only 8-byte aligned, as a tensor view with an
    odd storage offset is, instead of uploading a copy."""
    from arterynetwork_b200.engine import VRGEngine
    for k in env:
        monkeypatch.setenv(k, "1")
    try:
        eng = VRGEngine(data.shape, H=H, max_segment_size=max_seg, iter_max=iter_max, intensity="f64_dense")
    finally:
        for k in env:
            monkeypatch.delenv(k)
    with eng:
        if unaligned:
            import torch
            d = torch.empty(data.size + 1, dtype=torch.float64, device="cuda")[1:]
            assert d.data_ptr() % 16 == 8
            d.copy_(torch.from_numpy(np.ascontiguousarray(data, dtype=np.float64).ravel()))
            v = torch.from_numpy(np.ascontiguousarray(vm, dtype=np.uint8)).cuda()
            eng.attach_device(d.data_ptr(), v.data_ptr())
        else:
            eng.upload(np.asarray(data, dtype=np.float64), np.asarray(vm, dtype=np.uint8))
        eng.init()
        out = dict(eng.run())
        out["labels"] = eng.labels()
        out["trace"] = eng.trace()
        out["table"] = eng.table()
    return out


def assert_same_run(a, b):
    for k in COUNTERS:
        assert a[k] == b[k], k
    assert np.array_equal(a["labels"], b["labels"]) and np.array_equal(a["trace"], b["trace"])
    for x, y in zip(a["table"], b["table"]):  # levels and the two normalised sums, bit for bit
        assert np.array_equal(np.asarray(x).view(np.uint64), np.asarray(y).view(np.uint64))


def oracle_table_changes(data, vm, H, max_seg):
    from oracle.vrg_oracle import vrg_oracle
    ref = vrg_oracle(data, vm, H=H, max_segment_size=max_seg, record_tables=True)
    changes = 0
    for (pa, qa), (pb, qb) in zip(ref["tables"][:-1], ref["tables"][1:]):
        changes += not np.array_equal(np.asarray(pa) >= np.asarray(qa), np.asarray(pb) >= np.asarray(qb))
    return ref, changes


@pytest.mark.parametrize("name", TABLE_NAMES)
def test_cached_sweeps_equal_refresh_sweeps_on_every_fixture(name, monkeypatch):
    """Default run vs VRG_NO_DCACHE=1 vs the pipelined run: bit-equal, equal to the fixture.  Refreshes: one per run plus one
    per change of the oracle's decision table; with the switch, every sweep."""
    g = load_golden(name)
    args = (g["data"], g["value_map_in"], g["H"], g["max_segment_size"], monkeypatch)
    a = run_dense(*args)
    b = run_dense(*args, env=("VRG_NO_DCACHE",))
    p = run_dense(*args, env=("VRG_PIPELINE",))
    assert_same_run(a, b)
    assert_same_run(a, p)
    assert a["iterations"] == g["iterations"] and np.array_equal(a["trace"], g["trace"])
    assert np.array_equal(a["labels"], g["labels"])
    assert b["dense_refresh_sweeps"] == b["sweeps"]
    assert a["dense_refresh_sweeps"] == p["dense_refresh_sweeps"] and 1 <= a["dense_refresh_sweeps"] < a["sweeps"]
    if g["data"].size <= 64 ** 3:  # within reach of the NumPy oracle
        _, changes = oracle_table_changes(g["data"], g["value_map_in"], g["H"], g["max_segment_size"])
        assert a["dense_refresh_sweeps"] == 1 + changes


def test_table_changes_refresh_the_plane_on_every_path(monkeypatch):
    """tests/random_cases.table_shift_case: the decision table changes in the middle of the run.  In order, pipelined and
    with the separate kernels the result equals the oracle's, and each change costs exactly one refresh sweep."""
    from random_cases import table_shift_case
    data, vm = table_shift_case()
    ref, changes = oracle_table_changes(data, vm, 2.25, 10 ** 9)
    assert changes >= 2
    runs = {env: run_dense(data, vm, 2.25, 10 ** 9, monkeypatch, env=env)
            for env in ((), ("VRG_PIPELINE",), ("VRG_NO_FUSED_TAIL",), ("VRG_NO_DCACHE",))}
    for env, o in runs.items():
        assert o["iterations"] == ref["iterations"] and o["exit_reason"] == ref["exit"], env
        assert np.array_equal(o["labels"], ref["labels"]) and np.array_equal(o["trace"], ref["trace"]), env
        assert_same_run(o, runs[()])
    assert runs[("VRG_PIPELINE",)]["redone_sweeps"] == changes
    for env in ((), ("VRG_PIPELINE",), ("VRG_NO_FUSED_TAIL",)):
        assert runs[env]["dense_refresh_sweeps"] == 1 + changes, env
    assert runs[("VRG_NO_DCACHE",)]["dense_refresh_sweeps"] == runs[("VRG_NO_DCACHE",)]["sweeps"]


@pytest.mark.parametrize("in_place", [False, True])
def test_new_data_on_the_same_handle_is_never_served_from_the_old_plane(in_place, monkeypatch):
    """Run on data A, then on data B of the same shape (the mirror image of A, same level set) on the same handle: by a new
    attach, or by overwriting the attached device buffers in place.  The second run must equal a fresh handle on B and the
    fixture, mirrored."""
    import torch
    from arterynetwork_b200.engine import VRGEngine
    g = load_golden("forest_two_trees")
    A, vA = np.ascontiguousarray(g["data"], dtype=np.float64), g["value_map_in"].astype(np.uint8)
    B, vB = np.ascontiguousarray(A[:, ::-1, ::-1]), np.ascontiguousarray(vA[:, ::-1, ::-1])
    want = np.ascontiguousarray(g["labels"][:, ::-1, ::-1])
    fresh = run_dense(B, vB, g["H"], g["max_segment_size"], monkeypatch, env=("VRG_NO_DCACHE",))
    assert np.array_equal(fresh["labels"], want)
    dA, vdA = torch.from_numpy(A).cuda(), torch.from_numpy(vA).cuda()
    dB, vdB = torch.from_numpy(B).cuda(), torch.from_numpy(vB).cuda()
    with VRGEngine(A.shape, H=g["H"], max_segment_size=g["max_segment_size"], intensity="f64_dense") as eng:
        eng.attach_device(dA.data_ptr(), vdA.data_ptr())
        eng.init()
        ra = eng.run()
        assert ra["iterations"] == g["iterations"] and np.array_equal(eng.labels(), g["labels"])
        if in_place:
            dA.copy_(dB); vdA.copy_(vdB)
            torch.cuda.synchronize()
        else:
            eng.attach_device(dB.data_ptr(), vdB.data_ptr())
        eng.init()
        rb = eng.run()
        assert rb["dense_refresh_sweeps"] >= 1 and rb["dense_refresh_sweeps"] < rb["sweeps"]
        for k in COUNTERS:
            assert rb[k] == fresh[k], k
        assert np.array_equal(eng.labels(), want) and np.array_equal(eng.trace(), fresh["trace"])


def _phantom(shape, kw):
    from arterynetwork_b200.phantom import make_phantom
    data, vm, _ = make_phantom(shape, seed=5, **kw)
    return data, vm


@pytest.mark.parametrize("case", ["odd_x", "wide_1024", "unaligned", "label4"])
def test_every_sweep_variant_keeps_and_reads_the_plane(case, monkeypatch):
    """The refresh kernels other than the TMA ring of the bench shape: the plain-load kernel (odd X, and an even X attached
    from an 8-byte aligned buffer), a whole row per warp (X = 1024), and a label-4 input (excluded mask, separate kernels
    behind the sweep).  Default equals VRG_NO_DCACHE=1 equals the oracle, and the cache is used."""
    if case == "odd_x":
        from random_cases import table_shift_case
        data, vm = table_shift_case()
        data, vm = np.ascontiguousarray(data[:, :, :61]), np.ascontiguousarray(vm[:, :, :61])
        from oracle.vrg_oracle import vrg_oracle
        ref = vrg_oracle(data, vm, H=2.25, max_segment_size=10 ** 9)
        H, ms = 2.25, 10 ** 9
    elif case == "wide_1024":
        from oracle.c_oracle import vrg_oracle_c
        data, vm = _phantom((20, 24, 1024), dict(cell=(20, 24, 128), margin=3, depth=2, root_r2=4, min_len=8, max_len=40))
        ref = vrg_oracle_c(data, vm, max_segment_size=10 ** 12)
        H, ms = 2.25, 10 ** 12
    else:
        g = load_golden("forest40" if case == "unaligned" else "excl32")
        data, vm, H, ms = g["data"], g["value_map_in"], g["H"], g["max_segment_size"]
        ref = {"iterations": g["iterations"], "trace": g["trace"], "labels": g["labels"]}
    unaligned = case == "unaligned"
    if unaligned:  # the refresh must be the plain-load kernel, not the TMA ring it would take on aligned data
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            a = run_dense(data, vm, H, ms, monkeypatch, unaligned=True)
        assert any("k_sweep_dense_ldg" in e.name for e in prof.events())
    else:
        a = run_dense(data, vm, H, ms, monkeypatch)
    b = run_dense(data, vm, H, ms, monkeypatch, env=("VRG_NO_DCACHE",), unaligned=unaligned)
    assert_same_run(a, b)
    assert a["iterations"] == ref["iterations"] > 3
    assert np.array_equal(a["trace"], ref["trace"]) and np.array_equal(a["labels"], ref["labels"])
    assert 1 <= a["dense_refresh_sweeps"] < a["sweeps"] and b["dense_refresh_sweeps"] == b["sweeps"]


@pytest.mark.parametrize("name", sorted(os.path.splitext(f)[0] for f in os.listdir(UPDATE_DIR) if f.endswith(".npz")))
def test_caller_flips_in_dense_mode_refresh_the_plane(name, monkeypatch):
    """The update() call-by-call recordings on a dense handle: one sweep fills the plane, the recorded flips of the call are
    applied (vrg_apply_flips), and the result equals the reference's call; the run that continues from there on the same
    handle must not reuse the plane (its first sweep is a refresh) and equals a fresh VRG_NO_DCACHE run from that state."""
    from arterynetwork_b200.engine import VRGEngine
    f = np.load(os.path.join(UPDATE_DIR, name + ".npz"))
    k = f["k"].astype(np.int64)
    data = k.astype(np.float64) if bool(f["data_is_int"]) else k.astype(np.float64) / int(f["quantum"])
    H = float(f["H"])
    for c in range(1, int(f["n_calls"])):
        seg_in = np.unpackbits(f["c%d_seg_in" % c])[: k.size].reshape(k.shape).astype(bool)
        vm8 = np.full(k.shape, 3, dtype=np.uint8)
        vm8[f["c%d_vm_in" % c] == 4] = 4
        vm8[seg_in] = 0
        vm_out = f["c%d_vm_out" % c].astype(np.uint8)
        with VRGEngine(k.shape, H=H, max_segment_size=2 ** 62, intensity="f64_dense") as eng:
            eng.upload(data, vm8)
            eng.init()
            eng.enqueue_decide()
            assert eng.poll()["dense_refresh_sweeps"] == 1
            applied = eng.apply_flips(np.asarray(f["c%d_flips" % c], dtype=np.int64).reshape(-1, 3))
            assert np.array_equal(eng.labels(), vm_out), c
            r = eng.run()
            if r["sweeps"] > applied["sweeps"]:  # the run went on from the caller's update
                assert r["dense_refresh_sweeps"] >= 2, c
            labels = eng.labels()
        fresh = run_dense(data, vm_out, H, 2 ** 62, monkeypatch, env=("VRG_NO_DCACHE",))
        assert np.array_equal(labels, fresh["labels"]), c
        assert r["n_in"] == fresh["n_in"] and r["n_out"] == fresh["n_out"], c
