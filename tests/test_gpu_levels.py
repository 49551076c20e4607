"""Every size class of the level table against the C oracle, in all three sweep modes (B200 only).

The host picks kernels and launch shapes from the table size L (distinct levels, or span / step + 1 on a lattice):
- the Parzen kernel matrix `kmat` up to 2048 levels, `exp` inside every table evaluation above;
- the fused tail stages both histograms in shared memory up to 4096 levels, and reads them from global memory above;
- the fused tail builds the table in one pass while ceil(L / 32) <= SMs - 1, in several passes above;
- the init histogram: `k_init_hist_shared` (16-byte aligned rows, table beside the TMA ring), `k_init_hist_private`
  (L <= 880), `k_init_hist` with shared copies (L <= 6144), `k_init_hist` with global atomics;
- the dense sweep: TMA ring, one warp per whole row (X = 1024 while the table words fit beside its stages), plain loads;
- lattice (`rint`) or binary-search level lookup; `index` keeps the slot as uint16 (slot 65535 at L = 65536);
- 65536 distinct levels are accepted, 65537 raise LevelsError.

CASES names the class each case is for; every run checks with torch.profiler that it took that path, and
test_cases_reach_every_branch_in_every_mode checks that the cases together reach every branch.  The inputs are a tube along x
in noise, quantised to the case's levels (make_case); the C oracle (oracle/vrg_oracle.c) is the reference for the run, and a
long-double sum over float64 Parzen terms is the reference for the table."""
import contextlib
import functools
import io
import re

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

MODES = ["f64_dense", "f64_band", "index"]
A = 0.3989422804014327  # (2*pi)**-0.5, the reference's float64 constant
H = 2.25
MAX_SEG = 10 ** 12
COUNTERS = ("iterations", "exit_reason", "n_in", "n_out", "n_excluded", "sweeps", "q_cancelled", "q_add_to_inside",
            "q_remove_to_outside", "q_cancel_repromoted")
QUIRKS = {"q_add_to_inside": "add_to_inside", "q_remove_to_outside": "remove_to_outside",
          "q_cancel_repromoted": "cancel_repromoted", "q_cancelled": "cancelled"}

# The host's thresholds (csrc/vrg_b200.cu, vrg_tail.cuh).
KMAT_MAX = 2048
TAIL_STAGE_MAX = 4096
HIST_COPIES_MAX = 6144  # k_init_hist keeps min(8, 48 KB / (8 L)) shared copies: none above this
HIST_SHARED_MAX = (6916, 7108)  # k_init_hist_shared with rows of 64 fp64 / uint16 values (table beside a two-stage ring)


def _case(name, shape, levels, lattice=True, slots=None, lo=0.0, edges=False, excl=False, iter_max=200, hist=None,
          dense=None):
    """`levels` intensities are present; on a lattice they sit on `slots` (default: `levels`) slots, with two adjacent slots
    and both ends fixing the step.  `lo` squeezes every intensity into the upper (1 - lo) of the level range, which moves the
    decision's crossover into the table's last words.  `edges`: a quarter of the voxels just outside the tube take the lowest
    level and a quarter of the tube the highest, so both end slots hold band voxels.  `excl`: the darkest background voxels
    are label 4; the input then runs on the separate kernels instead of the fused tail.  `hist` = the init histogram branch
    for (f64 modes, index); `dense` = the f64_dense refresh sweep."""
    return dict(name=name, shape=shape, levels=levels, lattice=lattice, slots=slots or levels, lo=lo, edges=edges,
                excl=excl, iter_max=iter_max, hist=hist, dense=dense)


CASES = [
    _case("L880_oddx", (24, 40, 63), 880, hist=("private", "private"), dense="ldg"),
    _case("L881_oddx", (24, 40, 63), 881, hist=("copies", "copies"), dense="ldg"),
    _case("L2048", (24, 40, 64), 2048, hist=("shared", "shared"), dense="tma"),
    _case("L2049", (24, 40, 64), 2049, hist=("shared", "shared"), dense="tma"),
    _case("L4096_oddx", (24, 40, 63), 4096, lattice=False, hist=("copies", "copies"), dense="ldg"),
    _case("L4097", (24, 40, 64), 4097, lattice=False, hist=("shared", "shared"), dense="tma"),
    _case("L4704", (24, 40, 64), 4704, hist=("shared", "shared"), dense="tma"),
    _case("L4705", (24, 40, 64), 4705, edges=True, hist=("shared", "shared"), dense="tma"),
    _case("L6144_oddx", (32, 48, 95), 6144, lattice=False, lo=0.5, hist=("copies", "copies"), dense="ldg"),
    _case("L6145_oddx", (32, 48, 95), 6145, lattice=False, lo=0.5, hist=("global", "global"), dense="ldg"),
    _case("L6145_excluded", (32, 48, 95), 6145, lattice=False, lo=0.5, excl=True, hist=("global", "global"), dense="ldg"),
    # k_init_hist_shared keeps the table beside its TMA ring: up to 6916 levels with fp64 rows of 64, 7108 with uint16 ones
    _case("L6916", (24, 40, 64), 6916, lo=0.5, hist=("shared", "shared"), dense="tma"),
    _case("L6917", (24, 40, 64), 6917, lo=0.5, hist=("global", "shared"), dense="tma"),
    _case("L7108", (24, 40, 64), 7108, lo=0.5, hist=("global", "shared"), dense="tma"),
    _case("L7109", (24, 40, 64), 7109, lo=0.5, hist=("global", "global"), dense="tma"),
    _case("X960", (12, 16, 960), 3000, hist=("shared", "shared"), dense="tma"),
    _case("X1024_L18432", (12, 16, 1024), 3000, slots=18432, lo=0.5, hist=("global", "global"), dense="wide"),
    _case("X1024_L18433", (12, 16, 1024), 3000, slots=18433, lo=0.5, hist=("global", "global"), dense="tma"),
    _case("L65536_sparse", (24, 40, 64), 3000, slots=65536, lo=0.9, edges=True, hist=("global", "global"), dense="tma"),
    _case("L65536_full", (48, 48, 64), 65536, iter_max=3, hist=("global", "global"), dense="tma"),
    _case("L65536_nonlattice", (48, 48, 64), 65536, lattice=False, iter_max=3, hist=("global", "global"), dense="tma"),
]
BY_NAME = {c["name"]: c for c in CASES}


def make_case(c, seed=1):
    """Vessel N(0.75, 0.06), background N(0.35, 0.10) of the level range; every level once in the first voxels; intensities
    spread over 4 units (lattice: slot * 4 / (slots - 1); otherwise sorted uniform values); a 2x2x2 seed in the tube."""
    rng = np.random.default_rng(seed)
    Z, Y, X = c["shape"]
    K = c["levels"]
    cz, cy, cx = Z // 2, Y // 2, X // 2
    half = min(cx - 3, 28)  # the tube's length, so that every shape takes about 30 iterations
    z, y, x = np.ogrid[:Z, :Y, :X]
    r2 = (z - cz) ** 2 + (y - cy) ** 2
    along = np.abs(x - cx + 0.5) < half
    tube = (r2 <= 9) & along
    v = np.where(tube, rng.normal(0.75, 0.06, c["shape"]), rng.normal(0.35, 0.10, c["shape"]))
    dark = v < 0.2
    v = c["lo"] + (1.0 - c["lo"]) * v
    k = np.clip(np.rint(v * (K - 1)), 0, K - 1).astype(np.int64)
    if c["edges"]:
        ring = (r2 > 9) & (r2 <= 13) & along
        k[ring & (rng.random(c["shape"]) < 0.25)] = 0
        k[tube & (rng.random(c["shape"]) < 0.25)] = K - 1
    flat = k.reshape(-1)
    flat[:K] = rng.permutation(K)
    if c["lattice"]:
        n = c["slots"]
        sl = np.round(np.linspace(0, n - 1, K)).astype(np.int64)
        sl[1] = 1
        lv = sl * (4.0 / (n - 1))
    else:
        lv = np.sort(rng.uniform(0.0, 4.0, K))
        assert len(np.unique(lv)) == K
    vm = np.full(c["shape"], 3, np.uint8)
    if c["excl"]:
        vm[dark] = 4
    vm[cz - 1:cz + 1, cy - 1:cy + 1, cx - 1:cx + 1] = 0
    return lv[k], vm


def table_size(c):
    return c["slots"] if c["lattice"] else c["levels"]


def sms():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def table_passes(L, n_sms):
    """Passes of the fused tail over the table words: its last min(LW, SMs - 1) blocks build one word each per pass."""
    lw = (L + 31) // 32
    t = min(lw, n_sms - 1)
    return -(-lw // t), t


def hist_kernel(declared):
    """The init histogram kernel's name from the declared branch; shared copies and global atomics are both k_init_hist, told
    apart by the shared memory of its launch."""
    return {"shared": "k_init_hist_shared", "private": "k_init_hist_private"}.get(declared, "k_init_hist")


def classes(c, mode, n_sms):
    """The branches case `c` is declared to reach in `mode`.  Staging and table passes belong to the fused tail, which label 4
    turns off."""
    L = table_size(c)
    npass, _ = table_passes(L, n_sms)
    out = {"kmat": L <= KMAT_MAX, "lattice": c["lattice"], "excluded": c["excl"], "hist": c["hist"][1 if mode == "index" else 0]}
    if not c["excl"]:
        out.update(staged=L <= TAIL_STAGE_MAX, multipass=npass > 1)
    if mode == "f64_dense":
        out["dense"] = "wide_fallback" if c["dense"] == "tma" and c["shape"][2] > 30 * 32 else c["dense"]
    return out


@functools.lru_cache(maxsize=None)
def case_data(name):
    return make_case(BY_NAME[name])


@functools.lru_cache(maxsize=None)
def oracle(name):
    from oracle.c_oracle import vrg_oracle_c
    data, vm = case_data(name)
    return vrg_oracle_c(data, vm, H=H, max_segment_size=MAX_SEG, iter_max=BY_NAME[name]["iter_max"], record_tables=True)


def decisions(ref):
    """The oracle's decision tables: a capped run (exit 3) records one row per applied update and a last empty one."""
    n = ref["iterations"] - (1 if ref["exit"] == 3 else 0)
    return ref["tables"][:n]


def table_changes(ref):
    bits = [np.asarray(a) >= np.asarray(b) for a, b in decisions(ref)]
    return sum(not np.array_equal(p, q) for p, q in zip(bits[:-1], bits[1:]))


def slots_of(levels, c):
    """Table slot of each sorted distinct level."""
    if not c["lattice"]:
        return np.arange(len(levels))
    return np.rint((levels - levels[0]) / (levels[1] - levels[0])).astype(np.int64)


def run(data, vm, mode, monkeypatch, env=(), iter_max=200, profile=False, H=H):
    """One run on a fresh handle, the switches `env` set while the handle is created.  With `profile`, also the names of the
    kernels that ran."""
    from arterynetwork_b200.engine import VRGEngine
    for k in env:
        monkeypatch.setenv(k, "1")
    try:
        eng = VRGEngine(data.shape, H=H, max_segment_size=MAX_SEG, iter_max=iter_max, intensity=mode)
    finally:
        for k in env:
            monkeypatch.delenv(k)
    names = None
    with eng:
        if profile:
            import json
            import tempfile
            from torch.profiler import ProfilerActivity, profile as prof_ctx
            with prof_ctx(activities=[ProfilerActivity.CUDA]) as prof:
                eng.upload(np.asarray(data, dtype=np.float64), np.asarray(vm, dtype=np.uint8))
                eng.init()
                out = dict(eng.run())
            with tempfile.TemporaryDirectory() as tmp:
                prof.export_chrome_trace(tmp + "/trace.json")
                with open(tmp + "/trace.json") as f:
                    trace = json.load(f)
            kernels = [e for e in trace["traceEvents"] if e.get("cat") == "kernel"]
            names = {e["name"] for e in kernels}
            out["hist_smem"] = {e["args"]["shared memory"] for e in kernels if re.search(r"\bk_init_hist<", e["name"])}
        else:
            eng.upload(np.asarray(data, dtype=np.float64), np.asarray(vm, dtype=np.uint8))
            eng.init()
            out = dict(eng.run())
        out["labels"] = eng.labels()
        out["trace"] = eng.trace()
        out["table"] = eng.table()
    out["kernels"] = names
    return out


def assert_same_run(a, b, what):
    for k in COUNTERS:
        assert a[k] == b[k], (what, k)
    assert np.array_equal(a["labels"], b["labels"]) and np.array_equal(a["trace"], b["trace"]), what
    for x, y in zip(a["table"], b["table"]):
        assert np.array_equal(np.asarray(x).view(np.uint64), np.asarray(y).view(np.uint64)), what


def assert_equals_oracle(o, ref, what):
    assert o["iterations"] == ref["iterations"] and o["exit_reason"] == ref["exit"], what
    assert np.array_equal(o["trace"], ref["trace"]), what
    assert np.array_equal(o["labels"], ref["labels"]), what
    assert o["n_in"] == int((ref["labels"] <= 1).sum()) and o["n_excluded"] == int((ref["labels"] == 4).sum()), what
    assert o["n_out"] == ref["labels"].size - o["n_in"] - o["n_excluded"], what
    for k, q in QUIRKS.items():
        assert o[k] == ref["quirk_potential"][q], (what, k)


def observed_classes(names):
    """The branches a run took, from its kernel names."""
    names = list(names)
    out = {"kmat": any(re.search(r"\bk_kmat\b", n) for n in names), "tail": any(re.search(r"\bk_tail<", n) for n in names)}
    hist = {k for k in ("k_init_hist_shared", "k_init_hist_private") if any(k + "<" in n for n in names)}
    if any(re.search(r"\bk_init_hist<", n) for n in names):
        hist.add("k_init_hist")
    out["hist"] = hist
    dense = set()
    for n in names:
        m = re.search(r"\bk_sweep_dense<(true|false), (true|false)>", n)
        if m:
            dense.add("wide" if m.group(2) == "true" else "tma")
        elif re.search(r"\bk_sweep_dense<(true|false)>", n):
            dense.add("tma")
        if "k_sweep_dense_ldg" in n:
            dense.add("ldg")
    out["dense"] = dense
    return out


def reference_sums(levels, hin, hout, rows, mhH):
    """Exact-order-free Parzen sums at levels[rows]: float64 terms A * exp(-0.5 H d^2), as the reference evaluates them,
    multiplied by the integer counts and summed in long double."""
    hin_l, hout_l = hin.astype(np.longdouble), hout.astype(np.longdouble)
    si, so = np.empty(len(rows), np.longdouble), np.empty(len(rows), np.longdouble)
    for s in range(0, len(rows), 64):
        r = rows[s:s + 64]
        d = levels[None, :] - levels[r, None]
        kv = (A * np.exp(mhH * (d * d))).astype(np.longdouble)
        si[s:s + 64] = (kv * hin_l[None, :]).sum(axis=1)
        so[s:s + 64] = (kv * hout_l[None, :]).sum(axis=1)
    return si, so


def check_final_table(table, ref, c, data):
    """The run's final table at every present level (about 1024 of them on a 65536-level table: both ends, every level a band
    voxel holds, the levels around each crossover, and an even spread) against long-double sums from the oracle's final labels.
    rtol = (L + 4) * 2^-53 bounds a float64 sum of L positive terms."""
    lv, pin, pout = table
    L = table_size(c)
    assert len(lv) == L
    levels, inv = np.unique(data, return_inverse=True)
    inv = inv.reshape(-1)
    lab = ref["labels"].reshape(-1)
    hin = np.bincount(inv[lab <= 1], minlength=len(levels))
    hout = np.bincount(inv[(lab == 2) | (lab == 3)], minlength=len(levels))
    n_in, n_out = int(hin.sum()), int(hout.sum())
    slot = slots_of(levels, c)
    assert np.array_equal(lv[slot], levels)
    present = np.flatnonzero(hin + hout)
    if len(present) > 8192:
        bits = np.asarray(pin[slot] >= pout[slot])
        band = np.unique(inv[(lab == 1) | (lab == 2)])
        cross = np.flatnonzero(bits[1:] != bits[:-1])
        pick = np.concatenate([[0, len(levels) - 1], band, cross, cross + 1, cross - 1, cross + 2,
                               np.linspace(0, len(levels) - 1, 1024).astype(np.int64)])
        present = np.intersect1d(np.unique(pick), present)
        assert len(present) >= 1000
    si, so = reference_sums(levels, hin, hout, present, -0.5 * H)
    rtol = (L + 4) * 2.0 ** -53
    got_in, got_out = pin[slot[present]].astype(np.longdouble), pout[slot[present]].astype(np.longdouble)
    want_in, want_out = si / n_in, so / n_out
    err = max(float(np.max(np.abs(got_in - want_in) / want_in)), float(np.max(np.abs(got_out - want_out) / want_out)))
    assert err <= rtol, (c["name"], err, rtol)
    return len(present)


def check_oracle_case(c, ref, data, n_sms):
    """What makes the case a test of its class: decisions far from ties, a run long enough, and (several table passes) the
    decision changing in a word of the last pass, so a fault there changes the result."""
    tabs = decisions(ref)
    margin = min(float(np.min(np.abs(a - b) / np.maximum(a, b))) for a, b in tabs)
    assert margin > 1e-9, (c["name"], margin)
    assert not c["excl"] or (ref["labels"] == 4).any(), c["name"]
    if ref["exit"] == 3:
        assert ref["iterations"] == c["iter_max"] + 1
    else:
        assert ref["exit"] == 0 and ref["iterations"] >= 20, (c["name"], ref["iterations"])
    L = table_size(c)
    npass, t = table_passes(L, n_sms)
    levels = np.unique(data)
    word = slots_of(levels, c) // 32
    seg_words = word[np.searchsorted(levels, data[ref["labels"] <= 1])]
    assert seg_words.max() >= (npass - 1) * t, c["name"]  # the vessel's levels reach the last pass's words
    if npass > 1 and ref["exit"] == 0 and (L + 31) // 32 - (npass - 1) * t > 1:  # a one-word last pass holds only the top level
        late = word >= (npass - 1) * t
        bits = [np.asarray(a)[late] >= np.asarray(b)[late] for a, b in tabs]
        assert any(not np.array_equal(p, q) for p, q in zip(bits[:-1], bits[1:])), c["name"]


def test_cases_reach_every_branch_in_every_mode():
    """Together the cases reach both sides of every host choice in every mode, so moving a threshold cannot quietly move all
    of them into one branch.  (Each case's own test checks with the profiler that it takes its declared branches.)"""
    n_sms = sms()
    for mode in MODES:
        seen = {}
        for c in CASES:
            for k, v in classes(c, mode, n_sms).items():
                seen.setdefault(k, set()).add(v)
        for k in ("kmat", "staged", "multipass", "lattice", "excluded"):
            assert seen[k] == {True, False}, (mode, k)
        assert seen["hist"] == {"shared", "private", "copies", "global"}, mode
        if mode == "f64_dense":
            assert seen["dense"] == {"tma", "wide", "ldg", "wide_fallback"}
        # just below and just above each threshold
        sizes = {table_size(c) for c in CASES}
        lw_max = n_sms - 1
        for below in (KMAT_MAX, TAIL_STAGE_MAX, 32 * lw_max, 880, HIST_COPIES_MAX, *HIST_SHARED_MAX, 18432, 65536):
            assert below in sizes and (below + 1 in sizes or below == 65536), below


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("name", [c["name"] for c in CASES])
def test_level_class_matches_oracle_in_every_variant(name, mode, monkeypatch):
    """Per case and mode: the branches the case is declared for are the ones that ran; the result equals the C oracle's
    (labels, iterations, exit, trace, region sizes, order-dependence counters); the pipelined run, the separate kernels and
    (dense) the refresh-only sweep are bit-identical to it; the refresh sweeps and repeated sweeps follow the oracle's table
    changes; and the final table equals long-double sums from the oracle's final labels."""
    c = BY_NAME[name]
    data, vm = case_data(name)
    ref = oracle(name)
    n_sms = sms()
    check_oracle_case(c, ref, data, n_sms)
    a = run(data, vm, mode, monkeypatch, iter_max=c["iter_max"], profile=True)
    assert a["n_levels"] == table_size(c)
    want = classes(c, mode, n_sms)
    got = observed_classes(a["kernels"])
    assert got["kmat"] == want["kmat"], (name, mode, sorted(a["kernels"]))
    assert got["tail"] == (not c["excl"]), (name, mode)  # label 4 takes the separate kernels
    assert got["hist"] == {hist_kernel(want["hist"])}, (name, mode, got["hist"])
    if want["hist"] in ("copies", "global"):
        assert len(a["hist_smem"]) == 1 and (a["hist_smem"].pop() > 0) == (want["hist"] == "copies"), (name, mode)
    if mode == "f64_dense":
        assert got["dense"] == {{"wide_fallback": "tma"}.get(want["dense"], want["dense"])}, (name, got["dense"])
    assert_equals_oracle(a, ref, (name, mode))
    variants = [("VRG_PIPELINE",), ("VRG_NO_FUSED_TAIL",)] + ([("VRG_NO_DCACHE",)] if mode == "f64_dense" else [])
    runs = {env: run(data, vm, mode, monkeypatch, env=env, iter_max=c["iter_max"]) for env in variants}
    for env, o in runs.items():
        assert_same_run(a, o, (name, mode, env))
    if ref["exit"] == 0:
        changes = table_changes(ref)
        if not c["excl"]:  # the pipelined run needs the fused tail
            assert runs[("VRG_PIPELINE",)]["redone_sweeps"] == changes
        if mode == "f64_dense":
            for o in (a, runs[("VRG_PIPELINE",)], runs[("VRG_NO_FUSED_TAIL",)]):
                assert o["dense_refresh_sweeps"] == 1 + changes, name
    if mode == "f64_dense":
        b = runs[("VRG_NO_DCACHE",)]
        assert b["dense_refresh_sweeps"] == b["sweeps"]
    check_final_table(a["table"], ref, c, data)


@pytest.mark.parametrize("name", ["L2049", "L4097", "L6145_oddx", "X1024_L18433", "L65536_sparse"])
def test_parzen_sums_of_every_iteration_through_the_step_api(name):
    """Host-driven steps (vrg_enqueue_decide -> vrg_get_table, k_table) against the oracle's table of every iteration at every
    present level.  Both are float64 sums of the same terms within (L + 4) * 2^-53 of the exact sum, so they agree to twice
    that."""
    from arterynetwork_b200.engine import VRGEngine
    c = BY_NAME[name]
    data, vm = case_data(name)
    ref = oracle(name)
    tabs = decisions(ref)
    levels = np.unique(data)
    slot = slots_of(levels, c)
    rtol = 2 * (table_size(c) + 4) * 2.0 ** -53
    it, worst = 0, 0.0
    with VRGEngine(data.shape, H=H, max_segment_size=MAX_SEG, intensity="f64_band") as eng:
        eng.upload(data, vm)
        eng.init()
        while True:
            eng.enqueue_decide()
            lv, pin, pout = eng.table()
            rin, rout = tabs[it]
            assert np.array_equal(lv[slot], levels)
            worst = max(worst, float(np.max(np.abs(pin[slot] - rin) / rin)), float(np.max(np.abs(pout[slot] - rout) / rout)))
            eng.enqueue_cancel(); eng.enqueue_absorb(); eng.enqueue_flip(); eng.enqueue_advance()
            it += 1
            if eng.poll()["exit_reason"] != -1:
                break
        assert eng.poll()["iterations"] == ref["iterations"] and np.array_equal(eng.labels(), ref["labels"])
    assert it == len(tabs)
    assert worst <= rtol, (worst, rtol)


def test_index_mode_reads_the_end_slots_of_a_65536_slot_lattice(monkeypatch):
    """uint16 slot 65535 and slot 0 both hold band voxels of the final labels, and the index run equals the oracle."""
    c = BY_NAME["L65536_sparse"]
    data, vm = case_data(c["name"])
    ref = oracle(c["name"])
    slot = slots_of(np.unique(data), c)[np.searchsorted(np.unique(data), data)]
    band = (ref["labels"] == 1) | (ref["labels"] == 2)
    assert slot.max() == 65535 and (band & (slot == 65535)).sum() > 0 and (band & (slot == 0)).sum() > 0
    o = run(data, vm, "index", monkeypatch)
    assert_equals_oracle(o, ref, "index")


def test_65537_levels_raise_and_the_dropin_takes_the_continuous_mode():
    """One level more than the table holds: LevelsError in every table mode; the drop-in falls back to the brute-force Parzen
    mode and equals the exact-sum oracle.  The segment cap ends the run after a few updates: the exact-sum oracle takes
    minutes for the whole run."""
    from arterynetwork_b200 import variationalRegionGrowing as mod
    from arterynetwork_b200._native import LevelsError
    from arterynetwork_b200.engine import VRGEngine
    from oracle.vrg_oracle import vrg_oracle_exact
    c = _case("L65537", (33, 45, 45), 65537, lattice=False)
    data, vm = make_case(c)
    assert len(np.unique(data)) == 65537
    for mode in MODES:
        with VRGEngine(data.shape, H=H, max_segment_size=MAX_SEG, intensity=mode) as eng:
            with pytest.raises(LevelsError):
                eng.upload(data, vm)
                eng.init()
                eng.run()
    ref = vrg_oracle_exact(data, vm, H=H, max_segment_size=300)
    assert ref["exit"] == 2 and ref["iterations"] >= 3
    vm64 = vm.astype(np.int64)
    with contextlib.redirect_stdout(io.StringIO()) as buf:
        segmented, seg_map, out = mod.variationalRegionGrowing(data, vm64, maxSegmentSize=300)
    assert buf.getvalue().startswith("Finished at iteration %d (Max segment size reached)\n" % ref["iterations"])
    assert out is vm64 and np.array_equal(vm64, ref["labels"]) and np.array_equal(seg_map == 1, ref["seg"])
    assert np.array_equal(segmented, np.argwhere(ref["seg"]))


def test_negative_and_positive_zero_are_one_level(monkeypatch):
    """-0.0 and +0.0 in one volume are one level, as with np.unique, in every mode; count_nonzero counts -0.0 as zero."""
    from arterynetwork_b200.engine import VRGEngine
    from oracle.c_oracle import vrg_oracle_c
    c = _case("zeros", (24, 40, 64), 64, edges=True)
    data, vm = make_case(c)
    zeros = np.flatnonzero(data == 0.0)
    assert len(zeros) > 100
    data.reshape(-1)[zeros[::2]] = -0.0
    assert np.signbit(data).sum() == len(zeros[::2])
    ref = vrg_oracle_c(data, vm, H=H, max_segment_size=MAX_SEG)
    assert ref["iterations"] >= 20
    for mode in MODES:
        o = run(data, vm, mode, monkeypatch)
        assert o["n_levels"] == len(np.unique(data)) == 64, mode
        assert_equals_oracle(o, ref, mode)
        with VRGEngine(data.shape, H=H, max_segment_size=MAX_SEG, intensity=mode) as eng:
            eng.upload(data, vm)
            assert eng.count_nonzero() == np.count_nonzero(data)


@pytest.mark.parametrize("mode", MODES)
def test_one_handle_across_table_classes(mode):
    """One handle: a small table (kmat), the 65536-slot lattice (no kmat, 2048 words), the small table again.  kmat is freed
    and allocated again, the CUDA graph captured again and the dense bit-plane refreshed; each run equals its oracle."""
    from arterynetwork_b200.engine import VRGEngine
    small = _case("small", BY_NAME["L65536_sparse"]["shape"], 300)
    runs = [(make_case(small), None), (case_data("L65536_sparse"), oracle("L65536_sparse")), (make_case(small), None)]
    from oracle.c_oracle import vrg_oracle_c
    with VRGEngine(small["shape"], H=H, max_segment_size=MAX_SEG, intensity=mode) as eng:
        for (data, vm), ref in runs:
            if ref is None:
                ref = vrg_oracle_c(data, vm, H=H, max_segment_size=MAX_SEG)
            eng.upload(data, vm)
            eng.init()
            o = dict(eng.run())
            o["labels"], o["trace"] = eng.labels(), eng.trace()
            assert_equals_oracle(o, ref, (mode, o["n_levels"]))
            if mode == "f64_dense":
                assert 1 <= o["dense_refresh_sweeps"] < o["sweeps"]


@pytest.mark.parametrize("dtype", ["int16", "uint16"])
@pytest.mark.parametrize("on_device", [False, True])
def test_dropin_with_integer_volumes(dtype, on_device):
    """What users pass: an int16 or uint16 volume of 3000 consecutive integer levels (-1500..1499 or 62000..64999), as a NumPy array and
    as CUDA tensors, at the default INTENSITY.  H suits the intensity scale: 2.25 / s^2 for s intensity units per unit of the
    recipe.  Labels, segmentedMap, segmented rows and stdout equal the oracle's."""
    from arterynetwork_b200 import variationalRegionGrowing as mod
    from oracle.c_oracle import vrg_oracle_c
    K = 3000
    c = _case("ints", (24, 40, 64), K)
    data, vm = make_case(c)
    k = np.rint(data * ((K - 1) / 4.0)).astype(np.int64)
    ints = (k - 1500).astype(np.int16) if dtype == "int16" else (k + 62000).astype(np.uint16)
    s = (K - 1) / 4.0
    h = 2.25 / s ** 2
    ref = vrg_oracle_c(ints.astype(np.float64), vm, H=h, max_segment_size=MAX_SEG)
    assert ref["iterations"] >= 20
    want_out = "Finished at iteration %d\nTotal segmented voxels: %d/%d\n" % (
        ref["iterations"], int(ref["seg"].sum()), int(np.count_nonzero(ints)))
    assert mod.INTENSITY == "index"
    vm64 = vm.astype(np.int64)
    if on_device:
        import torch
        d = torch.from_numpy(ints.astype(np.int32) if dtype == "uint16" else ints).cuda()
        if dtype == "uint16":
            d = d.to(torch.uint16)
        assert str(d.dtype) == "torch." + dtype
        v = torch.from_numpy(vm64).cuda()
        with contextlib.redirect_stdout(io.StringIO()) as buf:
            segmented, seg_map, out = mod.variationalRegionGrowing(d, v, H=h, maxSegmentSize=MAX_SEG)
        torch.cuda.synchronize()
        assert out is v
        out, seg_map, segmented = out.cpu().numpy(), seg_map.cpu().numpy(), segmented.cpu().numpy()
    else:
        with contextlib.redirect_stdout(io.StringIO()) as buf:
            segmented, seg_map, out = mod.variationalRegionGrowing(ints, vm64, H=h, maxSegmentSize=MAX_SEG)
        assert out is vm64
    assert buf.getvalue() == want_out
    assert np.array_equal(out, ref["labels"])
    assert seg_map.dtype == np.int64 and np.array_equal(seg_map == 1, ref["seg"])
    assert np.array_equal(segmented, np.argwhere(ref["seg"]))


@pytest.mark.parametrize("on_device", [False, True])
@pytest.mark.parametrize("name", ["L4097", "L65536_sparse"])
def test_update_init_branch_sums_on_tables_without_kmat(name, on_device):
    """update()'s init branch on a table without kmat, as host arrays and as CUDA tensors, from the oracle's final
    segmentation: valueMap comes back as the oracle's labels, and innerProb / outerProb hold at every band voxel the
    reference's unnormalised Parzen sums (VRG:154-155; on the device k_band_sums_dense builds them from the table) to
    (L + 4) * 2^-53 of the long-double sums, and 0 elsewhere."""
    from arterynetwork_b200 import variationalRegionGrowing as mod
    c = BY_NAME[name]
    data, _ = case_data(name)
    ref = oracle(name)
    lab = ref["labels"]
    assert table_size(c) > KMAT_MAX
    levels, inv = np.unique(data, return_inverse=True)
    inv = inv.reshape(data.shape)
    hin = np.bincount(inv[lab <= 1], minlength=len(levels))
    hout = np.bincount(inv[(lab == 2) | (lab == 3)], minlength=len(levels))
    band = (lab == 1) | (lab == 2)
    rows = np.unique(inv[band])
    si, so = reference_sums(levels, hin, hout, rows, -0.5 * H)
    want_in, want_out = si[np.searchsorted(rows, inv[band])], so[np.searchsorted(rows, inv[band])]
    seg_map, vm = (lab <= 1).astype(np.int64), lab.astype(np.int64)
    if on_device:
        import torch
        d, s, v = (torch.from_numpy(np.ascontiguousarray(x)).cuda() for x in (data, seg_map, vm))
        out = mod.update(d, None, s, v, H)
        vm_out, ip, op = out[2].cpu().numpy(), out[5].cpu().numpy(), out[6].cpu().numpy()
    else:
        out = mod.update(data, np.argwhere(lab <= 1), seg_map, vm, H)
        vm_out, ip, op = out[2], out[5], out[6]
    assert np.array_equal(vm_out, lab)
    assert not ip[~band].any() and not op[~band].any()
    rtol = (table_size(c) + 4) * 2.0 ** -53
    err = max(float(np.max(np.abs(ip[band] - want_in) / want_in)), float(np.max(np.abs(op[band] - want_out) / want_out)))
    assert err <= rtol, (err, rtol)


def _slab_worker(rank, world, port, transport, out_dir):
    import os
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    import torch
    import torch.distributed as dist
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    from arterynetwork_b200.distributed import DistributedVRG, GpuSlabEngine, slab_bounds
    from arterynetwork_b200.engine import VRGEngine
    data, vm = case_data("L65536_sparse")
    b = slab_bounds(data.shape[0], world)
    eng = VRGEngine(data.shape, H=H, max_segment_size=MAX_SEG, intensity="index", device=rank, z_begin=b[rank],
                    z_end=b[rank + 1])
    eng.set_stream(torch.cuda.current_stream().cuda_stream)
    eng.upload(data, vm)
    drv = DistributedVRG(GpuSlabEngine(eng, rank), rank, world, check_every=3, transport=transport)
    drv.prepare_levels()
    drv.init()
    res = drv.run()
    np.savez(os.path.join(out_dir, "r%d.npz" % rank), labels=eng.labels(), trace=drv.trace(), iterations=res["iterations"],
             exit=res["exit_reason"])
    dist.barrier()
    eng.close()
    dist.destroy_process_group()


@pytest.mark.parametrize("transport", ["p2p", "collective"])
def test_65536_slot_lattice_on_slabs(transport, tmp_path):
    """The 65536-slot lattice as z-slabs over the box's GPUs (2 to 4), both transports: the statistics vector (2 * 65536 + 8
    int64, 1 MB) fills its exchange slot exactly, and the table is built in several passes behind the exchange.  Labels,
    iterations, exit and trace equal the whole-volume oracle's."""
    import socket
    import torch
    import torch.multiprocessing as mp
    world = min(torch.cuda.device_count(), 4)
    if world < 2:
        pytest.skip("needs at least 2 GPUs")
    ref = oracle("L65536_sparse")
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    mp.spawn(_slab_worker, args=(world, port, transport, str(tmp_path)), nprocs=world, join=True)
    parts = [np.load(str(tmp_path / ("r%d.npz" % r))) for r in range(world)]
    assert np.array_equal(np.concatenate([p["labels"] for p in parts]), ref["labels"])
    for p in parts:
        assert int(p["iterations"]) == ref["iterations"] and int(p["exit"]) == ref["exit"]
        assert np.array_equal(p["trace"], ref["trace"])
