"""Step time of the f64_dense run with the decision bit-plane (default) and without it (VRG_NO_DCACHE=1), C3 and C4.

One process, one device-resident phantom per workload (bench.device_phantom), two handles on the same inputs: one created
with VRG_NO_DCACHE=1 (every sweep reads the fp64 volume), one without (only the refresh sweeps do).  A step is what bench.py
times: attach + level scan + init + all iterations, device-synchronised.  One warm-up step of each, then `--rounds` rounds
that alternate the two; medians are reported, and every step's label hash and trace must agree between the two.  Then one
profiled step of each (CUDA events around every sweep launch pair, plain stream launches):
  refresh_sweep_ms = the mean sweep of the VRG_NO_DCACHE step (every one of its sweeps is a refresh);
  cached_sweep_ms  = (sweeps x mean - refresh_sweep_ms) / (sweeps - 1) from the default step, which has one refresh.
Writes one JSON with the card's name, power limit and max SM clock beside the numbers.

    python scripts/dense_cache_time.py --out profiles/r3b_dense_cache_time.json
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

import bench  # noqa: E402
from arterynetwork_b200.engine import VRGEngine  # noqa: E402


def gpu_info():
    info = {"torch_name": torch.cuda.get_device_name(0)}
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clock = [x.strip() for x in out.split(",")]
        info.update(name=name, power_limit=power, max_sm_clock=clock)
    except Exception as e:  # noqa: BLE001 -- the numbers are still worth having; say why the card's data is missing
        info["nvidia_smi_error"] = repr(e)
    return info


def make_engine(shape, no_dcache):
    if no_dcache:
        os.environ["VRG_NO_DCACHE"] = "1"
    try:
        return VRGEngine(shape, max_segment_size=10 ** 15, intensity="f64_dense")
    finally:
        os.environ.pop("VRG_NO_DCACHE", None)


def step(eng, d, v):
    eng.attach_device(d.data_ptr(), v.data_ptr())
    eng.init()
    return eng.run()


def timed_step(eng, d, v):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    res = step(eng, d, v)
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) * 1e3, res, eng.labels_hash(), bench.trace_hash(eng.trace())


def profiled_step(eng, d, v):
    eng.profile(True)
    res = step(eng, d, v)
    torch.cuda.synchronize()
    prof = eng.get_profile()
    eng.profile(False)
    return res, prof


def measure(workload, rounds):
    shape = bench.WORKLOADS[workload]
    d, v = bench.device_phantom(shape, 0, 0, shape[0], 0)
    torch.cuda.synchronize()
    engines = {"default": make_engine(shape, False), "no_dcache": make_engine(shape, True)}
    ms = {k: [] for k in engines}
    seen = {}
    for k, eng in engines.items():  # warm-up: module load, graph capture
        timed_step(eng, d, v)
    for _ in range(rounds):
        for k, eng in engines.items():
            t, res, lh, th = timed_step(eng, d, v)
            ms[k].append(t)
            seen.setdefault(k, (lh, th, res))
            assert (lh, th) == seen[k][:2], "%s: outputs changed between steps" % k
    assert seen["default"][:2] == seen["no_dcache"][:2], "default and VRG_NO_DCACHE=1 computed different outputs"
    prof = {k: profiled_step(eng, d, v) for k, eng in engines.items()}
    res_d, prof_d = prof["default"]
    res_n, prof_n = prof["no_dcache"]
    refresh_ms = prof_n["decide_ms"] / max(1, prof_n["decide_launches"])
    n = prof_d["decide_launches"]
    mean_d = prof_d["decide_ms"] / max(1, n)
    row = {
        "workload": "%s %dx%dx%d" % (workload, shape[2], shape[1], shape[0]),
        "ms_per_step_default": statistics.median(ms["default"]), "ms_per_step_no_dcache": statistics.median(ms["no_dcache"]),
        "ms_per_step_all": ms, "rounds": rounds,
        "speedup": statistics.median(ms["no_dcache"]) / statistics.median(ms["default"]),
        "sweeps": seen["default"][2]["sweeps"], "iterations": seen["default"][2]["iterations"],
        "dense_refresh_sweeps": res_d["dense_refresh_sweeps"], "dense_refresh_sweeps_no_dcache": res_n["dense_refresh_sweeps"],
        "refresh_sweep_ms": refresh_ms, "mean_sweep_ms_default": mean_d,
        "cached_sweep_ms": (n * mean_d - refresh_ms) / (n - 1) if n > 1 else None,
        "profiled_sweeps": n,
        "tail_ms_per_launch_default": prof_d["cancel_ms"] / max(1, prof_d["cancel_launches"]),
        "labels_hash": "0x%016x" % seen["default"][0], "trace_hash": seen["default"][1],
        "outputs_equal": True,
    }
    for eng in engines.values():
        eng.close()
    del d, v
    torch.cuda.empty_cache()
    return row


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", default="c3,c4")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3b_dense_cache_time.json"))
    args = ap.parse_args()
    out = {"gpu": gpu_info(), "rows": [measure(w, args.rounds) for w in args.workloads.split(",")]}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
