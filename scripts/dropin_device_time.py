"""Wall time of the drop-in ``variationalRegionGrowing`` on CUDA tensors against the same call on host arrays.

C2 and C3 phantoms (bench.device_phantom), the valueMap as int64 (the reference's dtype) and as uint8, INTENSITY ``index``
and ``f64_dense``.  Each call is timed with torch.cuda.synchronize() on both sides: one warm-up call of each kind, then
``--repeats`` calls of each, the two kinds alternating in the same process; medians are reported.  Both calls must return
the same labels, segmentedMap and segmented rows (compared on the device).  Writes one JSON with the device name and power
limit beside the numbers.

    python scripts/dropin_device_time.py --out profiles/r3a_dropin_device_time.json
"""
import argparse
import contextlib
import io
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

import bench  # noqa: E402
from arterynetwork_b200 import variationalRegionGrowing as mod  # noqa: E402


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


def timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    with contextlib.redirect_stdout(io.StringIO()) as buf:
        out = fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t0, out, buf.getvalue(), dict(mod.LAST_RUN)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", default="c2,c3")
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3a_dropin_device_time.json"))
    args = ap.parse_args()
    mod.MAX_SECONDS = None
    rows = []
    for w in args.workloads.split(","):
        shape = bench.WORKLOADS[w]
        d, v8 = bench.device_phantom(shape, 0, 0, shape[0], 0)
        torch.cuda.synchronize()
        h_data, h_vm8 = d.cpu().numpy(), v8.cpu().numpy()
        for lab in ("int64", "uint8"):
            v_dev0 = v8.to(getattr(torch, lab))
            h_vm0 = h_vm8.astype(getattr(np, lab))
            for mode in ("index", "f64_dense"):
                mod.INTENSITY = mode
                state = {}

                def dev_call():
                    v = v_dev0.clone()
                    torch.cuda.synchronize()
                    t, (seg, segmap, _), out, run = timed(lambda: mod.variationalRegionGrowing(d, v, maxSegmentSize=10 ** 15))
                    state["dev"] = (v, segmap, seg, out)
                    return t, run

                def host_call():
                    v = h_vm0.copy()
                    t, (seg, segmap, _), out, run = timed(lambda: mod.variationalRegionGrowing(h_data, v, maxSegmentSize=10 ** 15))
                    state["host"] = (v, segmap, seg, out)
                    return t, run

                dev_call(); host_call()  # warm-up of both kinds
                t_dev, t_host, dev_runs, host_runs = [], [], [], []
                for _ in range(args.repeats):
                    t, r = host_call(); t_host.append(t); host_runs.append(r)
                    t, r = dev_call(); t_dev.append(t); dev_runs.append(r)
                hv, hmap, hseg, hout = state["host"]
                dv, dmap, dseg, dout = state["dev"]
                same = (torch.equal(dv, torch.from_numpy(hv).cuda()) and torch.equal(dmap, torch.from_numpy(hmap).cuda())
                        and torch.equal(dseg, torch.from_numpy(np.ascontiguousarray(hseg)).cuda()) and dout == hout)
                del state

                def median_stages(runs):
                    keys = runs[0]["host_seconds"].keys()
                    return {k: round(statistics.median(r["host_seconds"][k] for r in runs), 5) for k in keys}
                row = {"workload": w, "shape": list(shape), "value_map_dtype": lab, "intensity": mode,
                       "iterations": dev_runs[-1]["iterations"], "segmented": int(dev_runs[-1]["n_in"]),
                       "tensor_call_s": {"median": round(statistics.median(t_dev), 5), "all": [round(x, 5) for x in t_dev]},
                       "numpy_call_s": {"median": round(statistics.median(t_host), 5), "all": [round(x, 5) for x in t_host]},
                       "tensor_stages_median_s": median_stages(dev_runs), "numpy_stages_median_s": median_stages(host_runs),
                       "identical_results": bool(same)}
                print(json.dumps(row), flush=True)
                rows.append(row)
        del d, v8, h_data, h_vm8
        torch.cuda.empty_cache()
    doc = {"what": "drop-in variationalRegionGrowing wall time, CUDA tensors vs host arrays (same process, alternating); "
                   "torch.cuda.synchronize() on both sides of every call; torch's default stream",
           "gpu": gpu_info(), "repeats": args.repeats, "rows": rows}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(doc, f, indent=1)
    if not all(r["identical_results"] for r in rows):
        sys.exit("tensor and host calls differ")


if __name__ == "__main__":
    main()
