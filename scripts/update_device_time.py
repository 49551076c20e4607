"""Wall time of ``update()`` on CUDA tensors against the same call on host arrays, and the device time of k_band_sums_dense.

C2 and C3 phantoms (bench.device_phantom), both maps as int64 (the reference's dtype).  Two calls are timed: the init branch,
and the flips of the first decision (the reference driver's next update, VRG:79-88,109).  Each call is timed with
torch.cuda.synchronize() on both sides; the inputs are fresh copies made outside the timed window.  One warm-up call of each
kind, then ``--repeats`` calls of each, host and tensor alternating in the same process; medians are reported.  Tensor and
host results must agree bit for bit (labels, segmentedMap, the row lists and both sum volumes).

k_band_sums_dense (vrg_band_sums_device) is timed with CUDA events over ``--kernel-launches`` launches behind one warm-up; its
rate is reported against the 24.3 B per voxel it moves nominally (16 B written: two float64 volumes; 8 B of intensity read at
band voxels only, so in practice less; about 0.3 B of bit-planes) and against the 16 B it writes.  The device name and power
limit are recorded beside the numbers.

``--profile`` instead runs one tensor init call and one tensor flips call per workload under torch.profiler (a run of its
own) and lists every host<->device copy it recorded; none may be as large as the volume at one byte per voxel.

    python scripts/update_device_time.py --out profiles/r3c_update_device_time.json
    python scripts/update_device_time.py --profile --out profiles/r3c_update_device_copies.json
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

import bench  # noqa: E402
from arterynetwork_b200 import _native as nat  # noqa: E402
from arterynetwork_b200 import variationalRegionGrowing as mod  # noqa: E402
from arterynetwork_b200.engine import VRGEngine  # noqa: E402

BYTES_PER_VOXEL = 24.3
WRITTEN_PER_VOXEL = 16.0


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
    out = fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t0, out


def inputs(shape):
    """Host and device phantoms, the state after the host init call, and the first decision's flips."""
    d, v8 = bench.device_phantom(shape, 0, 0, shape[0], 0)
    torch.cuda.synchronize()
    h_data = d.cpu().numpy()
    h_vm = v8.cpu().numpy().astype(np.int64)
    del v8
    segmented = np.argwhere(h_vm == 0)
    h_seg = np.zeros(shape, dtype=np.int64)
    h_seg[tuple(segmented.T)] = 1
    vm1, seg1 = h_vm.copy(), h_seg.copy()
    out = mod.update(h_data, segmented, seg1, vm1, 2.25)
    _, seg_map, vm, ib, ob, ip, op = out
    allb = np.concatenate((ib, ob))
    n_in = np.count_nonzero(vm <= 1)
    n_out = np.count_nonzero((vm == 2) | (vm == 3))
    flips = allb[np.logical_xor(seg_map[tuple(allb.T)], ip[tuple(allb.T)] / n_in >= op[tuple(allb.T)] / n_out)]
    return d, h_data, h_vm, h_seg, segmented, (seg1, vm1, ib, ob), flips


def same(t_out, h_out):
    ok = True
    for t, h in zip(t_out, h_out):
        if isinstance(t, torch.Tensor):
            ok = ok and tuple(t.shape) == h.shape and torch.equal(t, torch.from_numpy(np.ascontiguousarray(h)).cuda())
    return bool(ok)


def band_sums_time(d, seg_t, vm_t, shape, launches):
    nvox = int(np.prod(shape))
    pin = torch.empty(shape, dtype=torch.float64, device="cuda")
    pout = torch.empty(shape, dtype=torch.float64, device="cuda")
    with VRGEngine(shape, max_segment_size=2 ** 62, intensity="f64_band") as eng:
        eng.set_stream(torch.cuda.current_stream().cuda_stream)
        eng.attach_state_typed(d.data_ptr(), seg_t.data_ptr(), nat.DTYPE_I64, vm_t.data_ptr(), nat.DTYPE_I64)
        eng.init()
        eng.enqueue_table()
        eng.poll()
        eng.band_sums_device(pin.data_ptr(), pout.data_ptr())  # warm-up
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(launches):
            eng.band_sums_device(pin.data_ptr(), pout.data_ptr())
        b.record()
        torch.cuda.synchronize()
    ms = a.elapsed_time(b) / launches
    return {"ms": round(ms, 4), "nominal_TBps": round(BYTES_PER_VOXEL * nvox / ms / 1e9, 3),
            "written_TBps": round(WRITTEN_PER_VOXEL * nvox / ms / 1e9, 3), "launches": launches}


def run_timing(args):
    rows = []
    for w in args.workloads.split(","):
        shape = bench.WORKLOADS[w]
        d, h_data, h_vm, h_seg, segmented, (seg1, vm1, ib, ob), flips = inputs(shape)
        flips_t = torch.from_numpy(flips).cuda()
        vm_t0, seg_t0 = torch.from_numpy(h_vm).cuda(), torch.from_numpy(h_seg).cuda()
        vm1_t0, seg1_t0 = torch.from_numpy(vm1).cuda(), torch.from_numpy(seg1).cuda()
        last = {}

        def host_init():
            vm, seg = h_vm.copy(), h_seg.copy()
            t, out = timed(lambda: mod.update(h_data, segmented, seg, vm, 2.25))
            last["host_init"] = out
            return t

        def dev_init():
            vm, seg = vm_t0.clone(), seg_t0.clone()
            t, out = timed(lambda: mod.update(d, segmented, seg, vm, 2.25))
            last["dev_init"] = out
            return t

        def host_flips():
            vm, seg = vm1.copy(), seg1.copy()
            ip, op = np.zeros(shape), np.zeros(shape)
            t, out = timed(lambda: mod.update(h_data, segmented, seg, vm, 2.25, flips, ib, ob, ip, op))
            last["host_flips"] = out
            return t

        def dev_flips():
            vm, seg = vm1_t0.clone(), seg1_t0.clone()
            ip = torch.zeros(shape, dtype=torch.float64, device="cuda")
            op = torch.zeros(shape, dtype=torch.float64, device="cuda")
            t, out = timed(lambda: mod.update(d, segmented, seg, vm, 2.25, flips_t, None, None, ip, op))
            last["dev_flips"] = out
            return t

        calls = {"host_init": host_init, "dev_init": dev_init, "host_flips": host_flips, "dev_flips": dev_flips}
        for fn in calls.values():
            fn()  # warm-up of every kind
        times = {k: [] for k in calls}
        for _ in range(args.repeats):
            for k, fn in calls.items():
                last.pop(k, None)
                times[k].append(fn())
        identical = {"init": same(last["dev_init"], last["host_init"]), "flips": same(last["dev_flips"], last["host_flips"])}
        kern = band_sums_time(d, seg_t0, vm_t0, shape, args.kernel_launches)
        row = {"workload": w, "shape": list(shape), "flips": int(len(flips)),
               "inner_band": int(len(last["host_flips"][3])), "outer_band": int(len(last["host_flips"][4])),
               **{k + "_s": {"median": round(statistics.median(v), 4), "all": [round(x, 4) for x in v]} for k, v in times.items()},
               "identical_results": identical, "k_band_sums_dense": kern}
        print(json.dumps(row), flush=True)
        rows.append(row)
        last.clear()
        del d, vm_t0, seg_t0, vm1_t0, seg1_t0, flips_t
        torch.cuda.empty_cache()
    return {"what": "update() wall time, CUDA tensors vs host arrays (same process, alternating, int64 maps, torch's default "
                    "stream, torch.cuda.synchronize() on both sides of every call); k_band_sums_dense device time by CUDA "
                    "events", "bytes_per_voxel_nominal": BYTES_PER_VOXEL, "repeats": args.repeats, "rows": rows}


def run_profile(args):
    from torch.profiler import ProfilerActivity, profile
    rows = []
    for w in args.workloads.split(","):
        shape = bench.WORKLOADS[w]
        nvox = int(np.prod(shape))
        d, h_data, h_vm, h_seg, segmented, (seg1, vm1, ib, ob), flips = inputs(shape)
        vm, seg = torch.from_numpy(h_vm).cuda(), torch.from_numpy(h_seg).cuda()
        vm1_t, seg1_t = torch.from_numpy(vm1).cuda(), torch.from_numpy(seg1).cuda()
        flips_t = torch.from_numpy(flips).cuda()
        mod.update(d, segmented, seg.clone(), vm.clone(), 2.25)  # warm-up outside the capture
        torch.cuda.synchronize()
        with tempfile.TemporaryDirectory() as tmp:
            with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
                mod.update(d, segmented, seg, vm, 2.25)
                mod.update(d, segmented, seg1_t, vm1_t, 2.25, flips_t)
                torch.cuda.synchronize()
            trace = os.path.join(tmp, "trace.json")
            prof.export_chrome_trace(trace)
            with open(trace) as f:
                events = json.load(f)["traceEvents"]
        copies = [{"name": e["name"], "bytes": int(e.get("args", {}).get("bytes", -1))}
                  for e in events if e.get("cat") == "gpu_memcpy"]
        kernels = sorted({e["name"] for e in events if e.get("cat") == "kernel"})
        h2d_d2h = [c for c in copies if "HtoD" in c["name"] or "DtoH" in c["name"]]
        row = {"workload": w, "shape": list(shape), "volume_bytes_at_1B_per_voxel": nvox, "copies_h2d_d2h": len(h2d_d2h),
               "largest_h2d_d2h_bytes": max([c["bytes"] for c in h2d_d2h], default=0),
               "total_h2d_d2h_bytes": sum(max(0, c["bytes"]) for c in h2d_d2h),
               "volume_sized_copies": [c for c in h2d_d2h if c["bytes"] < 0 or c["bytes"] >= nvox],
               "kernels": kernels}
        print(json.dumps({k: v for k, v in row.items() if k != "kernels"}), flush=True)
        rows.append(row)
        del d, vm, seg, vm1_t, seg1_t, flips_t
        torch.cuda.empty_cache()
    return {"what": "host<->device copies recorded by torch.profiler around one tensor init call and one tensor flips call",
            "rows": rows}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", default="c2,c3")
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--kernel-launches", type=int, default=20)
    ap.add_argument("--profile", action="store_true")
    ap.add_argument("--out", required=True)
    args = ap.parse_args()
    doc = run_profile(args) if args.profile else run_timing(args)
    doc["gpu"] = gpu_info()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(doc, f, indent=1)
    if args.profile:
        if any(r["volume_sized_copies"] for r in doc["rows"]):
            sys.exit("a volume-sized host<->device copy was recorded")
    elif not all(all(r["identical_results"].values()) for r in doc["rows"]):
        sys.exit("tensor and host calls differ")


if __name__ == "__main__":
    main()
