#!/usr/bin/env python
"""Timings of distance_transform_edt's feature-transform path (vrg_edt_ft_device) beside the default EDT, on one GPU,
device-resident inputs, CUDA events:

    python scripts/bench_edt_ft.py [--shapes c2,c3] [--reps 5] [--no-scipy]

Prints one JSON line.  For each shape (C2 = 170x512x512, the GBM-scan shape; C3 = 640x880x880) and each of the two masks
of scripts/bench_mask.py (the thin vessel mask of the phantom and a brain-sized solid ellipsoid), four calls:

    default        vrg_edt_device: distances, unit spacing
    dist           feature transform, distances only (indices never stored)
    idx_dist       indices and distances
    idx_dist_aniso indices and distances with sampling (0.8, 0.4, 0.4)

each as ms, with the bytes a call must move at least (1 B mask read; 8 B distances and 12 B indices written, as
requested) over the time, and that rate as a share of the device-to-device copy rate measured in the same run.
``equals_scipy`` (C2 only): idx_dist_aniso equals scipy.ndimage.distance_transform_edt(mask, sampling=(0.8, 0.4, 0.4),
return_indices=True) bit for bit on both masks, and dist equals the default EDT.  The card's name and power limit are read
in the same run."""
import argparse
import ctypes
import json
import os
import subprocess
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

SHAPES = {"c2": (170, 512, 512), "c3": (640, 880, 880)}
ANISO = (0.8, 0.4, 0.4)


def card():
    import torch
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit"], info["max_sm_clock"] = [v.strip() for v in out.split(",")]
    except Exception as e:  # the timing stands without it, but say why it is missing
        info["power_limit"] = "not read: %s" % e
    return info


def timed(fn, reps):
    import torch
    fn()
    torch.cuda.synchronize()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(reps):
        fn()
    e.record()
    torch.cuda.synchronize()
    return s.elapsed_time(e) / reps


def copy_peak_gbps(reps):
    """device-to-device copy of 4 GB (read + write counted), larger than L2"""
    import torch
    a = torch.empty(1 << 29, dtype=torch.float64, device="cuda")
    b = torch.empty_like(a)
    ms = timed(lambda: b.copy_(a), reps)
    return 2 * a.numel() * 8 / ms / 1e6


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--shapes", default="c2,c3")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--no-scipy", action="store_true")
    a = ap.parse_args()
    import torch
    import bench
    from arterynetwork_b200 import _native as nat
    lib = nat.load()
    torch.cuda.set_device(0)
    res = {"card": card(), "reps": a.reps, "copy_peak_GBps": copy_peak_gbps(a.reps), "sampling_aniso": ANISO}
    aniso = (ctypes.c_double * 3)(*ANISO)
    for key in a.shapes.split(","):
        shape = SHAPES[key]
        Z, Y, X = shape
        n = Z * Y * X
        d_data, _ = bench.device_phantom(shape, 0, 0, Z, 0)
        vessel = (d_data > 0.5).to(torch.uint8).contiguous()
        del d_data
        z, y, x = torch.meshgrid(torch.arange(Z, device="cuda"), torch.arange(Y, device="cuda"), torch.arange(X, device="cuda"), indexing="ij")
        brain = ((((z - Z / 2) / (Z / 2 - 2)) ** 2 + ((y - Y / 2) / (Y / 2 - 4)) ** 2 + ((x - X / 2) / (X / 2 - 4)) ** 2) <= 1.0).to(torch.uint8).contiguous()
        del z, y, x
        dist = torch.empty(shape, dtype=torch.float64, device="cuda")
        dist_ref = torch.empty_like(dist)
        idx = torch.empty((3,) + shape, dtype=torch.int32, device="cuda")
        shp = (nat.i64 * 3)(*shape)
        out = {"shape": shape, "voxels": n}
        for mname, m in (("vessel_mask", vessel), ("brain_mask", brain)):
            calls = {
                "default": (lambda: nat.check(lib.vrg_edt_device(0, m.data_ptr(), ctypes.addressof(shp), dist_ref.data_ptr(), None)), 9),
                "dist": (lambda: nat.check(lib.vrg_edt_ft_device(0, m.data_ptr(), ctypes.addressof(shp), None, dist.data_ptr(), None, None)), 9),
                "idx_dist": (lambda: nat.check(lib.vrg_edt_ft_device(0, m.data_ptr(), ctypes.addressof(shp), None, dist.data_ptr(),
                                                                     idx.data_ptr(), None)), 21),
                "idx_dist_aniso": (lambda: nat.check(lib.vrg_edt_ft_device(0, m.data_ptr(), ctypes.addressof(shp), ctypes.addressof(aniso),
                                                                           dist.data_ptr(), idx.data_ptr(), None)), 21),
            }
            r = {"foreground_fraction": float(m.float().mean())}
            for cname, (fn, bpv) in calls.items():
                ms = timed(fn, a.reps)
                gbps = bpv * n / ms / 1e6
                r[cname] = {"ms": round(ms, 4), "bytes_per_voxel": bpv, "GBps": round(gbps, 1),
                            "share_of_copy_peak": round(gbps / res["copy_peak_GBps"], 3)}
            calls["default"][0]()
            calls["dist"][0]()
            torch.cuda.synchronize()
            r["dist_equals_default"] = bool(torch.equal(dist, dist_ref))
            if key == "c2" and not a.no_scipy:
                from scipy import ndimage as ndi
                calls["idx_dist_aniso"][0]()
                torch.cuda.synchronize()
                rdt, rft = ndi.distance_transform_edt(m.cpu().numpy(), sampling=ANISO, return_indices=True)
                r["equals_scipy"] = bool(np.array_equal(idx.cpu().numpy(), rft) and np.array_equal(dist.cpu().numpy(), rdt))
            out[mname] = r
        res[key] = out
        del vessel, brain, dist, dist_ref, idx
        torch.cuda.empty_cache()
    if "c2" in res and not a.no_scipy:
        res["equals_scipy"] = all(res["c2"][k]["equals_scipy"] for k in ("vessel_mask", "brain_mask"))
    print(json.dumps(res))


if __name__ == "__main__":
    main()
