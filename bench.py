#!/usr/bin/env python
"""bench.py -- VRG Gvoxel-updates/s on the BASELINE.json configs (see DESIGN.md "Measurement").

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload c3] [--intensity f64_dense]
    python bench.py --impl reference ...      # CPU arm: the oracle port on the host cores
    python bench.py ... --dump-outputs DIR    # also write the last timed step's outputs as DIR/*.npy (dump_outputs)

One "step" is one complete variational region growing run (level scan + init
branch + every iteration to convergence) on the synthetic vessel-forest phantom
of the named shape.  ``value`` = N_voxels * sweeps / time with the inputs
resident in HBM, on the production path (``vrg_run`` replaying CUDA graphs);
``e2e`` is the same run through the C-ABI with HOST (pinned) buffers, the
host->device copies of intensities + labels and the device->host copy of the
result labels inside the timed region.  Under torchrun (N > 1) the named volume
is cut into z-slabs, one per rank.  Outside the timed regions every run also

* checks its result against ``oracle/vrg_oracle.c`` on the whole volume (labels
  through a position-sensitive hash per slab, trace, iteration count) -> ``parity``;
* runs the largest phantom's weak-scaling slab (config C5: 2048 x 2048 x 128
  planes per GPU) -> ``weak`` (its parity: the N-slab result against one GPU
  running the whole N-slab volume);
* times the reference-facing Python function itself on host arrays -> ``dropin_e2e``.

Prints ONE JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

WORKLOADS = {  # (Z, Y, X): BASELINE.json configs; the 640 / 170 / 1024 axis is the slab axis (SURVEY.md 8(e))
    "c1": (128, 128, 128),
    "c2": (170, 512, 512),
    "c3": (640, 880, 880),
    "c4": (1024, 1024, 1024),
    "c5": (1024, 2048, 2048),
}
ALGO_BYTES_PER_UPDATE = 10.0  # SURVEY.md 8(d): 8 B fp64 intensity + 1 B label read + 1 B label write
METRIC = "VRG Gvoxel-updates/s at 880x880x640, 1/2/4/8 B200; % of HBM roofline"
CPU_SAMPLE_PLANES = 128
ORACLE_MAX_VOXELS = 1.2e9  # whole-volume oracle parity up to here (C4: 1.07e9); larger volumes: one-GPU replica
HALO = 2
DUMP_SAMPLE = 1 << 21  # voxels whose labels --dump-outputs writes
DUMP_SEED = 20240601


def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured"
    except Exception:
        return 6650.0, "fallback"


class ClockSampler:
    """SM clock + throttle reasons during the timed region (B200_PROFILING.md): NVML polled every 10 ms from a thread
    (first sample taken synchronously in start(), so that even a 50 ms timed region is covered); nvidia-smi -lms as the
    fallback when the NVML binding is missing."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")
    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, index=0):
        self.rows, self.proc, self.index = [], None, index
        self.nvml, self.handle, self.stop_flag, self.thread = None, None, threading.Event(), None
        self.sm, self.mx, self.reasons = [], [], set()

    def _nvml_sample(self):
        n = self.nvml
        self.sm.append(float(n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM)))
        self.mx.append(float(n.nvmlDeviceGetMaxClockInfo(self.handle, n.NVML_CLOCK_SM)))
        try:
            mask = int(n.nvmlDeviceGetCurrentClocksEventReasons(self.handle))
        except Exception:
            mask = int(n.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle))
        for bit, name in self.REASONS.items():
            if mask & bit:
                self.reasons.add(name)

    def _nvml_loop(self):
        while not self.stop_flag.wait(0.01):
            try:
                self._nvml_sample()
            except Exception:
                return

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nvml = pynvml
            visible = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(visible.split(",")[self.index]) if visible and visible.split(",")[self.index].isdigit() else self.index
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self._nvml_sample()
            self.thread = threading.Thread(target=self._nvml_loop, daemon=True)
            self.thread.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.nvml is not None:
            self.stop_flag.set()
            self.thread.join(timeout=2)
            return {"sm_mhz": statistics.median(self.sm) if self.sm else None, "sm_max_mhz": max(self.mx) if self.mx else None,
                    "samples": len(self.sm), "reasons": sorted(self.reasons), "source": "nvml, 10 ms period"}
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
                for name, val in zip(names, r[5:9]):
                    if val.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons), "source": "nvidia-smi -lms 200"}


def forest_for(shape, seed):
    from arterynetwork_b200.phantom import forest_segments
    return forest_segments(shape, seed=seed)


def device_phantom(shape, seed, z0, nz, device):
    """fp64 intensities + uint8 seeds of planes [z0, z0+nz) generated on the device."""
    import ctypes
    import torch
    from arterynetwork_b200 import _native as nat
    segs, roots = forest_for(shape, seed)
    d = torch.empty((nz,) + tuple(shape[1:]), dtype=torch.float64, device="cuda:%d" % device)
    v = torch.empty((nz,) + tuple(shape[1:]), dtype=torch.uint8, device="cuda:%d" % device)
    shp = (ctypes.c_int64 * 3)(*shape)
    segs = np.ascontiguousarray(segs); roots = np.ascontiguousarray(roots)
    nat.check(nat.load().vrg_phantom_device(device, ctypes.addressof(shp), z0, nz, segs.ctypes.data, len(segs),
                                            roots.ctypes.data, len(roots), seed, 256, 31, 0, 0,
                                            d.data_ptr(), v.data_ptr()))
    return d, v


def host_phantom_via_device(shape, seed, device, chunk_planes=64):
    """The whole phantom in host memory (float64 + uint8), generated on the device chunk by chunk (bit-identical to the
    NumPy generator, tests/test_gpu_parity.py::test_device_phantom_equals_numpy_phantom -- and far faster)."""
    import torch
    data = np.empty(shape, dtype=np.float64)
    vm = np.empty(shape, dtype=np.uint8)
    for z0 in range(0, shape[0], chunk_planes):
        nz = min(chunk_planes, shape[0] - z0)
        d, v = device_phantom(shape, seed, z0, nz, device)
        torch.cuda.synchronize(device)
        data[z0:z0 + nz] = d.cpu().numpy()
        vm[z0:z0 + nz] = v.cpu().numpy()
        del d, v
    return data, vm


def cpu_sample(shape, seed):
    """Bounded CPU sample of the workload: a window of its planes (about 1e8 voxels at most) that holds seeds, as its
    own volume.  Returns (data, value_map, description, z0)."""
    from arterynetwork_b200.phantom import forest_segments, make_phantom
    nz = min(CPU_SAMPLE_PLANES, shape[0], max(8, int(1.0e8 // (shape[1] * shape[2]))))
    _, roots = forest_segments(shape, seed=seed)
    rz = int(roots[:, 0].min())
    z0 = 0 if rz + 2 <= nz else max(0, min(shape[0] - nz, rz - nz // 2))  # planes [0, nz) unless they hold no seed
    data, vm, _ = make_phantom(shape, seed=seed, z0=z0, nz=nz)
    return data, vm, "planes [%d,%d) of the %dx%dx%d phantom as a %dx%dx%d volume, run to convergence" % (
        z0, z0 + nz, shape[2], shape[1], shape[0], shape[2], shape[1], nz), z0


def reference_python_c1():
    """The unmodified reference's own time on config C1 (128^3), measured in the build container when the golden
    fixture was made (tests/golden/make_golden.py c1_128): the reference is pure Python and cannot travel to the GPU
    box, so this is a recorded number, not one measured in this run."""
    try:
        f = np.load(os.path.join(ROOT, "tests", "golden", "c1_128.npz"))
        sec, it = float(f["reference_wall_s"]), int(f["iterations"])
        return {"seconds": sec, "iterations": it, "Gvoxel_updates_per_s": 128 ** 3 * it / sec / 1e9, "cores": 1,
                "where": "build container, recorded in tests/golden/c1_128.npz (unmodified reference, NumPy %s)" % str(f["numpy_version"])}
    except Exception:
        return None


def time_cpu_port(data, vm, threads):
    from oracle.c_oracle import vrg_oracle_c
    t0 = time.perf_counter()
    o = vrg_oracle_c(data, vm, max_segment_size=10 ** 15, nthreads=threads)
    dt = time.perf_counter() - t0
    return data.size * o["iterations"] / dt / 1e9, dt, o["iterations"]


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    shape = WORKLOADS[args.workload]
    threads = os.cpu_count() or 1
    data, vm, sample, _ = cpu_sample(shape, args.seed)
    for _ in range(args.warmup):
        time_cpu_port(data, vm, threads)
    t0 = time.perf_counter()
    iters = 0
    for _ in range(args.steps):
        _, _, it = time_cpu_port(data, vm, threads)
        iters += it
    dt = time.perf_counter() - t0
    value = data.size * iters / dt / 1e9
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "Gvoxel-updates/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": "%s %dx%dx%d vessel-forest phantom, seed %d" % (args.workload, shape[2], shape[1], shape[0], args.seed)},
        "cpu_baseline": {"value": value, "unit": "Gvoxel-updates/s", "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "Gvoxel-updates/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "note": "the reference is pure Python and exists only in the build container; this arm times oracle/vrg_oracle.c, "
                "the C restatement pinned to the reference's golden outputs, on all host threads",
    }
    print(json.dumps(line))


def workload_shape(args, n_gpus):
    """(Z, Y, X) of the run: the named config, or under --scaling weak its planes / 8 per GPU."""
    Z, Y, X = WORKLOADS[args.workload]
    if args.scaling == "weak":
        Z = (Z // 8) * n_gpus
    return (Z, Y, X)


def kernel_source_sha():
    """Hash of the kernel sources: measurements read back from profiles/ (ncu DRAM traffic) are stamped with it."""
    h = hashlib.sha256()
    for name in ("vrg_kernels.cuh", "vrg_b200.cu"):
        with open(os.path.join(ROOT, "arterynetwork_b200", "csrc", name), "rb") as f:
            h.update(f.read())
    return h.hexdigest()[:16]


def recorded_traffic(workload, intensity):
    """DRAM bytes per sweep launch from the committed ncu capture -- only if it was taken on this very kernel source."""
    path = os.path.join(ROOT, "profiles", "traffic_%s_%s.json" % (workload, intensity))
    try:
        t = json.load(open(path))
    except Exception:
        return None, "no ncu capture committed for this workload"
    if t.get("kernel_source_sha") != kernel_source_sha():
        return None, "profiles/%s was captured on an older kernel source (%s)" % (os.path.basename(path), t.get("kernel_source_sha"))
    return t.get("dram_bytes_per_launch"), "ncu --set full, %s" % t.get("source", os.path.basename(path))


# ------------------------------------------------------------------------------------------------------------------
class Ctx:
    """Where this process runs: one rank of a torchrun launch, or alone."""

    def __init__(self, args):
        import torch
        self.torch = torch
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(self.local)
        self.dist = None
        self.gloo = None
        if self.world > 1:
            import torch.distributed as dist
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local))
            self.dist = dist
            self.gloo = dist.new_group(backend="gloo")  # host-side barriers: no kernel sits on the GPUs while rank 0 works
        self.stream = torch.cuda.Stream()  # CUDA graphs cannot be captured on the default stream

    def barrier(self):
        if self.dist is not None:
            self.dist.barrier()

    def host_barrier(self):
        if self.dist is not None:
            self.dist.barrier(group=self.gloo)

    def max_ms(self, ms):
        if self.dist is None:
            return ms
        t = self.torch.tensor([ms], device="cuda", dtype=self.torch.float64)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def sum_f64(self, a):
        """Element-wise sum of a float64 array over all ranks (the array itself when alone)."""
        if self.dist is None:
            return a
        t = self.torch.from_numpy(np.ascontiguousarray(a, dtype=np.float64)).cuda()
        self.dist.all_reduce(t)
        return t.cpu().numpy()

    def gather_i64(self, values):
        """All ranks' int64 vectors (same length), as a (world, n) array on every rank."""
        t = self.torch.tensor([int(v) - 2 ** 64 if int(v) >= 2 ** 63 else int(v) for v in values], dtype=self.torch.int64,
                              device="cuda")  # uint64 values travel as their two's-complement int64
        if self.dist is None:
            return t.cpu().numpy()[None]
        parts = [self.torch.empty_like(t) for _ in range(self.world)]
        self.dist.all_gather(parts, t)
        return self.torch.stack(parts).cpu().numpy()

    def close(self):
        if self.dist is not None:
            self.dist.destroy_process_group()


def trace_hash(trace):
    return hashlib.sha256(np.ascontiguousarray(trace, dtype=np.int64).tobytes()).hexdigest()[:16]


def dump_outputs(ctx, eng, trace, shape, z0, z1, out_dir):
    """Writes what the run left in `eng` as .npy files under out_dir (rank 0), at most about 25 MB whatever the volume:
    labels_sample (float32) = the labels at labels_sample_index (float64 flat voxel indices, the same ones every run),
    label_counts_per_plane (float64, Z x 5) = how many voxels of each plane carry label 0..4, and
    trace (float64, rows of n_flips, n_in, n_out per iteration)."""
    plane = shape[1] * shape[2]
    nvox = shape[0] * plane
    idx = np.unique(np.random.default_rng(DUMP_SEED).integers(0, nvox, size=min(nvox, DUMP_SAMPLE)))
    lab = eng.labels()  # own planes [z0, z1)
    mine = (idx >= z0 * plane) & (idx < z1 * plane)
    sample = np.zeros(idx.size)
    sample[mine] = lab.reshape(-1)[idx[mine] - z0 * plane]
    counts = np.zeros((shape[0], 5))
    for k in range(5):
        counts[z0:z1, k] = (lab == k).sum(axis=(1, 2))
    sample, counts = ctx.sum_f64(sample), ctx.sum_f64(counts)
    if ctx.rank == 0:
        os.makedirs(out_dir, exist_ok=True)
        np.save(os.path.join(out_dir, "labels_sample.npy"), sample.astype(np.float32))
        np.save(os.path.join(out_dir, "labels_sample_index.npy"), idx.astype(np.float64))
        np.save(os.path.join(out_dir, "label_counts_per_plane.npy"), counts)
        np.save(os.path.join(out_dir, "trace.npy"), np.asarray(trace, dtype=np.float64))


def bench_volume(ctx, shape, seed, intensity, steps, warmup, want_e2e, want_parity, sample_clocks=False, dump_dir=None):
    """Times the whole-volume run of `shape` over ctx.world z-slabs; returns the measurements of one JSON line.
    With `dump_dir`, the outputs of the last timed step are written there (dump_outputs)."""
    import torch
    from arterynetwork_b200 import _native as nat
    from arterynetwork_b200.distributed import DistributedVRG, GpuSlabEngine, slab_bounds
    from arterynetwork_b200.engine import VRGEngine
    rank, world, local = ctx.rank, ctx.world, ctx.local
    nvox = shape[0] * shape[1] * shape[2]
    b = slab_bounds(shape[0], world) if world > 1 else [0, shape[0]]
    z0, z1 = b[rank], b[rank + 1]
    e0, e1 = max(0, z0 - HALO), min(shape[0], z1 + HALO)
    d_data, d_vm = device_phantom(shape, seed, e0, e1 - e0, local)
    torch.cuda.synchronize()
    out = {}
    with torch.cuda.stream(ctx.stream):
        eng = VRGEngine(shape, max_segment_size=10 ** 15, intensity=intensity, device=local, z_begin=z0, z_end=z1)
        eng.set_stream(ctx.stream.cuda_stream)
        drv = DistributedVRG(GpuSlabEngine(eng, local), rank, world, check_every=8, transport="p2p") if world > 1 else None

        def run_after_inputs():
            if drv is None:
                eng.init()
                return eng.run()
            drv.prepare_levels()
            drv.init()
            return drv.run()

        def step():
            eng.attach_device(d_data.data_ptr(), d_vm.data_ptr())
            return run_after_inputs()

        def timed(fn, n):
            start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ctx.barrier()
            torch.cuda.synchronize()
            start.record()
            sweeps = 0
            for _ in range(n):
                sweeps += fn()["sweeps"]
            end.record()
            ctx.barrier()
            torch.cuda.synchronize()
            return ctx.max_ms(start.elapsed_time(end)), sweeps  # device time, max over ranks

        for _ in range(warmup):
            step()
        sampler = ClockSampler(local) if (sample_clocks and rank == 0) else None
        if sampler:
            sampler.start()
        l0 = eng.poll()["kernel_launches"]
        ms, sweeps = timed(step, steps)
        res = eng.poll()
        launches = res["kernel_launches"] - l0
        out["clocks"] = sampler.stop() if sampler else None
        if dump_dir:
            dump_outputs(ctx, eng, drv.trace() if drv is not None else eng.trace(), shape, z0, z1, dump_dir)
        # per-launch time of the sweep: one extra step with CUDA events around every sweep launch (plain stream launches);
        # the same step gives the phases of the tail kernel (device clock) and a host-side split of the step
        eng.profile(True)
        ctx.barrier(); torch.cuda.synchronize()
        w0 = time.perf_counter()
        eng.attach_device(d_data.data_ptr(), d_vm.data_ptr())
        if drv is None:
            eng.set_levels(eng.scan_levels())  # vrg_init would do both; called here so that they can be timed on their own
        else:
            drv.prepare_levels()
        torch.cuda.synchronize(); w1 = time.perf_counter()
        eng.init() if drv is None else drv.init()
        torch.cuda.synchronize(); w2 = time.perf_counter()
        eng.run() if drv is None else drv.run()
        torch.cuda.synchronize(); w3 = time.perf_counter()
        prof = eng.get_profile()
        tp = eng.get_tail_profile()
        names = list(tp["first_block_us"])
        allr = ctx.gather_i64([int(tp["first_block_us"][k] * 1e3) for k in names] + [int(tp["last_block_us"][k] * 1e3) for k in names])
        per_rank = ctx.gather_i64([int(prof["decide_ms"] / max(1, prof["decide_launches"]) * 1e6),
                                   int(prof["cancel_ms"] / max(1, prof["cancel_launches"]) * 1e6)])
        prof["sweep_us_per_rank"] = [round(v / 1e3, 2) for v in per_rank[:, 0].tolist()]
        prof["tail_us_per_rank"] = [round(v / 1e3, 2) for v in per_rank[:, 1].tolist()]
        prof["tail_phases_us"] = {"launches": tp["launches"], "phases": names,
                                  "first_block_per_rank": [[round(v / 1e3, 2) for v in row[:len(names)]] for row in allr.tolist()],
                                  "last_block_per_rank": [[round(v / 1e3, 2) for v in row[len(names):]] for row in allr.tolist()]}
        prof["step_split_ms"] = {"levels": (w1 - w0) * 1e3, "init": (w2 - w1) * 1e3, "iterations_eager": (w3 - w2) * 1e3}
        eng.profile(False)
        out.update(ms=ms, sweeps=sweeps, res=res, prof=prof, launches=launches, value=nvox * sweeps / (ms * 1e-3) / 1e9,
                   planes=(z0, z1), local_vox=(min(shape[0], z1 + 1) - max(0, z0 - 1)) * shape[1] * shape[2])
        if want_e2e:
            # end to end through the C-ABI: every rank uploads its extended slab from pinned host memory, reads its labels back
            h_data = torch.empty(d_data.shape, dtype=torch.float64, pin_memory=True)
            h_vm = torch.empty(d_vm.shape, dtype=torch.uint8, pin_memory=True)
            h_out = torch.empty((z1 - z0,) + tuple(shape[1:]), dtype=torch.uint8, pin_memory=True)
            h_data.copy_(d_data); h_vm.copy_(d_vm)
            torch.cuda.synchronize()

            def e2e_step():
                eng.upload(h_data.numpy(), h_vm.numpy())
                r = run_after_inputs()
                nat.check(eng.lib.vrg_download_labels(eng._h, h_out.data_ptr()))
                return r
            for _ in range(max(1, min(warmup, 2))):
                e2e_step()
            e2e_ms, e2e_sweeps = timed(e2e_step, steps)
            io = ctx.gather_i64([h_data.numel() * 8 + h_vm.numel(), h_out.numel()]).sum(axis=0)
            out["e2e"] = {"value": nvox * e2e_sweeps / (e2e_ms * 1e-3) / 1e9, "unit": "Gvoxel-updates/s",
                          "h2d_bytes_per_step": int(io[0]), "d2h_bytes_per_step": int(io[1]),
                          "ms_per_step": e2e_ms / steps, "intensity_mode": intensity}
            del h_data, h_vm, h_out
            step()  # back on the resident inputs for the parity read-out below
        # ---- parity, outside every timed region ----------------------------------------------------------------
        my_hash = eng.labels_hash()
        trace = drv.trace() if drv is not None else eng.trace()
        hashes = ctx.gather_i64([my_hash]).astype(np.uint64)[:, 0]
        thash = ctx.gather_i64([int(trace_hash(trace), 16) >> 1])[:, 0]
        parity = {"labels_hash": "0x%016x" % (int(hashes.sum(dtype=np.uint64)) & (2 ** 64 - 1)),
                  "trace_hash": trace_hash(trace), "ranks_agree_on_trace": bool((thash == thash[0]).all()),
                  "iterations": int(res["iterations"]), "quirk_counters": {k: res[k] for k in res if k.startswith("q_")}}
        if want_parity and rank == 0:
            t0 = time.perf_counter()
            if nvox <= ORACLE_MAX_VOXELS:
                from oracle.c_oracle import hash_labels, vrg_oracle_c
                h_d, h_v = host_phantom_via_device(shape, seed, local)
                ref = vrg_oracle_c(h_d, h_v, max_segment_size=10 ** 15, nthreads=os.cpu_count() or 1)
                ref_hashes = [hash_labels(ref["labels"][b[r]:b[r + 1]], base=b[r] * shape[1] * shape[2]) for r in range(world)]
                ok = [int(ref_hashes[r]) == int(hashes[r]) for r in range(world)]
                parity.update(against="oracle/vrg_oracle.c on the whole %dx%dx%d volume (%d host threads)" % (
                                  shape[2], shape[1], shape[0], os.cpu_count() or 1),
                              labels_equal_per_slab=ok, trace_equal=bool(np.array_equal(ref["trace"], trace)),
                              iterations_equal=bool(ref["iterations"] == res["iterations"]),
                              oracle_quirk_potential=ref["quirk_potential"])
                parity["oracle"] = bool(all(ok) and parity["trace_equal"] and parity["iterations_equal"] and parity["ranks_agree_on_trace"])
                out["host_volume"] = (h_d, h_v, ref)
            else:
                # too large for a host-side oracle: the same volume on ONE GPU (this rank's), whole, as the reference run
                dd, vv = device_phantom(shape, seed, 0, shape[0], local)
                with VRGEngine(shape, max_segment_size=10 ** 15, intensity=intensity, device=local) as one:
                    one.set_stream(ctx.stream.cuda_stream)
                    one.attach_device(dd.data_ptr(), vv.data_ptr())
                    one.init()
                    r1 = one.run()
                    h1, t1 = one.labels_hash(), one.trace()
                del dd, vv
                same = (h1 == (int(hashes.sum(dtype=np.uint64)) & (2 ** 64 - 1)))
                parity.update(against="the whole %dx%dx%d volume on one GPU (too large for the host oracle)" % (shape[2], shape[1], shape[0]),
                              labels_equal=bool(same), trace_equal=bool(np.array_equal(t1, trace)),
                              iterations_equal=bool(r1["iterations"] == res["iterations"]))
                parity["oracle"] = None
                parity["single_gpu"] = bool(same and parity["trace_equal"] and parity["iterations_equal"] and parity["ranks_agree_on_trace"])
            parity["seconds"] = time.perf_counter() - t0
        ctx.host_barrier()
        out["parity"] = parity
        eng.close()
    del d_data, d_vm
    torch.cuda.empty_cache()
    return out


def roofline_of(r, peak, peak_kind, traffic=None, traffic_source=None, kernel="k_sweep_dense"):
    prof = r["prof"]
    per_launch_ms = prof["decide_ms"] / max(1, prof["decide_launches"])
    algo = ALGO_BYTES_PER_UPDATE * r["local_vox"]
    achieved = algo / (per_launch_ms * 1e-3) / 1e9
    sweeps_per_step = r["sweeps"] / max(1, r["steps"])
    return {"bound": "hbm", "kernel": kernel, "achieved": achieved, "peak": peak, "peak_kind": peak_kind, "unit": "GB/s",
            "frac": achieved / peak, "traffic": traffic, "traffic_source": traffic_source,
            "algorithmic_bytes_per_launch": algo, "ms_per_launch": per_launch_ms, "launches_timed": prof["decide_launches"],
            "timed": "CUDA events around every sweep launch of one extra step on plain stream launches (the timed steps replay CUDA graphs)",
            "share_of_step": per_launch_ms * sweeps_per_step / (r["ms"] / max(1, r["steps"])),
            "tail_ms_per_launch": prof["cancel_ms"] / max(1, prof["cancel_launches"]),
            "tail_phases_us": prof.get("tail_phases_us"), "step_split_ms": prof.get("step_split_ms"),
            "sweep_us_per_rank": prof.get("sweep_us_per_rank"), "tail_us_per_rank_eager": prof.get("tail_us_per_rank"),
            "note": "rank 0's slab (own planes +-1)"}


def dropin_e2e(ctx, shape, seed, devices, ref_labels=None, host=None):
    """Wall time of the reference-facing call itself -- variationalRegionGrowing(dataArray, valueMap) with NumPy arrays in
    host memory (float64 volume, int64 valueMap as the reference's own tests build it), everything included: label
    conversion, uploads, level scan, init, iterations, label / int64 segmentedMap downloads, argwhere-style coordinates,
    count_nonzero, the two printed lines."""
    import contextlib
    import io
    from arterynetwork_b200 import variationalRegionGrowing as mod
    data, vm8 = host if host is not None else host_phantom_via_device(shape, seed, ctx.local)
    vm = vm8.astype(np.int64)  # np.full(shape, 3) in the reference's tests is int64
    keep = (mod.DEVICES, mod.INTENSITY, mod.MAX_SECONDS)
    mod.DEVICES, mod.MAX_SECONDS = (list(devices) if len(devices) > 1 else None), None
    mod.DEVICE = devices[0]
    out = {}
    try:
        for mode in ("index", "f64_dense"):
            mod.INTENSITY = mode
            best = None
            for _ in range(2):  # first call warms the CUDA context / module load of a cold process
                v = vm.copy()
                buf = io.StringIO()
                t0 = time.perf_counter()
                with contextlib.redirect_stdout(buf):
                    segmented, seg_map, v_out = mod.variationalRegionGrowing(data, v, maxSegmentSize=10 ** 15)
                dt = time.perf_counter() - t0
                best = dt if best is None else min(best, dt)
            sweeps = mod.LAST_RUN["sweeps"]
            nvox = data.size
            entry = {"seconds": best, "Gvoxel_updates_per_s": nvox * sweeps / best / 1e9, "sweeps": sweeps,
                     "stdout": buf.getvalue().strip().splitlines(), "n_gpus": len(devices),
                     "host_seconds_last_call": {k: round(x, 4) for k, x in mod.LAST_RUN.get("host_seconds", {}).items()}}
            if ref_labels is not None:
                entry["labels_equal_oracle"] = bool(np.array_equal(v_out, ref_labels))
            out[mode] = entry
    finally:
        mod.DEVICES, mod.INTENSITY, mod.MAX_SECONDS = keep
    return out


def run_ours(args):
    ctx = Ctx(args)
    import torch
    rank, world = ctx.rank, ctx.world
    peak, peak_kind = measured_peak()
    shape = workload_shape(args, world)
    nvox = shape[0] * shape[1] * shape[2]
    prim = bench_volume(ctx, shape, args.seed, args.intensity, args.steps, args.warmup, want_e2e=True,
                        want_parity=not args.no_parity, sample_clocks=True, dump_dir=args.dump_outputs)
    prim["steps"] = args.steps
    modes = None
    if world == 1 and not args.quick:
        modes = {}
        for m in ("f64_band", "index"):
            if m == args.intensity:
                continue
            st = max(1, min(args.steps, 3))
            r = bench_volume(ctx, shape, args.seed, m, st, 2, want_e2e=False, want_parity=False)
            r["steps"] = st
            modes[m] = {"value": r["value"], "ms_per_step": r["ms"] / st,
                        "roofline_frac_10B": roofline_of(r, peak, peak_kind)["frac"],
                        "decide_ms_per_launch": r["prof"]["decide_ms"] / max(1, r["prof"]["decide_launches"]),
                        "labels_equal_primary": r["parity"]["labels_hash"] == prim["parity"]["labels_hash"]}
    # weak scaling on the largest phantom (BASELINE.json configs[4]): 2048 x 2048 x 128 planes per GPU
    weak = None
    if not args.quick and args.workload == "c3" and args.scaling == "strong":
        Zw, Yw, Xw = WORKLOADS["c5"]
        wshape = ((Zw // 8) * world, Yw, Xw)
        st = max(1, min(args.steps, 3))
        w = bench_volume(ctx, wshape, args.seed, args.intensity, st, 2, want_e2e=False, want_parity=not args.no_parity)
        w["steps"] = st
        weak = {"workload": "c5 weak: %dx%dx%d (2048x2048x128 planes per GPU)" % (Xw, Yw, wshape[0]), "value": w["value"],
                "unit": "Gvoxel-updates/s", "n_gpus": world, "steps": st, "warmup": 2, "ms_per_step": w["ms"] / st,
                "sweeps_per_step": w["sweeps"] // st, "scaling": "weak",
                "roofline_frac": roofline_of(w, peak, peak_kind)["frac"], "parity": w["parity"],
                "note": "weak-scaling efficiency at N GPUs = this value / (N x the value of the N = 1 run's `weak`)"}
    # the reference-facing Python call on host arrays (rank 0 drives every GPU of the run from one process)
    dropin = None
    if not args.quick:
        if rank == 0:
            dropin = {}
            host = prim.get("host_volume")
            dropin["c3" if args.workload == "c3" else args.workload] = dropin_e2e(
                ctx, shape, args.seed, list(range(world)), ref_labels=host[2]["labels"] if host else None,
                host=(host[0], host[1]) if host else None)
            if world == 1 and args.workload != "c2":
                dropin["c2"] = dropin_e2e(ctx, WORKLOADS["c2"], args.seed, [0])
        ctx.host_barrier()
    prim.pop("host_volume", None)
    if rank == 0:
        traffic, traffic_source = recorded_traffic(args.workload, args.intensity) if world == 1 else (None, None)
        z0, z1 = prim["planes"]
        line = {
            "metric": METRIC, "value": prim["value"], "unit": "Gvoxel-updates/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": prim["ms"] / args.steps, "higher_is_better": True, "scaling": args.scaling,
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": "%s %dx%dx%d vessel-forest phantom, seed %d" % (args.workload, shape[2], shape[1], shape[0], args.seed),
                       "intensity_mode": args.intensity, "sweeps_per_step": prim["sweeps"] // args.steps,
                       "segmented_voxels": prim["res"]["n_in"], "levels": prim["res"]["n_levels"],
                       "partition": "z-slabs, %d planes per rank, halo %d, peer-memory transport" % (z1 - z0, HALO) if world > 1 else "one volume",
                       "cuda_graph": True,
                       "l2": "inputs (%.1f GB per GPU) larger than L2; no flush" % (nvox * 9 / 1e9 / world),
                       "step": "attach resident inputs (zero-copy) + level scan%s + init + all iterations" % (
                           "/all-gather" if world > 1 else "")},
            "clocks": prim["clocks"],
            "e2e": prim["e2e"],
            "gpu_launches": prim["launches"],
            "roofline": roofline_of(prim, peak, peak_kind, traffic, traffic_source,
                                    "k_sweep_dense" if args.intensity == "f64_dense" else "k_sweep_band"),
            "parity": prim["parity"],
            "weak": weak,
            "dropin_e2e": dropin,
        }
        if modes is not None:
            modes[args.intensity] = {"value": prim["value"], "ms_per_step": prim["ms"] / args.steps,
                                     "roofline_frac_10B": line["roofline"]["frac"],
                                     "decide_ms_per_launch": line["roofline"]["ms_per_launch"], "labels_equal_primary": True}
            line["modes"] = modes
        if world == 1:
            # CPU baseline (rank 0, N=1): the oracle port on a bounded sample of the same phantom
            data_s, vm_s, sample, z0_s = cpu_sample(shape, args.seed)
            threads = os.cpu_count() or 1
            cpu_val, cpu_dt, cpu_it = time_cpu_port(data_s, vm_s, threads)
            line["cpu_baseline"] = {"value": cpu_val, "unit": "Gvoxel-updates/s", "cores": threads, "kind": "port",
                                    "sample": sample, "seconds": cpu_dt, "iterations": cpu_it,
                                    "reference_python_c1": reference_python_c1()}
        print(json.dumps(line))
    ctx.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c3", choices=sorted(WORKLOADS))
    ap.add_argument("--intensity", default="f64_dense", choices=["f64_dense", "f64_band", "index"])
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--scaling", default="strong", choices=["strong", "weak"],
                    help="strong: the named volume over N slabs (the BASELINE metric); weak: every GPU gets 1/8 of the "
                         "named volume's planes, i.e. the volume grows with N (c5: 2048x2048x128 per GPU)")
    ap.add_argument("--quick", action="store_true", help="primary measurement only (no secondary modes, weak slab, drop-in timing)")
    ap.add_argument("--no-parity", action="store_true", help="skip the whole-volume oracle comparison")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step as DIR/<name>.npy, to compare two builds output for output")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.impl == "reference":
        if args.dump_outputs:
            ap.error("--dump-outputs writes the GPU path's outputs; the reference arm has none")
        return run_reference_arm(args)
    return run_ours(args)


if __name__ == "__main__":
    main()
