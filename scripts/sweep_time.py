#!/usr/bin/env python
"""Timings of the dense sweep on arbitrary volume shapes (one process, several shapes):

    python scripts/sweep_time.py 640x880x880 82x880x880 128x2048x2048

Each item is ZxYxX.  Prints one JSON line per shape: mean k_sweep_dense time (CUDA events on the launch stream), whole-run
time with CUDA graphs, iterations."""
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench  # noqa: E402


def main():
    import torch
    from arterynetwork_b200.engine import VRGEngine
    torch.cuda.set_device(0)
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    for item in sys.argv[1:]:
        shape = tuple(int(t) for t in item.split("x"))
        d, v = bench.device_phantom(shape, 0, 0, shape[0], 0)
        torch.cuda.synchronize()
        nvox = shape[0] * shape[1] * shape[2]
        with VRGEngine(shape, max_segment_size=10 ** 15, intensity="f64_dense") as eng:
            eng.set_stream(stream.cuda_stream)

            def step():
                eng.attach_device(d.data_ptr(), v.data_ptr())
                eng.init()
                return eng.run()
            step(); step()
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            s.record()
            res = step()
            e.record()
            torch.cuda.synchronize()
            ms_graph = s.elapsed_time(e)
            eng.profile(True)
            s.record()
            res = step()
            e.record()
            torch.cuda.synchronize()
            ms_eager = s.elapsed_time(e)
            prof = eng.get_profile()
            tail = eng.get_tail_profile()
            eng.profile(False)
        per = prof["decide_ms"] / max(1, prof["decide_launches"])
        print(json.dumps({"shape": shape, "sweeps": res["sweeps"], "sweep_ms": per,
                          "sweep_10B_GBps": 10.0 * nvox / (per * 1e-3) / 1e9, "real_8B_GBps": 8.13 * nvox / (per * 1e-3) / 1e9,
                          "cancel_ms": prof["cancel_ms"] / max(1, prof["cancel_launches"]), "tail_phases_us": tail,
                          "run_ms_graph": ms_graph, "run_ms_eager_profiled": ms_eager,
                          "Gvox_s_graph": nvox * res["sweeps"] / ms_graph / 1e6,
                          "per_iter_us_graph": 1e3 * ms_graph / res["sweeps"]}), flush=True)
        del d, v
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
