"""CPU: the parts of bench.py's contract that need no GPU -- the reference arm's JSON line, the bounded CPU sample, the
workload shapes."""
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402


def test_reference_arm_prints_one_json_line_with_the_contract_keys():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "c1",
                          "--steps", "1", "--warmup", "0"], capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == bench.METRIC and d["unit"] == "Gvoxel-updates/s"
    assert d["higher_is_better"] is True and d["steps"] == 1 and d["warmup"] == 0 and d["value"] > 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["gpu_launches"] == 0


def test_reference_arm_is_silent_on_other_ranks():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1",
                          "--warmup", "0"], capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_bad_arguments_are_refused():
    for extra in (["--steps", "0"], ["--warmup", "-1"], ["--impl", "reference", "--dump-outputs", "x"]):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + extra, capture_output=True, text=True,
                             timeout=120, cwd=ROOT)
        assert out.returncode == 2 and out.stdout == "", (extra, out.stderr[-500:])


def test_dump_outputs_writes_a_fixed_sample_the_plane_counts_and_the_trace(tmp_path):
    shape = (6, 7, 9)
    labels = np.random.default_rng(1).integers(0, 5, size=shape, dtype=np.uint8)
    trace = np.array([[-1, 8, 370], [3, 11, 367]])

    class Ctx:
        rank = 0

        @staticmethod
        def sum_f64(a):
            return a

    class Eng:
        @staticmethod
        def labels():
            return labels.copy()

    for d in ("a", "b"):
        bench.dump_outputs(Ctx, Eng, trace, shape, 0, shape[0], str(tmp_path / d))
    a = {n: np.load(str(tmp_path / "a" / (n + ".npy"))) for n in ("labels_sample", "labels_sample_index", "label_counts_per_plane", "trace")}
    for n, v in a.items():
        assert v.dtype in (np.float32, np.float64)
        assert np.array_equal(v, np.load(str(tmp_path / "b" / (n + ".npy"))))
    idx = a["labels_sample_index"].astype(np.int64)
    assert np.array_equal(a["labels_sample"], labels.ravel()[idx])
    assert np.array_equal(a["label_counts_per_plane"], [[np.count_nonzero(p == k) for k in range(5)] for p in labels])
    assert np.array_equal(a["trace"], trace)
    # the two sample files stay the same size on every workload, far below 64 MB
    assert bench.DUMP_SAMPLE * (4 + 8) + bench.WORKLOADS["c5"][0] * 5 * 8 < 32 * 2 ** 20


def test_cpu_sample_is_bounded_and_holds_seeds():
    for name in ("c2", "c3", "c5"):
        shape = bench.WORKLOADS[name]
        from arterynetwork_b200.phantom import forest_segments
        _, roots = forest_segments(shape, seed=0)
        nz = min(bench.CPU_SAMPLE_PLANES, shape[0], max(8, int(1.0e8 // (shape[1] * shape[2]))))
        assert nz * shape[1] * shape[2] <= 1.3e8
        rz = int(roots[:, 0].min())
        z0 = 0 if rz + 2 <= nz else max(0, min(shape[0] - nz, rz - nz // 2))
        assert z0 <= rz and rz + 2 <= z0 + nz  # a whole 2x2x2 seed cube lies inside the window


def test_workload_shapes():
    class A:
        workload, scaling = "c5", "weak"
    assert bench.workload_shape(A, 1) == (128, 2048, 2048) and bench.workload_shape(A, 8) == bench.WORKLOADS["c5"]
    A.scaling = "strong"
    assert bench.workload_shape(A, 4) == bench.WORKLOADS["c5"]
    assert bench.WORKLOADS["c3"] == (640, 880, 880) and bench.ALGO_BYTES_PER_UPDATE == 10.0
    r = bench.reference_python_c1()
    assert r is not None and r["cores"] == 1 and 500 < r["seconds"] < 700 and np.isclose(r["Gvoxel_updates_per_s"], 128 ** 3 * r["iterations"] / r["seconds"] / 1e9)
