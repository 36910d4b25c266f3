"""The CPU-runnable arms of bench.py: `--impl reference` (the oracle port on the host cores,
one JSON line with the contract's keys) and `--workload loader` (host C++ loader vs the
reference's pandas body).  The GPU arm is exercised on the GPU box by the driver."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(*args):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], cwd=ROOT,
                         capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, f"stdout must carry exactly one JSON line, got {len(lines)}"
    return json.loads(lines[0])


def test_reference_arm_prints_the_contract_line():
    d = _run("--impl", "reference", "--genes", "300", "--ref-batch", "8", "--steps", "1",
             "--warmup", "0")
    assert d["impl"] == "reference" and d["metric"] == "BiGAN train cells/sec"
    assert d["unit"] == "cells/s" and d["higher_is_better"] is True and d["value"] > 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"] == {"value": d["value"], "unit": "cells/s", "h2d_bytes_per_step": 0,
                        "d2h_bytes_per_step": 0}
    assert "workload" in d["config"]


def test_reference_arm_classify_and_encode_workloads():
    c = _run("--impl", "reference", "--workload", "classify", "--genes", "200", "--ref-batch", "6",
             "--steps", "1", "--warmup", "0")
    assert "ClassifyCellBiGan" in c["config"]["workload"] and c["value"] > 0
    e = _run("--impl", "reference", "--workload", "encode", "--genes", "200")
    assert e["metric"] == "encode cells/sec" and e["value"] > 0


def test_loader_workload_matches_the_reference_body():
    d = _run("--workload", "loader", "--loader-cells", "40", "--genes", "600", "--steps", "1")
    assert d["metric"] == "load_matrix nnz/sec" and d["matches_reference_pandas_body"] is True
    assert d["cpu_baseline"]["kind"] == "reference" and d["value"] > 0 and d["gpu_launches"] == 0


def test_argument_checks():
    for args in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", "d"],
                 ["--workload", "encode", "--dump-outputs", "d"]):
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], cwd=ROOT,
                           capture_output=True, text=True, timeout=120)
        assert r.returncode == 2 and r.stdout == "", (args, r.stderr)


def test_dump_outputs_writes_a_fixed_sample_of_every_network(tmp_path):
    """bench.dump_outputs on stand-in networks whose every weight holds its own flat index:
    the sample is the same positions on every call, sorted, drawn across all arrays."""
    import numpy as np
    import bench

    class Net:
        def __init__(self, shapes):
            self.arrays, n = [], 0
            for s in shapes:
                size = int(np.prod(s))
                self.arrays.append(np.arange(n, n + size, dtype=np.float32).reshape(s))
                n += size

        def get_weights(self):
            return [a.copy() for a in self.arrays]

    class Engine:
        nets = {"G": Net([(300, 200), (200,), (40,)]), "E": Net([(7, 5), (5,)]), "D": Net([(9,)])}

    a, b = tmp_path / "a", tmp_path / "b"
    bench.dump_outputs(str(a), [0.5, 0.25, 2.0], Engine(), 0, sample=1000)
    bench.dump_outputs(str(b), [0.5, 0.25, 2.0], Engine(), 0, sample=1000)
    assert sorted(os.listdir(a)) == ["D_weights.npy", "E_weights.npy", "G_weights.npy", "losses.npy"]
    losses = np.load(a / "losses.npy")
    assert losses.dtype == np.float64 and losses.tolist() == [0.5, 0.25, 2.0]
    g = np.load(a / "G_weights.npy")
    assert g.dtype == np.float32 and len(g) == 1000 and (np.diff(g) > 0).all()
    assert g.max() >= 300 * 200                         # reaches past the first array
    assert np.load(a / "E_weights.npy").tolist() == list(range(40))   # smaller than the sample
    for name in os.listdir(a):
        assert np.array_equal(np.load(a / name), np.load(b / name))
    bench.dump_outputs(str(tmp_path / "c"), [0.0] * 3, Engine(), 1)   # other ranks write nothing
    assert not (tmp_path / "c").exists()


def test_stdout_is_parked_on_stderr_while_libraries_initialise():
    """bench.stdout_to_stderr: C-level (buffered printf) and Python-level writes made inside the
    block land on stderr; stdout keeps only what is printed afterwards."""
    code = (
        "import sys, ctypes; sys.path.insert(0, %r); import bench\n"
        "libc = ctypes.CDLL(None)\n"
        "with bench.stdout_to_stderr():\n"
        "    libc.printf(b'NCCL version x.y\\n'); print('python banner')\n"
        "print('{\"ok\": 1}', flush=True)\n" % ROOT)
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stderr
    assert r.stdout == '{"ok": 1}\n'
    assert "NCCL version x.y" in r.stderr and "python banner" in r.stderr
