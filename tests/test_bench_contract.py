"""CPU: the bench contract.  (1) `bench.py --impl reference` runs without a GPU and prints ONE JSON line with the keys
the driver reads (same `config.workload` string as our arm).  (2) The committed round-2 bench lines (profiles/) carry
the blocks the task statement asks for -- roofline, e2e, parity (green), cfg5 -- at every N."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_runs_on_cpu_and_matches_the_contract():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "poisson32",
                          "--steps", "1", "--warmup", "0"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
              "dtype", "data", "config", "impl", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["impl"] == "reference" and d["unit"] == "it/s" and d["value"] > 0 and d["higher_is_better"] is True
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    sys.path.insert(0, ROOT)
    import bench
    assert d["config"]["workload"] == bench.workload_name(*bench.WORKLOADS["poisson32"])


@pytest.mark.parametrize("fn,n", [("r2_bench_n1_default_final.json", 1), ("r2_bench_n2_final.json", 2), ("r2_bench_n4_final.json", 4),
                                  ("r2_bench_n8_final.json", 8)])
def test_committed_bench_lines_carry_green_parity_and_cfg5(fn, n):
    path = os.path.join(ROOT, "profiles", fn)
    if not os.path.exists(path):
        pytest.skip(fn + " not committed")
    d = json.loads(open(path).read().strip().splitlines()[-1])
    assert d["n_gpus"] == n and d["metric"] == "CG iterations/s" and d["dtype"] == "f64"
    assert d["roofline"]["bound"] == "hbm" and 0 < d["roofline"]["frac"] <= 1.0
    assert d["parity"]["ok"] is True and d["parity"]["max_rel_dev"] <= 1e-6 and d["parity"]["iters_compared"] >= 100
    assert d["e2e"]["value"] > 0 and d["e2e"]["h2d_bytes_per_step"] > 0 and d["gpu_launches"] > 0
    assert d["cfg5"]["parity"]["ok"] is True and d["cfg5"]["value"] > 0 and d["cfg5"]["n_gpus"] == n
    assert not d["clocks"]["reasons"] or set(d["clocks"]["reasons"]) <= {"sw_power_cap"}
    if n == 1:
        assert d["cpu_baseline"]["value"] > 0
        assert {e["solver"] for e in d["extra"]} == {"gmres(30)", "bicgstab"}
    else:
        assert d["parity"]["ranks_agree"] is True and d["cfg5"]["parity"]["ranks_agree"] is True


def test_bench_helpers_on_cpu():
    """The pieces of bench.py that do not need a GPU: the config-4 matrix assembled with torch ops (here on the CPU
    device) equals the SciPy assembly entry by entry; the parity block is green for the oracle's own history and red
    for a perturbed one; the golden parity reads the committed cfg5 history."""
    import numpy as np
    import torch
    sys.path[:0] = [ROOT, os.path.join(ROOT, "krylov.jl_b200")]
    import bench
    from krylov_b200 import problems as P
    from krylov_b200.problems import div_grad_csr
    from oracle import oracle as O
    n = 5000
    rp, ci, va = P.random_csr(n, 20, seed=1234, dtype=np.float32)
    drp, dci, dva = bench.device_random_csr(torch, torch.device("cpu"), n)
    assert np.array_equal(drp.numpy(), rp) and np.array_equal(dci.numpy(), ci) and np.array_equal(dva.numpy(), va)
    N, iters = 12, 30
    rp, ci, va = div_grad_csr(N)
    _, _, _, hist = O.cg_timed(rp, ci, va, np.ones(N ** 3), iters, 1, history=True)
    ok = bench.parity_block(list(hist), N, iters)
    assert ok["ok"] and ok["niter_equal"] and ok["iters_compared"] == iters and ok["max_rel_dev"] <= 1e-10      # OpenMP reduction order differs between thread counts
    bad = bench.parity_block(list(hist * (1 + 1e-5)), N, iters)
    assert bad["ok"] is False and bad["max_rel_dev"] > 1e-6
    short = bench.parity_block(list(hist[:-3]), N, iters)
    assert short["ok"] is False and short["niter_equal"] is False
    gold = json.load(open(os.path.join(ROOT, "tests", "golden", "bench_cg_poisson464.json")))
    g = bench.golden_parity(gold["residuals"], "bench_cg_poisson464")
    assert g["ok"] and g["iters_compared"] == bench.WORKLOADS["poisson464"][1]
    assert bench.golden_parity([1.0, 2.0], "no_such_file")["ok"] is None
    assert bench.algorithmic_bytes_cg(215 ** 3, 7 * 215 ** 3 - 6 * 215 ** 2) == 1586811804        # SURVEY.md 8(d)


def test_dump_outputs_writes_a_fixed_sample_of_the_solution(tmp_path):
    """--dump-outputs: non-empty float64 .npy files, under 64 MB in all, and the same seeded positions from run to run
    so that two builds can be compared entry by entry."""
    import types
    import numpy as np
    import torch
    sys.path.insert(0, ROOT)
    import bench
    n = 3 * bench.DUMP_SAMPLE + 7
    x = torch.arange(n, dtype=torch.float64) * 0.5
    stats = types.SimpleNamespace(niter=200, solved=False)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), x, stats)
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == ["niter.npy", "solved.npy", "x.npy", "x_index.npy"]
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in files) <= 64 << 20
    for f in files:
        a, b = np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f)
        assert a.dtype == np.float64 and a.size > 0 and np.array_equal(a, b), f
    idx, xs = np.load(tmp_path / "a" / "x_index.npy"), np.load(tmp_path / "a" / "x.npy")
    assert len(idx) == bench.DUMP_SAMPLE and np.all(np.diff(idx) > 0) and 0 <= idx[0] and idx[-1] < n
    k = np.arange(bench.DUMP_SAMPLE)
    lo, hi = k * n // bench.DUMP_SAMPLE, (k + 1) * n // bench.DUMP_SAMPLE
    assert np.all((lo <= idx) & (idx < hi))                          # one position per stratum, the last ending at n
    assert idx[-1] >= n - (n + bench.DUMP_SAMPLE - 1) // bench.DUMP_SAMPLE
    assert np.array_equal(xs, idx * 0.5)
    assert np.load(tmp_path / "a" / "niter.npy").tolist() == [200.0]
    small = torch.ones(10, dtype=torch.float64)
    bench.dump_outputs(str(tmp_path / "c"), small, types.SimpleNamespace(niter=3, solved=True))
    assert np.array_equal(np.load(tmp_path / "c" / "x.npy"), np.ones(10))
    assert np.load(tmp_path / "c" / "solved.npy").tolist() == [1.0]


@pytest.mark.parametrize("argv,env", [(["--steps", "0"], {}), (["--warmup", "-1"], {}),
                                      (["--impl", "reference", "--dump-outputs", "d"], {}),
                                      (["--dump-outputs", "d"], {"WORLD_SIZE": "2"})])
def test_bench_rejects_bad_arguments(argv, env, tmp_path):
    """A step count below 1, a negative warm-up, and --dump-outputs outside the single-GPU timed path are usage
    errors (exit 2) raised before any work starts, and nothing is written."""
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + argv, capture_output=True, text=True,
                         timeout=120, cwd=tmp_path, env=dict(os.environ, **env))
    assert out.returncode == 2 and "error:" in out.stderr and not out.stdout, (out.returncode, out.stderr[-500:])
    assert not os.listdir(tmp_path)
