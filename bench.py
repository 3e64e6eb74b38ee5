#!/usr/bin/env python
"""bench.py -- the hot-path benchmark (contract: task statement section 4).

Metric (BASELINE.json): CG iterations/s on the 3-D 7-point Poisson matrix
get_div_grad(N,N,N), N = 215 (n = 9 938 375, nnz = 69 291 275), Float64, b = ones,
and the achieved fraction of the HBM roofline.

A "step" is one cg!(ws, A, b; atol=0, rtol=0, itmax=ITERS) solve = ITERS = 200 fused
iterations (SURVEY.md 8(d); one persistent cooperative launch per 32 iterations).  `value` is timed with CUDA events on the
workspace's own stream with A and b resident in HBM; `e2e` times the same solve
through the reference-facing C ABI (krylov_solve / krylov_get_x) with pinned HOST
buffers for b and x.  The matrix (871 MB) is far larger than L2 (126 MB), so
every iteration streams it from HBM: no explicit L2 flush is needed.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload poisson215]
                    [--dump-outputs DIR]

--dump-outputs DIR writes what the last timed solve returned to its caller as DIR/<name>.npy (see
dump_outputs), so that two builds can be compared output for output on identical inputs.  It is refused for
--impl reference and for multi-rank runs (--gpus N > 1 under torchrun): only the single-GPU timed path dumps.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "krylov.jl_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402

WORKLOADS = {
    # name: (N, iterations per step)
    "poisson215": (215, 200),     # BASELINE config 2  (n ~ 1e7); SURVEY.md 8(d): timing run atol = rtol = 0, itmax = 200
    "poisson464": (464, 100),     # BASELINE config 5  (n ~ 1e8); SURVEY.md 8(d): 100 iterations at 1, 2, 4, 8 GPUs
    "poisson32": (32, 79),        # BASELINE config 1  (CPU-runnable reference case)
}
FALLBACK_HBM_GBS = 6650.0         # B200_PROFILING.md fallback when MEASURED_PEAKS.json is absent
DUMP_SAMPLE = 1 << 21             # entries of x written by --dump-outputs: 16 MB of values + 16 MB of positions


def workload_name(N, iters):
    """The SAME string in both arms (ours / --impl reference) and at every N: the driver compares `config.workload`."""
    return (f"cg! on get_div_grad({N},{N},{N}) Float64 CSR (n = {N ** 3}, nnz = {7 * N ** 3 - 6 * N ** 2}), b = ones, "
            f"atol = rtol = 0, itmax = {iters} per step")


def algorithmic_bytes_cg(n, nnz, v=8, i=4):
    """SURVEY.md section 8(d): B_cg = nnz(v+i) + (n+1)i + 9nv per fused CG iteration."""
    return nnz * (v + i) + (n + 1) * i + 9 * n * v


def hbm_peak():
    try:
        pk = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        return float(pk["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return FALLBACK_HBM_GBS, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons during the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.rows, self.proc, self.idx = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "20", "-i", str(self.idx)], stdout=subprocess.PIPE, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx = float(r[2])
                for name, col in (("hw_slowdown", 5), ("hw_thermal_slowdown", 6), ("sw_thermal_slowdown", 7), ("sw_power_cap", 8)):
                    if r[col].lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


def build_problem(N, torch, device, k_lo=0, k_hi=None):
    from krylov_b200.problems import div_grad_csr
    rp, ci, va = div_grad_csr(N, xp=torch, device=device, k_lo=k_lo, k_hi=k_hi)
    return rp, ci, va


_CPU_PROBLEM = {}


def cpu_leg(N, iters, threads, budget_s=20.0):
    """Times the CPU restatement of the same loop (oracle/, kind 'port') on a bounded sample of the workload:
    the same matrix, fewer iterations (sized for ~10-30 s)."""
    from krylov_b200.problems import div_grad_csr
    from oracle import oracle as O
    if N not in _CPU_PROBLEM:
        _CPU_PROBLEM[N] = div_grad_csr(N) + (np.ones(N ** 3),)
    rp, ci, va, b = _CPU_PROBLEM[N]
    t, _, _ = O.cg_timed(rp, ci, va, b, 2, threads)           # calibrate
    per_it = max(t / 2, 1e-6)
    k = int(max(3, min(iters, budget_s / per_it)))
    t, _, rn = O.cg_timed(rp, ci, va, b, k, threads)
    return dict(value=k / t, unit="it/s", cores=threads, kind="port",
                sample=f"{k} iterations of cg.jl:195-268 on get_div_grad({N},{N},{N}), b=ones, {threads} thread(s), "
                       f"{t:.2f} s wall"), k, t


def best_cpu_threads(N):
    """The thread count at which the CPU port runs fastest on this host (2 iterations per candidate): cpu_count()
    can exceed what the container may really use (a 128-thread run measured SLOWER than 1 thread on a GPU box), and
    the reference arm is meant to be the best the host can do."""
    from krylov_b200.problems import div_grad_csr
    from oracle import oracle as O
    if N not in _CPU_PROBLEM:
        _CPU_PROBLEM[N] = div_grad_csr(N) + (np.ones(N ** 3),)
    rp, ci, va, b = _CPU_PROBLEM[N]
    try:
        avail = len(os.sched_getaffinity(0))
    except AttributeError:
        avail = os.cpu_count() or 1
    cands = sorted({t for t in (1, 2, 4, 8, 16, 32, 64, avail) if t <= avail})
    best, best_t, sweep = 1, float("inf"), {}
    for t in cands:
        sec, _, _ = O.cg_timed(rp, ci, va, b, 2, t)
        sweep[t] = round(2 / sec, 2)
        if sec < best_t:
            best, best_t = t, sec
    return best, sweep


def affinity_threads(cap=32):
    try:
        avail = len(os.sched_getaffinity(0))
    except AttributeError:
        avail = os.cpu_count() or 1
    return max(1, min(cap, avail))


def parity_block(gpu_hist, N, iters, tol=1e-6):
    """Residual-norm history of the GPU solve vs the CPU oracle's on the SAME benchmark-size problem (outside the
    timed region): the oracle runs `iters` iterations of cg.jl:195-268 with OpenMP (its dots then differ from the
    sequential order by O(eps), far below the 1e-6 bar of north_star)."""
    from krylov_b200.problems import div_grad_csr
    from oracle import oracle as O
    if N not in _CPU_PROBLEM:
        _CPU_PROBLEM[N] = div_grad_csr(N) + (np.ones(N ** 3),)
    rp, ci, va, b = _CPU_PROBLEM[N]
    threads = affinity_threads()
    t, _, _, hist = O.cg_timed(rp, ci, va, b, iters, threads, history=True)
    g = np.asarray(gpu_hist, dtype=np.float64)
    k = min(len(g), len(hist))
    rel = np.abs(g[:k] - hist[:k]) / np.maximum(np.abs(hist[:k]), 1e-300)
    dev = float(rel.max()) if k else float("inf")
    return dict(against="oracle (CPU restatement of cg.jl:195-268), same matrix and b", iters_compared=k - 1,
                niter_equal=bool(len(g) == len(hist)), max_rel_dev=dev, tol=tol, ok=bool(len(g) == len(hist) and dev <= tol),
                oracle_threads=threads, oracle_seconds=round(t, 2))


def golden_parity(gpu_hist, name, tol=1e-6):
    """cfg5 (n ~ 1e8) is too large for an in-run oracle solve: compare with the committed oracle history
    (tests/golden/<name>.json, generated by tests/golden/gen_bench_golden.py)."""
    path = os.path.join(ROOT, "tests", "golden", name + ".json")
    if not os.path.exists(path):
        return dict(against=path, ok=None, note="golden file missing")
    gold = np.asarray(json.load(open(path))["residuals"], dtype=np.float64)
    g = np.asarray(gpu_hist, dtype=np.float64)
    k = min(len(g), len(gold))
    rel = np.abs(g[:k] - gold[:k]) / np.maximum(np.abs(gold[:k]), 1e-300)
    dev = float(rel.max()) if k else float("inf")
    return dict(against=f"tests/golden/{name}.json (oracle history)", iters_compared=k - 1, max_rel_dev=dev, tol=tol,
                ok=bool(k > 1 and dev <= tol))


def device_random_csr(torch, dev, n, per_row=20, seed=1234, shift=3.0):
    """BASELINE config 4 matrix (problems.random_csr: numpy default_rng(seed), indices first, then values,
    duplicates summed, +shift on the diagonal) ASSEMBLED on the GPU: the host only draws the random numbers.
    tests/test_gpu_formats.py checks it entry by entry against the SciPy assembly."""
    rng = np.random.default_rng(seed)
    cols = rng.integers(0, n, size=(n, per_row), dtype=np.int64)
    vals = rng.uniform(-1.0, 1.0, size=(n, per_row)).astype(np.float32)
    c = torch.from_numpy(cols.reshape(-1)).to(dev)
    v = torch.from_numpy(vals.reshape(-1)).to(dev)
    del cols, vals
    r = torch.arange(n, device=dev, dtype=torch.int64).repeat_interleave(per_row)
    d = torch.arange(n, device=dev, dtype=torch.int64)
    key = torch.cat([r * n + c, d * n + d])
    val = torch.cat([v, torch.full((n,), shift, dtype=torch.float32, device=dev)])
    del r, c, v
    key, order = torch.sort(key, stable=True)
    val = val[order]
    del order
    ukey, inv = torch.unique_consecutive(key, return_inverse=True)
    out = torch.zeros(ukey.numel(), dtype=torch.float32, device=dev)
    out.index_add_(0, inv, val)
    rows = ukey // n
    ci = (ukey - rows * n).to(torch.int32)
    counts = torch.bincount(rows, minlength=n)
    rp = torch.zeros(n + 1, dtype=torch.int64, device=dev)
    rp[1:] = torch.cumsum(counts, 0)
    return rp.to(torch.int32), ci, out


def dump_outputs(out_dir, x, stats):
    """Writes what one solve returned to its caller, in float64: x.npy (the solution; above DUMP_SAMPLE entries a
    fixed, seeded stratified sample of it), x_index.npy (the positions of those entries), niter.npy and solved.npy.
    The timed solve keeps no residual history, so there are no residual norms to write.  The strata split [0, n)
    into DUMP_SAMPLE contiguous ranges that cover it to the last entry, and one seeded position is drawn from each."""
    import torch
    n = int(x.numel())
    if n > DUMP_SAMPLE:
        bounds = np.arange(DUMP_SAMPLE + 1, dtype=np.int64) * n // DUMP_SAMPLE
        idx = bounds[:-1] + np.random.default_rng(0).integers(0, np.diff(bounds))
    else:
        idx = np.arange(n, dtype=np.int64)
    xs = x[torch.from_numpy(idx).to(x.device)].cpu().numpy()
    os.makedirs(out_dir, exist_ok=True)
    for name, a in (("x", xs), ("x_index", idx), ("niter", [stats.niter]), ("solved", [stats.solved])):
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(a, dtype=np.float64))


def extra_records(kb, torch, dev, peak):
    """BASELINE configs 3 and 4 on the same GPU (it/s + fraction of their own algorithmic-byte roofline,
    SURVEY.md 8d).  Not the headline metric: reported under "extra" on the N = 1 line."""
    from krylov_b200 import problems as P
    out = []

    def timed(ws, b, reps, **kw):
        st = torch.cuda.ExternalStream(kb.lib().krylov_b200_stream(ws._h), device=dev)
        for _ in range(2):
            ws.solve(None, b, **kw)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        l0 = ws.launches
        e0.record(st)
        for _ in range(reps):
            ws.solve(None, b, **kw)
        e1.record(st)
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) * 1e-3 / reps, ws.stats.niter, (ws.launches - l0) / reps

    # cfg3: gmres!(memory = 30, restart) on kron_unsymmetric(215), b = A*ones; 2 full cycles per solve
    N = 215
    rp, ci, va = P.kron_unsymmetric_csr(N, xp=torch, device=dev)
    n, nnz = N ** 3, int(va.numel())
    b = P.csr_matvec_ones(rp, ci, va)
    torch.cuda.synchronize()
    ws = kb.GmresWorkspace(n, n, np.float64, memory=30, device="cuda")
    ws.set_operator((rp, ci, va))
    sec, niter, launches = timed(ws, b, 3, atol=0.0, rtol=0.0, itmax=60, restart=True)
    ws.free()
    B = nnz * 12 + (n + 1) * 4 + 2 * n * 8 + 64 * n * 8
    its = niter / sec
    out.append(dict(solver="gmres(30)", config="cfg3: kron_unsymmetric(215) Float64, restart, 60 inner iterations per solve",
                    value=its, unit="it/s", launches_per_iteration=launches / niter,
                    roofline=dict(bound="hbm", bytes_per_iteration=B, achieved=B * its / 1e9, peak=peak, unit="GB/s",
                                  frac=B * its / 1e9 / peak, note="B_spmv + 64 n v (cycle average of the MGS sweep)")))
    del rp, ci, va, b
    torch.cuda.empty_cache()
    # cfg4: bicgstab! Float32 on the random CSR (n = 5e6, 20 draws/row + diagonal), b = A*ones; 50 iterations
    n = 5_000_000
    t0 = time.perf_counter()
    rp, ci, va = device_random_csr(torch, dev, n)
    nnz = int(va.numel())
    b = P.csr_matvec_ones(rp, ci, va)
    torch.cuda.synchronize()
    gen_s = time.perf_counter() - t0
    ws = kb.BicgstabWorkspace(n, n, np.float32, device="cuda")
    ws.set_operator((rp, ci, va))
    sec, niter, launches = timed(ws, b, 3, atol=0.0, rtol=0.0, itmax=50)
    ws.free()
    B = 2 * (nnz * 8 + (n + 1) * 4) + 20 * n * 4
    its = niter / sec
    out.append(dict(solver="bicgstab", config=f"cfg4: random CSR n={n} nnz={nnz} Float32, 50 iterations per solve",
                    value=its, unit="it/s", launches_per_iteration=launches / niter, matrix_generate_s=round(gen_s, 2),
                    roofline=dict(bound="hbm", bytes_per_iteration=B, achieved=B * its / 1e9, peak=peak, unit="GB/s",
                                  frac=B * its / 1e9 / peak,
                                  note="2 x matrix + 20 n v; the x gather of a uniformly RANDOM matrix is bound by the L1 "
                                       "sector rate (one 32-B sector per nonzero: 118 M sectors per SpMV, l1tex 84 % of "
                                       "peak, DRAM 30 %): profiles/r2_ncu_bicgstab_spmv.txt")))
    del rp, ci, va, b
    torch.cuda.empty_cache()
    return out


def cfg5_single(kb, torch, dev, steps, peak):
    """BASELINE config 5 (get_div_grad(464): n = 99 897 344) on ONE GPU -- the denominator of north_star's
    ">= 6x at 8 GPUs"; the multi-GPU runs carry the same key (krylov_b200/dist.py)."""
    N, iters = WORKLOADS["poisson464"]
    n, nnz = N ** 3, 7 * N ** 3 - 6 * N ** 2
    rp, ci, va = build_problem(N, torch, dev)
    b = torch.ones(n, dtype=torch.float64, device=dev)
    ws = kb.CgWorkspace(n, n, np.float64, device="cuda")
    ws.set_operator((rp, ci, va))
    del rp, ci, va
    torch.cuda.empty_cache()
    kw = dict(atol=0.0, rtol=0.0, itmax=iters)
    stream = torch.cuda.ExternalStream(kb.lib().krylov_b200_stream(ws._h), device=dev)
    for _ in range(3):
        ws.solve(None, b, **kw)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record(stream)
    for _ in range(steps):
        ws.solve(None, b, **kw)
    e1.record(stream)
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    ws.solve(None, b, history=True, **kw)
    hist = list(ws.stats.residuals)
    ws.free()
    del b
    torch.cuda.empty_cache()
    v = steps * iters / (ms * 1e-3)
    B = algorithmic_bytes_cg(n, nnz)
    return dict(workload=f"cg! on get_div_grad({N},{N},{N}) (n = {n}, nnz = {nnz}) on 1 GPU, {iters} iterations per step, "
                         f"{steps} steps", value=v, unit="it/s", n_gpus=1, ms_per_step=ms / steps, frac=B * v / 1e9 / peak,
                bytes_per_iteration=B, parity=golden_parity(hist, "bench_cg_poisson464"),
                speedup_note="north_star target: value at 8 GPUs >= 6 x this value (same key on the N=8 line)")


def run_reference(args):
    """--impl reference: the reference's CPU path.  Julia is not in this image, so the timed code is the
    oracle port (oracle/krylov_oracle.c), threaded over all host cores it can use."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    N, iters = WORKLOADS[args.workload]
    threads, sweep = best_cpu_threads(N)
    n, nnz = N ** 3, 7 * N ** 3 - 6 * N ** 2
    total_it, total_t = 0, 0.0
    leg = None
    for s in range(args.warmup + args.steps):
        leg, k, t = cpu_leg(N, iters, threads, budget_s=max(2.0, 60.0 / max(1, args.warmup + args.steps)))
        if s >= args.warmup:
            total_it += k; total_t += t
    v = total_it / total_t
    line = dict(metric="CG iterations/s", value=v, unit="it/s", n_gpus=args.gpus, steps=args.steps, warmup=args.warmup,
                ms_per_step=1e3 * total_t / args.steps, higher_is_better=True, scaling="strong", vs_baseline=None,
                dtype="f64", data="synthetic", impl="reference",
                config=dict(workload=workload_name(N, iters), n=n, nnz=nnz, iters_per_step=iters,
                            implementation="Julia absent: CPU restatement (oracle port) of src/cg.jl:195-268, OpenMP; thread count = "
                                           "fastest of a 2-iteration sweep; each step is a bounded sample of the workload's iterations",
                            thread_sweep_it_per_s=sweep),
                cpu_baseline=dict(leg, value=v),
                e2e=dict(value=v, unit="it/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0), gpu_launches=0)
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=os.environ.get("KB200_WORKLOAD", "poisson215"), choices=sorted(WORKLOADS))
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg and the parity block")
    ap.add_argument("--no-extra", action="store_true", help="skip the cfg3 / cfg4 extra records")
    ap.add_argument("--no-cfg5", dest="no_cfg5", action="store_true", help="skip the cfg5 (n ~ 1e8) record")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed solve returned as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and (args.impl == "reference" or int(os.environ.get("WORLD_SIZE", "1")) > 1):
        ap.error("--dump-outputs is supported for the single-process GPU run (--impl ours, one rank)")
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import krylov_b200 as kb
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        from krylov_b200 import dist
        return dist.bench_main(args, WORKLOADS, algorithmic_bytes_cg, hbm_peak, ClockSampler, parity_block, golden_parity, workload_name)
    if kb.device_count() < 1:
        raise SystemExit("bench.py needs a B200: libkrylov_b200 has no CPU path")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    N, iters = WORKLOADS[args.workload]
    n, nnz = N ** 3, 7 * N ** 3 - 6 * N ** 2
    t0 = time.perf_counter()
    rp, ci, va = build_problem(N, torch, dev)
    assert int(va.numel()) == nnz
    gen_s = time.perf_counter() - t0
    b = torch.ones(n, dtype=torch.float64, device=dev)

    # ---- device-resident arm (value) --------------------------------------
    ws = kb.CgWorkspace(n, n, np.float64, device="cuda")
    t0 = time.perf_counter()
    ws.set_operator((rp, ci, va))
    upload_s = time.perf_counter() - t0
    stream = torch.cuda.ExternalStream(kb.lib().krylov_b200_stream(ws._h), device=dev)
    solve_kw = dict(atol=0.0, rtol=0.0, itmax=iters)
    for _ in range(args.warmup):
        ws.solve(None, b, **solve_kw)
    sampler = ClockSampler(local)
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    l0 = ws.launches
    torch.cuda.synchronize()
    e0.record(stream)
    for _ in range(args.steps):
        ws.solve(None, b, **solve_kw)
    e1.record(stream)
    torch.cuda.synchronize()
    clocks = sampler.stop()
    launches = ws.launches - l0
    assert ws.stats.niter == iters, ws.stats
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, ws.x, ws.stats)
    ms = e0.elapsed_time(e1)
    its = args.steps * iters
    value = its / (ms * 1e-3)
    B = algorithmic_bytes_cg(n, nnz)
    peak, peak_src = hbm_peak()
    achieved = B * its / (ms * 1e-3) / 1e9
    # phase breakdown of the persistent kernel (cg_persist): phase A = SpMV + p update + <p,Ap> (+ x update),
    # phase B = r update + <r,r>; each measured inside the kernel (%globaltimer), its closing grid barrier included
    ws.solve(None, b, time_kernels=True, **solve_kw)
    k1_ms, k2_ms, timed = ws.kernel_times
    B_k1 = nnz * 12 + (n + 1) * 4 + 6 * n * 8      # matrix + read r,p,x + write p,Ap,x  (x update rides in phase A)
    B_k2 = 3 * n * 8                               # read r,Ap + write r
    kernels = dict(phase_a=dict(ms=k1_ms, bytes=B_k1, GBs=B_k1 / (k1_ms * 1e-3) / 1e9 if k1_ms else None),
                   phase_b=dict(ms=k2_ms, bytes=B_k2, GBs=B_k2 / (k2_ms * 1e-3) / 1e9 if k2_ms else None),
                   timed_iterations=timed, share_a=k1_ms / (k1_ms + k2_ms) if k1_ms else None,
                   kernel="cg_persist (one cooperative launch per 32 iterations)")
    # history of the same solve for the parity block (not timed)
    ws.solve(None, b, history=True, **solve_kw)
    gpu_hist = list(ws.stats.residuals)

    # ---- end-to-end arm: C ABI with pinned host buffers ---------------------
    wsh = kb.CgWorkspace(n, n, np.float64, device="host")
    wsh.share_operator(ws)
    bh = torch.ones(n, dtype=torch.float64).pin_memory()
    xh = torch.empty(n, dtype=torch.float64).pin_memory()
    bh_np, xh_np = bh.numpy(), xh.numpy()
    import ctypes as C
    for _ in range(max(1, args.warmup - 1)):
        wsh.solve(None, bh_np, **solve_kw)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        wsh.solve(None, bh_np, **solve_kw)                                   # H2D of b inside
        kb.lib().krylov_get_x(wsh._h, C.c_void_p(xh.data_ptr()), n)          # D2H of x inside
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    e2e = dict(value=its / e2e_s, unit="it/s", h2d_bytes_per_step=n * 8, d2h_bytes_per_step=n * 8,
               ms_per_step=1e3 * e2e_s / args.steps)

    # DRAM traffic per fused iteration from the committed ncu --set full capture of this same command
    # (profiles/r1_ncu_cg_final.txt); only meaningful for the workload it was taken on
    traffic = None
    try:
        if args.workload == "poisson215":
            traffic = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))["bytes_per_iteration"]
    except Exception:
        pass
    line = dict(metric="CG iterations/s", value=value, unit="it/s", n_gpus=1, steps=args.steps, warmup=args.warmup,
                ms_per_step=ms / args.steps, higher_is_better=True, scaling="strong", vs_baseline=None, dtype="f64",
                data="synthetic",
                config=dict(workload=workload_name(N, iters), n=n, nnz=nnz, iters_per_step=iters,
                            implementation="cg! fused: persistent cooperative kernel (32 iterations per launch), int32 CSR resident in HBM",
                            l2="inputs larger than L2 (matrix 0.87 GB vs 126 MB): no flush needed",
                            matrix_upload_s=round(upload_s, 3), matrix_generate_s=round(gen_s, 3)),
                roofline=dict(bound="hbm", achieved=achieved, peak=peak, unit="GB/s", frac=achieved / peak, traffic=traffic,
                              traffic_source="static: ncu --set full capture of this command, profiles/ncu_traffic.json",
                              peak_source=peak_src, bytes_per_iteration=B,
                              note="unit = one fused CG iteration (cg_k1 + cg_k2); B_cg from SURVEY.md 8(d)",
                              kernels=kernels),
                clocks=clocks, e2e=e2e, gpu_launches=int(launches))
    ws.free(); wsh.free()
    del rp, ci, va
    torch.cuda.empty_cache()
    if not args.no_extra and args.workload == "poisson215":
        try:
            line["extra"] = extra_records(kb, torch, dev, peak)
        except Exception as ex:
            line["extra"] = [dict(error=f"{type(ex).__name__}: {ex}")]
    if not args.no_cfg5 and args.workload == "poisson215":
        try:
            line["cfg5"] = cfg5_single(kb, torch, dev, max(2, args.steps // 2), peak)
        except Exception as ex:
            line["cfg5"] = dict(error=f"{type(ex).__name__}: {ex}")
    parity_ok = True
    if not args.no_cpu:
        try:
            leg, _, _ = cpu_leg(N, iters, 1, budget_s=15.0)
            line["cpu_baseline"] = leg
        except Exception as ex:  # the CPU leg must never cost the GPU number
            line["cpu_baseline"] = dict(value=None, unit="it/s", cores=1, kind="port", sample=f"failed: {ex}")
        try:
            line["parity"] = golden_parity(gpu_hist, "bench_cg_poisson464") if N > 300 else parity_block(gpu_hist, N, iters)
            parity_ok = line["parity"].get("ok") is not False and (line.get("cfg5", {}).get("parity") or {}).get("ok") is not False
        except Exception as ex:
            line["parity"] = dict(ok=None, note=f"failed: {type(ex).__name__}: {ex}")
    print(json.dumps(line))
    if not parity_ok:
        raise SystemExit("parity FAILED: GPU residual history deviates from the oracle by more than 1e-6 (see the line above)")


if __name__ == "__main__":
    main()
