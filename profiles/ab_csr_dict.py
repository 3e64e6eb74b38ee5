"""Alternating A/B of the flagship benchmark between two built trees: the CSR stream (parent tree) and the
dictionary-encoded stream (this tree).

    python profiles/ab_csr_dict.py --base <parent tree> [--runs 5] [--out DIR]

Each run is `python bench.py --no-cpu --no-extra --no-cfg5 --steps 20 --warmup 3 --dump-outputs ...` in that
tree (20 x 200 CG iterations on get_div_grad(215): a timed window of about a second).  The arms alternate
base, branch, base, ... so that drift of the shared machine lands on both.  Prints, and writes to DIR/ab.json,
median / min / max of `value` per arm, the phase split of each arm's median run, the fraction of the HBM peak the
dictionary byte model reaches (bench.py's roofline uses the CSR model B_cg, which overstates the bytes of the
encoded stream), and whether the two arms' dumped outputs (sampled x, niter, solved) are identical."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CMD = ["--no-cpu", "--no-extra", "--no-cfg5", "--steps", "20", "--warmup", "3"]


def dict_bytes_per_iteration(n, nnz):
    """One code byte per nonzero + rowptr + the 9 vector passes of the fused iteration (DESIGN.md section 3)."""
    return nnz * 1 + (n + 1) * 4 + 9 * n * 8


def run(tree, dump):
    p = subprocess.run([sys.executable, "bench.py", *CMD, "--dump-outputs", dump], cwd=tree, capture_output=True,
                       text=True)
    if p.returncode != 0:
        sys.stderr.write(p.stdout[-4000:] + p.stderr[-4000:])
        raise SystemExit(f"bench.py failed in {tree}")
    return json.loads([l for l in p.stdout.splitlines() if l.startswith("{")][-1])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--base", required=True, help="tree of the parent commit, built")
    ap.add_argument("--runs", type=int, default=5)
    ap.add_argument("--out", help="directory for the dumped outputs and ab.json (default: a new temporary directory)")
    args = ap.parse_args()
    args.out = os.path.abspath(args.out or tempfile.mkdtemp(prefix="ab_csr_dict_"))   # bench.py runs in each tree
    arms = {"base": os.path.abspath(args.base), "branch": ROOT}
    res = {a: [] for a in arms}
    for i in range(args.runs):
        for a, tree in arms.items():
            line = run(tree, os.path.join(args.out, a))
            res[a].append(line)
            print(f"run {i} {a:6s} {line['value']:9.1f} it/s  phase A {line['roofline']['kernels']['phase_a']['ms'] * 1e3:6.1f} us"
                  f"  phase B {line['roofline']['kernels']['phase_b']['ms'] * 1e3:5.1f} us", flush=True)
    summary = {}
    for a, lines in res.items():
        v = [l["value"] for l in lines]
        med = sorted(lines, key=lambda l: l["value"])[len(lines) // 2]
        n, nnz, peak = med["config"]["n"], med["config"]["nnz"], med["roofline"]["peak"]
        summary[a] = dict(values=v, median=statistics.median(v), min=min(v), max=max(v),
                          phase_a_us=med["roofline"]["kernels"]["phase_a"]["ms"] * 1e3,
                          phase_b_us=med["roofline"]["kernels"]["phase_b"]["ms"] * 1e3,
                          frac_csr_model=med["roofline"]["frac"],
                          frac_dict_model=dict_bytes_per_iteration(n, nnz) * statistics.median(v) / 1e9 / peak,
                          peak_GBs=peak, clocks=med.get("clocks"))
    summary["speedup_median"] = summary["branch"]["median"] / summary["base"]["median"]
    summary["every_branch_run_faster"] = summary["branch"]["min"] > summary["base"]["max"]
    same = {}
    for name in ("x", "x_index", "niter", "solved"):
        a = np.load(os.path.join(args.out, "base", name + ".npy"))
        b = np.load(os.path.join(args.out, "branch", name + ".npy"))
        same[name] = bool(np.array_equal(a, b))
    summary["outputs_identical"] = same
    os.makedirs(args.out, exist_ok=True)
    json.dump(summary, open(os.path.join(args.out, "ab.json"), "w"), indent=1)
    print(json.dumps(summary, indent=1))
    print(f"outputs and ab.json in {args.out}")


if __name__ == "__main__":
    main()
