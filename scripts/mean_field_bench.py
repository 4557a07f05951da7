"""
Stage timings of mean-field DCA on the GPU (CUDA events per stage: counts, covariance, SPD inverse = Cholesky +
triangular inverse + X^T X, couplings/fields, DI, scores) at three sizes, the achieved fp64 rate of the counts
and of the inverse (operations from the shapes over the event time), and a CPU arm on the same matrices (numpy
inv of the covariance; the float64 oracle for the whole fit at the smallest size).  Writes one JSON line to
stdout and to --out.

    python scripts/mean_field_bench.py --out /tmp/mean_field_bench.json [--sizes 50000x200,50000x500,...]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def gpu_identity():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except OSError:
        out = ""
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="50000x200,50000x500,50000x800")
    ap.add_argument("--repeats", type=int, default=2)
    ap.add_argument("--cpu-oracle-max-L", type=int, default=200)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    from evcouplings_b200 import msa, synthetic
    from evcouplings_b200.engine import CudaEngine
    import mf_oracle as mo
    eng = CudaEngine()
    q, pc, theta = 21, 0.5, 0.8
    rows = []
    for spec in a.sizes.split(","):
        N, L = (int(v) for v in spec.split("x"))
        codes = synthetic.synthetic_msa_codes(N, L, 2)
        counts = eng.hamming_counts(codes, msa.identity_threshold_count(theta, L))
        w = 1.0 / counts.astype(np.float64)
        n = L * (q - 1)
        runs = []
        for r in range(a.repeats + 1):           # first run warms up every shape
            t = {}
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            res = eng.mean_field(codes, w, q, pc, timings=t)
            t["total_wall_ms"] = (time.perf_counter() - t0) * 1e3
            if r:
                runs.append(t)
        best = {k: min(rr[k] for rr in runs) for k in runs[0]}
        inv_flops = float(n) ** 3                 # n^3/3 Cholesky + n^3/3 triangular inverse + n^3/3 X^T X
        count_flops = float(N) * (L * q) * (L * q + 64)   # lower tiles of the (Lq)^2 one-hot product
        row = dict(N=N, L=L, q=q, n=n, stage_ms=best, runs=runs,
                   inverse_fp64_tflops=inv_flops / (best["inverse"] * 1e-3) / 1e12,
                   counts_fp64_tflops=count_flops / (best["counts"] * 1e-3) / 1e12,
                   di_iterations_mean=float(res["di_iters"].mean()), di_iterations_max=int(res["di_iters"].max()))
        # CPU arm: numpy inv of a covariance matrix of the same size n
        if L <= a.cpu_oracle_max_L:
            t0 = time.perf_counter()
            o = mo.fit(codes, w, q, pc, di=True)
            row["cpu_oracle_fit_s"] = time.perf_counter() - t0
            C = o["C"]
            row["max_abs_err_J_vs_oracle"] = float(np.abs(res["J_tri"] - mo.tri(o["J"])).max())
            row["max_abs_err_di_vs_oracle"] = float(np.abs(res["di"] - mo.tri(o["di"])).max())
            row["cpu_inv_matrix"] = "the same covariance matrix"
        else:
            # the float64 one-hot product over all N sequences would take the CPU arm minutes; the inverse is
            # timed on the covariance of the first 5,000 sequences (same n, similar conditioning)
            fi, fij = mo.frequencies(codes[:5000], w[:5000], q)
            C = mo.covariance(fi, fij, pc)[1]
            del fi, fij
            row["cpu_inv_matrix"] = "covariance of the first 5000 sequences"
        t0 = time.perf_counter()
        np.linalg.inv(C)
        row["cpu_numpy_inv_s"] = time.perf_counter() - t0
        del C
        rows.append(row)
        print(json.dumps({k: v for k, v in row.items() if k != "runs"}), file=sys.stderr, flush=True)
    out = dict(workload="mean_field", device=gpu_identity(), torch_threads=torch.get_num_threads(),
               cpu_count=os.cpu_count(), sizes=rows,
               note="stage_ms: best of --repeats after one warm-up run, CUDA events; inverse = Cholesky + "
                    "triangular inverse + X^T X in one call (synchronous); CPU arm: numpy on the same host")
    line = json.dumps(out)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
