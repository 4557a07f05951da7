#!/usr/bin/env python
"""
bench.py -- headline benchmark of the PLM hot path (BASELINE.json metric).

Metric: PLM gradient evaluations expressed as cell-ops/s, one cell-op = one (n, i, j, a) term,
N * L^2 * q per objective+gradient evaluation (SURVEY.md 8d).  Workload at 1 GPU = BASELINE
configs[1]: synthetic MSA N=50,000, L=200, q=21 (gap is a state), fp32.  A "step" is one evaluation
of the objective and its full gradient (expand -> forward -> backward -> symmetrise -> all-reduce ->
regulariser) for a fixed parameter vector.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--scaling weak|strong]
                    [--precision fp32|bf16] [--seqs N --sites L] [--workload plm|hamming|fit]
                    [--dump-outputs DIR]

--dump-outputs DIR: after the timed steps, write what the timed path computed in its last step as DIR/<name>.npy
(float32 / float64): for `plm` the gradient (`gradient`) and [-loglk, objective] (`fx`), for `hamming` the
neighbour counts (`counts`).  Inputs are seeded, so two builds run with the same arguments can be compared
output for output.

N > 1: launched by torchrun, one rank per GPU; sequences sharded over ranks, ONE NCCL all-reduce of
[gradient, -loglk] (n + 4 floats) per step.  Default `weak`: 50,000 sequences per GPU (the 8-GPU point is the
Pfam-scale sharded case, BASELINE configs[3] territory); `--scaling strong` keeps N=50,000 total (the size the
BASELINE metric is quoted on).

`--impl reference`: the reference's plmc C/OpenMP binary is not available (source not vendored, no
network), so the CPU arm times oracle/plm_oracle_c.c -- a site-parallel C/OpenMP fp32 port of the
same objective (kind "port") -- on ALL host cores (thread count set explicitly: torchrun exports
OMP_NUM_THREADS=1), on the FULL 50,000-sequence workload, one evaluation per step.

The default N=1 line also carries three sub-records so that the driver's single run records them:
`hamming` (BASELINE configs[2], pruned and un-pruned kernel time, integer-pipe roofline), `fit` (device L-BFGS
ms/iteration) and `run_plmc_e2e` (alignment file -> reweighting -> 100 iterations -> .model/_ECs.txt).
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_PER_GPU, L, Q = 50000, 200, 21
LAMBDA_H, LAMBDA_J = 0.01, 0.01 * (Q - 1) * (L - 1)
SEED = 2
METRIC = "PLM gradient evals/s as N*L^2*q cell-ops/s"
UNIT = "cell-ops/s"
ACC_SAMPLE_N = 5000
CPU_BUDGET_S = 150.0
DUMP_LIMIT_BYTES = 64 << 20
DUMP_SEED = 0


def host_threads():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(p) as f:
            d = json.load(f)
        return {"hbm": float(d["hbm_gbs"]), "hbm_src": "measured (MEASURED_PEAKS.json hbm_gbs)",
                "tf": float(d["bf16_tflops"]), "tf_src": "measured (MEASURED_PEAKS.json bf16_tflops, cuBLAS burst)",
                "tf_sustained": float(d.get("bf16_tflops_sustained", 0.0)) or None,
                "sm_max_mhz": float(d.get("sm_max_mhz", 1965.0))}
    except Exception:
        return {"hbm": 6650.0, "hbm_src": "fallback (B200_PROFILING.md 6.65 TB/s)", "tf": 1590.0,
                "tf_src": "fallback (B200_PROFILING.md 1.59 PFLOP/s)", "tf_sustained": 1400.0, "sm_max_mhz": 1965.0}


class ClockSampler(threading.Thread):
    """SM clock / throttle reasons during the timed region.  NVML (a few hundred samples per second, so that even a
    0.1 s timed region is covered); falls back to polling nvidia-smi (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        super().__init__(daemon=True)
        self.gpu_index = gpu_index
        self.samples = []       # (sm_mhz, max_mhz, power_w, hw_slow, hw_thermal, sw_thermal, sw_power)
        self.stop_flag = threading.Event()
        self.source = "nvml"
        self.nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            idx = gpu_index
            if vis:
                try:
                    idx = int(vis.split(",")[gpu_index])
                except Exception:
                    idx = gpu_index
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(idx)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
            self.nvml = pynvml
        except Exception:
            self.source = "nvidia-smi"

    def _nvml_sample(self):
        n = self.nvml
        sm = float(n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM))
        try:
            pw = n.nvmlDeviceGetPowerUsage(self.handle) / 1000.0
        except Exception:
            pw = 0.0
        try:
            r = n.nvmlDeviceGetCurrentClocksEventReasons(self.handle)
        except Exception:
            r = n.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle)
        self.samples.append((sm, self.max_mhz, pw, bool(r & 0x8), bool(r & 0x40), bool(r & 0x20), bool(r & 0x4)))

    def run(self):
        while not self.stop_flag.is_set():
            try:
                if self.nvml is not None:
                    self._nvml_sample()
                    self.stop_flag.wait(0.004)
                    continue
                out = subprocess.run(["nvidia-smi", "-i", str(self.gpu_index), "--query-gpu=" + self.Q,
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5)
                p = [x.strip() for x in out.stdout.strip().split(",")]
                if len(p) >= 7:
                    act = [x.lower().startswith("active") for x in p[3:7]]
                    self.samples.append((float(p[0]), float(p[1]), float(p[2]), act[0], act[1], act[2], act[3]))
            except Exception:
                pass
            self.stop_flag.wait(0.05)

    def summary(self):
        self.stop_flag.set()
        self.join(timeout=6)
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0, "source": self.source}
        sm = sorted(s[0] for s in self.samples)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for k, n in enumerate(names) if any(s[3 + k] for s in self.samples)]
        return {"sm_mhz": sm[len(sm) // 2], "sm_min_mhz": sm[0], "sm_max_mhz": float(self.samples[0][1]),
                "power_w_max": max(s[2] for s in self.samples), "reasons": reasons, "samples": len(sm),
                "source": self.source}


def make_inputs(n_total):
    from evcouplings_b200 import synthetic
    codes = synthetic.synthetic_msa_codes(n_total, L, SEED)
    n = L * Q + L * (L - 1) // 2 * Q * Q
    x = np.random.default_rng(SEED).normal(0.0, 0.05, n).astype(np.float32)
    return codes, x


def dump_outputs(directory, arrays):
    """Writes each array as DIR/<name>.npy.  An array too large for the DUMP_LIMIT_BYTES budget left by the others
    is replaced by a fixed, seeded sample of its elements (<name>.npy) and their flat positions (<name>_index.npy,
    float64).  Returns the names written."""
    os.makedirs(directory, exist_ok=True)
    budget = DUMP_LIMIT_BYTES
    written = []
    for name, a in sorted(arrays.items(), key=lambda kv: kv[1].nbytes):
        a = np.ascontiguousarray(a)
        if a.nbytes > budget:
            a = a.reshape(-1)
            k = budget // (a.itemsize + 8)
            idx = np.unique(np.random.default_rng(DUMP_SEED).integers(0, a.size, k))
            np.save(os.path.join(directory, name + "_index.npy"), idx.astype(np.float64))
            written.append(name + "_index")
            budget -= idx.size * 8
            a = a[idx]
        np.save(os.path.join(directory, name + ".npy"), a)
        written.append(name)
        budget -= a.nbytes
    return written


def cpu_arm(codes, x, weights, steps, warmup, budget_s=CPU_BUDGET_S):
    """Times the C/OpenMP fp32 port on the given sequences with ALL host threads (set explicitly).
    Returns (cell-ops/s, seconds per evaluation, threads, steps actually timed)."""
    from oracle import c_oracle as co
    co.build()
    threads = host_threads()
    w = np.ascontiguousarray(weights, dtype=np.float32)
    t0 = time.perf_counter()
    for _ in range(max(1, warmup)):
        co.plm_eval(codes, w, x, Q, LAMBDA_H, LAMBDA_J, "f32", nthreads=threads)
    dt_warm = (time.perf_counter() - t0) / max(1, warmup)
    steps = max(1, min(steps, int(budget_s / max(dt_warm, 1e-3))))
    t0 = time.perf_counter()
    for _ in range(steps):
        co.plm_eval(codes, w, x, Q, LAMBDA_H, LAMBDA_J, "f32", nthreads=threads)
    dt = (time.perf_counter() - t0) / steps
    cells = float(codes.shape[0]) * L * L * Q
    return cells / dt, dt, threads, steps


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    codes, x = make_inputs(N_PER_GPU)
    weights = np.random.default_rng(SEED + 1).uniform(0.05, 1.0, N_PER_GPU).astype(np.float32)
    value, dt, threads, steps = cpu_arm(codes, x, weights, max(1, args.steps), max(1, min(args.warmup, 2)))
    sample = ("the full workload: all %d sequences (same generator/seed), L=%d q=%d, one fx+gradient evaluation per "
              "step; %d steps timed (capped to %.0f s of CPU work)" % (N_PER_GPU, L, Q, steps, CPU_BUDGET_S))
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": steps, "warmup": max(1, min(args.warmup, 2)), "ms_per_step": dt * 1e3, "higher_is_better": True,
        "scaling": args.scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "PLM fx+gradient, synthetic MSA N=%d L=%d q=%d fp32 (BASELINE configs[1])"
                   % (N_PER_GPU, L, Q), "cpu_sample": sample, "same_config": True},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample,
                         "note": "plmc itself is not vendored/buildable; C/OpenMP fp32 restatement "
                                 "(oracle/plm_oracle_c.c), site-parallel like plmc's OpenMP build; thread count set "
                                 "explicitly (torchrun exports OMP_NUM_THREADS=1)"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


def _nccl_env():
    """NCCL's INIT lines (rank / nranks / topology) are wanted on STDERR so that the driver can count ranks, and
    stdout must stay ONE JSON line (NCCL prints its version banner and, without a debug file, everything to stdout).
    NCCL therefore logs into a per-rank temporary file that _nccl_log_to_stderr() copies to stderr at the end."""
    os.environ["NCCL_DEBUG"] = os.environ.get("EVC_NCCL_DEBUG", "INFO")
    os.environ["NCCL_DEBUG_SUBSYS"] = os.environ.get("EVC_NCCL_DEBUG_SUBSYS", "INIT")
    d = tempfile.mkdtemp(prefix="evc_nccl_")
    os.environ["NCCL_DEBUG_FILE"] = os.path.join(d, "nccl.%h.%p.log")
    return d


def _nccl_log_to_stderr(d):
    try:
        for name in sorted(os.listdir(d)):
            with open(os.path.join(d, name)) as f:
                for ln in f:
                    if "NCCL" in ln:
                        sys.stderr.write(ln)
            os.unlink(os.path.join(d, name))
        os.rmdir(d)
        sys.stderr.flush()
    except Exception:
        pass


def hamming_subrecord(engine, peaks, steps=3):
    """BASELINE configs[2] (N=200k, L=300) on this GPU: pruned (product) and un-pruned kernel time."""
    import ctypes
    import torch
    from evcouplings_b200 import msa, synthetic, _lib
    lib = engine.lib
    N, Lh = 200000, 300
    codes = synthetic.synthetic_msa_codes(N, Lh, 3)
    thr = msa.identity_threshold_count(0.8, Lh)
    d_codes = torch.from_numpy(codes).to(engine.device)
    words = lib.evc_hamming_plane_words(N, Lh)
    d_planes = torch.empty(words, dtype=torch.int32, device=engine.device)
    d_counts = torch.zeros(N, dtype=torch.int32, device=engine.device)
    _lib.check(lib.evc_hamming_pack(engine.ptr(d_codes), N, Lh, engine.ptr(d_planes), engine.stream()), "pack")
    ntiles = lib.evc_hamming_num_tiles(N)

    def timed():
        _lib.check(lib.evc_hamming_count_tiles(engine.ptr(d_planes), N, Lh, thr, 0, ntiles, engine.ptr(d_counts),
                                               engine.stream()), "count")
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            d_counts.zero_()
            _lib.check(lib.evc_hamming_count_tiles(engine.ptr(d_planes), N, Lh, thr, 0, ntiles,
                                                   engine.ptr(d_counts), engine.stream()), "count")
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / steps

    ms = timed()
    pairs = 0.5 * N * (N - 1)
    Wd = -(-Lh // 32)
    # integer-pipe roofline: per 32-site word of a pair 5 x (XOR, OR/accumulate) folded into 5 LOP3 + 1 IADD on the
    # ALU pipe (64 lanes/clk/SM) and 1 POPC on the XU pipe (16 lanes/clk/SM): the ALU pipe bounds it
    alu_ops = pairs * Wd * 6.0
    sms = 148
    peak_ops = 64.0 * sms * peaks["sm_max_mhz"] * 1e6
    rec = {"metric": "Hamming reweighting pairs/s", "value": pairs / (ms * 1e-3), "unit": "pairs/s",
           "ms_per_step": ms, "steps": steps,
           "config": {"workload": "pairwise Hamming reweighting N=%d L=%d theta=0.8 (BASELINE configs[2])" % (N, Lh)},
           "roofline": {"bound": "int-alu", "kernel": "hamming_tile_kernel<FILTER> + hamming_verify_kernel",
                        "achieved": alu_ops / (ms * 1e-3) / 1e12, "peak": peak_ops / 1e12, "unit": "Tops/s (int32 ALU)",
                        "frac": alu_ops / (ms * 1e-3) / peak_ops, "traffic": None,
                        "algorithmic_ops_per_launch": alu_ops,
                        "note": "algorithmic = un-pruned op count (N(N-1)/2 pairs x ceil(L/32) words x 6 ALU ops); "
                                "the product kernels prune exactly (two-phase filter, early termination), so frac can "
                                "exceed 1; the un-pruned run of the same kernel is in `unpruned`; bit-planes are "
                                "L2-resident (40 MB), HBM is not the bound",
                        "site_compares_per_s": pairs * Lh / (ms * 1e-3)}}
    return rec, (codes, thr, d_counts.cpu().numpy())


def run_b200(args):
    import ctypes
    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    nccl_dir = _nccl_env()
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        sys.stderr.write("[bench] rank %d / %d on cuda:%d, backend nccl %s\n"
                         % (rank, world, local_rank, ".".join(str(v) for v in torch.cuda.nccl.version())))
    else:
        torch.cuda.set_device(0)
    from evcouplings_b200 import msa
    from evcouplings_b200.engine import CudaEngine

    engine = CudaEngine()
    n_total = N_PER_GPU * world if args.scaling == "weak" else N_PER_GPU
    codes, x = make_inputs(n_total)
    n = x.size
    peaks = measured_peaks()

    # sequence weights from the real reweighting pass (hot path (b)), untimed setup
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    counts = engine.hamming_counts(codes, msa.identity_threshold_count(0.8, L))
    torch.cuda.synchronize()
    t_ham = time.perf_counter() - t0
    weights = (1.0 / counts).astype(np.float32)

    prob = engine.plm_problem(codes, weights, Q, -1, LAMBDA_H, LAMBDA_J, backward=args.backward,
                              forward=args.forward, precision=args.precision)
    prob.set_x(x)
    engine.lib.evc_plm_set_profiling(prob.handle, 1)
    cells = float(n_total) * L * L * Q
    n_local = prob.shard[1] - prob.shard[0]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident throughput (`value`) ------------------------------------------------
    for _ in range(args.warmup):
        prob.evaluate_async(prob.x)
    barrier()
    sampler = ClockSampler(local_rank)
    sampler.start()
    launches0 = engine.kernel_launches
    prob.time_collective, prob.collective_events = world > 1, []
    stage = np.zeros(5, dtype=np.float32)
    stage_sum = np.zeros(5, dtype=np.float64)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(args.steps):
        prob.evaluate_async(prob.x)
        engine.lib.evc_plm_last_stage_ms(prob.handle, stage.ctypes.data_as(ctypes.c_void_p))
        stage_sum += stage
    ev1.record()
    barrier()
    ms_total = ev0.elapsed_time(ev1)
    if args.dump_outputs and rank == 0:
        # the last timed step's results, before anything else reuses the buffers
        outputs = {"gradient": prob.g.cpu().numpy(), "fx": prob.fxbuf.cpu().numpy()}
    launches = engine.kernel_launches - launches0
    t = torch.tensor([ms_total], dtype=torch.float64, device=engine.device)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_step = float(t.item()) / args.steps
    clocks = sampler.summary()
    value = cells / (ms_step * 1e-3)
    stage_ms = stage_sum / args.steps
    fx_check = prob.fxbuf.tolist()

    # ---- rank consistency: after the all-reduce every rank must hold the same objective and gradient ----
    consistency = None
    comm = None
    prob.time_collective = False
    if world > 1:
        # where the multi-GPU step goes: compute per rank (sum of the stage timers) and the collective as THIS rank
        # sees it (its duration includes waiting for the slowest rank)
        coll_ms = float(np.mean([a.elapsed_time(b) for a, b in prob.collective_events])) if prob.collective_events else 0.0
        mine = torch.tensor([float(stage_ms.sum()), coll_ms], dtype=torch.float64, device=engine.device)
        allr = [torch.zeros_like(mine) for _ in range(world)]
        dist.all_gather(allr, mine)
        comp = [float(t_[0]) for t_ in allr]
        coll = [float(t_[1]) for t_ in allr]
        comm = {"compute_ms_per_rank": comp, "collective_ms_per_rank_incl_wait": coll,
                "collective_ms_min_over_ranks": min(coll),
                "note": "one all-reduce of %d floats per step; the minimum over ranks of the collective's duration is the "
                        "best estimate of the transfer itself (the slowest rank does not wait)" % (n + 4)}
        chk = torch.stack([prob.fxbuf[0], prob.fxbuf[1], prob.g.double().sum(), prob.g.double().abs().sum()])
        gathered = [torch.zeros_like(chk) for _ in range(world)]
        dist.all_gather(gathered, chk)
        consistency = {"fx_identical_on_all_ranks": bool(all(torch.equal(gathered[0][:2], t_[:2]) for t_ in gathered)),
                       "gradient_checksums_identical_on_all_ranks":
                           bool(all(torch.equal(gathered[0][2:], t_[2:]) for t_ in gathered))}

    # ---- end to end through the public host API (host buffers, H2D + D2H inside) --------------
    x_pin = torch.from_numpy(x).pin_memory()
    g_pin = torch.empty(n, dtype=torch.float32).pin_memory()
    for _ in range(min(args.warmup, 3)):
        prob.evaluate_host(x_pin, g_pin)
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        fx_e2e = prob.evaluate_host(x_pin, g_pin)
    barrier()
    e2e_s = (time.perf_counter() - t0) / args.steps
    te = torch.tensor([e2e_s], dtype=torch.float64, device=engine.device)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_value = cells / float(te.item())

    # ---- roofline of the dominant kernel -------------------------------------------------------
    # SURVEY 8d figures.  Dense (tensor-core) path: 2*N*(L*q)^2 algorithmic flop per GEMM launch (4*N*(Lq)^2 per
    # evaluation).  fp32 mode: each algorithmic product is executed as two bf16 products (hi + lo split of the
    # real-valued operand); bf16 mode: one.  Gather path / HBM accounting: 8 B per cell-op per evaluation.
    local_cells = float(n_local) * L * L * Q
    lq = float(L * Q)
    names = ["expand", {"tc": "tc_gemm_persistent_kernel<1,*> (forward logits)", "tcfused": "tc_fwd_fused_kernel",
                       "gather": "plm_fwd_kernel"}[prob.forward],
             "plm_softmax_kernel", "tc_gemm_persistent_kernel<0,*> (backward)" if prob.backward == "tc" else "plm_bwd_kernel",
             "finalize"]
    dom = 1 if stage_ms[1] >= stage_ms[3] else 3
    dom_is_tc = (prob.forward in ("tc", "tcfused")) if dom == 1 else (prob.backward == "tc")
    hbm_whole = (8.0 * local_cells + n_local * L) / (ms_step * 1e-3) / 1e9
    traffic, traffic_src = ncu_traffic(names[dom], args.precision) if (world == 1 and n_local == 50000 and L == 200) else (None, None)
    products = 1.0 if args.precision == "bf16" else 2.0
    if dom_is_tc:
        alg_flops = 2.0 * n_local * lq * lq
        pad_m = -(-int(lq) // 128) * 128
        pad_n192 = -(-int(lq) // 192) * 192
        if dom == 1:
            rows = {"tc": pad_m, "tcfused": -(-L // 8) * 176}[prob.forward]
            kk = -(-int(lq) // 64) * 64
            seqs = -(-n_local // (192 if prob.forward == "tc" else 128)) * (192 if prob.forward == "tc" else 128)
            exec_flops = products * 2.0 * rows * kk * seqs
        else:
            exec_flops = products * 2.0 * pad_m * pad_n192 * (-(-n_local // 64) * 64)
        achieved = alg_flops / (stage_ms[dom] * 1e-3) / 1e12
        roofline = {"bound": "tensor", "kernel": names[dom], "achieved": achieved, "peak": peaks["tf"], "unit": "TFLOP/s",
                    "frac": achieved / peaks["tf"], "traffic": traffic, "traffic_source": traffic_src,
                    "peak_source": peaks["tf_src"], "algorithmic_flops_per_launch": alg_flops,
                    "executed": {"flops_per_launch": exec_flops, "tflops": exec_flops / (stage_ms[dom] * 1e-3) / 1e12,
                                 "frac_of_peak": exec_flops / (stage_ms[dom] * 1e-3) / 1e12 / peaks["tf"],
                                 "note": ("each algorithmic product = 2 bf16 products (hi+lo split keeps 16 mantissa "
                                          "bits of J / of the residuals), " if products == 2.0 else
                                          "bf16 tiles: one bf16 product per algorithmic product, ") +
                                         "tiles padded to 128/192/64"}}
    else:
        alg_bytes = 4.0 * local_cells + (float(n_local) * L if dom == 1 else 0.0)
        achieved = alg_bytes / (stage_ms[dom] * 1e-3) / 1e9
        roofline = {"bound": "hbm", "kernel": names[dom], "achieved": achieved, "peak": peaks["hbm"], "unit": "GB/s",
                    "frac": achieved / peaks["hbm"], "traffic": traffic, "traffic_source": traffic_src,
                    "peak_source": peaks["hbm_src"], "algorithmic_bytes_per_launch": alg_bytes,
                    "note": "on-chip-bound kernel: achieved > peak means the gathered bytes are served from shared "
                            "memory, not HBM (see DESIGN.md, profiles/)"}
    roofline["stage_ms"] = {k: float(v) for k, v in zip(names, stage_ms)}
    roofline["whole_evaluation_tensor"] = {
        "algorithmic_tflops": 2.0 * 2.0 * n_local * lq * lq / (ms_step * 1e-3) / 1e12,
        "frac_of_peak": 2.0 * 2.0 * n_local * lq * lq / (ms_step * 1e-3) / 1e12 / peaks["tf"]}
    roofline["hbm_accounting_whole_eval"] = {
        "algorithmic_bytes": 8.0 * local_cells + n_local * L, "achieved_GBps": hbm_whole, "peak_GBps": peaks["hbm"],
        "frac": hbm_whole / peaks["hbm"],
        "note": "north-star accounting (8 B per cell-op); >1 because the work is done on-chip (tensor cores / "
                "shared memory); not a physical fraction"}

    dtype = ("f32" if (prob.forward == "gather" and prob.backward == "gather") else
             "f32 parameters/accumulation; tensor-core products as bf16 hi+lo pairs (16 mantissa bits)"
             if args.precision != "bf16" else
             "bf16 tiles (one bf16 product per term), f32 parameters/accumulation (BASELINE configs[4] mode)")
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": args.scaling,
        "vs_baseline": None, "dtype": dtype, "data": "synthetic",
        "config": {"workload": ("PLM fx+gradient, synthetic MSA N=%d%s L=%d q=%d %s"
                                % (N_PER_GPU if args.scaling == "weak" else n_total,
                                   " per GPU (sharded, N_total=%d)" % n_total if (world > 1 and args.scaling == "weak")
                                   else (" total (sharded over %d GPUs)" % world if world > 1 else ""), L, Q,
                                   "fp32" if args.precision != "bf16" else "bf16 tiles"))
                   + (" (BASELINE configs[1])" if (N_PER_GPU, L) == (50000, 200) else " (non-default shape)"),
                   "global_sequences": n_total, "precision": args.precision,
                   "parallelism": "dp%d (sequence shards, 1 NCCL all-reduce of %d floats = [g, -loglk] per step)"
                   % (world, n + 4) if world > 1 else "single GPU",
                   "l2": "inputs larger than L2 (one-hot operands 2x%.0f MB, logits %.0f MB, residuals %.0f MB per step)"
                   % (n_local * lq * 2 / 1e6, n_local * lq * 4 / 1e6, n_local * lq * 2 * products / 1e6),
                   "lambda_h": LAMBDA_H, "lambda_J": LAMBDA_J, "n_params": n, "forward": prob.forward,
                   "backward": prob.backward},
        "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": UNIT, "ms_per_step": float(te.item()) * 1e3,
                "h2d_bytes_per_step": int(4 * n), "d2h_bytes_per_step": int(4 * n + 16)},
        "gpu_launches": int(launches),
        "roofline": roofline,
        "fx": {"negloglk": fx_check[0], "objective": fx_check[1], "e2e_objective": fx_e2e},
        "hamming_setup": {"pairs_per_s": 0.5 * n_total * (n_total - 1) / t_ham, "seconds": t_ham, "N": n_total,
                          "note": "includes H2D + packing; untimed setup, not the benchmarked step"},
    }
    if consistency is not None:
        line["rank_consistency"] = consistency
    if comm is not None:
        line["communication"] = comm

    # ---- correctness of the timed path (every world size; the oracle is the checker only) ----
    if rank == 0:
        try:
            from oracle import c_oracle as co
            solo = CudaEngine(standalone=True)
            ns = min(ACC_SAMPLE_N, n_total)
            sub = solo.plm_problem(codes[:ns], weights[:ns], Q, -1, 0.0, 0.0, backward=prob.backward,
                                   forward=prob.forward, precision=args.precision)
            sub.set_x(x)
            fs = sub.evaluate(sub.x)
            gs = sub.g.cpu().numpy().astype(np.float64)
            sub.close()
            f64, g64, _ = co.plm_eval(codes[:ns], weights[:ns].astype(np.float64), x.astype(np.float64), Q, 0.0, 0.0,
                                      "f64", nthreads=host_threads())
            _, g32, _ = co.plm_eval(codes[:ns], weights[:ns], x, Q, 0.0, 0.0, "f32", nthreads=host_threads())
            line["accuracy"] = {
                "sample": "%d sequences of the workload, data term only, vs float64 oracle" % ns,
                "grad_rel_l2_err": float(np.linalg.norm(gs - g64) / np.linalg.norm(g64)),
                "fx_rel_err": float(abs(fs - f64) / abs(f64)),
                "cpu_fp32_port_grad_rel_l2_err": float(np.linalg.norm(g32 - g64) / np.linalg.norm(g64)),
            }
            if world > 1:
                # the sharded evaluation against ONE GPU evaluating all n_total sequences
                whole = solo.plm_problem(codes, weights, Q, -1, LAMBDA_H, LAMBDA_J, backward=prob.backward,
                                         forward=prob.forward, precision=args.precision)
                whole.set_x(x)
                fw = whole.evaluate(whole.x)
                gw = whole.g.double()
                gd = prob.g.double()
                line["accuracy"]["sharded_vs_single_gpu"] = {
                    "fx_rel_diff": float(abs(fw - fx_check[1]) / abs(fw)),
                    "grad_rel_l2_diff": float(((gw - gd).norm() / gw.norm()).item()),
                    "note": "same %d sequences evaluated by rank 0 alone; differences are summation order only" % n_total}
                whole.close()
        except Exception as e:      # the checker must never break the bench line
            line["accuracy"] = {"error": "%s: %s" % (type(e).__name__, e)}

    if rank == 0 and world == 1 and not args.no_subrecords:
        # CPU port beside it: the FULL workload, all host threads, bounded to ~20 s
        try:
            cb_value, cb_dt, threads, cb_steps = cpu_arm(codes, x, weights, 2, 1, budget_s=20.0)
            line["cpu_baseline"] = {"value": cb_value, "unit": UNIT, "cores": threads, "kind": "port",
                                    "sample": "the full workload (all %d sequences), %d timed evaluations after 1 "
                                              "warm-up (%.2f s each)" % (n_total, cb_steps, cb_dt)}
        except Exception as e:
            line["cpu_baseline"] = {"error": str(e)}
        try:
            line["fit"] = fit_subrecord(prob, x, ms_step)
        except Exception as e:
            line["fit"] = {"error": "%s: %s" % (type(e).__name__, e)}
    prob.close()
    if rank == 0 and world == 1 and not args.no_subrecords and (N_PER_GPU, L) == (50000, 200):
        try:
            line["run_plmc_e2e"] = run_plmc_subrecord(codes, line.get("cpu_baseline", {}))
        except Exception as e:
            line["run_plmc_e2e"] = {"error": "%s: %s" % (type(e).__name__, e)}
        try:
            rec, _ = hamming_subrecord(engine, peaks)
            line["hamming"] = rec
            line["hamming"]["unpruned"] = hamming_unpruned_ms()
        except Exception as e:
            line["hamming"] = {"error": "%s: %s" % (type(e).__name__, e)}
    if args.dump_outputs and rank == 0:
        line["dumped_outputs"] = dump_outputs(args.dump_outputs, outputs)
    if world > 1:
        dist.destroy_process_group()
    _nccl_log_to_stderr(nccl_dir)
    if rank == 0:
        print(json.dumps(line))
        sys.stdout.flush()


def ncu_traffic(kernel_name, precision):
    """DRAM bytes per launch of the dominant kernel from the newest committed `ncu --set full` extract
    (profiles/r2_ncu_traffic.json, written by profiles/summarize_ncu.py from the .ncu-rep of this round)."""
    path = os.path.join(ROOT, "profiles", "r2_ncu_traffic.json")
    if not kernel_name.startswith("tc_gemm_persistent_kernel"):
        return None, None           # the table holds the default-path GEMMs only
    try:
        with open(path) as f:
            table = json.load(f)
        key = ("fwd" if "forward" in kernel_name or "fused" in kernel_name else "bwd") + ("_bf16" if precision == "bf16" else "_fp32")
        ent = table.get(key)
        if ent is None:
            return None, None
        return float(ent["dram_bytes_read"]) + float(ent["dram_bytes_write"]), "profiles/r2_ncu_traffic.json[%s] (%s)" % (key, ent.get("capture", "?"))
    except Exception:
        return None, None


def fit_subrecord(prob, x, ms_eval, iterations=40):
    """Device-resident L-BFGS (evc_plm_fit): ms per iteration next to ms per evaluation."""
    import torch
    from evcouplings_b200 import lbfgs
    x0 = np.zeros_like(x)
    prob.fit(x0, lbfgs.default_params(max_iterations=2, epsilon=1e-9, m=6))     # allocates the workspace (untimed)
    params = lbfgs.default_params(max_iterations=iterations, epsilon=1e-9, m=6)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    res = prob.fit(x0, params)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    return {"driver": "evc_plm_fit (L-BFGS loop inside libevcplm, 48 B D2H per evaluation)", "iterations": res.iterations,
            "evaluations": res.evaluations, "ms_per_iteration": dt * 1e3 / max(1, res.iterations),
            "ms_per_evaluation_in_fit": dt * 1e3 / max(1, res.evaluations), "ms_per_evaluation_bench": ms_eval,
            "status": res.status, "fx": res.fx}


def run_plmc_subrecord(codes, cpu_baseline, iterations=100):
    """End to end through the reference-facing entry point: A2M file -> ingest -> reweighting -> f_i/f_ij ->
    100 L-BFGS iterations -> .model + _ECs.txt, wall clock."""
    from evcouplings_b200 import synthetic, tools
    d = tempfile.mkdtemp(prefix="evc_bench_")
    a2m = os.path.join(d, "cfg2.a2m")
    synthetic.write_a2m(a2m, codes)
    t0 = time.perf_counter()
    res, run = tools.run_plmc(a2m, os.path.join(d, "cfg2_ECs.txt"), os.path.join(d, "cfg2.model"),
                              focus_seq="seq0/1-%d" % L, theta=0.8, ignore_gaps=False, iterations=iterations,
                              lambda_h=LAMBDA_H, lambda_J=LAMBDA_J, return_run=True, num_gpus=1)
    wall = time.perf_counter() - t0
    sizes = {k: os.path.getsize(os.path.join(d, k)) for k in os.listdir(d)}
    for k in list(sizes):
        os.unlink(os.path.join(d, k))
    os.rmdir(d)
    rec = {"what": "evcouplings_b200.run_plmc on the config-2 alignment written as A2M (%d x %d), %d iterations"
                   % (codes.shape[0], codes.shape[1], iterations),
           "wall_s": wall, "timings_s": {k: float(v) for k, v in run.timings.items()},
           "iterations": int(run.lbfgs.iterations), "evaluations": int(run.lbfgs.evaluations),
           "status": run.lbfgs.status, "n_eff": run.n_eff, "output_bytes": sizes}
    if "value" in cpu_baseline:
        cells = float(codes.shape[0]) * L * L * Q
        per_eval = cells / cpu_baseline["value"]
        rec["cpu_port_estimate_s"] = {"optimisation": per_eval * int(run.lbfgs.evaluations),
                                      "note": "CPU port: measured s/evaluation (cpu_baseline) x the same number of "
                                              "evaluations; ingest and file writing are the same host code"}
    return rec


def hamming_unpruned_ms():
    """Un-pruned time of the Hamming tile kernel (early termination and the two-phase filter disabled through the
    library's bench hook, which is read once per process => separate process)."""
    code = ("import sys, json; sys.path.insert(0, %r)\nimport bench, torch\n"
            "from evcouplings_b200.engine import CudaEngine\ntorch.cuda.set_device(0)\n"
            "rec, _ = bench.hamming_subrecord(CudaEngine(), bench.measured_peaks(), steps=2)\n"
            "print('UNPRUNED ' + json.dumps({'ms_per_step': rec['ms_per_step'], 'frac': rec['roofline']['frac']}))\n" % ROOT)
    env = dict(os.environ)
    env["EVC_HAMMING_NO_PRUNE"] = "1"
    p = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=env, timeout=600)
    for ln in p.stdout.splitlines():
        if ln.startswith("UNPRUNED "):
            return json.loads(ln[len("UNPRUNED "):])
    return {"error": p.stderr[-500:]}


def run_hamming(args):
    """Secondary workload (BASELINE configs[2]): O(N^2 L) Hamming reweighting, N=200,000 L=300.
    Device-resident timing of the tile kernels (planes already packed in HBM)."""
    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    nccl_dir = _nccl_env()
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    from evcouplings_b200 import msa, synthetic, _lib
    from evcouplings_b200.engine import CudaEngine, shard_bounds
    engine = CudaEngine()
    lib = engine.lib
    peaks = measured_peaks()
    if args.hamming_pabp:
        c = np.load(os.path.join(ROOT, "tests", "golden", "pabp_codes.npz"))
        codes = np.ascontiguousarray(c["codes"])
        N, Lh = codes.shape
        label = "PABP_YEAST real alignment (valid rows, %d x %d, shipped with the reference)" % (N, Lh)
    else:
        N, Lh = args.hamming_n, 300
        codes = synthetic.synthetic_msa_codes(N, Lh, 3)
        label = "synthetic N=%d L=%d (BASELINE configs[2])" % (N, Lh)
    thr = msa.identity_threshold_count(0.8, Lh)
    d_codes = torch.from_numpy(codes).to(engine.device)
    words = lib.evc_hamming_plane_words(N, Lh)
    d_planes = torch.empty(words, dtype=torch.int32, device=engine.device)
    d_counts = torch.zeros(N, dtype=torch.int32, device=engine.device)
    _lib.check(lib.evc_hamming_pack(engine.ptr(d_codes), N, Lh, engine.ptr(d_planes), engine.stream()), "pack")
    ntiles = lib.evc_hamming_num_tiles(N)
    lo, hi = shard_bounds(ntiles, world, rank)
    steps, warm = max(1, args.steps), max(1, min(args.warmup, 2))
    for _ in range(warm):
        _lib.check(lib.evc_hamming_count_tiles(engine.ptr(d_planes), N, Lh, thr, lo, hi, engine.ptr(d_counts),
                                               engine.stream()), "count")
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    sampler = ClockSampler(local_rank)
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        d_counts.zero_()
        _lib.check(lib.evc_hamming_count_tiles(engine.ptr(d_planes), N, Lh, thr, lo, hi, engine.ptr(d_counts),
                                               engine.stream()), "count")
        if world > 1:
            dist.all_reduce(d_counts)
    e1.record()
    torch.cuda.synchronize()
    t = torch.tensor([e0.elapsed_time(e1) / steps], dtype=torch.float64, device=engine.device)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    clocks = sampler.summary()
    pairs = 0.5 * N * (N - 1)
    Wd = -(-Lh // 32)
    alu_ops = pairs * Wd * 6.0
    peak_ops = 64.0 * 148 * peaks["sm_max_mhz"] * 1e6 * world
    line = {"metric": "Hamming reweighting pairs/s", "value": pairs / (ms * 1e-3), "unit": "pairs/s", "n_gpus": world,
            "steps": steps, "warmup": warm, "ms_per_step": ms, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "u8 (5 bit-planes, u32 words)", "data": "real" if args.hamming_pabp else "synthetic",
            "config": {"workload": "pairwise Hamming reweighting, " + label + ", theta=0.8",
                       "l2": "bit-plane buffer %.0f MB is L2-resident by design; integer-pipe bound" % (words * 4 / 1e6),
                       "pruning": "disabled (EVC_HAMMING_NO_PRUNE)" if os.environ.get("EVC_HAMMING_NO_PRUNE") else
                                  "exact two-phase filter + early termination (product default)"},
            "clocks": clocks, "gpu_launches": steps,
            "roofline": {"bound": "int-alu", "kernel": "hamming_tile_kernel", "achieved": alu_ops / (ms * 1e-3) / 1e12,
                         "peak": peak_ops / 1e12, "unit": "Tops/s (int32 ALU)", "frac": alu_ops / (ms * 1e-3) / peak_ops,
                         "traffic": None, "algorithmic_ops_per_launch": alu_ops,
                         "note": "algorithmic = un-pruned op count (pairs x ceil(L/32) words x (5 LOP3 + IADD)); ALU pipe "
                                 "64 lanes/clk/SM x 148 SMs x max SM clock; exact pruning lets frac exceed 1",
                         "site_compares_per_s": pairs * Lh / (ms * 1e-3)}}
    if rank == 0 and world == 1:
        from oracle import c_oracle as co
        rows = 256
        t0 = time.perf_counter()
        ref = co.hamming_counts(codes, thr, rows=(0, rows), nthreads=host_threads())
        dt = time.perf_counter() - t0
        got = d_counts.cpu().numpy()
        line["cpu_baseline"] = {"value": rows * N / dt / 2, "unit": "pairs/s", "cores": host_threads(), "kind": "port",
                                "sample": "%d of %d rows against all columns (%.1f s); unordered-pair equivalent" % (rows, N, dt)}
        line["parity_sample_rows_exact"] = bool(np.array_equal(got[:rows], ref))
    if args.dump_outputs and rank == 0:
        line["dumped_outputs"] = dump_outputs(args.dump_outputs, {"counts": d_counts.cpu().numpy().astype(np.float64)})
    if world > 1:
        dist.destroy_process_group()
    _nccl_log_to_stderr(nccl_dir)
    if rank == 0:
        print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="plm", choices=["plm", "hamming"])
    ap.add_argument("--hamming-n", type=int, default=200000)
    ap.add_argument("--hamming-pabp", action="store_true", help="Hamming workload on the real PABP alignment")
    ap.add_argument("--seqs", type=int, default=None, help="sequences per GPU (default 50000 = BASELINE configs[1])")
    ap.add_argument("--sites", type=int, default=None, help="alignment length L (default 200)")
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200, help="timed evaluations (default 200 = about 1 s)")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"])
    ap.add_argument("--precision", default="fp32", choices=["fp32", "bf16"],
                    help="tensor-core products: fp32-equivalent bf16 hi+lo pairs (default) or bf16 tiles")
    ap.add_argument("--forward", default=None, choices=["gather", "tc", "tcfused"],
                    help="forward kernel of the data term (default: engine default / EVC_FORWARD)")
    ap.add_argument("--backward", default=None, choices=["gather", "tc"],
                    help="backward kernel of the data term (default: engine default / EVC_BACKWARD)")
    ap.add_argument("--no-subrecords", action="store_true", help="skip the hamming / fit / run_plmc sub-records")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's outputs as DIR/<name>.npy (at most 64 MB in all)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs applies to --impl b200")
    global N_PER_GPU, L, LAMBDA_J
    if args.seqs:
        N_PER_GPU = args.seqs
    if args.sites:
        L = args.sites
        LAMBDA_J = 0.01 * (Q - 1) * (L - 1)
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    if args.workload == "hamming":
        run_hamming(args)
    elif args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
