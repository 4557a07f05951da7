"""
GPU parity tests (-m gpu): the CUDA path, called through the C ABI of libevcplm.so, against the CPU
oracle (oracle/) on the same seeded inputs and against the committed golden fixtures.  Integer work
(Hamming counts) must be bit-exact; floating point is fp32 on the device and is compared with the
float64 oracle at the tolerances written in each test.
"""
import ctypes
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from evcouplings_b200 import _lib, lbfgs, model_io, msa, synthetic, tools  # noqa: E402
from oracle import c_oracle as co  # noqa: E402
from oracle import plm_oracle as po  # noqa: E402


@pytest.fixture(scope="module")
def lib():
    l = _lib.load()
    _lib.require_device()
    return l


@pytest.fixture(scope="module")
def engine(lib):
    from evcouplings_b200.engine import CudaEngine
    return CudaEngine()


def gpu_hamming(lib, codes, thr):
    codes = np.ascontiguousarray(codes, dtype=np.uint8)
    N, L = codes.shape
    out = np.zeros(N, dtype=np.int32)
    _lib.check(lib.evc_hamming_counts(codes.ctypes.data_as(ctypes.c_void_p), N, L, thr, 0,
                                      out.ctypes.data_as(ctypes.c_void_p)), "evc_hamming_counts")
    return out


def gpu_eval_host(lib, codes, w, x, q, gap_code, lam_h, lam_J, tc=False, tcf=False, fused=False):
    codes = np.ascontiguousarray(codes, dtype=np.uint8)
    w = np.ascontiguousarray(w, dtype=np.float32)
    x = np.ascontiguousarray(x, dtype=np.float32)
    N, L = codes.shape
    h = ctypes.c_void_p()
    _lib.check(lib.evc_plm_create(ctypes.byref(h), codes.ctypes.data_as(ctypes.c_void_p), N, L, q, gap_code,
                                  w.ctypes.data_as(ctypes.c_void_p), 0), "evc_plm_create")
    try:
        if tc:
            _lib.check(lib.evc_plm_set_backward(h, 1), "evc_plm_set_backward")
        if tcf:
            _lib.check(lib.evc_plm_set_forward(h, 2 if fused else 1), "evc_plm_set_forward")
        assert lib.evc_plm_num_params(h) == x.size
        g = np.zeros_like(x)
        fx = np.zeros(2, dtype=np.float64)
        _lib.check(lib.evc_plm_eval_host(h, x.ctypes.data_as(ctypes.c_void_p), g.ctypes.data_as(ctypes.c_void_p),
                                         fx.ctypes.data_as(ctypes.c_void_p), lam_h, lam_J), "evc_plm_eval_host")
    finally:
        lib.evc_plm_destroy(h)
    return fx[1], g, fx[0]


# ------------------------------------------------------------------------------------------------
# (b) Hamming reweighting: bit-exact
# ------------------------------------------------------------------------------------------------
def test_hamming_golden_intree_twins(lib, golden_dir):
    """against counts produced by the reference's own num_cluster_members (alignment.py:1192-1233)"""
    d = np.load(os.path.join(golden_dir, "intree_twins.npz"))
    for name in ("cfg1", "tie", "odd"):
        codes = d[name + "_codes"]
        thr = msa.identity_threshold_count(float(d[name + "_theta"]), codes.shape[1])
        assert np.array_equal(gpu_hamming(lib, codes, thr), d[name + "_counts"])


@pytest.mark.parametrize("N,L,theta,seed", [(1, 5, 0.8, 0), (2, 31, 0.5, 1), (127, 32, 0.8, 2), (129, 33, 0.8, 3),
                                            (1000, 97, 0.7, 4), (3001, 200, 0.8, 5), (5000, 300, 0.8, 6),
                                            (777, 800, 0.9, 7)])
def test_hamming_vs_oracle(lib, N, L, theta, seed):
    codes = synthetic.synthetic_msa_codes(N, L, seed)
    thr = msa.identity_threshold_count(theta, L)
    assert np.array_equal(gpu_hamming(lib, codes, thr), co.hamming_counts(codes, thr))


def test_hamming_edge_thresholds(lib):
    codes = synthetic.synthetic_msa_codes(300, 40, 11)
    codes[17] = codes[3]                      # exact duplicates
    assert (gpu_hamming(lib, codes, 0) == 300).all()            # everything is a neighbour
    got = gpu_hamming(lib, codes, 40)                           # only exact duplicates
    assert np.array_equal(got, co.hamming_counts(codes, 40)) and got[17] >= 2
    assert (gpu_hamming(lib, codes, 41) == 0).all()             # unreachable threshold
    all_gap = np.zeros((50, 64), dtype=np.uint8)
    assert (gpu_hamming(lib, all_gap, 64) == 50).all()          # gap == gap is an identity
    hi = np.full((40, 10), 31, dtype=np.uint8)                  # largest representable code
    assert (gpu_hamming(lib, hi, 10) == 40).all()


def test_hamming_two_phase_overflow_falls_back_exactly(tmp_path):
    """long alignment (two-phase filter + verify) with a candidate buffer forced to 100 entries: the overflow
    path must fall back to the single-phase kernel and still be exact (run in a subprocess: env-controlled)."""
    import subprocess, sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    code = (
        "import sys, ctypes, numpy as np; sys.path.insert(0, %r)\n"
        "from evcouplings_b200 import _lib, msa, synthetic\nfrom oracle import c_oracle as co\n"
        "lib = _lib.load(); codes = synthetic.synthetic_msa_codes(3000, 300, 6)\n"
        "thr = msa.identity_threshold_count(0.8, 300); out = np.zeros(3000, dtype=np.int32)\n"
        "_lib.check(lib.evc_hamming_counts(codes.ctypes.data_as(ctypes.c_void_p), 3000, 300, thr, 0,"
        " out.ctypes.data_as(ctypes.c_void_p)), 'hamming')\n"
        "assert np.array_equal(out, co.hamming_counts(codes, thr)); print('exact')\n" % root)
    for cap in ("100", None):
        env = dict(os.environ)
        if cap:
            env["EVC_HAMMING_CAND_CAP"] = cap
        p = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=env, timeout=300)
        assert p.returncode == 0 and "exact" in p.stdout, p.stderr[-2000:]


def test_hamming_pabp_golden_counts(lib, golden_dir):
    """exact equality with the neighbour counts plmc itself stored (golden PABP run), full 151,496 x 82"""
    c = np.load(os.path.join(golden_dir, "pabp_codes.npz"))
    valid = np.unpackbits(c["valid_packed"])[: int(c["n_total"])].astype(bool)
    gold = c["golden_counts_all"][valid]
    got = gpu_hamming(lib, c["codes"], msa.identity_threshold_count(0.8, 82))
    assert np.array_equal(got, gold)
    assert abs((1.0 / got).sum() - 18615.48) < 0.01


def test_hamming_full_size_sampled_rows(lib):
    """BASELINE config 3 shape (N=200k, L=300): every sampled row equals the oracle's count."""
    N, L = 200000, 300
    codes = synthetic.synthetic_msa_codes(N, L, 3)
    thr = msa.identity_threshold_count(0.8, L)
    got = gpu_hamming(lib, codes, thr)
    for r0 in (0, 99968, N - 48):
        ref = co.hamming_counts(codes, thr, rows=(r0, r0 + 48))
        assert np.array_equal(got[r0:r0 + 48], ref)
    assert got.min() >= 1


# ------------------------------------------------------------------------------------------------
# (a) PLM objective + gradient: fp32 device vs float64 oracle
# ------------------------------------------------------------------------------------------------
def _check_eval(lib, N, L, q, gap, seed, lam_h=0.01, lam_J=2.0, xscale=0.1, tc=False, tcf=False, fused=False):
    rng = np.random.default_rng(seed)
    codes = synthetic.synthetic_msa_codes(N, L, seed)
    if gap:
        codes = synthetic.to_ignore_gaps_codes(codes)
    if q in (4, 5):
        codes = (codes % 5).astype(np.uint8)
        if gap:
            codes = np.where(codes == 4, 4, codes).astype(np.uint8)   # 4 == gap code for q=4
    w = rng.uniform(0.05, 1.0, N).astype(np.float32)
    n = L * q + L * (L - 1) // 2 * q * q
    x = rng.normal(0, xscale, n).astype(np.float32)
    fx, g, nll = gpu_eval_host(lib, codes, w, x, q, q if gap else -1, lam_h, lam_J, tc=tc, tcf=tcf, fused=fused)
    fx64, g64, nll64 = co.plm_eval(codes, w.astype(np.float64), x.astype(np.float64), q, lam_h, lam_J, "f64")
    # tolerance: fp32 accumulation over N sequences; measured error of the CPU fp32 port is the yardstick
    fx32, g32, _ = co.plm_eval(codes, w, x, q, lam_h, lam_J, "f32")
    err_gpu = np.abs(g - g64).max()
    err_c32 = np.abs(g32 - g64).max()
    scale = np.abs(g64).max()
    assert abs(fx - fx64) <= 2e-6 * abs(fx64), (fx, fx64)
    assert abs(nll - nll64) <= 2e-6 * abs(nll64)
    # gather / tensor-core backward: <= 3x the fp32 CPU port.  Tensor-core FORWARD: the couplings enter the
    # tcgen05 GEMM as bf16 hi + lo (16 mantissa bits, |dJ| <= 2^-17 |J|), stated tolerance 5x / 4e-6 * max|g|
    fac, rel = (5.0, 4e-6) if tcf else (3.0, 2e-6)
    assert err_gpu <= max(fac * err_c32, rel * scale), (err_gpu, err_c32, scale)
    assert np.linalg.norm(g - g64) <= 5e-6 * np.linalg.norm(g64)
    print("eval parity N=%d L=%d q=%d tc=%s tcf=%s: max err %.3e (C fp32 port %.3e), rel L2 %.3e, fx rel %.3e"
          % (N, L, q, tc, tcf, err_gpu, err_c32, np.linalg.norm(g - g64) / np.linalg.norm(g64),
             abs(fx - fx64) / abs(fx64)))
    return err_gpu, err_c32


@pytest.mark.parametrize("N,L,q,gap,seed", [
    (200, 40, 21, False, 1),        # BASELINE config 1 shape
    (200, 40, 20, True, 1),         # ... with ignore_gaps (pipeline default)
    (1, 2, 21, False, 2),           # smallest legal problem
    (513, 33, 21, False, 3),        # ragged: N not a tile multiple, L not a multiple of 4
    (2049, 26, 20, True, 4),        # crosses a backward tile (2048) by one sequence
    (700, 97, 21, False, 5),
    (3000, 64, 20, True, 6),
    (300, 30, 5, False, 7),         # nucleotide alphabets
    (300, 30, 4, True, 8),
])
def test_plm_eval_vs_oracle(lib, N, L, q, gap, seed):
    _check_eval(lib, N, L, q, gap, seed)


@pytest.mark.parametrize("N,L,q,gap,seed", [
    (200, 40, 21, False, 1), (200, 40, 20, True, 1), (1, 2, 21, False, 2), (513, 33, 21, False, 3),
    (2049, 26, 20, True, 4), (700, 97, 21, False, 5), (3000, 64, 20, True, 6), (300, 30, 5, False, 7),
])
def test_plm_eval_tensor_core_backward_vs_oracle(lib, N, L, q, gap, seed):
    """same tolerance as the gather path: the bf16 hi/lo split of the residuals (16 mantissa bits, fp32
    accumulation in TMEM) must not be worse than 3x the error of a plain fp32 CPU evaluation."""
    _check_eval(lib, N, L, q, gap, seed, tc=True)


@pytest.mark.parametrize("N,L,q,gap,seed,xscale", [
    (200, 40, 21, False, 1, 0.1), (200, 40, 20, True, 1, 0.1), (1, 2, 21, False, 2, 0.1),
    (513, 33, 21, False, 3, 0.1), (2049, 26, 20, True, 4, 0.1), (700, 97, 21, False, 5, 0.1),
    (3000, 64, 20, True, 6, 0.1), (300, 30, 5, False, 7, 0.1), (400, 24, 21, False, 10, 1.0),
])
def test_plm_eval_tensor_core_forward_vs_oracle(lib, N, L, q, gap, seed, xscale):
    """forward logits on tcgen05 with the couplings split in bf16 hi + lo (16 mantissa bits): same tolerance;
    both the unfused (logits matrix + softmax kernel) and the fused-epilogue variants"""
    _check_eval(lib, N, L, q, gap, seed, xscale=xscale, tcf=True)
    _check_eval(lib, N, L, q, gap, seed, xscale=xscale, tcf=True, fused=True)


@pytest.mark.parametrize("N,L,q,gap,seed", [
    (3000, 500, 20, True, 41),      # BASELINE configs[3] site count (Pfam-scale L=500), ignore_gaps
    (1500, 800, 21, False, 42),     # BASELINE configs[4] site count (EVcomplex L=800)
])
def test_plm_eval_large_L_shapes(lib, N, L, q, gap, seed):
    """geometry of the long-alignment configs (more sites than one shared-memory row block / many GEMM tiles)"""
    _check_eval(lib, N, L, q, gap, seed, tcf=True)
    _check_eval(lib, N, L, q, gap, seed, tcf=True, fused=True)      # falls back to the unfused path for L*q > 8192
    _check_eval(lib, N, L, q, gap, seed, tc=False, tcf=False)


def test_plm_eval_zero_and_large_params(lib):
    _check_eval(lib, 400, 24, 21, False, 9, xscale=0.0)          # x = 0: uniform softmax
    _check_eval(lib, 400, 24, 21, False, 10, xscale=1.0)         # large couplings: peaked softmax


def test_plm_eval_all_gap_column_ignore_gaps(lib):
    """a column that is entirely gaps contributes nothing and receives no data gradient"""
    codes = synthetic.to_ignore_gaps_codes(synthetic.synthetic_msa_codes(256, 12, 3))
    codes[:, 5] = 20
    w = np.ones(256, dtype=np.float32)
    n = 12 * 20 + 66 * 400
    x = np.random.default_rng(0).normal(0, 0.1, n).astype(np.float32)
    fx, g, nll = gpu_eval_host(lib, codes, w, x, 20, 20, 0.0, 0.0)
    fx64, g64, _ = co.plm_eval(codes, w.astype(np.float64), x.astype(np.float64), 20, 0.0, 0.0, "f64")
    assert np.abs(g - g64).max() < 1e-4
    assert np.abs(g[5 * 20:6 * 20]).max() == 0.0


def test_plm_create_rejects_bad_arguments(lib):
    codes = np.zeros((4, 6), dtype=np.uint8)
    w = np.ones(4, dtype=np.float32)
    h = ctypes.c_void_p()
    for q, gap in ((7, -1), (21, 5)):
        rc = lib.evc_plm_create(ctypes.byref(h), codes.ctypes.data_as(ctypes.c_void_p), 4, 6, q, gap,
                                w.ctypes.data_as(ctypes.c_void_p), 0)
        assert rc != 0 and lib.evc_last_error()
    rc = lib.evc_plm_create(ctypes.byref(h), codes.ctypes.data_as(ctypes.c_void_p), 0, 6, 21, -1,
                            w.ctypes.data_as(ctypes.c_void_p), 0)
    assert rc != 0


def test_weighted_counts_vs_oracle(engine):
    for gap in (False, True):
        codes = synthetic.synthetic_msa_codes(900, 30, 21)
        if gap:
            codes = synthetic.to_ignore_gaps_codes(codes)
        q = 20 if gap else 21
        w = (1.0 / co.hamming_counts(codes, 24)).astype(np.float32)
        prob = engine.plm_problem(codes, w, q, q if gap else -1, 0.01, 1.0)
        fic, fijc = prob.weighted_counts()
        prob.close()
        fi, fij = model_io.normalise_frequencies(fic, fijc, float(w.sum()), gap)
        fi_o, fij_o = po.frequencies(codes, w.astype(np.float64), q, q if gap else -1)
        assert np.abs(fi - fi_o).max() < 2e-6 and np.abs(fij - fij_o).max() < 2e-6


def test_pabp_frequencies_golden(engine, golden_dir):
    """f_i / f_ij from the CUDA path vs the values plmc wrote into the golden .model (<= 1e-6 + fp32 noise)"""
    c = np.load(os.path.join(golden_dir, "pabp_codes.npz"))
    g = np.load(os.path.join(golden_dir, "pabp_golden.npz"))
    valid = np.unpackbits(c["valid_packed"])[: int(c["n_total"])].astype(bool)
    w = (1.0 / c["golden_counts_all"][valid]).astype(np.float32)
    prob = engine.plm_problem(c["codes"], w, 20, 20, 0.01, 16.2)
    fic, fijc = prob.weighted_counts()
    prob.close()
    fi, fij = model_io.normalise_frequencies(fic, fijc, float(w.sum()), True)
    assert np.abs(fi - g["fi"]).max() < 5e-6
    assert np.abs(fij[g["fij_pair_index"]] - g["fij_blocks"]).max() < 5e-6


def test_pabp_gradient_balance_at_golden_optimum(engine, golden_dir):
    """SURVEY row a7 pin, on the device: at plmc's own (h, J) the data gradient balances 2*lambda_J*J."""
    c = np.load(os.path.join(golden_dir, "pabp_codes.npz"))
    g = np.load(os.path.join(golden_dir, "pabp_golden.npz"))
    valid = np.unpackbits(c["valid_packed"])[: int(c["n_total"])].astype(bool)
    w = (1.0 / c["golden_counts_all"][valid]).astype(np.float32)
    prob = engine.plm_problem(c["codes"], w, 20, 20, 0.0, 0.0)
    x = np.concatenate([g["h"].ravel(), g["J"].ravel()]).astype(np.float32)
    prob.set_x(x)
    prob.evaluate(prob.x)
    grad = prob.g.cpu().numpy()
    prob.close()
    gJ = grad[82 * 20:].reshape(-1, 20, 20)
    for k in g["fij_pair_index"]:
        J = g["J"][k].astype(np.float64)
        m = np.abs(J) > 0.02
        assert 0.9 < np.median(-gJ[k][m] / (2 * 16.2 * J[m])) < 1.1


# ------------------------------------------------------------------------------------------------
# a8: device L-BFGS algebra vs numpy
# ------------------------------------------------------------------------------------------------
def test_lbfgs_vector_algebra(engine):
    import torch
    codes = synthetic.synthetic_msa_codes(64, 9, 2)
    prob = engine.plm_problem(codes, np.ones(64, dtype=np.float32), 21, -1, 0.01, 1.0, m=4)
    prob._ensure_python_space()       # vectors of the Python driver (the default fit runs inside libevcplm)
    n, m = prob.n, 4
    rng = np.random.default_rng(0)
    a, b = rng.normal(size=n).astype(np.float32), rng.normal(size=n).astype(np.float32)
    ta, tb = torch.from_numpy(a).cuda(), torch.from_numpy(b).cuda()
    assert abs(prob.dot(ta, tb) - float(np.dot(a.astype(np.float64), b.astype(np.float64)))) < 1e-9 * n
    prob.axpby(ta, tb, 0.5, 2.0)
    assert np.allclose(ta.cpu().numpy(), 0.5 * b + 2.0 * a, rtol=1e-6, atol=1e-6)
    # build a history of 6 updates in a ring of 4 and compare the direction with a numpy two-loop
    from cpu_engine import OracleProblem
    ref = OracleProblem(codes, np.ones(64), 21, -1, 0.01, 1.0, m=m)
    end = 0
    for k in range(1, 7):
        xp, gp = rng.normal(size=n).astype(np.float32), rng.normal(size=n).astype(np.float32)
        s = (0.1 * rng.normal(size=n)).astype(np.float32)
        xn = xp + s
        gn = (gp + s * rng.uniform(0.5, 2.0, n).astype(np.float32)).astype(np.float32)   # y.s > 0
        prob.x.copy_(torch.from_numpy(xn)); prob.g.copy_(torch.from_numpy(gn))
        prob.xp.copy_(torch.from_numpy(xp)); prob.gp.copy_(torch.from_numpy(gp))
        prob.update_pair(end, prob.xp, prob.gp)
        ref.x[:], ref.g[:] = xn, gn
        ref.update_pair(end, (xn - s.astype(np.float64)) * 0 + xp, gp.astype(np.float64))
        end = (end + 1) % m
        bound = min(m, k)
        prob.direction(prob.d, bound, end)
        ref.direction(ref.d, bound, end)
        got = prob.d.cpu().numpy()
        assert np.linalg.norm(got - ref.d) <= 2e-5 * np.linalg.norm(ref.d), k
    prob.close()


# ------------------------------------------------------------------------------------------------
# end to end through run_plmc (the reference-facing plugin)
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("ignore_gaps", [False, True])
def test_run_plmc_config1_vs_oracle_optimum(engine, tmp_path, ignore_gaps):
    """BASELINE config 1 (N=200, L=40): fitted h, J and EC scores vs the float64 oracle optimum.
    Tolerances (north star): CN rms <= 1e-4; parameters max abs <= 2e-3."""
    N, L = 200, 40
    codes = synthetic.synthetic_msa_codes(N, L, 1)
    a2m = tmp_path / "cfg1.a2m"
    synthetic.write_a2m(str(a2m), codes)
    q = 20 if ignore_gaps else 21
    lam_J = 0.01 * (q - 1) * (L - 1)
    res, run = tools.run_plmc(str(a2m), str(tmp_path / "o_ECs.txt"), str(tmp_path / "o.model"), focus_seq="seq0/1-40",
                              theta=0.8, ignore_gaps=ignore_gaps, iterations=3000, lambda_h=0.01, lambda_J=lam_J,
                              engine=engine, return_run=True, epsilon=1e-5)
    ali = run.alignment
    counts_o = co.hamming_counts(ali.codes, msa.identity_threshold_count(0.8, L))
    assert np.array_equal(run.counts, counts_o)
    w = 1.0 / counts_o
    xo, info = po.fit(ali.codes, w, q, 0.01, lam_J, ali.gap_code, x0=tools.initial_point(
        po.frequencies(ali.codes, w, q, ali.gap_code)[0], w.sum(), L, q).astype(np.float64), max_iter=4000,
        objective_fn=lambda v: co.plm_eval(ali.codes, w, v, q, 0.01, lam_J, "f64"))
    m = po.read_model(str(tmp_path / "o.model"))
    x = np.concatenate([m["h"].ravel(), m["J"].ravel()]).astype(np.float64)
    cn = np.loadtxt(str(tmp_path / "o_ECs.txt"), usecols=5)
    cn_o = po.cn_scores(xo[L * q:].reshape(-1, q, q), L)
    nh = L * q
    f_gpu = po.objective(x, ali.codes, w, q, 0.01, lam_J, ali.gap_code)[0]
    f_opt = po.objective(xo, ali.codes, w, q, 0.01, lam_J, ali.gap_code)[0]
    dJ, dh = np.abs(x[nh:] - xo[nh:]).max(), np.abs(x[:nh] - xo[:nh]).max()
    print("status", res.optimization_status, "iters", run.lbfgs.iterations, "evals", run.lbfgs.evaluations,
          "max|dJ|", dJ, "max|dh|", dh, "rel objective gap", (f_gpu - f_opt) / f_opt,
          "cn rms", np.sqrt(np.mean((cn - cn_o) ** 2)), "cn max", np.abs(cn - cn_o).max())
    # stated fp32 tolerances: EC (cn) rms <= 1e-4 (north star); couplings max abs <= 2e-3; fields max abs
    # <= 0.1 (lambda_h = 0.01 leaves h almost flat: the objective gap below is what convergence means);
    # objective within 1e-6 relative of the float64 optimum
    assert np.sqrt(np.mean((cn - cn_o) ** 2)) <= 1e-4
    assert dJ <= 2e-3 and dh <= 0.1
    assert 0 <= (f_gpu - f_opt) / f_opt <= 1e-6
    assert res.num_valid_seqs == N and res.num_valid_sites == L
    fi_o, fij_o = po.frequencies(ali.codes, w, q, ali.gap_code)
    assert np.abs(m["fi"] - fi_o).max() < 2e-6 and np.abs(m["fij"] - fij_o).max() < 2e-6


def test_run_plmc_iteration_capped_trajectory_matches_host_logic(engine, tmp_path):
    """same L-BFGS control logic, device vs oracle backend, 15 iterations from the same start:
    trajectories agree to fp32 noise (fx within 1e-5 relative at every iteration)."""
    from cpu_engine import OracleEngine
    codes = synthetic.synthetic_msa_codes(300, 24, 4)
    a2m = tmp_path / "t.a2m"
    synthetic.write_a2m(str(a2m), codes)
    kw = dict(focus_seq="seq0", theta=0.8, iterations=15, lambda_h=0.01, lambda_J=0.01 * 20 * 23, return_run=True)
    r1, run1 = tools.run_plmc(str(a2m), str(tmp_path / "g_ECs.txt"), str(tmp_path / "g.model"), engine=engine, **kw)
    r2, run2 = tools.run_plmc(str(a2m), str(tmp_path / "c_ECs.txt"), str(tmp_path / "c.model"),
                              engine=OracleEngine(), **kw)
    f1 = r1.iteration_table["fx"].astype(float).values
    f2 = r2.iteration_table["fx"].astype(float).values
    assert len(f1) == len(f2) == 15
    assert np.abs(f1 - f2).max() <= 1e-5 * np.abs(f2).max()
    assert np.abs(run1.x - run2.x).max() < 5e-4


# ------------------------------------------------------------------------------------------------
# full BASELINE size (config 2: N=50k, L=200, q=21): size-independent properties
# ------------------------------------------------------------------------------------------------
def test_full_size_properties(engine):
    import torch
    N, L, q = 50000, 200, 21
    codes = synthetic.synthetic_msa_codes(N, L, 2)
    rng = np.random.default_rng(2)
    w = rng.uniform(0.05, 1.0, N).astype(np.float32)
    n = L * q + L * (L - 1) // 2 * q * q
    x = rng.normal(0, 0.05, n).astype(np.float32)
    full = engine.plm_problem(codes, w, q, -1, 0.0, 0.0)
    full.set_x(x)
    f_full = full.evaluate(full.x)
    g_full = full.g.clone()
    # (1) shards add up: data term is a sum over sequences
    half = N // 2 + 77
    pa = engine.plm_problem(codes[:half], w[:half], q, -1, 0.0, 0.0)
    pb = engine.plm_problem(codes[half:], w[half:], q, -1, 0.0, 0.0)
    pa.set_x(x); pb.set_x(x)
    fa, fb = pa.evaluate(pa.x), pb.evaluate(pb.x)
    assert abs((fa + fb) - f_full) <= 1e-9 * abs(f_full) + 1e-3
    gsum = pa.g + pb.g
    assert float((gsum - g_full).norm() / g_full.norm()) < 1e-5      # fp32 accumulation order differs
    pa.close(); pb.close()
    # (2) linear in the weights
    p2 = engine.plm_problem(codes, 2.0 * w, q, -1, 0.0, 0.0)
    p2.set_x(x)
    f2 = p2.evaluate(p2.x)
    assert abs(f2 - 2 * f_full) <= 1e-7 * abs(f_full)
    assert float((p2.g - 2 * g_full).norm() / g_full.norm()) < 1e-5
    p2.close()
    # (3) gradient is the derivative of fx along a random direction (central difference)
    d = torch.from_numpy(rng.normal(0, 1.0, n).astype(np.float32)).cuda()
    d /= d.norm()
    eps = 1e-1            # fx carries ~1e-7 relative noise (fp32 logits): use a wide central difference
    xs = torch.from_numpy(x).cuda()
    fp = full.evaluate(xs + eps * d)
    fm = full.evaluate(xs - eps * d)
    dd = float((g_full.double() * d.double()).sum())
    assert abs((fp - fm) / (2 * eps) - dd) <= 1e-2 * abs(dd) + 0.5
    # (4) the full-size gradient itself against the float64 oracle (C/OpenMP port, all host cores)
    fo_full, go_full, _ = co.plm_eval(codes, w.astype(np.float64), x.astype(np.float64), q, 0.0, 0.0, "f64")
    assert abs(f_full - fo_full) <= 2e-6 * abs(fo_full)
    gfh = g_full.cpu().numpy()
    rel = np.linalg.norm(gfh - go_full) / np.linalg.norm(go_full)
    print("full-size gradient vs float64 oracle: rel L2 err %.3e, max abs %.3e (max |g| %.3e)"
          % (rel, np.abs(gfh - go_full).max(), np.abs(go_full).max()))
    assert rel <= 1e-5
    # (5) sampled sequences subset against the oracle at full L (N_sub = 1500)
    full.close()
    sub = engine.plm_problem(codes[:1500], w[:1500], q, -1, 0.0, 0.0)
    sub.set_x(x)
    fs = sub.evaluate(sub.x)
    fo, go, _ = co.plm_eval(codes[:1500], w[:1500].astype(np.float64), x.astype(np.float64), q, 0.0, 0.0, "f64")
    assert abs(fs - fo) <= 2e-6 * abs(fo)
    assert np.linalg.norm(sub.g.cpu().numpy() - go) <= 5e-6 * np.linalg.norm(go)
    sub.close()


# ------------------------------------------------------------------------------------------------
# full BASELINE sizes of configs 4 (per-GPU share, L=500) and 5 (N=100k, L=800): tile scheduler, K-chunk promotion
# over 100k sequences, L*q = 16,800 -- against the float64 oracle through the shard-additivity identity
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("N,L,precision", [(62500, 500, "fp32"), (100000, 800, "fp32"), (100000, 800, "bf16")])
def test_full_size_config4_config5_shapes(engine, N, L, precision):
    import torch
    q, ns = 21, 2000
    codes = synthetic.synthetic_msa_codes(N, L, 4 if L == 500 else 5)
    rng = np.random.default_rng(L)
    w = rng.uniform(0.05, 1.0, N).astype(np.float32)
    n = L * q + L * (L - 1) // 2 * q * q
    x = rng.normal(0, 0.02, n).astype(np.float32)
    full = engine.plm_problem(codes, w, q, -1, 0.0, 0.0, precision=precision)
    full.set_x(x)
    f_full = full.evaluate(full.x)
    g_full = full.g.clone()
    full.close()
    rest = engine.plm_problem(codes[ns:], w[ns:], q, -1, 0.0, 0.0, precision=precision)
    rest.set_x(x)
    f_rest = rest.evaluate(rest.x)
    g_part = (g_full - rest.g).cpu().numpy().astype(np.float64)      # = gradient of the first ns sequences
    gnorm = float(g_full.double().norm())
    rest.close()
    del g_full
    torch.cuda.empty_cache()
    fo, go, _ = co.plm_eval(codes[:ns], w[:ns].astype(np.float64), x.astype(np.float64), q, 0.0, 0.0, "f64")
    err = np.linalg.norm(g_part - go)
    print("N=%d L=%d %s: |g_full - g_rest - g_oracle(first %d)| / |g_full| = %.3e; fx identity rel %.3e"
          % (N, L, precision, ns, err / gnorm, abs((f_full - f_rest) - fo) / abs(f_full)))
    # stated tolerances.  fp32-equivalent products: 2e-5 of |g_full| (two fp32 GPU gradients are subtracted);
    # bf16 tiles (BASELINE configs[4] mode): 8-bit mantissa products => 5e-3 of |g_full|, fx 1e-3 of the slice
    if precision == "fp32":
        assert err <= 2e-5 * gnorm
        assert abs((f_full - f_rest) - fo) <= 2e-6 * abs(f_full)
    else:
        assert err <= 5e-3 * gnorm
        assert abs((f_full - f_rest) - fo) <= 1e-3 * abs(fo) + 2e-6 * abs(f_full)


# ------------------------------------------------------------------------------------------------
# precision mode 1 ("bf16 tiles / fp32 parameters", BASELINE configs[4]; SURVEY 8b `precision`)
# ------------------------------------------------------------------------------------------------
def test_precision_bf16_tiles_vs_fp32_mode(engine):
    """One bf16 product per term instead of the hi+lo pair.  Stated tolerance against the fp32-equivalent run of
    the SAME kernels at the same point: gradient rel. L2 <= 5e-3, objective rel. <= 1e-4 (bf16 keeps 8 mantissa
    bits of each coupling / residual; the one-hot operand stays exact; accumulation stays fp32).  Measured on the
    B200: gradient 4.7e-4 here, 8.1e-4 at config 2, 1.2e-3 at config 5; objective 8e-7."""
    N, L, q = 6000, 120, 21
    codes = synthetic.synthetic_msa_codes(N, L, 11)
    rng = np.random.default_rng(11)
    w = rng.uniform(0.05, 1.0, N).astype(np.float32)
    n = L * q + L * (L - 1) // 2 * q * q
    x = rng.normal(0, 0.05, n).astype(np.float32)
    res = {}
    for prec in ("fp32", "bf16"):
        p = engine.plm_problem(codes, w, q, -1, 0.01, 5.0, precision=prec)
        p.set_x(x)
        res[prec] = (p.evaluate(p.x), p.g.cpu().numpy().astype(np.float64))
        p.close()
    fo, go, _ = co.plm_eval(codes, w.astype(np.float64), x.astype(np.float64), q, 0.01, 5.0, "f64")
    e32 = np.linalg.norm(res["fp32"][1] - go) / np.linalg.norm(go)
    e16 = np.linalg.norm(res["bf16"][1] - go) / np.linalg.norm(go)
    f16 = abs(res["bf16"][0] - fo) / abs(fo)
    print("gradient rel L2 vs float64 oracle: fp32 mode %.2e, bf16 tiles %.2e; fx rel (bf16) %.2e" % (e32, e16, f16))
    assert e32 <= 5e-6
    assert e16 <= 5e-3 and f16 <= 1e-4
    assert np.linalg.norm(res["bf16"][1] - res["fp32"][1]) <= 5e-3 * np.linalg.norm(res["fp32"][1])


def test_precision_schedule_auto_reaches_the_fp32_optimum(engine, tmp_path):
    """precision="auto": bf16 tiles until |g|/|x| < 10 eps, then fp32-equivalent products to convergence.  The fitted
    EC scores must agree with the pure fp32 run within the north-star tolerance (rms <= 1e-4)."""
    N, L = 400, 40
    codes = synthetic.synthetic_msa_codes(N, L, 12)
    a2m = tmp_path / "p.a2m"
    synthetic.write_a2m(str(a2m), codes)
    lam_J = 0.01 * 20 * (L - 1)
    out = {}
    for prec in ("fp32", "auto", "bf16"):
        res, run = tools.run_plmc(str(a2m), str(tmp_path / (prec + "_ECs.txt")), str(tmp_path / (prec + ".model")),
                                  focus_seq="seq0", theta=0.8, iterations=2000, lambda_h=0.01, lambda_J=lam_J,
                                  engine=engine, return_run=True, epsilon=1e-5, precision=prec)
        out[prec] = (np.loadtxt(str(tmp_path / (prec + "_ECs.txt")), usecols=5), res, run)
        print(prec, res.optimization_status, run.lbfgs.iterations, run.lbfgs.evaluations)
    rms_auto = np.sqrt(np.mean((out["auto"][0] - out["fp32"][0]) ** 2))
    rms_bf16 = np.sqrt(np.mean((out["bf16"][0] - out["fp32"][0]) ** 2))
    print("EC rms vs the fp32 run: auto %.2e, bf16-only %.2e" % (rms_auto, rms_bf16))
    # at epsilon = 1e-5 the fp32 evaluation noise ends these runs in the line search (LBFGSERR_ROUNDING_ERROR: fx
    # differences fall below 1e-7 * fx) before the gradient criterion triggers; what is asserted is WHERE they end up:
    # against each other and against the float64 optimum of the same objective
    ali = out["auto"][2].alignment
    w = 1.0 / co.hamming_counts(ali.codes, msa.identity_threshold_count(0.8, L))
    xo, _ = po.fit(ali.codes, w, 21, 0.01, lam_J, ali.gap_code, x0=tools.initial_point(
        po.frequencies(ali.codes, w, 21, ali.gap_code)[0], w.sum(), L, 21).astype(np.float64), max_iter=4000,
        objective_fn=lambda v: co.plm_eval(ali.codes, w, v, 21, 0.01, lam_J, "f64"))
    cn_opt = po.cn_scores(xo[L * 21:].reshape(-1, 21, 21), L)
    rms_opt = {k: float(np.sqrt(np.mean((out[k][0] - cn_opt) ** 2))) for k in out}
    print("EC rms vs the float64 optimum:", rms_opt)
    assert rms_opt["fp32"] <= 1e-4 and rms_opt["auto"] <= 1e-4
    assert rms_auto <= 1e-4          # measured 8e-6
    assert rms_bf16 <= 2e-3          # bf16 tiles alone: stated (looser) tolerance, measured 3.5e-4


# ------------------------------------------------------------------------------------------------
# a8: the device-resident L-BFGS (evc_plm_fit) against the Python driver of the same algorithm
# ------------------------------------------------------------------------------------------------
def test_device_fit_matches_python_driver(engine):
    N, L, q = 1200, 30, 21
    codes = synthetic.synthetic_msa_codes(N, L, 13)
    w = (1.0 / co.hamming_counts(codes, msa.identity_threshold_count(0.8, L))).astype(np.float32)
    params = lbfgs.default_params(max_iterations=25, epsilon=1e-9, m=6)
    traces = {}
    xs = {}
    for driver in ("device", "python"):
        p = engine.plm_problem(codes, w, q, -1, 0.01, 0.01 * 20 * (L - 1))
        tr = []
        res = p.fit(np.zeros(p.n, dtype=np.float32), params, progress=lambda k, fx, xn, gn, st, nls: tr.append((fx, gn, st, nls)) and False,
                    driver=driver)
        traces[driver] = (np.array(tr), res)
        xs[driver] = p.get_x()
        p.close()
    td, tp = traces["device"][0], traces["python"][0]
    assert traces["device"][1].status == traces["python"][1].status == "LBFGSERR_MAXIMUMITERATION"
    assert len(td) == len(tp) == 25
    assert np.abs(td[:, 0] - tp[:, 0]).max() <= 1e-6 * np.abs(tp[:, 0]).max()       # fx per iteration
    assert np.array_equal(td[:, 3], tp[:, 3])                                         # line-search evaluations
    assert np.abs(xs["device"] - xs["python"]).max() <= 1e-4
    assert traces["device"][1].evaluations == traces["python"][1].evaluations


def test_create_rejects_out_of_range_codes(lib):
    codes = synthetic.synthetic_msa_codes(64, 8, 1)
    codes[5, 3] = 21                                   # q = 21 without an ignored gap: valid codes are 0..20
    w = np.ones(64, dtype=np.float32)
    h = ctypes.c_void_p()
    rc = lib.evc_plm_create(ctypes.byref(h), codes.ctypes.data_as(ctypes.c_void_p), 64, 8, 21, -1,
                            w.ctypes.data_as(ctypes.c_void_p), 0)
    assert rc != 0 and b"out of range" in lib.evc_last_error()


# ------------------------------------------------------------------------------------------------
# 8(f3): GPU drop-ins of the reference's in-tree numba twins
# ------------------------------------------------------------------------------------------------
def test_intree_twin_dropins_vs_reference_outputs(engine, golden_dir):
    """evcouplings_b200.alignment.{num_cluster_members, frequencies, pair_frequencies} against the outputs of
    the reference's own functions (alignment.py:1078-1233) stored by tests/golden/make_golden.py"""
    from evcouplings_b200 import alignment as ga
    d = np.load(os.path.join(golden_dir, "intree_twins.npz"))
    for name in ("cfg1", "tie", "odd"):
        codes = d[name + "_codes"].astype(np.int64)
        theta = float(d[name + "_theta"])
        counts = ga.num_cluster_members(codes, theta, engine=engine)
        assert counts.dtype == np.float64 and np.array_equal(counts, d[name + "_counts"].astype(np.float64))
        w = 1.0 / counts
        fi = ga.frequencies(codes, w, 21, engine=engine)
        assert np.abs(fi - d[name + "_fi"]).max() < 2e-6
        fij = ga.pair_frequencies(codes, w, 21, fi, engine=engine)
        L = codes.shape[1]
        iu, ju = np.triu_indices(L, 1)
        assert np.abs(fij[iu, ju] - d[name + "_fij_tri"]).max() < 2e-6
        assert np.abs(fij[ju, iu] - d[name + "_fij_tri"].transpose(0, 2, 1)).max() < 2e-6
        assert np.allclose(fij[3, 3][np.arange(21), np.arange(21)], fi[3])


def test_identities_to_seq_and_set_weights_vs_reference_class(engine, golden_dir):
    """f3: identities_to_seq (alignment.py:1156-1189) and Alignment.set_weights (:899-930) drop-ins.  The
    reference's own numba function and Alignment class are the comparison (their outputs on a seeded alignment
    stored by tests/golden/make_golden.py); the definition (row-wise equality count) always is."""
    import types
    from evcouplings_b200 import alignment as ga
    rng = np.random.default_rng(5)
    for N, L in ((1, 1), (257, 33), (5000, 301)):
        m = rng.integers(0, 21, size=(N, L))
        s = m[rng.integers(0, N)].copy()
        got = ga.identities_to_seq(s, m, engine=engine)
        assert got.dtype == np.float64 and np.array_equal(got, (m == s[None, :]).sum(axis=1).astype(np.float64))
    with pytest.raises(ValueError):
        ga.frequencies(np.full((4, 3), 21), np.ones(4), 21, engine=engine)        # symbol out of range
    d = np.load(os.path.join(golden_dir, "reference_boundary.npz"))
    mapped = d["ali_matrix_mapped"].astype(np.int64)
    # the reference's Alignment.matrix_mapped of synthetic_msa_codes(300, 25, 9) is those codes
    assert np.array_equal(mapped, synthetic.synthetic_msa_codes(300, 25, 9).astype(np.int64))
    ali = types.SimpleNamespace(matrix_mapped=mapped, _frequencies=d["ali_frequencies_unweighted"],
                                _pair_frequencies=None)
    ga.set_weights(ali, 0.8, engine=engine)
    assert np.array_equal(ali.num_cluster_members, d["ali_num_cluster_members"])
    assert np.array_equal(ali.weights, d["ali_weights"])
    # the drop-in resets the cached frequencies like the reference does: the next access is weighted
    assert ali._frequencies is None and ali._pair_frequencies is None
    fw = ga.frequencies(mapped, ali.weights, 21, engine=engine)
    assert np.allclose(fw, d["ali_frequencies"]) and not np.allclose(fw, d["ali_frequencies_unweighted"])
    assert np.array_equal(ga.identities_to_seq(mapped[0], mapped, engine=engine), d["ali_identities_to_first"])


# ------------------------------------------------------------------------------------------------
# the real thing: fit the golden PABP alignment and compare with what plmc itself produced
# ------------------------------------------------------------------------------------------------
def test_pabp_fit_vs_real_plmc_ecs(engine, golden_dir):
    """SURVEY 8(c) check (v).  Same data, weights and regularisation as the plmc run shipped with the
    reference (N=151,496, L=82, q=20, lambda_h=0.01, lambda_J=16.2).  plmc stopped unconverged after 200
    iterations (its own gradient balance is only ~0.97), so this is reported, and gated loosely:
    EC (cn) rms < 0.03 on scores of O(1), and the top-L contacts are essentially the same set."""
    from evcouplings_b200 import lbfgs as lb
    c = np.load(os.path.join(golden_dir, "pabp_codes.npz"))
    g = np.load(os.path.join(golden_dir, "pabp_golden.npz"))
    valid = np.unpackbits(c["valid_packed"])[: int(c["n_total"])].astype(bool)
    codes = c["codes"]
    counts = engine.hamming_counts(codes, msa.identity_threshold_count(0.8, 82))
    assert np.array_equal(counts, c["golden_counts_all"][valid])
    w = (1.0 / counts).astype(np.float32)
    L, q = 82, 20
    prob = engine.plm_problem(codes, w, q, q, 0.01, 16.2)
    fic, fijc = prob.weighted_counts()
    fi, _ = model_io.normalise_frequencies(fic, fijc, float(w.sum()), True)
    x0 = tools.initial_point(fi, float(w.sum()), L, q)
    rows = []
    res = prob.fit(x0, lb.default_params(max_iterations=400, epsilon=1e-4),
                   lambda k, fx, xn, gn, step, nls: rows.append((k, fx, gn / max(1.0, xn))) and False)
    x = prob.get_x()
    fn = prob.fn_scores()
    # objective of plmc's own parameters under our evaluation, for reference
    xg = np.concatenate([g["h"].ravel(), g["J"].ravel()]).astype(np.float32)
    prob.set_x(xg)
    f_golden = prob.evaluate(prob.x)
    prob.close()
    cn = model_io.apc_cn_scores(fn, L)
    gold = g["ec_cn"]
    rms = float(np.sqrt(np.mean((cn - gold) ** 2)))
    iu, ju = np.triu_indices(L, 1)
    far = (ju - iu) >= 6
    top = lambda v: set(np.argsort(-np.where(far, v, -1e9))[:L])
    overlap = len(top(cn) & top(gold)) / float(L)
    corr = float(np.corrcoef(cn, gold)[0, 1])
    dJ = float(np.abs(x[L * q:] - g["J"].ravel()).max())
    print("PABP fit: %s after %d iterations (%d evaluations), fx=%.3f vs plmc parameters fx=%.3f; "
          "EC rms vs plmc %.4f, max %.4f, pearson %.5f, top-L long-range overlap %.3f, max|dJ| %.4f"
          % (res.status, res.iterations, res.evaluations, res.fx, f_golden, rms, np.abs(cn - gold).max(), corr,
             overlap, dJ))
    assert res.fx <= f_golden + 1e-6 * abs(f_golden)      # we are at least as converged as plmc was
    assert rms < 0.03 and corr > 0.995 and overlap >= 0.9


# ------------------------------------------------------------------------------------------------
# 8(f1) EC scoring / 8(f2) energies on the device vs the reference's CouplingsModel outputs
# ------------------------------------------------------------------------------------------------
def _golden_models(golden_dir):
    from evcouplings_b200 import model_ops
    tiny = model_ops.read_model(os.path.join(golden_dir, "tiny.model"))
    g = np.load(os.path.join(golden_dir, "pabp_golden.npz"))
    L, q = 82, 20
    pabp = dict(L=L, q=q, alphabet=str(g["alphabet"]), target_seq=str(g["target_seq"]), index_list=g["index_list"],
                fi=g["fi"], h=g["h"], J=g["J"], fij=np.zeros((L * (L - 1) // 2, q, q), dtype=np.float32))
    return dict(tiny=tiny, pabp=pabp)


def test_model_reader_matches_reference_reader(golden_dir):
    from evcouplings_b200 import model_ops
    m = model_ops.read_model(os.path.join(golden_dir, "tiny.model"))
    r = np.load(os.path.join(golden_dir, "tiny_ref_read.npz"))
    assert np.array_equal(m["J"].astype(np.float64), r["ref_J_tri"]) and np.array_equal(m["h"].astype(np.float64), r["ref_h"])
    assert np.array_equal(m["fij"].astype(np.float64), r["ref_fij_tri"]) and m["alphabet"] == str(r["ref_alphabet"])


def test_ec_table_vs_reference_calculate_ecs(engine, golden_dir):
    """FN (zero-sum gauge), CN (APC), MI raw/APC of CouplingsModel._calculate_ecs (model.py:777-827)"""
    from evcouplings_b200 import model_ops
    ref = np.load(os.path.join(golden_dir, "model_consumers.npz"))
    models = _golden_models(golden_dir)
    for name in ("tiny", "pabp"):
        m = models[name]
        fn_raw, fn_zs, mi = model_ops.pair_scores(m, engine)
        assert np.abs(fn_zs - ref[name + "_fn"]).max() < 2e-6
        tab = model_ops.ec_table(m, engine).sort_values(by=["i", "j"])
        assert np.abs(tab["cn"].values - ref[name + "_cn"]).max() < 5e-6
        assert np.abs(fn_raw - np.sqrt((m["J"].astype(np.float64) ** 2).sum(axis=(1, 2)))).max() < 2e-6
        if name == "tiny":
            assert np.abs(mi - ref["tiny_mi_raw"]).max() < 2e-6
            assert np.abs(tab["mi_apc"].values - ref["tiny_mi_apc"]).max() < 5e-6
    # PABP: the zero-sum CN is the score the reference's CouplingsModel reports (differs from plmc's _ECs.txt)
    g = np.load(os.path.join(golden_dir, "pabp_golden.npz"))
    tab = model_ops.ec_table(models["pabp"], engine).sort_values(by=["i", "j"])
    assert np.abs(tab["cn"].values - g["ref_cn_zero_sum"]).max() < 5e-6


def test_hamiltonians_and_mutants_vs_reference(engine, golden_dir):
    """_hamiltonians / _single_mutant_hamiltonians / _delta_hamiltonian (model.py:25-176) incl. the notebook
    known answers H(target) = 312.19741128035912 and smm(127, 'E') = -7.6052584765675419"""
    from evcouplings_b200 import model_ops
    ref = np.load(os.path.join(golden_dir, "model_consumers.npz"))
    models = _golden_models(golden_dir)
    for name in ("tiny", "pabp"):
        m = models[name]
        H = model_ops.hamiltonians(m, [str(s) for s in ref[name + "_seqs"]], engine)
        assert H.shape == ref[name + "_H"].shape
        assert np.abs(H - ref[name + "_H"]).max() < 2e-4 * max(1.0, np.abs(ref[name + "_H"]).max())
        smm = model_ops.single_mutant_matrix(m, engine)
        assert np.abs(smm - ref[name + "_smm"]).max() < 5e-4
        variants = [[(int(a), b, c) for a, b, c in (s.split(",") for s in str(v).split(";"))]
                    for v in ref[name + "_variants"]]
        dH = model_ops.delta_hamiltonians(m, variants, engine)
        assert np.abs(dH - ref[name + "_dH"]).max() < 5e-4
    Hp = model_ops.hamiltonians(models["pabp"], [models["pabp"]["target_seq"]], engine)
    assert abs(Hp[0, 0] - 312.19741128035912) < 2e-4
    smm = model_ops.single_mutant_matrix(models["pabp"], engine)
    assert abs(smm[127 - 123, "ACDEFGHIKLMNPQRSTVWY".index("E"), 0] - (-7.6052584765675419)) < 5e-4
    # throughput case: many sequences at once
    rng = np.random.default_rng(0)
    big = rng.integers(0, 20, size=(20000, 82)).astype(np.uint8)
    Hb = model_ops.hamiltonians(models["pabp"], big, engine)
    J = po.full_couplings(models["pabp"]["J"].astype(np.float64), 82, 20)
    k = 777
    hj = sum(J[i, j, big[k, i], big[k, j]] for i in range(82) for j in range(i + 1, 82))
    hh = sum(models["pabp"]["h"][i, big[k, i]] for i in range(82))
    assert abs(Hb[k, 1] - hj) < 2e-4 * max(1.0, abs(hj)) and abs(Hb[k, 2] - hh) < 1e-4


def test_plmc_compatible_executable_on_gpu(tmp_path):
    """bin/evcplm-plmc with the argv the reference builds (tools.py:202-262): files written, stderr parses"""
    import subprocess, sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    codes = synthetic.synthetic_msa_codes(200, 40, 1)
    a2m = str(tmp_path / "cfg1.a2m")
    synthetic.write_a2m(a2m, codes)
    ecs, model = str(tmp_path / "o_ECs.txt"), str(tmp_path / "o.model")
    cmd = [sys.executable, os.path.join(root, "bin", "evcplm-plmc"), "-c", ecs, "-o", model, "-f", "seq0", "-g",
           "-m", "25", "-t", "0.2", "-lh", "0.01", "-le", "7.41", "-n", "8", a2m]
    p = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stderr
    it, fields = tools.parse_plmc_log(p.stderr)
    assert fields[1:6] == (200, 200, 40, 40, 1) and len(it) == 25
    m = po.read_model(model)
    assert (m["L"], m["q"], m["num_iter"]) == (40, 20, 25) and abs(m["lambda_J"] - 7.41) < 1e-5
    assert len(open(ecs).read().strip().split("\n")) == 780
