"""Mean-field DCA on the GPU (csrc/mean_field.cu through evcouplings_b200.mean_field) against the float64 oracle
(tests/mf_oracle.py) and the reference's own outputs (tests/golden/mean_field_golden.npz)."""
import ctypes
import io
import json
import os

import numpy as np
import pytest

import mf_oracle as mo
from test_mean_field_host import GOLDEN, case_codes, load_golden, reference_ec_text

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def engine():
    from evcouplings_b200.engine import CudaEngine
    return CudaEngine()


def _dev(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def test_weighted_counts_f64(engine):
    import torch
    from evcouplings_b200 import _lib, synthetic
    codes = synthetic.synthetic_msa_codes(3000, 30, 5)
    w = 1.0 / np.random.default_rng(1).integers(1, 40, size=len(codes)).astype(np.float64)
    q, L = 21, 30
    F = torch.empty((L * q, L * q), dtype=torch.float64, device="cuda")
    d_codes, d_w = _dev(codes), _dev(w)           # kept alive until the kernel has run
    _lib.check(engine.lib.evc_mf_weighted_counts_f64(engine.ptr(d_codes), engine.ptr(d_w), len(codes), L, q,
                                                     float(w.sum()), engine.ptr(F), engine.stream()), "counts")
    fi, fij = mo.frequencies(codes, w, q)
    ref = fij.transpose(0, 2, 1, 3).reshape(L * q, L * q)
    got = F.cpu().numpy()
    nz = ref != 0
    assert np.all(got[~nz] == 0)
    assert np.max(np.abs(got[nz] - ref[nz]) / ref[nz]) <= 1e-7


def _spd(n, cond, seed):
    """Q diag(geomspace(1, 1/cond)) Q^T on the device (test input generation only)."""
    import torch
    g = torch.Generator(device="cuda").manual_seed(seed)
    Q, _ = torch.linalg.qr(torch.randn((n, n), dtype=torch.float64, device="cuda", generator=g))
    ev = torch.logspace(0.0, -np.log10(cond), n, dtype=torch.float64, device="cuda")
    A = (Q * ev) @ Q.T
    return (A + A.T) / 2


@pytest.mark.parametrize("n", [1640, 4000, 10000])
def test_spd_inverse(engine, n):
    import torch
    from evcouplings_b200 import _lib
    A = _spd(n, 1e4, n)
    X = A.clone()
    work = torch.empty_like(X)
    info = ctypes.c_int32(-1)
    _lib.check(engine.lib.evc_spd_inverse_f64(engine.ptr(X), n, engine.ptr(work), ctypes.byref(info),
                                              engine.stream()), "evc_spd_inverse_f64")
    assert info.value == 0
    err = float((A @ X - torch.eye(n, dtype=torch.float64, device="cuda")).abs().max())
    print("n=%d  max|AX - I| = %.2e" % (n, err))
    assert err <= 1e-9


def test_spd_inverse_rejects_indefinite(engine):
    import torch
    from evcouplings_b200 import _lib
    n = 300
    A = _spd(n, 10.0, 3)
    A[150, 150] = -5.0                            # not positive definite
    dA = A.clone()
    work = torch.empty_like(dA)
    info = ctypes.c_int32(0)
    rc = engine.lib.evc_spd_inverse_f64(engine.ptr(dA), n, engine.ptr(work), ctypes.byref(info), engine.stream())
    assert rc == _lib.EVC_NOT_SPD and 1 <= info.value <= n
    assert ("column %d" % info.value).encode() in engine.lib.evc_last_error()
    torch.cuda.synchronize()                      # the device is still usable
    assert float(torch.ones(4, device="cuda").sum()) == 4.0


def test_di_kernel_matches_oracle(engine):
    import torch
    from evcouplings_b200 import _lib
    g = load_golden()
    codes, alphabet, theta, pc, _ = case_codes(g, "pabp")
    w = g["pabp_weights"]
    o = mo.fit(codes, w, len(alphabet), pc)
    L, q = o["h"].shape
    J_tri = mo.tri(o["J"])
    npairs = len(J_tri)
    di = torch.empty(npairs, dtype=torch.float64, device="cuda")
    it = torch.empty(npairs, dtype=torch.int32, device="cuda")
    d_J, d_rfi = _dev(J_tri), _dev(o["rfi"])      # kept alive until the kernel has run
    _lib.check(engine.lib.evc_mf_di_scores(engine.ptr(d_J), engine.ptr(d_rfi), L, q, engine.ptr(di), engine.ptr(it),
                                           engine.stream()), "evc_mf_di_scores")
    diff_iters = int((it.cpu().numpy() != mo.tri(o["di_iters"])).sum())
    print("DI: max abs err %.2e; pairs with a different iteration count: %d of %d"
          % (np.abs(di.cpu().numpy() - mo.tri(o["di"])).max(), diff_iters, npairs))
    assert np.abs(di.cpu().numpy() - mo.tri(o["di"])).max() <= 1e-9


def _top(scores, L, tol):
    """Top-L pair indices by score; pairs tied within tol with the L-th score are interchangeable."""
    order = np.argsort(-scores, kind="stable")
    cut = scores[order[L - 1]]
    return set(order[:L]), set(np.nonzero(np.abs(scores - cut) <= tol)[0])


def _same_top(a, b, L, tol=2e-6):
    ta, tie_a = _top(a, L, tol)
    tb, tie_b = _top(b, L, tol)
    return (ta ^ tb) <= (tie_a | tie_b)


@pytest.mark.parametrize("case", ["pabp", "syn", "rna"])
def test_end_to_end_against_reference(engine, case, tmp_path):
    from evcouplings_b200.mean_field import fit_codes
    from evcouplings_b200 import model_ops
    g = load_golden()
    codes, alphabet, theta, pc, index_list = case_codes(g, case)
    m = fit_codes(codes, alphabet, index_list, theta, pc, engine)
    p = case + "_"
    assert m.N_valid == int(g[p + "N_valid"]) and np.array_equal(m.index_list, g[p + "index_list"])
    assert np.allclose(m.weights, g[p + "weights"], rtol=0, atol=0)
    assert abs(m.N_eff - float(g[p + "N_eff"])) <= 1e-9
    jmax = float(g[p + "J_absmax"])
    J = m.J_tri.reshape(-1)[g[p + "J_sample_idx"]]
    assert np.abs(J - g[p + "J_sample"]).max() <= 1e-5 * jmax
    assert np.abs(m.h_i - g[p + "h_i"]).max() <= 1e-5 * jmax
    assert np.abs(m.regularized_f_i - g[p + "regularized_f_i"]).max() <= 1e-9
    iu, ju = np.triu_indices(m.L, 1)
    for name, got in (("di", m.di_scores), ("mi_raw", m.mi_scores_raw), ("mi_apc", m.mi_scores_apc),
                      ("cn", m.cn_scores)):
        err = np.abs(got[iu, ju] - g[p + name]).max()
        print("%s %s max abs err %.2e" % (case, name, err))
        assert err <= 2e-6, (name, err)
    assert _same_top(m.di_scores[iu, ju], g[p + "di"], m.L)
    assert _same_top(m.cn_scores[iu, ju], g[p + "cn"], m.L)
    ec = tmp_path / "ECs.txt"
    m.to_raw_ec_file(str(ec))
    got = np.loadtxt(str(ec), dtype=str)
    ref = np.loadtxt(io.StringIO(reference_ec_text(g, case)), dtype=str)
    assert np.array_equal(got[:, :4], ref[:, :4])
    assert np.abs(got[:, 4:].astype(float) - ref[:, 4:].astype(float)).max() <= 2e-6 + 1e-6
    # the model file reads back as the reference's reader read its own file
    mf = tmp_path / "mf.model"
    m.to_file(str(mf))
    r = model_ops.read_model(str(mf))
    hdr = json.loads(str(g[p + "file_header"]))
    assert (r["L"], r["q"], r["n_valid"], r["n_invalid"]) == (hdr["L"], hdr["q"], hdr["N_valid"], hdr["N_invalid"])
    assert abs(-r["lambda_h"] - hdr["pseudo_count"]) <= 1e-7 and r["alphabet"] == hdr["alphabet"]
    assert r["target_seq"] == hdr["target_seq"] and np.array_equal(r["index_list"], g[p + "file_index_list"])
    assert np.allclose(r["weights"], g[p + "file_weights"], rtol=1e-6)
    assert np.abs(r["J"].reshape(-1)[g[p + "J_sample_idx"]] - g[p + "file_J_sample"]).max() <= 1e-5 * jmax
    assert np.abs(r["fij"].reshape(-1)[g[p + "J_sample_idx"]] - g[p + "file_fij_sample"]).max() <= 1e-6
    assert np.abs(r["fi"] - g[p + "file_f_i"]).max() <= 1e-6


def test_duck_typed_alignment_object(engine):
    """MeanFieldDCA takes any object with the reference Alignment's matrix / ids / alphabet."""
    from evcouplings_b200 import MeanFieldDCA
    g = load_golden()
    text = str(g["syn_alignment_text"])
    recs = [r.split("\n", 1) for r in text.split(">")[1:]]

    class Ali(object):
        ids = [r[0] for r in recs]
        matrix = np.array([list(r[1].strip()) for r in recs])
        alphabet = str(g["syn_alphabet"])
        _match_gap, _insert_gap = "-", "."

    theta, pc = g["syn_params"]
    m = MeanFieldDCA(Ali(), engine=engine).fit(theta=theta, pseudo_count=pc)
    iu, ju = np.triu_indices(m.L, 1)
    assert np.abs(m.di_scores[iu, ju] - g["syn_di"]).max() <= 2e-6


def test_large_synthetic_against_oracle(engine):
    """N = 50,000, L = 200 (n = 4,000) against the float64 oracle (DI on a sample of pairs)."""
    from evcouplings_b200 import msa, synthetic
    from evcouplings_b200.mean_field import fit_codes
    codes = synthetic.synthetic_msa_codes(50000, 200, 2)
    L, q, pc = 200, 21, 0.5
    m = fit_codes(codes, msa.ALPHABET_PROTEIN, np.arange(1, L + 1), 0.8, pc, engine)
    o = mo.fit(codes, m.weights, q, pc, di=False)
    jmax = np.abs(o["J"]).max()
    assert np.abs(m.J_tri - mo.tri(o["J"])).max() <= 1e-5 * jmax
    assert np.abs(m.h_i - o["h"]).max() <= 1e-5 * jmax
    iu, ju = np.triu_indices(L, 1)
    for name, got in (("mi_raw", m.mi_scores_raw), ("mi_apc", m.mi_scores_apc), ("cn", m.cn_scores)):
        assert np.abs(got[iu, ju] - o[name][iu, ju]).max() <= 2e-6, name
    rng = np.random.default_rng(0)
    for p in rng.choice(len(iu), size=300, replace=False):
        i, j = iu[p], ju[p]
        E = np.exp(o["J"][i, j])
        u, v, _ = mo.two_site(E, o["rfi"][i], o["rfi"][j])
        P = E * np.outer(u, v)
        P /= P.sum()
        di = np.sum(P * np.log((P + mo.TINY) / (np.outer(o["rfi"][i], o["rfi"][j]) + mo.TINY)))
        assert abs(m.di_scores[i, j] - di) <= 2e-6
    assert os.path.exists(GOLDEN)
