"""
Drop-in boundary on the GPU (-m gpu): the calls the reference's OWN couplings protocol and its OWN run_plmc make
into our boundary, recorded with the unmodified reference (tests/golden/make_golden.py, reference_boundary),
are replayed over the CUDA engine, and what we return and write is checked against what the reference's stage
code and readers made of it (see tests/reference_golden.py).

  1. primary plug point: evcouplings.couplings.protocol.run(protocol="standard") (protocol.py:363-429 ->
     infer_plmc :56-257) calling evcouplings_b200.run_plmc (CudaEngine, default tcgen05 path);
  2. secondary plug point: the argv the reference's run_plmc (tools.py:126-307) builds drives bin/evcplm-plmc,
     i.e. the real executable with the real engine, and its stderr is parsed as the reference parses it.
"""
import os
import subprocess

import numpy as np
import pytest

import reference_golden as rg

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def ref():
    return rg.load()


@pytest.fixture(scope="module")
def engine():
    from evcouplings_b200.engine import CudaEngine
    return CudaEngine()


@pytest.mark.parametrize("ignore_gaps", [True, False])
def test_reference_standard_protocol_over_cuda_engine(ref, engine, tmp_path, ignore_gaps):
    """BASELINE configs[0] (N=200, L=40) through the reference's stage driver's call, numerics on the B200."""
    from evcouplings_b200 import synthetic, tools
    from cpu_engine import OracleEngine
    from oracle import plm_oracle as po
    meta, arr = ref
    name = "standard_it40_ig%d" % int(ignore_gaps)
    rec = meta[name]
    N, L = 200, 40
    codes = synthetic.synthetic_msa_codes(N, L, 1)
    a2m = str(tmp_path / "cfg1.a2m")
    synthetic.write_a2m(a2m, codes)
    args = [rg.subst(a, tmp_path) for a in rec["args"]]
    kwargs = {k: rg.subst(v, tmp_path) for k, v in rec["kwargs"].items()}
    q_eff = 20 if ignore_gaps else 21
    lam_J = 0.01 * (q_eff - 1) * (L - 1)
    assert abs(kwargs["lambda_J"] - lam_J) < 1e-12           # protocol.py:157-179
    assert kwargs["iterations"] == 40
    res, run = tools.run_plmc(*args, engine=engine, return_run=True, num_gpus=1, **kwargs)
    rg.check_result_as_protocol_reads_it(meta, rec, res, run)
    assert rec["outcfg"]["num_sites"] == L and rec["outcfg"]["num_valid_sequences"] == N
    # the reference's readers on the files the CUDA engine wrote
    m = rg.check_model_as_reference_reads_it(rec, res.param_file, run)
    assert m["L"] == L and m["q"] == q_eff and m["n_valid"] == N
    J = m["J"].astype(np.float64)
    ecs = rg.check_ecs_as_reference_reads_them(arr, name, res.couplings_file, J, L)
    assert np.abs(ecs["cn"] - po.cn_scores(J, L)).max() < 2e-6
    it_own = rg.check_log_as_reference_parses_it(rec, run.log, 40)
    assert rec["log_fields"][-1] == "LBFGSERR_MAXIMUMITERATION"
    # same host logic over the float64 oracle backend from the same start, same iteration cap: the objective the
    # CUDA engine reached is the oracle's to fp32 noise (device L-BFGS = the same algorithm)
    r2, run2 = tools.run_plmc(a2m, str(tmp_path / "c_ECs.txt"), str(tmp_path / "c.model"), focus_seq="seq0/1-40",
                              theta=0.8, ignore_gaps=ignore_gaps, iterations=40, lambda_h=0.01, lambda_J=lam_J,
                              engine=OracleEngine(), return_run=True)
    f1 = it_own["fx"].astype(float).values
    f2 = r2.iteration_table["fx"].astype(float).values
    assert np.abs(f1 - f2).max() <= 2e-5 * np.abs(f2).max()
    cn2 = np.loadtxt(str(tmp_path / "c_ECs.txt"), usecols=5)
    assert np.sqrt(np.mean((ecs["cn"] - cn2) ** 2)) < 2e-3
    # and so are the ECs the reference read from the oracle run when the fixture was recorded
    assert np.sqrt(np.mean((ecs["cn"] - arr[name + "_ecs_cn"]) ** 2)) < 2e-3


def test_unmodified_reference_run_plmc_over_real_executable(ref, tmp_path):
    """The reference's run_plmc argv (subprocess + stderr scraping) over bin/evcplm-plmc with the CUDA engine."""
    from evcouplings_b200 import synthetic, tools
    from oracle import plm_oracle as po
    meta, _ = ref
    rec = meta["cli_gpu"]
    codes = synthetic.synthetic_msa_codes(300, 24, 3)
    synthetic.write_a2m(str(tmp_path / "in.a2m"), codes)
    argv = [rg.subst(a, tmp_path) for a in rec["argv"]]
    env = dict(os.environ, EVC_NUM_GPUS="1")
    p = subprocess.run([os.path.join(ROOT, "bin", "evcplm-plmc")] + argv, capture_output=True, text=True, env=env)
    assert p.returncode == 0, p.stderr
    it, fields = tools.parse_plmc_log(p.stderr)
    want = rec["result"]
    ecs, model = rg.subst(want["couplings_file"], tmp_path), rg.subst(want["param_file"], tmp_path)
    assert os.path.getsize(ecs) > 0 and os.path.getsize(model) > 0
    got = dict(zip(["focus_seq_index", "num_valid_seqs", "num_total_seqs", "num_valid_sites", "num_total_sites",
                    "region_start", "effective_samples", "optimization_status"], fields))
    assert abs(got.pop("effective_samples") - want["effective_samples"]) < 0.06
    assert got == {k: v for k, v in want.items() if k in got}
    assert got["num_valid_seqs"] == 300 and got["num_total_seqs"] == 300 and got["num_valid_sites"] == 24
    assert got["focus_seq_index"] == 1 and got["region_start"] == 1
    assert got["optimization_status"] == "LBFGSERR_MAXIMUMITERATION"
    assert list(it.columns) == rec["iter_columns"] and len(it) == rec["iter_len"] == 20
    m = po.read_model(model)
    assert (m["L"], m["q"], m["num_iter"]) == (24, 20, 20) and abs(m["lambda_J"] - 4.0) < 1e-6
    assert abs(fields[6] - m["n_eff"]) < 0.06
    fx = it["fx"].astype(float).values
    assert np.all(np.diff(fx) <= 1e-6 * np.abs(fx[:-1]))          # monotone descent
