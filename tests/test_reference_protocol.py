"""
Drop-in boundary test (CPU): the calls the reference's OWN couplings protocol
(evcouplings/couplings/protocol.py:363-429 ``standard`` -> ``infer_plmc`` :56-257, and ``complex``) makes into
``run_plmc``, and the argv its own ``run_plmc`` (tools.py:126-307) builds for a plmc executable, are replayed
from the fixture recorded with the unmodified reference (tests/golden/make_golden.py, reference_boundary);
what we return and write is checked against what the reference's stage code and readers (CouplingsModel
model.py:317-400, read_raw_ec_file pairs.py:34-65, parse_plmc_log tools.py:20-108) made of it.  The numerical
engine injected here is the test-only oracle engine; the same host code runs over the CUDA engine in
tests/test_gpu_reference_protocol.py.
"""
import gzip
import os
import subprocess
import sys

import numpy as np
import pytest

import reference_golden as rg


@pytest.fixture(scope="module")
def ref():
    return rg.load()


@pytest.mark.parametrize("ignore_gaps", [True, False])
def test_reference_standard_protocol_over_our_run_plmc(ref, tmp_path, ignore_gaps):
    from evcouplings_b200 import synthetic, tools
    from cpu_engine import OracleEngine
    from oracle import plm_oracle as po
    meta, arr = ref
    name = "standard_it30_ig%d" % int(ignore_gaps)
    rec = meta[name]
    N, L = 200, 40                      # BASELINE configs[0]
    codes = synthetic.synthetic_msa_codes(N, L, 1)
    synthetic.write_a2m(str(tmp_path / "cfg1.a2m"), codes)
    args = [rg.subst(a, tmp_path) for a in rec["args"]]
    kwargs = {k: rg.subst(v, tmp_path) for k, v in rec["kwargs"].items()}

    # the protocol hands us lambda_J already scaled by (q_eff - 1) * (L - 1)   (protocol.py:157-179)
    q_eff = 20 if ignore_gaps else 21
    assert abs(kwargs["lambda_J"] - 0.01 * (q_eff - 1) * (L - 1)) < 1e-12
    assert kwargs["focus_seq"] == "seq0/1-40" and kwargs["theta"] == 0.8 and kwargs["iterations"] == 30
    res, run = tools.run_plmc(*args, engine=OracleEngine(), return_run=True, **kwargs)

    # stage outputs the rest of the pipeline consumes
    rg.check_result_as_protocol_reads_it(meta, rec, res, run)
    assert rec["outcfg"]["num_sites"] == L and rec["outcfg"]["num_valid_sequences"] == N
    res.iteration_table.to_csv(str(tmp_path / "job_iteration_table.csv"))

    # the reference's own readers on our files
    m = rg.check_model_as_reference_reads_it(rec, res.param_file, run)
    assert m["alphabet"] == ("ACDEFGHIKLMNPQRSTVWY" if ignore_gaps else "-ACDEFGHIKLMNPQRSTVWY")
    assert abs(m["theta"] - 0.2) < 1e-7 and abs(m["n_eff"] - run.n_eff) < 1e-2
    assert m["target_seq"] == run.alignment.target_seq
    # same oracle fit as when the reference read it
    J = m["J"].astype(np.float64)
    assert np.abs(m["h"] - arr[name + "_h"]).max() < 1e-5
    Jt = J.reshape(-1)
    assert np.abs(Jt[arr[name + "_J_idx"]] - arr[name + "_J"]).max() < 1e-5
    sums = np.array([Jt.sum(), np.abs(Jt).sum(), (Jt * Jt).sum()])
    assert np.all(np.abs(sums - arr[name + "_J_sums"]) <= 1e-5 * np.abs(arr[name + "_J_sums"]) + 1e-6)
    ecs = rg.check_ecs_as_reference_reads_them(arr, name, res.couplings_file, J, L)
    assert np.abs(ecs["cn"] - po.cn_scores(J, L)).max() < 1e-6
    assert np.abs(ecs["cn"] - arr[name + "_ecs_cn"]).max() < 1e-5
    # the reference's own log parser on our log agrees with ours
    it = rg.check_log_as_reference_parses_it(rec, run.log, 30)
    fx_ref = np.array([float(r[3]) for r in rec["iter_rows"]])
    assert np.abs(it["fx"].astype(float).values - fx_ref).max() <= 1e-5 * np.abs(fx_ref).max()


def test_reference_parse_of_realistic_failure_modes(ref):
    """mandatory log lines: the reference raises KeyError without them (tools.py:97-99); ours too."""
    from evcouplings_b200 import tools
    meta, _ = ref
    assert meta["parse_failure"] == "KeyError"
    with pytest.raises(KeyError):
        tools.parse_plmc_log("nothing useful")


def test_product_ingest_on_real_pabp_alignment(golden_dir, tmp_path):
    """product ingest on a seeded sample of the real A2M shipped with the reference (its focus record and 1,000
    others, 100 of them invalid) == the matching rows of the golden fixture (which the oracle's per-character
    restatement produced and plmc's own header / weights confirm: 151,496 valid + 545 invalid)."""
    from evcouplings_b200 import msa
    path = tmp_path / "PABP_YEAST_sample.a2m"
    with gzip.open(os.path.join(golden_dir, "pabp_sample.a2m.gz"), "rb") as f:
        path.write_bytes(f.read())
    rows = np.load(os.path.join(golden_dir, "pabp_sample_rows.npy"))
    ali = msa.load_alignment(str(path), focus="PABP_YEAST", ignore_gaps=True)
    c = np.load(os.path.join(golden_dir, "pabp_codes.npz"))
    valid_all = np.unpackbits(c["valid_packed"])[: int(c["n_total"])].astype(bool)
    valid = valid_all[rows]
    codes = c["codes"][(np.cumsum(valid_all) - 1)[rows[valid]]]
    assert np.array_equal(ali.valid, valid) and np.array_equal(ali.codes, codes)
    assert ali.target_seq == str(c["target_seq"]) and np.array_equal(ali.index_list, c["index_list"])
    assert (ali.n_valid, ali.n_total - ali.n_valid, ali.region_start, ali.num_total_sites) == \
        (int(valid.sum()), int((~valid).sum()), 115, 96)
    assert (~valid).sum() == 100


def test_unmodified_reference_run_plmc_over_plmc_compatible_cli(ref, tmp_path):
    """Secondary plug point: the argv the reference's OWN run_plmc (tools.py:126-307) builds drives our
    plmc-compatible executable; its stderr, parsed as the reference parses it, gives the reference's recorded
    PlmcResult.  The wrapper used here injects the test-only oracle engine; bin/evcplm-plmc is the same
    entry point with the CUDA engine."""
    import stat
    from evcouplings_b200 import synthetic, tools
    from oracle import plm_oracle as po
    meta, _ = ref
    rec = meta["cli_cpu"]
    codes = synthetic.synthetic_msa_codes(150, 16, 3)
    synthetic.write_a2m(str(tmp_path / "in.a2m"), codes)
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    wrapper = tmp_path / "plmc_test_wrapper"
    wrapper.write_text(
        "#!%s\nimport sys\nsys.path.insert(0, %r); sys.path.insert(0, %r)\n"
        "from cpu_engine import OracleEngine\nfrom evcouplings_b200.plmc_cli import main\n"
        "sys.exit(main(engine=OracleEngine()))\n" % (sys.executable, root, os.path.join(root, "tests")))
    wrapper.chmod(wrapper.stat().st_mode | stat.S_IEXEC)
    argv = [rg.subst(a, tmp_path) for a in rec["argv"]]
    p = subprocess.run([str(wrapper)] + argv, capture_output=True, text=True)
    assert p.returncode == 0, p.stderr
    it, fields = tools.parse_plmc_log(p.stderr)
    want = rec["result"]
    ecs, model = rg.subst(want["couplings_file"], tmp_path), rg.subst(want["param_file"], tmp_path)
    assert os.path.getsize(ecs) > 0 and os.path.getsize(model) > 0
    got = dict(zip(["focus_seq_index", "num_valid_seqs", "num_total_seqs", "num_valid_sites", "num_total_sites",
                    "region_start", "effective_samples", "optimization_status"], fields))
    assert abs(got.pop("effective_samples") - want["effective_samples"]) < 0.06
    assert got == {k: v for k, v in want.items() if k in got}
    assert got["num_valid_seqs"] == 150 and got["num_total_seqs"] == 150 and got["num_valid_sites"] == 16
    assert got["focus_seq_index"] == 1 and got["region_start"] == 1
    assert got["optimization_status"] == "LBFGSERR_MAXIMUMITERATION"
    assert list(it.columns) == rec["iter_columns"] and len(it) == rec["iter_len"] == 12
    m = po.read_model(model)
    assert (m["L"], m["q"], m["num_iter"]) == (16, 20, 12) and abs(m["theta"] - 0.2) < 1e-6
    assert abs(m["lambda_J"] - 2.5) < 1e-6 and abs(fields[6] - m["n_eff"]) < 0.06
    assert len(open(ecs).read().strip().split("\n")) == 16 * 15 // 2


def test_plmc_cli_argument_handling():
    from evcouplings_b200 import plmc_cli
    ali, o = plmc_cli.parse_args(["-c", "e.txt", "-o", "m.model", "-f", "SEQ", "-g", "-m", "100", "-t", "0.2",
                                  "-lh", "0.01", "-le", "16.2", "-n", "4", "in.a2m"])
    assert ali == "in.a2m" and o["couplings_file"] == "e.txt" and o["param_file"] == "m.model"
    assert o["focus_seq"] == "SEQ" and o["ignore_gaps"] and o["iterations"] == 100
    assert abs(o["theta"] - 0.8) < 1e-12 and o["lambda_h"] == 0.01 and o["lambda_J"] == 16.2 and o["cpu"] == "4"
    import io
    for bad in (["-c"], ["in.a2m"], ["-c", "e", "a", "b"], ["-zz", "1", "-c", "e", "a"]):
        assert plmc_cli.main(bad, stderr=io.StringIO()) == 2
    err = io.StringIO()
    assert plmc_cli.main(["-c", "/tmp/e.txt", "/nonexistent/file.a2m"], stderr=err) == 1 and "ResourceError" in err.getvalue()


def test_reference_complex_protocol_over_our_run_plmc(ref, tmp_path):
    """BASELINE configs[4] flavour (EVcomplex concatenated two-chain alignment): the call the reference's
    ``complex`` protocol (protocol.py:480-594; same infer_plmc -> run_plmc boundary, two segments, inter-chain
    EC table) makes is replayed over our run_plmc.  Small shapes here (2 x 12 sites); the engine itself is
    parity- and bench-tested at L=800 on the GPU."""
    from evcouplings_b200 import synthetic, tools
    from cpu_engine import OracleEngine
    meta, arr = ref
    rec = meta["complex"]
    N, L1, L2 = 160, 12, 12
    L = L1 + L2
    codes = synthetic.synthetic_msa_codes(N, L, 8)
    synthetic.write_a2m(str(tmp_path / "complex.a2m"), codes, focus_name="A_B")   # "A_B/1-24" like complex/alignment.py:85-92
    args = [rg.subst(a, tmp_path) for a in rec["args"]]
    kwargs = {k: rg.subst(v, tmp_path) for k, v in rec["kwargs"].items()}
    assert kwargs["focus_seq"] == "A_B/1-%d" % L
    res, run = tools.run_plmc(*args, engine=OracleEngine(), return_run=True, **kwargs)
    rg.check_result_as_protocol_reads_it(meta, rec, res, run)
    assert rec["outcfg"]["num_sites"] == L and rec["outcfg"]["num_valid_sequences"] == N
    m = rg.check_model_as_reference_reads_it(rec, res.param_file, run)
    assert m["L"] == L and m["q"] == 20
    ecs = rg.check_ecs_as_reference_reads_them(arr, "complex", res.couplings_file, m["J"], L)
    # the reference's inter-chain table: the raw ECs with i in segment A_1 and j in segment B_1
    inter = int(((ecs["i"] <= L1) & (ecs["j"] > L1)).sum())
    assert inter == rec["inter_ecs"]["rows"] == L1 * L2
    assert rec["inter_ecs"]["segment_i"] == ["A_1"] and rec["inter_ecs"]["segment_j"] == ["B_1"]
