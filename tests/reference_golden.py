"""
What the reference (EVcouplings) does at our boundary, replayed from tests/golden/reference_boundary.npz
(written by tests/golden/make_golden.py with the unmodified reference): the arguments its couplings protocol
passes to run_plmc, the argv its run_plmc builds for a plmc executable, and what its stage code, model reader,
EC reader and log parser made of what our run_plmc returned and wrote.
"""
import json
import os

import numpy as np

from oracle import plm_oracle as po

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_boundary.npz")


def load():
    d = np.load(GOLDEN)
    return json.loads(str(d["meta"])), d


def subst(v, tmp):
    """Recorded temporary paths are stored as {tmp}."""
    return v.replace("{tmp}", str(tmp)) if isinstance(v, str) else v


def check_result_as_protocol_reads_it(meta, rec, res, run):
    """protocol.py infer_plmc: PlmcResult._asdict(), iteration_table.to_csv, outcfg from four result fields."""
    assert list(res._fields) == meta["plmc_result_fields"]
    d = res._asdict()
    assert hasattr(d["iteration_table"], "to_csv")
    out = rec["outcfg"]
    assert (res.num_valid_sites, res.num_valid_seqs, res.region_start) == \
        (out["num_sites"], out["num_valid_sequences"], out["region_start"])
    assert abs(res.effective_samples - out["effective_sequences"]) < 0.06
    assert abs(res.effective_samples - run.n_eff) < 0.06
    for path in (res.couplings_file, res.param_file):
        assert os.path.getsize(path) > 0


def check_model_as_reference_reads_it(rec, path, run):
    """Header fields as the reference's CouplingsModel read them; h / J are the fitted x exactly (our reader
    and the reference's reader agree byte for byte: test_tiny_model_layout_vs_reference_reader)."""
    m = po.read_model(path)
    g = rec["model"]
    L, q = g["L"], g["num_symbols"]
    assert (m["L"], m["q"], m["n_valid"], m["alphabet"], m["target_seq"]) == \
        (L, q, g["N_valid"], g["alphabet"], g["target_seq"])
    assert np.float32(m["theta"]) == np.float32(g["theta"]) and abs(m["n_eff"] - g["N_eff"]) < 1e-2
    h = run.x[:L * q].reshape(L, q)
    J = run.x[L * q:].reshape(-1, q, q)
    assert np.array_equal(m["h"], h.astype(np.float32)) and np.array_equal(m["J"], J.astype(np.float32))
    return m


def read_ecs(path):
    """The raw EC file's columns as the reference's read_raw_ec_file reads them (i A_i j A_j fn cn)."""
    t = np.loadtxt(path, dtype=str, ndmin=2)
    return dict(i=t[:, 0].astype(int), A_i="".join(t[:, 1]), j=t[:, 2].astype(int), A_j="".join(t[:, 3]),
                cn=t[:, 5].astype(np.float64))


def check_ecs_as_reference_reads_them(arr, name, path, J, L):
    ecs = read_ecs(path)
    assert len(ecs["i"]) == L * (L - 1) // 2
    assert np.array_equal(ecs["i"], arr[name + "_ecs_ij"][0]) and np.array_equal(ecs["j"], arr[name + "_ecs_ij"][1])
    assert [ecs["A_i"], ecs["A_j"]] == [str(s) for s in arr[name + "_ecs_A"]]
    return ecs


def check_log_as_reference_parses_it(rec, log, iterations):
    """Our parser reproduces the reference parser's reading of the recorded log exactly; the fresh log has the
    same fields, columns and length."""
    from evcouplings_b200 import tools
    it_g, f_g = tools.parse_plmc_log(rec["log"])
    assert list(f_g) == rec["log_fields"]
    assert list(it_g.columns) == rec["iter_columns"] and it_g.values.tolist() == rec["iter_rows"]
    it, f = tools.parse_plmc_log(log)
    assert list(it.columns) == rec["iter_columns"] and len(it) == len(rec["iter_rows"]) == iterations
    assert list(f[:6]) == rec["log_fields"][:6] and f[7] == rec["log_fields"][7]
    assert abs(f[6] - rec["log_fields"][6]) < 0.06
    return it
