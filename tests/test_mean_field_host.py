"""Mean-field DCA host logic (no GPU): the float64 oracle against the reference's outputs on three alignments
(tests/golden/mean_field_golden.npz, written by tests/golden/make_mean_field_golden.py), site and sequence
selection, the EC file format and the mean-field .model header."""
import gzip
import json
import os

import numpy as np
import pytest

import mf_oracle as mo

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "mean_field_golden.npz")
_cache = {}


def load_golden():
    if "g" not in _cache:
        _cache["g"] = dict(np.load(GOLDEN))
    return _cache["g"]


def alignment_text(g, case):
    if case == "pabp":
        with gzip.open(os.path.join(os.path.dirname(GOLDEN), "pabp_sample.a2m.gz"), "rt") as f:
            return f.read()
    return str(g[case + "_alignment_text"])


def parse_text(text):
    ids, seqs = [], []
    for rec in text.split(">")[1:]:
        head, _, body = rec.partition("\n")
        ids.append(head.strip())
        seqs.append("".join(body.split()))
    raw = np.frombuffer("".join(seqs).encode("ascii"), dtype=np.uint8).reshape(len(seqs), -1)
    return ids, raw


def reference_ec_text(g, case):
    """The reference's raw EC file: stored as written (syn, rna), or, for PABP, the same format
    (``i A_i j A_j mi_raw mi_apc di cn``, six decimals) over the reference's stored scores."""
    p = case + "_"
    if p + "ec_text" in g:
        return str(g[p + "ec_text"])
    idx, ts = g[p + "index_list"], str(g[p + "target_seq"])
    iu, ju = np.triu_indices(len(idx), 1)
    cols = [g[p + k] for k in ("mi_raw", "mi_apc", "di", "cn")]
    return "".join(" ".join([str(idx[i]), ts[i], str(idx[j]), ts[j]] + ["{0:.6f}".format(c[k]) for c in cols]) + "\n"
                   for k, (i, j) in enumerate(zip(iu, ju)))


def case_codes(g, case):
    from evcouplings_b200.mean_field import select_alignment
    ids, raw = parse_text(alignment_text(g, case))
    alphabet = str(g[case + "_alphabet"])
    theta, pc = (float(v) for v in g[case + "_params"])
    codes, index_list, _ = select_alignment(raw, ids, alphabet)
    return codes, alphabet, theta, pc, index_list


@pytest.mark.parametrize("case", ["pabp", "syn", "rna"])
def test_oracle_reproduces_reference(case):
    g = load_golden()
    p = case + "_"
    codes, alphabet, theta, pc, index_list = case_codes(g, case)
    assert len(codes) == int(g[p + "N_valid"])
    assert np.array_equal(index_list, g[p + "index_list"])
    w = mo.cluster_weights(codes, theta)
    assert np.array_equal(w, g[p + "weights"])
    o = mo.fit(codes, w, len(alphabet), pc)
    assert abs(o["n_eff"] - float(g[p + "N_eff"])) <= 1e-9
    jmax = float(g[p + "J_absmax"])
    assert abs(np.abs(mo.tri(o["J"])).max() - jmax) <= 1e-9 * jmax
    assert np.abs(mo.tri(o["J"]).reshape(-1)[g[p + "J_sample_idx"]] - g[p + "J_sample"]).max() <= 1e-9 * jmax
    assert np.abs(o["h"] - g[p + "h_i"]).max() <= 1e-9 * jmax
    assert np.abs(o["rfi"] - g[p + "regularized_f_i"]).max() <= 1e-12
    for name in ("di", "mi_raw", "mi_apc", "cn"):
        assert np.abs(mo.tri(o[name]) - g[p + name]).max() <= 1e-9, name
    target = "".join(np.array(list(alphabet))[codes[0]])
    assert target == str(g[p + "target_seq"])


def test_selection_rules():
    """Sites: upper-case non-gap target columns; records: all site characters in the alphabet (case-sensitive,
    '.' and lower case in a site invalidate); index list from the target's /start-end."""
    from evcouplings_b200.mean_field import select_alignment
    text = ">t/5-12\nAcD-eFGH\n>a\nAcDxaF-H\n>b\nA.D-eFgH\n>c\nA.D-efGH\n>d\nAcXAeFGH\n>e\nAcD.eFGH\n"
    ids, raw = parse_text(text)
    codes, index_list, valid = select_alignment(raw, ids, "-ACDEFGHIKLMNPQRSTVWY")
    assert list(index_list) == [5, 7, 10, 11, 12]
    assert list(valid) == [True, True, False, False, False, True]
    assert codes.shape == (3, 5) and "".join("-ACDEFGHIKLMNPQRSTVWY"[c] for c in codes[1]) == "ADF-H"
    with pytest.raises(ValueError, match="residue range"):
        select_alignment(raw, ["t"] + ids[1:], "-ACDEFGHIKLMNPQRSTVWY")
    with pytest.raises(ValueError, match="does not match"):
        select_alignment(raw, ["t/5-20"] + ids[1:], "-ACDEFGHIKLMNPQRSTVWY")


def _model_from_oracle(case, tmp_path):
    from evcouplings_b200.mean_field import MeanFieldModel
    g = load_golden()
    codes, alphabet, theta, pc, index_list = case_codes(g, case)
    w = g[case + "_weights"]
    o = mo.fit(codes, w, len(alphabet), pc)
    res = dict(fi=o["fi"], rfi=o["rfi"], h=o["h"], fij_tri=mo.tri(o["fij"]), J_tri=mo.tri(o["J"]),
               di=mo.tri(o["di"]), fn=mo.tri(o["fn"]), mi=mo.tri(o["mi_raw"]), di_iters=mo.tri(o["di_iters"]))
    return g, MeanFieldModel(res, codes, w, alphabet, index_list, theta, pc)


def test_ec_file_format(tmp_path):
    g, m = _model_from_oracle("rna", tmp_path)
    path = tmp_path / "ECs.txt"
    m.to_raw_ec_file(str(path))
    lines = path.read_text().splitlines()
    ref = str(g["rna_ec_text"]).splitlines()
    assert len(lines) == len(ref) == m.L * (m.L - 1) // 2
    for a, b in zip(lines, ref):
        fa, fb = a.split(" "), b.split(" ")
        assert len(fa) == 8 and fa[:4] == fb[:4]
        assert all(len(x.split(".")[1]) == 6 for x in fa[4:])
        assert max(abs(float(x) - float(y)) for x, y in zip(fa[4:], fb[4:])) <= 1.5e-6


def test_mean_field_model_header_reads_back(tmp_path):
    from evcouplings_b200 import model_ops
    g, m = _model_from_oracle("syn", tmp_path)
    path = tmp_path / "mf.model"
    m.to_file(str(path))
    r = model_ops.read_model(str(path))
    hdr = json.loads(str(g["syn_file_header"]))
    assert hdr["class_name"] == "MeanFieldCouplingsModel"
    assert (r["L"], r["q"], r["n_valid"], r["n_invalid"], r["num_iter"]) == (hdr["L"], hdr["q"], hdr["N_valid"], 0, -1)
    assert r["lambda_J"] == r["lambda_group"] == -1.0
    assert abs(r["lambda_h"] + hdr["pseudo_count"]) <= 1e-7 and abs(r["theta"] - hdr["theta"]) <= 1e-7
    assert abs(r["n_eff"] - hdr["N_eff"]) <= 1e-3 and r["alphabet"] == hdr["alphabet"]
    assert r["target_seq"] == hdr["target_seq"] and np.array_equal(r["index_list"], g["syn_file_index_list"])
    assert np.allclose(r["weights"], g["syn_file_weights"], rtol=1e-6)
    assert np.allclose(r["fi"], g["syn_file_f_i"], atol=1e-7) and np.allclose(r["h"], g["syn_file_h_i"], atol=1e-4)
    idx = g["syn_J_sample_idx"]
    assert np.allclose(r["J"].reshape(-1)[idx], g["syn_file_J_sample"], atol=1e-4)
    assert np.allclose(r["fij"].reshape(-1)[idx], g["syn_file_fij_sample"], atol=1e-7)
    path64 = tmp_path / "mf64.model"
    m.to_file(str(path64), precision="float64")
    assert os.path.getsize(path64) > os.path.getsize(path)
    with pytest.raises(ValueError):
        m.to_file(str(tmp_path / "v1.model"), file_format="plmc_v1")


def test_shipped_library_has_the_fp64_mean_field_kernels():
    """SASS of the shipped library: the mean-field kernels are there and the tile GEMM runs on the fp64 FMA pipe."""
    import shutil
    import subprocess
    from evcouplings_b200 import _lib
    exe = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(exe):
        pytest.skip("cuobjdump not available")
    sass = subprocess.run([exe, "-sass", _lib.LIB_PATH], capture_output=True, text=True, timeout=600).stdout
    for name in ("mf_gemm_f64_kernel", "mf_potrf_block_kernel", "mf_trsm_lower_kernel", "mf_di_kernel",
                 "mf_fields_kernel", "mf_covariance_kernel"):
        assert name in sass, name
    gemm = sass[sass.index("mf_gemm_f64_kernel"):]
    gemm = gemm[:gemm.index("Function :", 20)] if "Function :" in gemm[20:] else gemm
    assert "DFMA" in gemm


@pytest.mark.parametrize("case", ["syn", "rna"])
def test_ec_text_rebuilt_from_scores_matches_reference_file(case):
    """The PABP EC file is compared in this format; where the reference's own file is stored it is reproduced."""
    g = load_golden()
    without_text = {k: v for k, v in g.items() if k != case + "_ec_text"}
    assert reference_ec_text(without_text, case) == str(g[case + "_ec_text"])
