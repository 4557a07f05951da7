"""
Generate tests/golden/mean_field_golden.npz: what the reference's mean-field DCA (MeanFieldDCA.fit and
MeanFieldCouplingsModel) computes on three inputs, run unmodified on the CPU:

    python tests/golden/make_mean_field_golden.py REFERENCE_DIR

    pabp  the seeded 1,000-record PABP sample (pabp_sample.a2m.gz), protein, theta 0.8, pseudo-count 0.5
    syn   a small synthetic protein alignment with insert columns and invalid records, theta 0.8, pseudo-count 0.1
    rna   a synthetic RNA alignment (alphabet -ACGU, q = 5), theta 0.8, pseudo-count 0.5

Per case (prefix "<case>_"): the alignment text (syn, rna), index list, N_valid, N_eff, weights, regularised f_i,
h_i, DI / MI raw / MI APC / CN (pairs i<j), a seeded sample of 1,000 J_ij tri-block entries (the full tensors
would make the fixture megabytes), the raw EC file text (syn, rna; the PABP file is the same format over the
stored scores), and the header and arrays of the reference's own plmc_v2 writer as its CouplingsModel reads them
back (float32, as written).  Only outputs are stored.
"""
import gzip
import json
import os
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, HERE)

import ref_harness  # noqa: E402
from evcouplings_b200 import synthetic  # noqa: E402

J_SAMPLE = 1000


def synthetic_text(N, L, seed, alphabet, q_res, n_insert, n_invalid):
    """A2M text: focus record first (header with a residue range), insert columns in lower case / '.', and a
    few records with a character outside the alphabet in a match column (invalid for mean-field DCA)."""
    rng = np.random.default_rng(seed)
    codes = synthetic.synthetic_msa_codes(N, L, seed, q_res=q_res)
    lut = np.frombuffer(alphabet.encode("ascii"), dtype=np.uint8)
    chars = lut[codes].copy()
    ins_at = np.sort(rng.choice(np.arange(1, L), size=n_insert, replace=False))
    lower = np.frombuffer(alphabet[1:].lower().encode("ascii"), dtype=np.uint8)
    cols = []
    for k in range(L):
        if k in ins_at:
            ins = lower[rng.integers(0, len(lower), size=N)]
            ins[rng.random(N) < 0.5] = ord(".")
            ins[0] = lower[0]
            cols.append(ins)
        cols.append(chars[:, k])
    mat = np.stack(cols, axis=1)
    bad = rng.choice(np.arange(1, N), size=n_invalid, replace=False)
    mat[bad, rng.integers(0, mat.shape[1], size=n_invalid)] = ord("X")
    width = mat.shape[1]
    lines = []
    for n in range(N):
        name = "target/11-%d" % (10 + width) if n == 0 else "seq%d" % n
        lines.append(">%s\n%s\n" % (name, bytes(mat[n]).decode("ascii")))
    return "".join(lines)


def run_case(text, alphabet, theta, pc):
    from evcouplings.align.alignment import Alignment
    from evcouplings.couplings.mean_field import MeanFieldDCA
    from evcouplings.couplings.model import CouplingsModel
    import io
    ali = Alignment.from_file(io.StringIO(text), alphabet=alphabet, format="fasta")
    model = MeanFieldDCA(ali).fit(theta=theta, pseudo_count=pc)
    L, q = model.L, model.num_symbols
    iu, ju = np.triu_indices(L, 1)
    J_tri = model.J_ij[iu, ju].reshape(-1)
    rng = np.random.default_rng(L * 1000 + q)
    sample = np.sort(rng.choice(J_tri.size, size=min(J_SAMPLE, J_tri.size), replace=False)).astype(np.int32)
    out = dict(
        index_list=np.asarray(model.index_list), N_valid=model.N_valid, N_eff=model.N_eff,
        weights=np.asarray(model.weights, dtype=np.float64), target_seq=np.array("".join(model.target_seq)),
        regularized_f_i=model.regularized_f_i, h_i=model.h_i, J_sample_idx=sample, J_sample=J_tri[sample],
        J_absmax=np.abs(J_tri).max(),
        di=model.di_scores[iu, ju], mi_raw=model.mi_scores_raw[iu, ju], mi_apc=model.mi_scores_apc[iu, ju],
        cn=model.cn_scores[iu, ju],
    )
    with tempfile.TemporaryDirectory() as tmp:
        ec = os.path.join(tmp, "ECs.txt")
        model.to_raw_ec_file(ec)
        out["ec_text"] = np.array(open(ec).read())
        mf = os.path.join(tmp, "mf.model")
        model.to_file(mf)
        back = CouplingsModel(mf)
        out["file_header"] = np.array(json.dumps(dict(
            L=int(back.L), q=int(back.num_symbols), N_valid=int(back.N_valid), N_invalid=int(back.N_invalid),
            num_iter=None if back.num_iter is None else int(back.num_iter), theta=float(back.theta),
            pseudo_count=float(back.pseudo_count), N_eff=float(back.N_eff), alphabet="".join(back.alphabet),
            target_seq="".join(back.target_seq), class_name=type(back).__name__)))
        out["file_weights"] = np.asarray(back.weights, dtype=np.float32)
        out["file_index_list"] = np.asarray(back.index_list)
        out["file_f_i"] = back.f_i.astype(np.float32)
        out["file_h_i"] = back.h_i.astype(np.float32)
        out["file_J_sample"] = back.J_ij[iu, ju].reshape(-1)[sample].astype(np.float32)
        out["file_fij_sample"] = back.f_ij[iu, ju].reshape(-1)[sample].astype(np.float32)
    return out


CASES = {
    # name: (alphabet, theta, pseudo-count)
    "pabp": ("-ACDEFGHIKLMNPQRSTVWY", 0.8, 0.5),
    "syn": ("-ACDEFGHIKLMNPQRSTVWY", 0.8, 0.1),
    "rna": ("-ACGU", 0.8, 0.5),
}


def case_text(name):
    if name == "pabp":
        with gzip.open(os.path.join(HERE, "pabp_sample.a2m.gz"), "rt") as f:
            return f.read()
    if name == "syn":
        return synthetic_text(400, 36, 11, CASES["syn"][0], 20, 4, 6)
    return synthetic_text(300, 48, 12, CASES["rna"][0], 4, 3, 5)


def main(reference_dir):
    ref_harness.set_root(reference_dir)
    ref_harness.install()
    store = {}
    for name, (alphabet, theta, pc) in CASES.items():
        text = case_text(name)
        res = run_case(text, alphabet, theta, pc)
        if name == "pabp":
            del res["ec_text"]
        else:
            res["alignment_text"] = np.array(text)
        res["params"] = np.array([theta, pc])
        res["alphabet"] = np.array(alphabet)
        for k, v in res.items():
            store["%s_%s" % (name, k)] = v
        print("%s: L=%d N_valid=%d N_eff=%.2f" % (name, len(res["index_list"]), res["N_valid"], res["N_eff"]))
    path = os.path.join(HERE, "mean_field_golden.npz")
    np.savez_compressed(path, **store)
    print("wrote %s (%d bytes)" % (path, os.path.getsize(path)))


if __name__ == "__main__":
    if len(sys.argv) != 2:
        sys.exit("usage: make_mean_field_golden.py REFERENCE_DIR")
    main(sys.argv[1])
