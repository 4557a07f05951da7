"""
Generate the committed golden fixtures in tests/golden/.

Needs an unmodified EVcouplings checkout:
    python tests/golden/make_golden.py REFERENCE_DIR [fixture ...]
(fixtures: pabp in_tree_twins tiny_model model_consumers pabp_sample reference_boundary; default all)

Sources of truth
  (1) the real plmc run shipped with the reference:
      REFERENCE_DIR/notebooks/example/PABP_YEAST.{a2m,model_params}, PABP_YEAST_ECs.txt
      (presumed command: plmc -f PABP_YEAST -g -m 200 -t 0.2 -lh 0.01 -le 16.2)
  (2) the reference's own Python, imported unmodified via ref_harness:
      evcouplings/align/alignment.py:1192-1233 num_cluster_members,
      :1078-1153 frequencies / pair_frequencies,
      evcouplings/couplings/model.py:317-400 CouplingsModel reader (+ cn/fn scores :744-827),
      evcouplings/couplings/tools.py:20-108 parse_plmc_log,
      evcouplings/couplings/protocol.py standard / complex and tools.py run_plmc driving our run_plmc and
      our plmc-compatible executable (reference_boundary).
Nothing from the reference's *source code* is copied; only its outputs on
seeded inputs are stored.
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, HERE)

import ref_harness  # noqa: E402
from oracle import plm_oracle as po  # noqa: E402

EX = None          # REFERENCE_DIR/notebooks/example, set in __main__


def pabp():
    ids, seqs = po.read_a2m(os.path.join(EX, "PABP_YEAST.a2m"))
    prep = po.prepare_alignment(ids, seqs, focus="PABP_YEAST", alphabet=None, ignore_gaps=True)
    gm = po.read_model(os.path.join(EX, "PABP_YEAST.model_params"))
    counts_all = gm["weights"].astype(np.int32)           # golden stores integer neighbour counts
    np.savez_compressed(
        os.path.join(HERE, "pabp_codes.npz"),
        codes=prep["codes"], valid_packed=np.packbits(prep["valid"]),
        n_total=prep["n_total"], golden_counts_all=counts_all,
        focus_cols=prep["focus_cols"], index_list=prep["index_list"],
        target_seq=np.array(prep["target_seq"]), region_start=prep["region_start"],
    )
    # EC text
    ec = np.loadtxt(os.path.join(EX, "PABP_YEAST_ECs.txt"), dtype=str)
    pairs = [(0, 1), (6, 8), (3, 60), (20, 21), (33, 70), (50, 81)]
    L = gm["L"]
    iu, ju = np.triu_indices(L, 1)
    pidx = np.array([np.nonzero((iu == i) & (ju == j))[0][0] for i, j in pairs])
    # reference reader KATs on the golden file
    ref_harness.install()
    from evcouplings.couplings.model import CouplingsModel
    cm = CouplingsModel(os.path.join(EX, "PABP_YEAST.model_params"))
    kat = dict(
        hi_127=float(cm.hi(127, cm.seq(127))),
        Jij_127_172=float(cm.Jij(127, 172, cm.seq(127), cm.seq(172))),
        ref_cn_zero_sum=cm.cn_scores[iu, ju].astype(np.float64),   # model.py:788-803 (zero-sum gauge first)
    )
    np.savez_compressed(
        os.path.join(HERE, "pabp_golden.npz"),
        hdr_i=np.array([gm["L"], gm["q"], gm["n_valid"], gm["n_invalid"], gm["num_iter"]], dtype=np.int32),
        hdr_f=np.array([gm["theta"], gm["lambda_h"], gm["lambda_J"], gm["lambda_group"], gm["n_eff"]],
                       dtype=np.float32),
        alphabet=np.array(gm["alphabet"]), target_seq=np.array(gm["target_seq"]),
        index_list=gm["index_list"], fi=gm["fi"], h=gm["h"], J=gm["J"],
        fij_pairs=np.array(pairs, dtype=np.int32), fij_pair_index=pidx, fij_blocks=gm["fij"][pidx],
        ec_i=ec[:, 0].astype(np.int32), ec_Ai=ec[:, 1], ec_j=ec[:, 2].astype(np.int32), ec_Aj=ec[:, 3],
        ec_cn=ec[:, 5].astype(np.float64),
        kat_hi_127=kat["hi_127"], kat_Jij_127_172=kat["Jij_127_172"],
        ref_cn_zero_sum=kat["ref_cn_zero_sum"],
    )
    print("pabp fixtures written; valid=%d" % prep["n_valid"])


def in_tree_twins():
    """Reference numba kernels on the seeded config-1 alignment (N=200, L=40, q=21)."""
    ref_harness.install()
    from evcouplings.align import alignment as al
    out = {}
    for name, (N, L, seed, theta) in dict(cfg1=(200, 40, 1, 0.8), tie=(300, 50, 7, 0.8),
                                          odd=(257, 33, 11, 0.7)).items():
        codes = po.synthetic_msa_codes(N, L, seed)
        m = codes.astype(np.int64)
        counts = al.num_cluster_members(m, theta)
        w = 1.0 / counts
        fi = al.frequencies(m, w, 21)
        fij = al.pair_frequencies(m, w, 21, fi)
        iu, ju = np.triu_indices(L, 1)
        out[name + "_codes"] = codes
        out[name + "_theta"] = theta
        out[name + "_counts"] = counts.astype(np.int32)
        out[name + "_fi"] = fi
        out[name + "_fij_tri"] = fij[iu, ju]
    np.savez_compressed(os.path.join(HERE, "intree_twins.npz"), **out)
    print("in-tree twin fixtures written")


def tiny_model():
    """Tiny model written in plmc_v2 layout, read back by the reference's CouplingsModel."""
    ref_harness.install()
    from evcouplings.couplings.model import CouplingsModel
    N, L, q = 60, 12, 21
    codes = po.synthetic_msa_codes(N, L, 21)
    counts = po.hamming_counts(codes, 0.8)
    w = po.sequence_weights(counts)
    fi, fij = po.frequencies(codes, w, q)
    x, res = po.fit(codes, w, q, 0.01, 0.01 * (q - 1) * (L - 1), max_iter=400)
    h, Jt = po.unpack(x, L, q)
    alphabet = po.ALPHABET_PROTEIN
    target = "".join(alphabet[c] for c in codes[0])
    index_list = np.arange(5, 5 + L, dtype=np.int32)
    path = os.path.join(HERE, "tiny.model")
    po.write_model(path, L, q, N, 0, int(res.nit), 0.2, 0.01, 0.01 * (q - 1) * (L - 1), 0.0, w.sum(),
                   alphabet, counts.astype(np.float32), target, index_list, fi, h, fij, Jt)
    ecs_path = os.path.join(HERE, "tiny_ECs.txt")
    po.write_ecs(ecs_path, Jt.astype(np.float32), L, index_list, target)
    cm = CouplingsModel(path)
    iu, ju = np.triu_indices(L, 1)
    from evcouplings.couplings.pairs import read_raw_ec_file
    ecs = read_raw_ec_file(ecs_path, sort=False)
    np.savez_compressed(
        os.path.join(HERE, "tiny_ref_read.npz"),
        codes=codes, counts=counts, x=x.astype(np.float64),
        ref_J_tri=cm.J_ij[iu, ju], ref_h=cm.h_i, ref_fi=cm.f_i, ref_fij_tri=cm.f_ij[iu, ju],
        ref_L=cm.L, ref_q=cm.num_symbols, ref_N_eff=cm.N_eff, ref_theta=cm.theta,
        ref_lambda_J=cm.lambda_J, ref_alphabet=np.array("".join(cm.alphabet)),
        ref_target=np.array("".join(cm.target_seq)), ref_index_list=cm.index_list,
        ref_fn=cm.fn_scores[iu, ju], ref_cn_zero_sum=cm.cn_scores[iu, ju],
        ecs_i=ecs["i"].values, ecs_j=ecs["j"].values, ecs_cn=ecs["cn"].values,
        ecs_Ai=ecs["A_i"].values.astype(str), ecs_Aj=ecs["A_j"].values.astype(str),
    )
    print("tiny model fixtures written; iters=%d" % res.nit)


def model_consumers():
    """Reference CouplingsModel outputs (model.py) on the tiny model and on the golden PABP model:
    ecs table scores, hamiltonians, single-mutant matrix, delta_hamiltonian."""
    ref_harness.install()
    from evcouplings.couplings.model import CouplingsModel
    rng = np.random.default_rng(5)
    out = {}
    for name, path in (("tiny", os.path.join(HERE, "tiny.model")),
                       ("pabp", os.path.join(EX, "PABP_YEAST.model_params"))):
        cm = CouplingsModel(path)
        L, q = cm.L, cm.num_symbols
        iu, ju = np.triu_indices(L, 1)
        alphabet = "".join(cm.alphabet)
        tgt = "".join(cm.target_seq)
        seqs = [tgt] + ["".join(alphabet[k] for k in rng.integers(0, q, L)) for _ in range(40)]
        # a few sequences close to the target
        for _ in range(20):
            s = list(tgt)
            for p in rng.integers(0, L, 3):
                s[p] = alphabet[rng.integers(0, q)]
            seqs.append("".join(s))
        out[name + "_seqs"] = np.array(seqs)
        out[name + "_H"] = cm.hamiltonians(seqs)
        out[name + "_smm"] = cm.single_mut_mat_full
        out[name + "_fn"] = cm.fn_scores[iu, ju]
        out[name + "_cn"] = cm.cn_scores[iu, ju]
        if name == "tiny":
            out[name + "_mi_raw"] = cm.mi_scores_raw[iu, ju]
            out[name + "_mi_apc"] = cm.mi_scores_apc[iu, ju]
        variants = []
        for _ in range(12):
            ps = sorted(set(int(p) for p in rng.integers(0, L, 2)))
            variants.append([(int(cm.index_list[p]), tgt[p], alphabet[rng.integers(0, q)]) for p in ps])
        out[name + "_var_pos"] = np.array([[v[0][0], v[-1][0]] for v in variants])
        out[name + "_variants"] = np.array([";".join("%d,%s,%s" % s for s in v) for v in variants])
        out[name + "_dH"] = np.array([cm.delta_hamiltonian(v) for v in variants])
    np.savez_compressed(os.path.join(HERE, "model_consumers.npz"), **out)
    print("model consumer fixtures written; PABP H(target) = %.10f, smm(127,E) = %.10f" % (
        out["pabp_H"][0, 0], out["pabp_smm"][127 - 123, "ACDEFGHIKLMNPQRSTVWY".index("E"), 0]))


def pabp_sample(n_valid=900, n_invalid=100):
    """A seeded sample of the real PABP_YEAST.a2m (focus record first, then records in file order) and the
    0-based record numbers it keeps; the expected codes / validity are rows of pabp_codes.npz."""
    import gzip
    c = np.load(os.path.join(HERE, "pabp_codes.npz"))
    valid = np.unpackbits(c["valid_packed"])[: int(c["n_total"])].astype(bool)
    rng = np.random.default_rng(2024)
    vi, ii = np.nonzero(valid[1:])[0] + 1, np.nonzero(~valid[1:])[0] + 1
    rows = np.sort(np.concatenate([[0], rng.choice(vi, n_valid, replace=False),
                                   rng.choice(ii, n_invalid, replace=False)])).astype(np.int32)
    keep, k, out = set(rows.tolist()), -1, []
    with open(os.path.join(EX, "PABP_YEAST.a2m")) as f:
        for line in f:
            if line.startswith(">"):
                k += 1
            if k in keep:
                out.append(line)
    with gzip.GzipFile(os.path.join(HERE, "pabp_sample.a2m.gz"), "wb", mtime=0) as f:
        f.write("".join(out).encode())
    np.save(os.path.join(HERE, "pabp_sample_rows.npy"), rows)
    print("pabp sample written: %d records" % len(rows))


def reference_boundary():
    """The reference's own couplings protocol (standard, complex), its own run_plmc and its readers, run over
    our run_plmc / plmc-compatible executable with the CPU oracle engine.  Stored: what the reference passes
    in (arguments, argv; temporary paths as {tmp}), and what its stage code, readers and log parser made of
    what we returned and wrote.  The tests replay the recorded calls without the reference."""
    import json
    import stat
    import tempfile
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    ref_harness.install()
    import evcouplings.couplings.tools as ct
    import evcouplings.couplings.protocol as cpr
    import evcouplings.couplings.model as cm
    import evcouplings.couplings.pairs as cp
    from evcouplings.align.alignment import Alignment, identities_to_seq
    from evcouplings_b200 import synthetic, tools
    from cpu_engine import OracleEngine
    meta = {"plmc_result_fields": list(ct.PlmcResult._fields)}
    arrays = {}
    rng = np.random.default_rng(17)

    def protocol_kwargs(prefix, a2m, L, ignore_gaps, iterations, cpu):
        return dict(
            protocol="standard", prefix=prefix, alignment_file=a2m, focus_mode=True,
            focus_sequence="seq0/1-%d" % L, theta=0.8, alphabet=None,
            segments=[["A_1", "aa", "seq0", 1, L, list(range(1, L + 1))]], ignore_gaps=ignore_gaps,
            iterations=iterations, lambda_h=0.01, lambda_J=0.01, lambda_J_times_Lq=True, lambda_group=None,
            scale_clusters=None, cpu=cpu, plmc="plmc", reuse_ecs=False, min_sequence_distance=6,
            frequencies_file=None, scoring_model="skewnormal")

    with tempfile.TemporaryDirectory() as tmp:
        def rel(v):
            return v.replace(tmp, "{tmp}") if isinstance(v, str) else v

        def run_protocol(kw):
            captured = {}

            def run_plmc(*a, **k):
                res, run = tools.run_plmc(*a, engine=OracleEngine(), return_run=True, **k)
                captured.update(args=[rel(v) for v in a], kwargs={n: rel(v) for n, v in k.items()}, run=run)
                return res

            original, ct.run_plmc = ct.run_plmc, run_plmc
            try:
                outcfg = cpr.run(**kw)
            finally:
                ct.run_plmc = original
            rec = {"args": captured["args"], "kwargs": captured["kwargs"],
                   "outcfg": {k: outcfg[k] for k in ("num_sites", "num_valid_sequences", "effective_sequences",
                                                       "region_start")},
                   "outcfg_keys": sorted(outcfg)}
            model = cm.CouplingsModel(outcfg["model_file"])
            rec["model"] = {"L": int(model.L), "num_symbols": int(model.num_symbols), "N_valid": int(model.N_valid),
                            "alphabet": "".join(model.alphabet), "theta": float(model.theta),
                            "N_eff": float(model.N_eff), "target_seq": "".join(model.target_seq)}
            it_ref, fields_ref = ct.parse_plmc_log(captured["run"].log)
            rec["log"] = captured["run"].log
            rec["log_fields"] = list(fields_ref)
            rec["iter_columns"] = list(it_ref.columns)
            rec["iter_rows"] = it_ref.values.tolist()
            ecs = cp.read_raw_ec_file(outcfg["raw_ec_file"], sort=False)
            return rec, outcfg, model, ecs

        # standard protocol, BASELINE configs[0]; (30 iterations, cpu=2) and (40 iterations, cpu=1)
        N, L = 200, 40
        codes = synthetic.synthetic_msa_codes(N, L, 1)
        a2m = os.path.join(tmp, "cfg1.a2m")
        synthetic.write_a2m(a2m, codes)
        for iterations, cpu in ((30, 2), (40, 1)):
            for ig in (True, False):
                name = "standard_it%d_ig%d" % (iterations, int(ig))
                prefix = os.path.join(tmp, name, "job")
                rec, outcfg, model, ecs = run_protocol(protocol_kwargs(prefix, a2m, L, ig, iterations, cpu))
                rec["files"] = sorted(os.path.relpath(os.path.join(dp, f), os.path.dirname(prefix))
                                      for dp, _, fs in os.walk(os.path.dirname(prefix)) for f in fs)
                meta[name] = rec
                iu, ju = np.triu_indices(L, 1)
                Jt = model.J_ij[iu, ju].reshape(-1)
                idx = np.sort(rng.choice(Jt.size, 600, replace=False)).astype(np.int32)
                arrays[name + "_h"] = model.h_i
                arrays[name + "_J_idx"], arrays[name + "_J"] = idx, Jt[idx]
                arrays[name + "_J_sums"] = np.array([Jt.sum(), np.abs(Jt).sum(), (Jt * Jt).sum()])
                arrays[name + "_ecs_ij"] = np.stack([ecs["i"].values, ecs["j"].values]).astype(np.int16)
                arrays[name + "_ecs_A"] = np.array(["".join(ecs["A_i"].astype(str)), "".join(ecs["A_j"].astype(str))])
                arrays[name + "_ecs_cn"] = ecs["cn"].values.astype(np.float64)

        # complex protocol (two segments of 12 sites)
        N, L1, L2 = 160, 12, 12
        codes = synthetic.synthetic_msa_codes(N, L1 + L2, 8)
        a2m = os.path.join(tmp, "complex.a2m")
        synthetic.write_a2m(a2m, codes, focus_name="A_B")
        kw = protocol_kwargs(os.path.join(tmp, "cx", "job"), a2m, L1 + L2, True, 30, 2)
        kw.update(protocol="complex", focus_sequence="A_B/1-%d" % (L1 + L2), use_all_ecs_for_scoring=False,
                  segments=[["A_1", "aa", "A", 1, L1, list(range(1, L1 + 1))],
                            ["B_1", "aa", "B", 1, L2, list(range(1, L2 + 1))]])
        rec, outcfg, model, ecs = run_protocol(kw)
        import pandas as pd
        inter = pd.read_csv(outcfg["inter_ec_file"])
        rec["inter_ecs"] = {"rows": len(inter), "segment_i": sorted(set(inter["segment_i"])),
                            "segment_j": sorted(set(inter["segment_j"]))}
        meta["complex"] = rec
        arrays["complex_ecs_ij"] = np.stack([ecs["i"].values, ecs["j"].values]).astype(np.int16)
        arrays["complex_ecs_A"] = np.array(["".join(ecs["A_i"].astype(str)), "".join(ecs["A_j"].astype(str))])

        # the reference's run_plmc (argv, subprocess, stderr parsing, file checks) over our executable
        codes = synthetic.synthetic_msa_codes(150, 16, 3)
        a2m = os.path.join(tmp, "in.a2m")
        synthetic.write_a2m(a2m, codes)
        argv_file = os.path.join(tmp, "argv.json")
        wrapper = os.path.join(tmp, "plmc_wrapper")
        with open(wrapper, "w") as f:
            f.write("#!%s\nimport json, sys\nsys.path.insert(0, %r); sys.path.insert(0, %r)\n"
                    "json.dump(sys.argv[1:], open(%r, 'w'))\n"
                    "from cpu_engine import OracleEngine\nfrom evcouplings_b200.plmc_cli import main\n"
                    "sys.exit(main(engine=OracleEngine()))\n"
                    % (sys.executable, ROOT, os.path.join(ROOT, "tests"), argv_file))
        os.chmod(wrapper, os.stat(wrapper).st_mode | stat.S_IEXEC)
        for name, L, n_it, lam_J in (("cli_cpu", 16, 12, 2.5), ("cli_gpu", 24, 20, 4.0)):
            if name == "cli_gpu":
                codes = synthetic.synthetic_msa_codes(300, 24, 3)
                synthetic.write_a2m(a2m, codes)
            ecs_path, model_path = os.path.join(tmp, name, "x_ECs.txt"), os.path.join(tmp, name, "x.model")
            res = ct.run_plmc(a2m, ecs_path, model_path, focus_seq="seq0/1-%d" % L, alphabet=None, theta=0.8,
                              scale=None, ignore_gaps=True, iterations=n_it, lambda_h=0.01, lambda_J=lam_J,
                              lambda_g=None, cpu=2, binary=wrapper)
            with open(argv_file) as f:
                argv = [rel(a) for a in json.load(f)]
            d = res._asdict()
            it = d.pop("iteration_table")
            meta[name] = {"argv": argv, "result": {k: rel(v) for k, v in d.items()},
                          "iter_columns": list(it.columns), "iter_len": len(it)}

    try:
        ct.parse_plmc_log("nothing useful")
        meta["parse_failure"] = None
    except Exception as e:
        meta["parse_failure"] = type(e).__name__

    # Alignment.set_weights / identities_to_seq on the reference's own class
    codes = synthetic.synthetic_msa_codes(300, 25, 9)
    seqs = ["".join(synthetic.ALPHABET[c] for c in row) for row in codes]
    ali = Alignment.from_dict({"s%d" % k: v for k, v in enumerate(seqs)})
    f_unweighted = ali.frequencies.copy()
    ali.set_weights(0.8)
    arrays["ali_matrix_mapped"] = ali.matrix_mapped.astype(np.int8)
    arrays["ali_num_cluster_members"] = ali.num_cluster_members
    arrays["ali_weights"] = ali.weights
    arrays["ali_frequencies_unweighted"] = f_unweighted
    arrays["ali_frequencies"] = ali.frequencies
    arrays["ali_identities_to_first"] = identities_to_seq(ali.matrix_mapped[0], ali.matrix_mapped)

    np.savez_compressed(os.path.join(HERE, "reference_boundary.npz"), meta=np.array(json.dumps(meta)), **arrays)
    print("reference boundary fixtures written")


FIXTURES = dict(pabp=pabp, in_tree_twins=in_tree_twins, tiny_model=tiny_model, model_consumers=model_consumers,
                pabp_sample=pabp_sample, reference_boundary=reference_boundary)


if __name__ == "__main__":
    if len(sys.argv) < 2:
        sys.exit(__doc__)
    ref_harness.set_root(sys.argv[1])
    EX = os.path.join(ref_harness.REFERENCE_ROOT, "notebooks", "example")
    for name in sys.argv[2:] or list(FIXTURES):
        FIXTURES[name]()
