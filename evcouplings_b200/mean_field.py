"""
Mean-field DCA on the GPU: the couplings stage's ``mean_field`` protocol (evcouplings/couplings/protocol.py,
evcouplings/couplings/mean_field.py) with every numerical step in fp64 CUDA kernels (csrc/mean_field.cu).

    import evcouplings.couplings.protocol as cp, evcouplings_b200
    cp.MeanFieldDCA = evcouplings_b200.MeanFieldDCA

Rules kept from the reference: the target is the first record; model sites are the columns where it has an
upper-case character that is not a gap ('-' or '.'); a record is valid when all its characters in those columns
are in the alphabet (case-sensitive); the index list numbers the target's columns from the ``/start-end`` of its
header.  Sequence weights are 1 / #neighbours at identity >= theta over the valid records.
"""
import re

import numpy as np

from . import model_io, model_ops, msa

ALPHABET_MAP = {"aa": msa.ALPHABET_PROTEIN, "dna": "-ACGT", "rna": "-ACGU"}


def _char_matrix(matrix):
    """(N, W) array of one-character strings (or bytes) -> uint8 characters."""
    m = np.asarray(matrix)
    if m.dtype.kind == "U":
        cp = np.ascontiguousarray(m).view(np.uint32).reshape(m.shape)
        if cp.size and int(cp.max()) > 127:
            raise ValueError("alignment contains non-ASCII characters")
        return cp.astype(np.uint8)
    if m.dtype.kind == "S":
        return np.ascontiguousarray(m).view(np.uint8).reshape(m.shape)
    return np.ascontiguousarray(m, dtype=np.uint8)


def _header_range(header):
    m = re.search(r"(.+)/(\d+)-(\d+)", header.split()[0] if header.split() else header)
    if m is None:
        raise ValueError("target header %r has no /start-end residue range" % header)
    return int(m.group(2)), int(m.group(3))


def select_alignment(raw, ids, alphabet, match_gap="-", insert_gap="."):
    """raw: (N, W) uint8 characters, target first.  Returns (codes (N_valid, L) uint8 in alphabet order,
    index_list (L,) int64, valid (N,) bool)."""
    raw = np.ascontiguousarray(raw, dtype=np.uint8)
    target = raw[0]
    focus = (target >= ord("A")) & (target <= ord("Z")) & (target != ord(match_gap)) & (target != ord(insert_gap))
    start, stop = _header_range(ids[0])
    if stop - start + 1 != raw.shape[1]:
        raise ValueError("target range %d-%d does not match the alignment width %d" % (start, stop, raw.shape[1]))
    cols = np.nonzero(focus)[0]
    if len(cols) < 2:
        raise ValueError("fewer than 2 model sites selected")
    index_list = np.arange(start, stop + 1)[focus]
    lut = np.full(256, 255, dtype=np.uint8)
    for k, ch in enumerate(alphabet):
        lut[ord(ch)] = k
    sub = np.ascontiguousarray(raw[:, cols])
    codes, valid = msa._encode_rows(sub, lut, np.arange(len(cols)))
    if len(codes) == 0:
        raise ValueError("no valid sequences")
    return codes, index_list, valid


class MeanFieldModel(object):
    """What the reference's MeanFieldCouplingsModel exposes to the protocol and its readers.  Pair quantities are
    kept packed (pairs i<j); the L x L x q x q tensors are built on first access."""

    def __init__(self, res, codes, weights, alphabet, index_list, theta, pseudo_count):
        L, q = res["h"].shape
        self.L, self.num_symbols = L, q
        self.N_valid = len(codes)
        self.N_invalid = 0
        self.weights = weights
        self.N_eff = float(weights.sum())
        self.alphabet = np.array(list(alphabet))
        self.index_list = np.asarray(index_list)
        self.target_seq = np.array(list(alphabet))[codes[0]]
        self.theta, self.pseudo_count = theta, pseudo_count
        self.f_i = res["fi"]
        self.regularized_f_i = res["rfi"]
        self.h_i = res["h"]
        self.J_tri = res["J_tri"]
        self.fij_tri = res["fij_tri"]
        self.di_iterations = res["di_iters"]
        self._iu, self._ju = np.triu_indices(L, 1)
        self.di_scores = self._square(res["di"])
        self.fn_scores = self._square(res["fn"])
        self.mi_scores_raw = self._square(res["mi"])
        self.cn_scores = model_ops.apc(self.fn_scores)
        self.mi_scores_apc = model_ops.apc(self.mi_scores_raw)
        self._J_ij = self._f_ij = None

    def _square(self, v):
        M = np.zeros((self.L, self.L))
        M[self._iu, self._ju] = v
        M[self._ju, self._iu] = v
        return M

    def _full(self, tri):
        T = np.zeros((self.L, self.L, self.num_symbols, self.num_symbols))
        T[self._iu, self._ju] = tri
        T[self._ju, self._iu] = tri.transpose(0, 2, 1)
        return T

    @property
    def J_ij(self):
        """L x L x q x q couplings (J_ji = J_ij^T; the i == i blocks are zero, as in the model file)."""
        if self._J_ij is None:
            self._J_ij = self._full(self.J_tri)
        return self._J_ij

    @property
    def f_ij(self):
        """L x L x q x q raw pair frequencies, f_ii = diag(f_i)."""
        if self._f_ij is None:
            F = self._full(self.fij_tri)
            F[np.arange(self.L), np.arange(self.L)] = [np.diag(r) for r in self.f_i]
            self._f_ij = F
        return self._f_ij

    def to_raw_ec_file(self, couplings_file):
        """``i A_i j A_j mi_raw mi_apc di cn``, six decimals, pairs i<j in row-major order."""
        idx, ts = self.index_list, self.target_seq
        with open(couplings_file, "w") as f:
            f.writelines("%s %s %s %s %.6f %.6f %.6f %.6f\n" % (
                idx[i], ts[i], idx[j], ts[j], self.mi_scores_raw[i, j], self.mi_scores_apc[i, j],
                self.di_scores[i, j], self.cn_scores[i, j]) for i, j in zip(self._iu, self._ju))

    def to_file(self, out_file, precision="float32", file_format="plmc_v2"):
        if file_format != "plmc_v2":
            raise ValueError("Illegal file format: %s. Valid option: plmc_v2." % file_format)
        model_io.write_mean_field_model_file(
            out_file, self.L, self.num_symbols, self.N_valid, self.theta, self.pseudo_count, self.N_eff,
            "".join(self.alphabet), self.weights, "".join(self.target_seq), self.index_list, self.f_i, self.h_i,
            self.fij_tri, self.J_tri, precision=precision)


def fit_codes(codes, alphabet, index_list, theta=0.8, pseudo_count=0.5, engine=None):
    """Mean-field DCA of encoded valid sequences (codes in alphabet order, target first)."""
    if engine is None:
        from .engine import CudaEngine
        engine = CudaEngine()
    codes = np.ascontiguousarray(codes, dtype=np.uint8)
    L = codes.shape[1]
    counts = engine.hamming_counts(codes, msa.identity_threshold_count(theta, L))
    weights = 1.0 / counts.astype(np.float64)
    res = engine.mean_field(codes, weights, len(alphabet), pseudo_count)
    return MeanFieldModel(res, codes, weights, alphabet, index_list, theta, pseudo_count)


class MeanFieldDCA(object):
    """Drop-in for the reference's MeanFieldDCA: ``MeanFieldDCA(alignment).fit(theta, pseudo_count)``.
    ``alignment`` needs what the reference's Alignment exposes: ``matrix`` (N x W characters, target first),
    ``ids``, ``alphabet`` and optionally ``_match_gap`` / ``_insert_gap``."""

    def __init__(self, alignment, engine=None):
        self.alphabet = "".join(alignment.alphabet)
        raw = _char_matrix(alignment.matrix)
        self.codes, self.index_list, self.valid = select_alignment(
            raw, list(alignment.ids), self.alphabet, getattr(alignment, "_match_gap", "-"),
            getattr(alignment, "_insert_gap", "."))
        self.engine = engine

    def fit(self, theta=0.8, pseudo_count=0.5):
        return fit_codes(self.codes, self.alphabet, self.index_list, theta, pseudo_count, self.engine)


def run_mean_field(alignment_file, raw_ec_file, model_file=None, focus_seq=None, alphabet=None, theta=0.8,
                   pseudo_count=0.5, engine=None):
    """File-level mean-field DCA: alignment (A2M/FASTA, target first, or the record named ``focus_seq``) ->
    raw EC file (and the plmc_v2 model file).  Returns the model."""
    alphabet = ALPHABET_MAP.get(alphabet, alphabet) if alphabet is not None else msa.ALPHABET_PROTEIN
    ids, raw = msa.read_fasta_matrix(alignment_file)
    if focus_seq is not None:
        k, _ = msa._find_focus(ids, focus_seq)
        order = np.r_[k, np.delete(np.arange(len(ids)), k)]
        raw, ids = raw[order], [ids[o] for o in order]
    codes, index_list, _ = select_alignment(raw, ids, alphabet)
    model = fit_codes(codes, alphabet, index_list, theta, pseudo_count, engine)
    model.to_raw_ec_file(raw_ec_file)
    if model_file is not None:
        model.to_file(model_file)
    return model


