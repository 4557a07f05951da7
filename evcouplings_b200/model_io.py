"""
Output files of the couplings stage, byte/format compatible with what plmc writes
and the reference reads:

* ``.model`` (plmc_v2 binary): layout defined by the reference's reader
  evcouplings/couplings/model.py:317-389 and writer :1200-1252.
* ``_ECs.txt``: text format read by evcouplings/couplings/pairs.py:55-58
  (``i A_i j A_j fn cn`` separated by single spaces, fn column literally 0).

EC score written to ``_ECs.txt`` (SURVEY.md 8a row a10, pinned against the golden
PABP_YEAST_ECs.txt): cn_ij = F_ij - c_i c_j / cbar with F_ij the Frobenius norm of
J_ij in the gauge of the file (no zero-sum shift), c_i the mean of F over j != i.
"""
import numpy as np


def apc_cn_scores(fn_tri, L):
    """fn_tri: Frobenius norms of the L(L-1)/2 blocks (pair order i<j row-major).  Returns cn (same order)."""
    F = np.zeros((L, L), dtype=np.float64)
    iu, ju = np.triu_indices(L, 1)
    F[iu, ju] = fn_tri
    F = F + F.T
    ci = F.sum(axis=1) / (L - 1)
    cbar = F.sum() / (L * (L - 1))
    if cbar == 0.0:
        return np.zeros(len(iu))
    return (F - np.outer(ci, ci) / cbar)[iu, ju]


def write_ec_file(path, fn_tri, L, index_list, target_seq):
    cn = apc_cn_scores(np.asarray(fn_tri, dtype=np.float64), L)
    iu, ju = np.triu_indices(L, 1)
    idx = np.asarray(index_list)
    lines = ["%d %s %d %s 0 %f\n" % (idx[i], target_seq[i], idx[j], target_seq[j], c)
             for i, j, c in zip(iu, ju, cn)]
    with open(path, "w") as f:
        f.writelines(lines)
    return cn


def write_model_file(path, L, q, n_valid, n_invalid, num_iter, theta_plmc, lambda_h, lambda_J, lambda_group,
                     n_eff, alphabet, weights_all, target_seq, index_list, fi, h, fij_tri, J_tri):
    """plmc_v2 layout, little endian, no padding:
    int32[5] L q N_valid N_invalid num_iter | float32[5] theta lambda_h lambda_J lambda_group N_eff |
    char[q] alphabet | float32[N] weights | char[L] target_seq | int32[L] index_list |
    float32[L][q] f_i | float32[L][q] h_i | float32[npairs][q][q] f_ij | float32[npairs][q][q] J_ij"""
    if lambda_h < 0:
        raise ValueError("lambda_h < 0 marks a mean-field model in this format; refusing to write it")
    _write_plmc_v2(path, L, q, n_valid, n_invalid, num_iter, theta_plmc, lambda_h, lambda_J, lambda_group, n_eff,
                   alphabet, weights_all, target_seq, index_list, fi, h, fij_tri, J_tri, "<f4")


def write_mean_field_model_file(path, L, q, n_valid, theta, pseudo_count, n_eff, alphabet, weights, target_seq,
                                index_list, fi, h, fij_tri, J_tri, precision="float32"):
    """A mean-field model in the plmc_v2 layout, as the reference's MeanFieldCouplingsModel.to_file writes it:
    lambda_h = -pseudo_count (the reference's reader takes lambda_h < 0 as "mean-field model"), lambda_J,
    lambda_group and num_iter = -1, N_invalid = 0 with the weights of the valid sequences only; the real-valued
    fields in ``precision`` (float16 / float32 / float64)."""
    dtype = np.dtype(precision).newbyteorder("<")
    if dtype.kind != "f":
        raise ValueError("precision must be a floating-point type")
    _write_plmc_v2(path, L, q, n_valid, 0, -1, theta, -pseudo_count, -1, -1, n_eff, alphabet, weights, target_seq,
                   index_list, fi, h, fij_tri, J_tri, dtype)


def _write_plmc_v2(path, L, q, n_valid, n_invalid, num_iter, theta, lambda_h, lambda_J, lambda_group, n_eff,
                   alphabet, weights_all, target_seq, index_list, fi, h, fij_tri, J_tri, dtype):
    alphabet = str(alphabet)
    target_seq = str(target_seq)
    npairs = L * (L - 1) // 2
    fi = np.asarray(fi, dtype=dtype).reshape(L, q)
    h = np.asarray(h, dtype=dtype).reshape(L, q)
    fij_tri = np.asarray(fij_tri, dtype=dtype).reshape(npairs, q, q)
    J_tri = np.asarray(J_tri, dtype=dtype).reshape(npairs, q, q)
    weights_all = np.asarray(weights_all, dtype=dtype)
    if len(alphabet) != q or len(target_seq) != L or len(index_list) != L:
        raise ValueError("inconsistent model dimensions")
    if weights_all.shape != (n_valid + n_invalid,):
        raise ValueError("weights must cover valid + invalid sequences")
    with open(path, "wb") as f:
        np.array([L, q, n_valid, n_invalid, num_iter], dtype="<i4").tofile(f)
        np.array([theta, lambda_h, lambda_J, lambda_group, n_eff], dtype=dtype).tofile(f)
        f.write(alphabet.encode("ascii"))
        weights_all.tofile(f)
        f.write(target_seq.encode("ascii"))
        np.asarray(index_list, dtype="<i4").tofile(f)
        fi.tofile(f)
        h.tofile(f)
        fij_tri.tofile(f)
        J_tri.tofile(f)


def model_file_size(L, q, n_seqs):
    return 40 + q + 4 * n_seqs + L + 4 * L + 8 * L * q + 8 * (L * (L - 1) // 2) * q * q


def normalise_frequencies(fi_counts, fij_counts, n_eff, ignore_gaps):
    """Weighted counts -> f_i, f_ij as stored in the .model (SURVEY.md row a6): divide by N_eff when the
    gap is a model state (evcouplings/align/alignment.py:1106,1144); with ignore_gaps normalise each
    site / pair over the non-gap weight."""
    fi_counts = np.asarray(fi_counts, dtype=np.float64)
    fij_counts = np.asarray(fij_counts, dtype=np.float64)
    if ignore_gaps:
        si = fi_counts.sum(axis=1, keepdims=True)
        sij = fij_counts.sum(axis=(1, 2), keepdims=True)
        fi = np.divide(fi_counts, si, out=np.zeros_like(fi_counts), where=si > 0)
        fij = np.divide(fij_counts, sij, out=np.zeros_like(fij_counts), where=sij > 0)
    else:
        fi = fi_counts / n_eff
        fij = fij_counts / n_eff
    return fi, fij
