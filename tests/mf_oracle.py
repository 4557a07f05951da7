"""
Mean-field DCA in numpy float64, restated from its formulas (the test oracle of evcouplings_b200.mean_field and
of the kernels in csrc/mean_field.cu).  Codes are (N, L) integers in alphabet order, gap first; the last state
q-1 is the reference state of the model.

    f_i, f_ij        weighted one-hot frequencies over N_eff = sum(w), f_ii = diag(f_i)
    rf_i             (1-pc) f_i + pc/q
    rf_ij            (1-pc) f_ij + pc/q^2  (i != j),   (1-pc) f_i[a] d_ab + (pc/q) d_ab  (i == j)
    C                rf_ij[a][b] - rf_i[a] rf_j[b],  a, b < q-1,  index i*(q-1)+a
    J_ij[a][b]       -inv(C)[(i,a),(j,b)],  0 on the last state
    h_i[a]           log(rf_i[a] / rf_i[q-1]) - sum_{j != i} sum_b J_ij[a][b] rf_j[b]
    DI_ij            two-site model P ~ exp(J_ij) * (u v^T) with u, v from the fixed point
                     u <- rf_i / (E v), v <- rf_j / (E^T u) (both from the previous iterate, each normalised to
                     sum 1, from 1/q, until the max-abs change is <= 1e-4); DI = sum P log((P+1e-100)/(rf_i rf_j^T+1e-100))
    FN, CN           Frobenius norm of the zero-sum-gauge J_ij, and its average product correction
    MI               sum_{p>0} f_ij log(f_ij / (f_i f_j^T)), and its average product correction
"""
import numpy as np

TINY = 1.0e-100
DI_EPSILON = 1.0e-4


def cluster_weights(codes, theta):
    """1 / #{t : identity(s, t) >= theta} (self included)."""
    codes = np.asarray(codes)
    N, L = codes.shape
    q = int(codes.max()) + 1
    X = np.zeros((N, L * q), dtype=np.float32)
    X[np.repeat(np.arange(N), L), (np.arange(L) * q + codes).ravel()] = 1.0
    ident = X @ X.T                                  # exact small integers in float32
    return 1.0 / (ident.astype(np.float64) / float(L) >= theta).sum(axis=1)


def frequencies(codes, w, q):
    """f_i (L, q) and f_ij (L, L, q, q), normalised by sum(w)."""
    codes = np.asarray(codes)
    N, L = codes.shape
    X = np.zeros((N, L * q))
    X[np.repeat(np.arange(N), L), (np.arange(L) * q + codes).ravel()] = 1.0
    F = (X * w[:, None]).T @ X / w.sum()
    fij = F.reshape(L, q, L, q).transpose(0, 2, 1, 3).copy()
    fi = np.einsum("iiaa->ia", fij).copy()
    return fi, fij


def covariance(fi, fij, pc):
    L, q = fi.shape
    rfi = (1.0 - pc) * fi + pc / q
    rfij = (1.0 - pc) * fij + pc / q ** 2
    for i in range(L):
        rfij[i, i] = np.diag((1.0 - pc) * fi[i] + pc / q)
    Q = q - 1
    C = (rfij[:, :, :Q, :Q] - rfi[:, None, :Q, None] * rfi[None, :, None, :Q])
    return rfi, C.transpose(0, 2, 1, 3).reshape(L * Q, L * Q)


def couplings_fields(Cinv, rfi):
    L, q = rfi.shape
    Q = q - 1
    J = np.zeros((L, L, q, q))
    J[:, :, :Q, :Q] = -Cinv.reshape(L, Q, L, Q).transpose(0, 2, 1, 3)
    Joff = J.copy()
    Joff[np.arange(L), np.arange(L)] = 0.0
    h = np.log(rfi / rfi[:, -1:]) - np.einsum("ijab,jb->ia", Joff, rfi)
    return J, h


def two_site(E, fi, fj):
    q = len(fi)
    u = np.full(q, 1.0 / q)
    v = np.full(q, 1.0 / q)
    diff, it = 1.0, 0
    while diff > DI_EPSILON:
        un = fi / (E @ v)
        vn = fj / (u @ E)
        un = un / un.sum()
        vn = vn / vn.sum()
        diff = max(np.abs(un - u).max(), np.abs(vn - v).max())
        u, v = un, vn
        it += 1
    return u, v, it


def direct_information(J, rfi):
    """DI (L, L) and the fixed-point iteration count of each pair (L, L)."""
    L, q = rfi.shape
    di = np.zeros((L, L))
    iters = np.zeros((L, L), dtype=np.int64)
    for i in range(L - 1):
        for j in range(i + 1, L):
            E = np.exp(J[i, j])
            u, v, it = two_site(E, rfi[i], rfi[j])
            P = E * np.outer(u, v)
            P = P / P.sum()
            di[i, j] = di[j, i] = np.sum(P * np.log((P + TINY) / (np.outer(rfi[i], rfi[j]) + TINY)))
            iters[i, j] = iters[j, i] = it
    return di, iters


def apc(M):
    L = M.shape[0]
    col = M.mean(axis=0) * L / (L - 1)
    out = M - np.outer(col, col) / (M.mean() * L / (L - 1))
    out[np.diag_indices(L)] = 0.0
    return out


def fn_mi(J, fi, fij):
    L, q = fi.shape
    J0 = (J - J.mean(axis=3, keepdims=True) - J.mean(axis=2, keepdims=True) + J.mean(axis=(2, 3), keepdims=True))
    fn = np.sqrt((J0 ** 2).sum(axis=(2, 3)))
    fn[np.diag_indices(L)] = 0.0
    m = fi[:, None, :, None] * fi[None, :, None, :]
    with np.errstate(divide="ignore", invalid="ignore"):
        t = np.where(fij > 0, fij * np.log(np.where(fij > 0, fij, 1.0) / np.where(fij > 0, m, 1.0)), 0.0)
    mi = t.sum(axis=(2, 3))
    mi[np.diag_indices(L)] = 0.0
    return fn, mi


def fit(codes, w, q, pc, di=True):
    """Everything the mean-field model holds, as float64 arrays (L x L matrices for the pair scores)."""
    w = np.asarray(w, dtype=np.float64)
    fi, fij = frequencies(codes, w, q)
    rfi, C = covariance(fi, fij, pc)
    Cinv = np.linalg.inv(C)
    J, h = couplings_fields(Cinv, rfi)
    fn, mi = fn_mi(J, fi, fij)
    out = dict(fi=fi, fij=fij, rfi=rfi, C=C, Cinv=Cinv, J=J, h=h, fn=fn, cn=apc(fn), mi_raw=mi, mi_apc=apc(mi),
               n_eff=w.sum())
    if di:
        out["di"], out["di_iters"] = direct_information(J, rfi)
    return out


def tri(M):
    """(L, L, ...) -> pairs i<j in row-major order."""
    iu, ju = np.triu_indices(M.shape[0], 1)
    return M[iu, ju]
