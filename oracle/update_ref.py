"""Extended-precision reference of one stacked EKF update (mc/update.m:3-32 with R = I), for the kernel tests.

`update_ref` evaluates the update in np.longdouble (80-bit extended on x86-64, eps 1.1e-19) from the compact inputs
the device works on: per feature h, z and the compact Jacobian Hc [2][13] (7 camera columns, then the 6 (inverse
depth) or 3 (Cartesian) columns of the feature's own block), and the list of selected features.  numpy has no
longdouble LAPACK, so the Cholesky factor and the triangular solve are written out here.

`fp64_same_form` runs the device's algebra in float64 (S = L L', W = inv(L) H P, x + W' inv(L) nu, J P J' - (W J')'(W J'),
then q / |q|).  Its error against `update_ref` is what one correct fp64 implementation of that algebra loses; the
kernel tests bound the device's error by a multiple of it.  The `mutation` argument breaks it on purpose, so that a
test can show that the bar would catch a kernel making the same mistake.

Errors are measured by `scaled_err`: |dx_i| / sqrt(P_ii) and |dP_ij| / sqrt(P_ii P_jj) with P the prior covariance, so
that an error confined to a block of small variance (the camera block) counts as much as one in a large block.
"""
import numpy as np
import scipy.linalg

from oracle import ekf_oracle as O

XV = 13
# The device's error may be at most BAR_MULT times the larger error of the two fp64 forms, and never needs to be below
# BAR_FLOOR (x and P separately, both measured by scaled_err against update_ref).
BAR_MULT = 8.0
BAR_FLOOR = 1e-15
MUTATIONS =("drop_last_row", "skip_last_column", "linv_fp32", "skip_normjac")


def feature_offsets(types):
    """State offset and block width of every feature (types: 1 = inverse depth, 2 = Cartesian, in feature order)."""
    off, w = [], []
    pos = XV
    for t in types:
        wt = 6 if int(t) == 1 else 3
        off.append(pos)
        w.append(wt)
        pos += wt
    return np.array(off, dtype=int), np.array(w, dtype=int), pos


def stack(types, h, z, Hc, sel, dtype=np.float64):
    """Dense H (2*len(sel) x n) scattered from the compact Jacobians, and nu = z - h, of the selected features."""
    off, w, n = feature_offsets(types)
    sel = [int(i) for i in sel]
    H = np.zeros((2 * len(sel), n), dtype=dtype)
    nu = np.zeros(2 * len(sel), dtype=dtype)
    for j, i in enumerate(sel):
        for r in range(2):
            H[2 * j + r, :7] = np.asarray(Hc[i][r][:7], dtype=dtype)
            H[2 * j + r, off[i]:off[i] + w[i]] = np.asarray(Hc[i][r][7:7 + w[i]], dtype=dtype)
            nu[2 * j + r] = dtype(z[i][r]) - dtype(h[i][r])
    return H, nu


def _normjac(q):
    r, x, y, zq = q
    nn = r * r + x * x + y * y + zq * zq
    sc = 1 / (nn * np.sqrt(nn))
    return sc * np.array([[x * x + y * y + zq * zq, -r * x, -r * y, -r * zq],
                          [-x * r, r * r + y * y + zq * zq, -x * y, -x * zq],
                          [-y * r, -y * x, r * r + x * x + zq * zq, -y * zq],
                          [-zq * r, -zq * x, -zq * y, r * r + x * x + y * y]], dtype=q.dtype)


def _apply_normjac(x, P, J):
    """P <- J P J' with J = blkdiag(I3, J, I), then q <- q / |q| (mc/update.m:18-24)."""
    P = P.copy()
    P[3:7, :] = J @ P[3:7, :]
    P[:, 3:7] = P[:, 3:7] @ J.T
    x = x.copy()
    q = x[3:7]
    x[3:7] = q / np.sqrt(np.sum(q * q))
    return x, P


def _chol_ld(S):
    k = S.shape[0]
    L = np.zeros_like(S)
    for j in range(k):
        d = S[j, j] - np.dot(L[j, :j], L[j, :j])
        if not d > 0:
            raise np.linalg.LinAlgError("S is not positive definite at pivot %d" % j)
        L[j, j] = np.sqrt(d)
        L[j + 1:, j] = (S[j + 1:, j] - L[j + 1:, :j] @ L[j, :j]) / L[j, j]
    return L


def _fwd_ld(L, B):
    """inv(L) B by forward substitution (B: k x m)."""
    X = np.zeros_like(B)
    for i in range(L.shape[0]):
        X[i] = (B[i] - L[i, :i] @ X[:i]) / L[i, i]
    return X


def update_ref(x, P, types, h, z, Hc, sel, which_prior=0, xp=None):
    """x+, P+ of mc/update.m:3-32 (R = I) in extended precision, returned as longdouble arrays.

    The update starts from x (which_prior = 0) or from xp (which_prior = 1, the li update's x_k_km1); P is the
    covariance it starts from either way.  No selected feature: the starting state is passed through."""
    ld = np.longdouble
    x0 = np.asarray(xp if which_prior else x, dtype=ld).copy()
    P0 = np.asarray(P, dtype=ld)
    n = P0.shape[0]
    if len(sel) == 0:
        return x0, P0.copy()
    off, w, n_f = feature_offsets(types)
    assert n_f == n, (n_f, n)
    H, nu = stack(types, h, z, Hc, sel, dtype=ld)
    k = H.shape[0]
    # H P through the (at most) 13 non-zero columns of each row
    HP = np.zeros((k, n), dtype=ld)
    for r in range(k):
        cols = np.nonzero(H[r])[0]
        HP[r] = H[r, cols] @ P0[cols]
    S = HP @ H.T + np.eye(k, dtype=ld)
    S = 0.5 * (S + S.T)
    L = _chol_ld(S)
    Wm = _fwd_ld(L, HP)                          # inv(L) H P
    y = _fwd_ld(L, nu[:, None])[:, 0]            # inv(L) nu
    x1 = x0 + Wm.T @ y                           # x + K nu,       K = P H' inv(S)
    P1 = P0 - Wm.T @ Wm                          # P - K S K'
    P1 = np.tril(P1) + np.tril(P1, -1).T
    return _apply_normjac(x1, P1, _normjac(x1[3:7]))


def fp64_same_form(x, P, types, h, z, Hc, sel, which_prior=0, xp=None, mutation=None):
    """The device's algebra in float64: S = L L', W = inv(L) H P, y = inv(L) nu, x+ = x + W'y, then
    P+ = J P J' - (W J')'(W J') and q / |q| with J = normJac(q+) (un-normalised q+).

    mutation (test of the bar's sensitivity): "drop_last_row" (the last stacked row is left out), "skip_last_column"
    (the last state entry and covariance row/column are not updated), "linv_fp32" (inv(L) rounded to float32),
    "skip_normjac" (no normalisation Jacobian on P)."""
    assert mutation is None or mutation in MUTATIONS, mutation
    x0 = np.array(xp if which_prior else x, dtype=np.float64)
    P0 = np.asarray(P, dtype=np.float64)
    if len(sel) == 0:
        return x0, P0.copy()
    H, nu = stack(types, h, z, Hc, sel)
    if mutation == "drop_last_row":
        H, nu = H[:-1], nu[:-1]
    k = H.shape[0]
    HP = H @ P0
    S = HP @ H.T + np.eye(k)
    L = np.linalg.cholesky(0.5 * (S + S.T))
    Li = scipy.linalg.solve_triangular(L, np.eye(k), lower=True)
    if mutation == "linv_fp32":
        Li = Li.astype(np.float32).astype(np.float64)
    Wm = Li @ HP
    y = Li @ nu
    if mutation == "skip_last_column":
        Wm[:, -1] = 0.0
    x1 = x0 + Wm.T @ y
    J = np.eye(4) if mutation == "skip_normjac" else _normjac(x1[3:7])
    Wm[:, 3:7] = Wm[:, 3:7] @ J.T
    JPJ = P0.copy()
    JPJ[3:7, :] = J @ JPJ[3:7, :]
    JPJ[:, 3:7] = JPJ[:, 3:7] @ J.T
    P1 = JPJ - Wm.T @ Wm
    P1 = np.tril(P1) + np.tril(P1, -1).T
    x1[3:7] = x1[3:7] / np.linalg.norm(x1[3:7])
    return x1, P1


def oracle_fp64(x, P, types, h, z, Hc, sel, which_prior=0, xp=None):
    """ekf_oracle.update (explicit inv(S), P - K S K') on the same inputs."""
    x0 = np.array(xp if which_prior else x, dtype=np.float64)
    P0 = np.asarray(P, dtype=np.float64)
    if len(sel) == 0:
        return x0, P0.copy()
    H, nu = stack(types, h, z, Hc, sel)
    xo, Po, _ = O.update(x0, P0, H, np.eye(len(nu)), nu, np.zeros_like(nu))
    return xo, Po


def random_filter(rng, types, n_pad=None):
    """Seeded inputs of one filter with the given feature types: x (unit quaternion), a second state xp, and
    P = A A' with row scales graded from 1e-6 (camera) to 1 (last feature), zero-padded to n_pad."""
    _, _, n = feature_offsets(types)
    n_pad = n if n_pad is None else n_pad
    R = rng.standard_normal((n, n)) / np.sqrt(n)
    d = 10.0 ** np.linspace(-6.0, 0.0, n)
    A = d[:, None] * np.linalg.cholesky(R @ R.T + 0.5 * np.eye(n))
    P = np.zeros((n_pad, n_pad))
    P[:n, :n] = np.tril(A @ A.T) + np.tril(A @ A.T, -1).T
    x = np.zeros(n_pad)
    xp = np.zeros(n_pad)
    for v in (x, xp):
        v[:n] = rng.standard_normal(n)
        v[3:7] /= np.linalg.norm(v[3:7])
    return x, xp, P


def random_features(rng, nfeat):
    """h, z [nfeat][2] and compact Jacobians Hc [nfeat][2][13] of order 1 (the columns past a Cartesian feature's
    3-wide block hold values too: the update must not read them)."""
    h = rng.standard_normal((nfeat, 2))
    z = h + rng.standard_normal((nfeat, 2))
    Hc = rng.standard_normal((nfeat, 2, 13))
    return h, z, Hc


def scattered_selection(rng, nfeat, ns):
    """ns of nfeat feature indices, ascending, always the first and the last one (the last one alone for ns = 1)."""
    if ns == 0:
        return []
    if ns == 1:
        return [nfeat - 1]
    mid = rng.choice(np.arange(1, nfeat - 1), ns - 2, replace=False) if ns > 2 else []
    return sorted([0, nfeat - 1] + [int(i) for i in mid])


def scaled_err(x, P, x_ref, P_ref, P_prior):
    """(max_i |x_i - x_ref_i| / sqrt(P_ii), max_ij |P_ij - P_ref_ij| / sqrt(P_ii P_jj)), P = P_prior."""
    d = np.sqrt(np.diag(np.asarray(P_prior, dtype=np.longdouble)))
    ex = np.abs(np.asarray(x, dtype=np.longdouble) - x_ref) / d
    eP = np.abs(np.asarray(P, dtype=np.longdouble) - P_ref) / np.outer(d, d)
    return float(ex.max()), float(eP.max())


def bar(x, P, types, h, z, Hc, sel, x_ref, P_ref, which_prior=0, xp=None):
    """(bar on the x error, bar on the P error) of one update: BAR_MULT times the larger scaled error of
    fp64_same_form and oracle_fp64 against the extended-precision result, at least BAR_FLOOR."""
    errs = [scaled_err(*f(x, P, types, h, z, Hc, sel, which_prior, xp), x_ref, P_ref, P)
            for f in (fp64_same_form, oracle_fp64)]
    return tuple(max(BAR_MULT * max(e[i] for e in errs), BAR_FLOOR) for i in range(2))
