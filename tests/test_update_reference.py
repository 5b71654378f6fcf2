"""The extended-precision reference of one stacked update (oracle/update_ref.py), checked without a GPU:
against mpmath at 40 digits, against the fp64 forms, and the sensitivity of the bar the kernel tests use."""
import mpmath
import numpy as np
import pytest

from oracle import update_ref as U


def _case(seed, types, sel):
    rng = np.random.default_rng(seed)
    types = np.asarray(types)
    x, xp, P = U.random_filter(rng, types)
    h, z, Hc = U.random_features(rng, len(types))
    return x, xp, P, types, h, z, Hc, list(sel)


def _mp_update(x0, P, types, h, z, Hc, sel):
    """mc/update.m:3-32 (R = I) in mpmath at 40 digits, the textbook form: K = P H' inv(S), P - K S K', J P J'."""
    mpmath.mp.dps = 40
    H, _ = U.stack(types, h, z, Hc, sel)
    nu = [mpmath.mpf(z[i][r]) - mpmath.mpf(h[i][r]) for i in sel for r in range(2)]
    n, k = P.shape[0], H.shape[0]
    Hm = mpmath.matrix(H.tolist())
    Pm = mpmath.matrix(P.tolist())
    S = Hm * Pm * Hm.T + mpmath.eye(k)
    K = Pm * Hm.T * mpmath.inverse(S)
    x1 = mpmath.matrix(x0.tolist()) + K * mpmath.matrix(nu)
    P1 = Pm - K * S * K.T
    q = [x1[3 + i] for i in range(4)]
    r, a, b, c = q
    nn = r * r + a * a + b * b + c * c
    J = mpmath.matrix([[a * a + b * b + c * c, -r * a, -r * b, -r * c],
                       [-a * r, r * r + b * b + c * c, -a * b, -a * c],
                       [-b * r, -b * a, r * r + a * a + c * c, -b * c],
                       [-c * r, -c * a, -c * b, r * r + a * a + b * b]]) * nn ** mpmath.mpf(-1.5)
    Jf = mpmath.eye(n)
    for i in range(4):
        for j in range(4):
            Jf[3 + i, 3 + j] = J[i, j]
    P1 = Jf * P1 * Jf.T
    nq = mpmath.sqrt(nn)
    for i in range(4):
        x1[3 + i] = x1[3 + i] / nq
    return x1, P1


@pytest.mark.parametrize("types,sel,which_prior", [
    ([1], [0], 0),                       # n = 19, k = 2
    ([2], [0], 1),                       # n = 16, k = 2
    ([2, 2, 1], [0, 2], 0),              # n = 25, k = 4
    ([1, 2, 1, 1], [0, 1, 2, 3], 1),     # n = 34, k = 8
    ([1, 1, 2, 1, 2, 2, 1], [0, 3, 6], 0),   # n = 40, k = 6
])
def test_reference_matches_mpmath(types, sel, which_prior):
    x, xp, P, types, h, z, Hc, sel = _case(11 + len(types), types, sel)
    xr, Pr = U.update_ref(x, P, types, h, z, Hc, sel, which_prior, xp)
    xm, Pm = _mp_update(xp if which_prior else x, P, types, h, z, Hc, sel)
    n = P.shape[0]
    d = [mpmath.sqrt(mpmath.mpf(P[i, i])) for i in range(n)]
    # x relative to the larger of |x_i| and its prior deviation; P relative to sqrt(P_ii P_jj)
    ex = max(abs(mpmath.mpf(float(xr[i])) + mpmath.mpf(float(xr[i] - np.longdouble(float(xr[i])))) - xm[i])
             / max(abs(xm[i]), d[i]) for i in range(n))
    eP = max(abs(mpmath.mpf(float(Pr[i, j])) + mpmath.mpf(float(Pr[i, j] - np.longdouble(float(Pr[i, j])))) - Pm[i, j])
             / (d[i] * d[j]) for i in range(n) for j in range(n))
    assert ex <= 1e-17 and eP <= 1e-17, (float(ex), float(eP))


# shapes of the kernel tests: small and large k, mixed maps, n on and off the 64-wide tiles
FP64_SHAPES = [(40, 1), (100, 17), (100, 33), (130, 56), (100, 100)]


def _shape_case(seed, nfeat, ns):
    rng = np.random.default_rng(seed)
    return _case(seed, rng.choice([1, 2], nfeat), U.scattered_selection(rng, nfeat, ns))


@pytest.mark.parametrize("nfeat,ns", FP64_SHAPES)
def test_reference_agrees_with_fp64(nfeat, ns):
    """Both fp64 forms stay within a few hundred fp64 roundings of the reference (scaled errors): the reference and the
    fp64 arithmetic describe the same update, and what separates them is rounding."""
    x, xp, P, types, h, z, Hc, sel = _shape_case(1000 + nfeat + ns, nfeat, ns)
    xr, Pr = U.update_ref(x, P, types, h, z, Hc, sel)
    bound = 512 * np.finfo(np.float64).eps * (2 * ns + 13)
    for f in (U.fp64_same_form, U.oracle_fp64):
        xf, Pf = f(x, P, types, h, z, Hc, sel)
        ex, eP = U.scaled_err(xf, Pf, xr, Pr, P)
        # x_i itself is stored in fp64: its error is measured against the larger of |x_i| and sqrt(P_ii)
        ex_abs = np.abs(xf - xr) / np.maximum(np.abs(xr), np.sqrt(np.diag(P)))
        assert eP <= bound and float(ex_abs.max()) <= bound, (f.__name__, float(ex_abs.max()), eP, bound)
        assert eP > 0.0 and ex > 0.0   # the reference is not itself fp64


@pytest.mark.parametrize("mutation", U.MUTATIONS)
def test_bar_catches_mutations(mutation):
    """Each mistake a kernel could make, applied to the fp64 form, fails the kernel tests' bar by at least 100x."""
    for nfeat, ns in [(40, 17), (100, 33)]:
        x, xp, P, types, h, z, Hc, sel = _shape_case(2000 + nfeat, nfeat, ns)
        xr, Pr = U.update_ref(x, P, types, h, z, Hc, sel)
        bx, bP = U.bar(x, P, types, h, z, Hc, sel, xr, Pr)
        ex0, eP0 = U.scaled_err(*U.fp64_same_form(x, P, types, h, z, Hc, sel), xr, Pr, P)
        assert ex0 <= bx and eP0 <= bP
        ex, eP = U.scaled_err(*U.fp64_same_form(x, P, types, h, z, Hc, sel, mutation=mutation), xr, Pr, P)
        assert max(ex / bx, eP / bP) >= 100.0, (mutation, ex, bx, eP, bP)
