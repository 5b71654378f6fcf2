"""The EKF update kernels (launch_update, k_update.cu) against the extended-precision reference of oracle/update_ref.py,
at every stacked size k where the choice of Cholesky, W or S-pair kernel changes, and at state sizes n on both sides of
the 64-wide tile and 8-wide block edges of the covariance downdate.

A case is a batch in which every filter gets its own (n, k): seeded x, P = A A' with row scales from 1e-6 (camera) to
1, compact Jacobians of order 1, and a scattered selection of k / 2 features that always holds the first and the last
one.  Each case runs the li update (which_prior = 1) and then the hi update (which_prior = 0) through the C ABI; each
update's reference starts from the device state downloaded just before it.  Per filter the device's error, scaled by
the prior (|dx_i| / sqrt(P_ii), |dP_ij| / sqrt(P_ii P_jj)), must stay within update_ref.bar: 8x the error of the same
algebra in fp64 or of ekf_oracle.update, whichever is larger.  Exact on every filter: P bit-symmetric, rows and
columns [n, n_max) zero, and a filter without a selected feature keeps its state bit for bit.

`chol_variant` / `w_variant` / `pairs_variant` restate the selection rule of launch_update; every context asserts that
the variants it targets receive filters on both sides of their bounds, and a profiler run asserts that they launched.
"""
import numpy as np
import pytest

from oracle import update_ref as U

pytestmark = pytest.mark.gpu

F_HAS_H, F_LI, F_HI = 1, 8, 16
WORST = {}   # (context, update, kernel family) -> worst device / fp64 error ratio


# ---- the selection rule of launch_update (k_update.cu, common.cuh) ---------------------------------------------------
def lockstep(B, N):
    return B < 128 and 2 * N >= 256


def chol_variant(B, N, hi, k):
    """(kernel, KMIN, KM): the Cholesky kernel that takes a filter with k stacked rows, and the k range it takes."""
    kmax = 2 * N
    if k == 0:
        return None
    if lockstep(B, N):
        return ("k_cb", 0, kmax)
    use_mid = kmax > 112
    large = use_mid and kmax > 144
    kres = 200 if large else 144
    if k > kres:
        return ("k_chol", kres, kmax)
    if hi and k <= 32:
        return ("k_chol_w32", 0, 32)
    bounds = ([0, 112, 144, 200] if use_mid else [0, 144]) if not hi else ([32, 48, 112, 144, 200] if use_mid else [32, 48, 144])
    for lo, up in zip(bounds, bounds[1:]):
        if lo < k <= up:
            return ("k_chol_sm<%d,%d>" % (up, lo), lo, up)
    raise AssertionError((B, N, hi, k))


def w_variant(k):
    if k == 0:
        return None
    return ("k_w_small", 0, 32) if k <= 32 else ("k_gemm/%d" % ((k + 63) // 64), 32, None)


def pairs_variant(B, N):
    return "k_upd_pairs" if B < 296 else ("k_upd_S staged" if N <= 128 else "k_upd_S unstaged")


def assert_bounds_covered(B, N, ks, hi, targets):
    """Each targeted Cholesky variant receives a filter at its lowest and highest k and one just outside each bound
    (where such a k exists: 0 <= k <= 2 N)."""
    kmax = 2 * N
    got = {}
    for k in ks:
        v = chol_variant(B, N, hi, k)
        if v is not None:
            got.setdefault(v[0], set()).add(k)
    for name in targets:
        lo, up = next(chol_variant(B, N, hi, k)[1:] for k in ks if chol_variant(B, N, hi, k) and chol_variant(B, N, hi, k)[0] == name)
        up = min(up, kmax)
        need_in = {lo + 2, up}
        need_out = {k for k in (lo, up + 2) if 0 <= k <= kmax}
        assert need_in <= got[name], (name, sorted(got[name]), need_in)
        assert need_out <= set(ks), (name, need_out)


# ---- cases ------------------------------------------------------------------------------------------------------------
class Case:
    """Feature types, x, xp, P of every filter of a batch (n_max padded), and per update the features and selection."""

    def __init__(self, seed, N, ks, nfeat=None, n_max=None, cart=0.5, types=None):
        rng = np.random.default_rng(seed)
        self.N, self.B = N, len(ks)
        self.types = np.zeros((self.B, N), dtype=np.uint8)
        self.nfeat = []
        for b, k in enumerate(ks):
            if types is not None:
                t = types[b]
            else:
                nf = nfeat[b] if nfeat is not None else min(N, k // 2 + int(rng.integers(0, 6)))
                t = np.where(rng.random(nf) < cart, 2, 1)
            self.types[b, :len(t)] = t
            self.nfeat.append(len(t))
        self.n = [U.feature_offsets(self.types[b, :self.nfeat[b]])[2] for b in range(self.B)]
        self.n_max = n_max or min(13 + 6 * N, max(self.n) + 5)
        self.x = np.zeros((self.B, self.n_max))
        self.xp = np.zeros((self.B, self.n_max))
        self.P = np.zeros((self.B, self.n_max, self.n_max))
        for b in range(self.B):
            x, xp, P = U.random_filter(rng, self.types[b, :self.nfeat[b]])
            n = self.n[b]
            self.x[b, :n], self.xp[b, :n], self.P[b, :n, :n] = x, xp, P
        self.rng = rng

    def features(self, ks):
        """h, z, Hc and the selection of one update, k[b] / 2 scattered features per filter."""
        h = np.zeros((self.B, self.N, 2))
        z = np.zeros((self.B, self.N, 2))
        Hc = np.zeros((self.B, self.N, 2, 13))
        sel = []
        for b, k in enumerate(ks):
            nf = self.nfeat[b]
            assert k // 2 <= nf, (b, k, nf)
            if nf:
                h[b, :nf], z[b, :nf], Hc[b, :nf] = U.random_features(self.rng, nf)
            sel.append(U.scattered_selection(self.rng, nf, k // 2))
        return h, z, Hc, sel

    def upload(self, bank, b0=0, nb=None):
        nb = self.B - b0 if nb is None else nb
        s = slice(b0, b0 + nb)
        bank.upload_feature_types(self.types[s], np.array(self.nfeat[s], dtype=np.int32), b0=b0)
        bank.upload_state(self.x[s], self.P[s], b0=b0)
        bank.upload_state(self.xp[s], which=1, b0=b0)


def make_bank(case, B=None):
    import ekf_slam_b200 as pkg
    return pkg.FilterBank(B or case.B, case.N, case.n_max)


def run_update(bank, case, ks, hi, tag, check=True, feats=None):
    """One masked update of every filter of the bank (the first len(ks) filters carry the case; the rest are left with
    no selected feature).  Returns the device's x, P after it."""
    B = bank.B
    h, z, Hc, sel = feats if feats is not None else case.features(ks)
    bit, other = (F_HI, F_LI) if hi else (F_LI, F_HI)
    flags = np.zeros((case.B, case.N), dtype=np.uint8)
    for b in range(case.B):
        flags[b, :case.nfeat[b]] = F_HAS_H | other      # not selected by this update's mask
        flags[b, sel[b]] = F_HAS_H | bit
    x0, P0, _ = bank.download_state()
    xp0 = bank.download_state(which=1, want_P=False)[0]
    bank.upload_features(h=h, Hc=Hc, z=z, flags=flags)
    bank.hp(need=F_HAS_H | bit)
    which_prior = 0 if hi else 1
    bank.update_masked(bit, which_prior)
    x1, P1, _ = bank.download_state()
    st = bank.download_stats()
    if not check:
        return x1, P1
    assert B == case.B
    for b in range(B):
        n, k = case.n[b], 2 * len(sel[b])
        assert st["n_hi" if hi else "n_li"][b] == k // 2, (tag, b)
        assert st["status"][b] == 0, (tag, b, st["status"][b])
        assert np.array_equal(P1[b], P1[b].T), (tag, b, "P not bit-symmetric")
        assert not P1[b, n:].any() and not P1[b, :, n:].any() and not x1[b, n:].any(), (tag, b, "padding written")
        if k == 0:
            assert np.array_equal(P1[b], P0[b]), (tag, b)
            assert np.array_equal(x1[b, :n], (xp0 if which_prior else x0)[b, :n]), (tag, b)
            continue
        args = (x0[b, :n], P0[b, :n, :n], case.types[b, :case.nfeat[b]], h[b], z[b], Hc[b], sel[b])
        xr, Pr = U.update_ref(*args, which_prior, xp0[b, :n])
        bx, bP = U.bar(*args, xr, Pr, which_prior, xp0[b, :n])
        ex, eP = U.scaled_err(x1[b, :n], P1[b, :n, :n], xr, Pr, P0[b, :n, :n])
        fam = (tag, "hi" if hi else "li", chol_variant(B, case.N, hi, k)[0] + " + " + w_variant(k)[0])
        ratio = max(ex / bx, eP / bP) * U.BAR_MULT
        WORST[fam] = max(WORST.get(fam, 0.0), ratio)
        assert ex <= bx and eP <= bP, "%s filter %d (n %d, k %d): x %.2e (bar %.2e), P %.2e (bar %.2e)" % (
            fam, b, n, k, ex, bx, eP, bP)
    return x1, P1


def run_case(case, ks_li, ks_hi, tag, bank=None):
    own = bank is None
    bank = bank or make_bank(case)
    case.upload(bank)
    run_update(bank, case, ks_li, False, tag)
    run_update(bank, case, ks_hi, True, tag)
    if own:
        bank.close()


def launched_kernels(fn):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
    return {e.name.replace(" ", "") for e in prof.events()}


def has_kernel(names, stem, *targs):
    """Demangled `stem<a,b,...` or mangled `stemILia...` among the launched kernel names."""
    if stem.endswith("("):   # a plain function of that exact name
        dem, man = stem, "%d%s7DevView" % (len(stem) - 1, stem[:-1])
    else:
        dem = stem + ("<" + ",".join(str(a) for a in targs) if targs else "")
        man = "%d%s" % (len(stem), stem) + ("I" + "".join("Li%dE" % a for a in targs) if targs else "")
    return any(dem in s or man in s for s in names)


@pytest.fixture(scope="module", autouse=True)
def report():
    yield
    print("\nworst device / fp64 error ratio per context, update and kernel family:")
    for fam in sorted(WORST):
        print("  %-14s %s  %-34s %.2f" % (fam[0], fam[1], fam[2], WORST[fam]))


# ---- contexts ---------------------------------------------------------------------------------------------------------
def _fill(ks, B, seed):
    """ks on the first filters, 0-3 selected features on the rest (at least one filter with none)."""
    rng = np.random.default_rng(seed)
    fill = [0] + [2 * int(v) for v in rng.integers(0, 4, B - len(ks) - 1)] if B > len(ks) else []
    return list(ks) + fill


K_N56 = [2, 4, 30, 32, 34, 46, 48, 50, 62, 64, 66, 110, 112]
K_N100 = [2, 32, 34, 48, 50, 64, 66, 110, 112, 114, 128, 130, 142, 144, 146, 192, 194, 198, 200]


def test_b24_n56_small_kernels():
    """kmax 112: li k_chol_sm<144,0>; hi k_chol_w32 / k_chol_sm<48,32> / k_chol_sm<144,48>; k_w_small and k_gemm with one
    and two row tiles; the pair loop as k_upd_pairs."""
    B, N = 24, 56
    ks = _fill(K_N56, B, 1)
    assert_bounds_covered(B, N, ks, False, ["k_chol_sm<144,0>"])
    assert_bounds_covered(B, N, ks, True, ["k_chol_w32", "k_chol_sm<48,32>", "k_chol_sm<144,48>"])
    assert {64, 66} <= set(ks) and {32, 34} <= set(ks)
    case = Case(10, N, ks)
    names = launched_kernels(lambda: run_case(case, ks, ks, "B24 N56"))
    for stem, args in [("k_chol_sm", (144, 256, 0)), ("k_chol_w32", ()), ("k_chol_sm", (48, 128, 32)),
                       ("k_chol_sm", (144, 256, 48)), ("k_w_small", ()), ("k_gemm", ()), ("k_upd_pairs", ()),
                       ("k_downdate_ws2", ())]:
        assert has_kernel(names, stem, *args), (stem, args, sorted(n for n in names if n.startswith("void")))


def test_b24_n100_resident_variants():
    """kmax 200: every resident Cholesky variant on its stream, both KMIN sets; k_gemm up to four row tiles."""
    B, N = 24, 100
    ks = _fill(K_N100, B, 2)
    assert_bounds_covered(B, N, ks, False, ["k_chol_sm<112,0>", "k_chol_sm<144,112>", "k_chol_sm<200,144>"])
    assert_bounds_covered(B, N, ks, True, ["k_chol_w32", "k_chol_sm<48,32>", "k_chol_sm<112,48>", "k_chol_sm<144,112>",
                                           "k_chol_sm<200,144>"])
    case = Case(20, N, ks)
    names = launched_kernels(lambda: run_case(case, ks, ks, "B24 N100"))
    for args in [(112, 256, 0), (144, 256, 112), (200, 512, 144), (48, 128, 32), (112, 256, 48)]:
        assert has_kernel(names, "k_chol_sm", *args), args
    assert has_kernel(names, "k_chol_w32") and not has_kernel(names, "k_chol(")


def _sweep_filters():
    """(types, k) per filter: n = 13 + 6 a + 3 c on both sides of the 64-wide tiles and 8-wide blocks of the downdate,
    inverse-depth and Cartesian features mixed, each n at a small k (<= 32) and a large one (> 64)."""
    out = [(np.array([2]), 2), (np.array([1]), 2)]   # n = 16, 19
    for r in (1, 7, 8, 9, 31, 32, 33, 57, 63, 0):
        n = next(n for n in range(r, 614, 64) if n >= 211 and (n - 13) % 3 == 0)
        m = (n - 13) // 3                      # 3-wide units: a inverse-depth features (2 units), c Cartesian (1 unit)
        a = max(1, m - 100, min(m - 65, m // 3))
        t = np.array([1] * a + [2] * (m - 2 * a))
        np.random.default_rng(r).shuffle(t)
        assert 65 <= len(t) <= 100 and U.feature_offsets(t)[2] == n
        out += [(t, 32 - 2 * (r % 2)), (t, 130)]
    return out


def test_state_size_sweep_downdate_edges():
    """n mod 64 in {1, 7, 8, 9, 31, 32, 33, 57, 63, 0} (full, STRIP and masked-diagonal downdate tiles; every 8x8 block
    mask) and n < 64, at kmax 200."""
    N = 100
    filt = _sweep_filters()
    ks = [k for _, k in filt]
    case = Case(30, N, ks, types=[t for t, _ in filt], n_max=13 + 6 * N)
    assert {1, 7, 8, 9, 31, 32, 33, 57, 63, 0} <= {n % 64 for n in case.n} and min(case.n) < 64
    run_case(case, ks, ks, "n sweep")


def test_b8_n120_global_chol():
    """kmax 240: the global-memory k_chol behind the resident variants (k > 200), four k_gemm row tiles."""
    B, N = 8, 120
    ks = [144, 146, 192, 194, 200, 202, 238, 240]
    assert_bounds_covered(B, N, ks, False, ["k_chol", "k_chol_sm<200,144>"])
    case = Case(40, N, ks, cart=0.8)
    names = launched_kernels(lambda: run_case(case, ks, ks, "B8 N120"))
    assert has_kernel(names, "k_chol(") and has_kernel(names, "k_chol_sm", 200, 512, 144)


K_LOCK = [0, 2, 62, 64, 66, 128, 130, 256, 258, 280]


def test_b8_n140_lockstep():
    """The lock-step chain (k_cb_*, k_mk_y / k_mk_cv / k_mk_fin) across its 64-row panels, the 64-row CV_ROWS and
    128-column chunks, with ragged k below kact; then a batch with every k <= 62 and one with every k = 0."""
    B, N = 8, 140
    batches = [K_LOCK[:8], K_LOCK[2:], [2, 62, 30, 0, 60, 34, 4, 62], [0] * 8]
    assert lockstep(B, N)
    bank = None
    for i, ks in enumerate(batches):
        case = Case(50 + i, N, ks, nfeat=[140] * 8 if i < 2 else None, n_max=13 + 6 * N, cart=0.7)
        bank = bank or make_bank(case)
        if i == 0:
            names = launched_kernels(lambda: run_case(case, ks, ks, "B8 N140", bank))
            for stem in ("k_cb_diagpanel", "k_cb_trail", "k_cb_inv", "k_mk_y", "k_mk_cv", "k_mk_fin"):
                assert has_kernel(names, stem), stem
        else:
            run_case(case, ks, ks, "B8 N140", bank)
    bank.close()


def test_lockstep_switch_b127_b128():
    """kmax 256: B = 127 runs the lock-step Cholesky, B = 128 the per-filter kernels (k_chol for k > 200); the same
    inputs on both sides."""
    N = 128
    ks = _fill([256, 254, 200, 202, 130, 64], 128, 6)
    case = Case(60, N, ks, cart=0.8)
    assert lockstep(127, N) and not lockstep(128, N)
    run_case(case, ks, ks, "B128 N128")
    sub = Case(60, N, ks, cart=0.8)
    for name in ("types", "x", "xp", "P"):
        setattr(sub, name, getattr(case, name)[:127])
    sub.nfeat, sub.n, sub.B = case.nfeat[:127], case.n[:127], 127
    sub.rng = np.random.default_rng(61)
    run_case(sub, ks[:127], ks[:127], "B127 N128")


def test_b296_n100_staged_pairs():
    """B >= 296: the pair loop inside k_upd_S, staged (N_max <= 128); large k on six filters, fillers elsewhere."""
    B, N = 296, 100
    ks = _fill([34, 112, 114, 144, 146, 200], B, 7)
    assert pairs_variant(B, N) == "k_upd_S staged"
    case = Case(70, N, ks)
    names = launched_kernels(lambda: run_case(case, ks, ks, "B296 N100"))
    assert has_kernel(names, "k_upd_S") and not has_kernel(names, "k_upd_pairs")


def test_b296_n130_unstaged_pairs():
    """B >= 296, N_max > 128: the unstaged pair loop in k_upd_S; k > 200 in the non-lock-step k_chol."""
    B, N = 296, 130
    ks = _fill([34, 112, 146, 202, 260], B, 8)
    assert pairs_variant(B, N) == "k_upd_S unstaged" and chol_variant(B, N, False, 260)[0] == "k_chol"
    case = Case(80, N, ks, cart=0.8)
    names = launched_kernels(lambda: run_case(case, ks, ks, "B296 N130"))
    assert has_kernel(names, "k_chol(") and not has_kernel(names, "k_upd_pairs") and not has_kernel(names, "k_cb_inv")


def test_stale_buffers_across_updates():
    """Three li + hi updates in a row on one context, k permuted between the filters each time (a filter moves between
    kernels, a smaller k follows a larger one), and two filters' maps shrunk before the third: G, W, inv(L) still hold
    rows and columns of the earlier updates."""
    B, N = 24, 100
    ks = _fill(K_N100, B, 9)
    case = Case(90, N, ks, nfeat=[N] * B)
    bank = make_bank(case)
    case.upload(bank)
    rng = np.random.default_rng(91)
    prev = ks
    for step in range(3):
        if step == 2:
            # shrink filters 0 and 1 (the largest k of the last update among them) to 7 and 40 features
            x, P, _ = bank.download_state()
            xp = bank.download_state(which=1, want_P=False)[0]
            for b, nf in ((0, 7), (1, 40)):
                t = case.types[b, :nf].copy()
                n = U.feature_offsets(t)[2]
                case.types[b] = 0
                case.types[b, :nf] = t
                case.nfeat[b], case.n[b] = nf, n
                x[b, n:], xp[b, n:], P[b, n:], P[b, :, n:] = 0, 0, 0, 0
                bank.upload_feature_types(case.types[b:b + 1], np.array([nf], dtype=np.int32), b0=b)
                bank.upload_state(x[b:b + 1], P[b:b + 1], b0=b)
                bank.upload_state(xp[b:b + 1], which=1, b0=b)
        kl = list(rng.permutation(ks))
        kl = [min(k, 2 * case.nfeat[b]) for b, k in enumerate(kl)]
        assert any(a < b for a, b in zip(kl, prev))
        kh = list(rng.permutation(kl))
        kh = [min(k, 2 * case.nfeat[b]) for b, k in enumerate(kh)]
        run_update(bank, case, kl, False, "stale %d" % step)
        run_update(bank, case, kh, True, "stale %d" % step)
        prev = kh
    bank.close()


@pytest.mark.parametrize("B,N", [(24, 100), (8, 140)])
def test_filter_independence(B, N):
    """A filter's result does not depend on the other filters of the batch: the even filters keep their inputs, the odd
    ones get new values (and, per filter, a different k), and the even filters' x and P stay bit-identical.  In the
    lock-step context the launch loops run to the batch's largest k (kact), so there the odd filters keep their k."""
    ks = _fill(K_N100, B, 10)[:B] if N == 100 else K_LOCK[:B]
    runs = []
    for variant in range(2):
        case = Case(100, N, ks, nfeat=[N] * B, n_max=13 + 6 * N)
        other = Case(200 + variant, N, ks, nfeat=[N] * B, n_max=13 + 6 * N)
        f_li, f_hi = case.features(ks), case.features(ks)
        o_li, o_hi = other.features(ks), other.features(ks)
        k2 = ks if lockstep(B, N) else [ks[(b + 2) % B] if b % 2 else k for b, k in enumerate(ks)]
        if variant:
            for b in range(1, B, 2):
                case.x[b], case.xp[b], case.P[b] = other.x[b], other.xp[b], other.P[b]
        feats = []
        for f, o in ((f_li, o_li), (f_hi, o_hi)):
            h, z, Hc, sel = [np.array(a) if i < 3 else list(a) for i, a in enumerate(f)]
            if variant:
                rng = np.random.default_rng(300)
                for b in range(1, B, 2):
                    h[b], z[b], Hc[b] = o[0][b], o[1][b], o[2][b]
                    sel[b] = U.scattered_selection(rng, N, k2[b] // 2)
            feats.append((h, z, Hc, sel))
        bank = make_bank(case)
        case.upload(bank)
        run_update(bank, case, None, False, "indep", check=False, feats=feats[0])
        x, P = run_update(bank, case, None, True, "indep", check=False, feats=feats[1])
        runs.append((x[0::2].copy(), P[0::2].copy()))
        bank.close()
    assert np.array_equal(runs[0][0], runs[1][0]) and np.array_equal(runs[0][1], runs[1][1])
