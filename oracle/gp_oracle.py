"""TEST INFRASTRUCTURE ONLY -- CPU (numpy/scipy, float64) restatement of the Spearmint GP-EI hot path.

This is the parity oracle for ``spearmint_b200``.  It is *not* part of the product: only
``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s ``cpu_baseline`` / ``--impl reference``
legs may import it.  The product path never routes through it.

Pinning: the reference ships no tests or golden vectors (SURVEY.md section 4), so this file is
pinned against the reference ITSELF, executed in the build container through
``oracle/ref_shim.py``: ``tests/golden/make_golden.py`` froze the reference's outputs into
``tests/golden/*.npz`` and ``tests/test_oracle_golden.py`` checks every function here against
them (rtol 1e-9 or tighter); ``tests/test_oracle_vs_reference.py`` re-checks against the
reference's outputs on a second set of seeded inputs (``tests/golden/make_golden_live.py``).

Reference files restated (paths relative to ``/root/reference/spearmint/spearmint``):
  GP   = gp.py                          OPT  = chooser/GPEIOptChooser.py
  PSEC = chooser/GPEIperSecChooser.py   UTIL = util.py
A hyper-sample is the reference's tuple ``(mean, noise, amp2, ls)`` (OPT:628).
"""
import numpy as np
import scipy.linalg as spla
import scipy.stats as sps

KINDS = ("SE", "ARDSE", "Matern32", "Matern52")
JITTER = 1e-6  # OPT:209-210


# ----------------------------------------------------------------------------- kernels
def dist2(ls, x1, x2=None):
    """Scaled squared distances via the expanded form, clamped at 0 (GP:34-54)."""
    a = x1 / ls
    b = a if x2 is None else x2 / ls
    na = np.sum(a * a, axis=1)
    nb = np.sum(b * b, axis=1)
    cross = np.dot(a, 2 * b.T)
    return np.maximum(-(cross - na[:, None] - nb[None, :]), 0.0)


def kernel(kind, ls, x1, x2=None):
    """Correlation matrix k(x1,x2) for the four stationary kernels of gp.py.

    SE ignores ``ls`` (GP:87-93), ARDSE GP:95-100, Matern32 GP:107-113, Matern52 GP:120-127.
    """
    if kind == "SE":
        ls = np.ones_like(ls)
    r2 = dist2(ls, x1, x2)
    if kind in ("SE", "ARDSE"):
        return np.exp(-0.5 * r2)
    if kind == "Matern32":
        r = np.sqrt(r2) * np.sqrt(3.0)
        return (1.0 + r) * np.exp(-r)
    if kind == "Matern52":
        r2 = np.abs(r2)
        r = np.sqrt(r2)
        s5 = np.sqrt(5.0)
        return (1.0 + s5 * r + (5.0 / 3.0) * r2) * np.exp(-s5 * r)
    raise ValueError(kind)


def grad_dist2(ls, x1, x2):
    """d r2[i,j] / d x2-side sign convention of GP:56-85: gX[i,j,d] = (2/ls_d) (x1_id - x2_jd)/ls_d."""
    a = x1 / ls
    b = x2 / ls
    return 2.0 * (a[:, None, :] - b[None, :, :]) / ls


def grad_kernel(kind, ls, x1, x2):
    """The reference's ``grad_<kernel>`` (GP:102-105, 115-118, 129-132): dk/dr2 * grad_dist2."""
    if kind == "SE":
        ls = np.ones_like(ls)
    r2 = dist2(ls, x1, x2)
    if kind in ("SE", "ARDSE"):
        w = -0.5 * np.exp(-0.5 * r2)
    elif kind == "Matern32":
        w = -1.5 * np.exp(-np.sqrt(3.0) * np.sqrt(r2))
    elif kind == "Matern52":
        r = np.sqrt(r2)
        s5 = np.sqrt(5.0)
        w = -(5.0 / 6.0) * np.exp(-s5 * r) * (1.0 + s5 * r)
    else:
        raise ValueError(kind)
    return w[:, :, None] * grad_dist2(ls, x1, x2)


def cov(kind, amp2, ls, x1, x2=None):
    """amp2*(k + 1e-6 I) for the self case, amp2*k for the cross case (OPT:207-212, PSEC:145-150)."""
    if x2 is None:
        return amp2 * (kernel(kind, ls, x1) + JITTER * np.eye(x1.shape[0]))
    return amp2 * kernel(kind, ls, x1, x2)


# ----------------------------------------------------------------------------- EI
def _ei_from_moments(best, m, s):
    u = (best - m) / s
    return s * (u * sps.norm.cdf(u) + sps.norm.pdf(u))


def predict(kind, hyper, comp, cand, vals):
    """No-pending predictive mean / variance at candidates (OPT:534-548). Returns (m, v, L, alpha)."""
    mean, noise, amp2, ls = hyper
    n = comp.shape[0]
    K = cov(kind, amp2, ls, comp) + noise * np.eye(n)
    L = spla.cholesky(K, lower=True)
    alpha = spla.cho_solve((L, True), vals - mean)
    Kx = cov(kind, amp2, ls, comp, cand)
    beta = spla.solve_triangular(L, Kx, lower=True)
    m = np.dot(Kx.T, alpha) + mean
    v = amp2 * (1 + JITTER) - np.sum(beta ** 2, axis=0)
    return m, v, L, alpha


def fantasies(kind, hyper, comp, pend, vals, normals):
    """Pending-fantasy prologue (OPT:558-597).

    ``normals`` is the (P,F) standard-normal block the reference draws with
    ``npr.set_state(self.randomstate); npr.randn(P, F)`` (OPT:588-589).
    Returns (comp_pend, L_joint, fant_vals[(N+P),F], bests[F]).
    """
    mean, noise, amp2, ls = hyper
    n = comp.shape[0]
    cp = np.concatenate((comp, pend))
    Lj = spla.cholesky(cov(kind, amp2, ls, cp) + noise * np.eye(cp.shape[0]), lower=True)
    Kp = cov(kind, amp2, ls, comp, pend)
    Kpp = cov(kind, amp2, ls, pend)
    Lo = Lj[:n, :n]
    alpha = spla.cho_solve((Lo, True), vals - mean)
    beta = spla.cho_solve((Lo, True), Kp)
    pm = np.dot(Kp.T, alpha) + mean
    pK = Kpp - np.dot(Kp.T, beta)
    pL = spla.cholesky(pK, lower=True)
    pf = np.dot(pL, normals) + pm[:, None]
    fant = np.concatenate((np.tile(vals[:, None], (1, normals.shape[1])), pf))
    return cp, Lj, fant, np.min(fant, axis=0)


def compute_ei(kind, hyper, comp, pend, cand, vals, normals=None):
    """GPEIOptChooser.compute_ei for one hyper-sample (OPT:527-619); identical math in GPEI:178-266."""
    mean, noise, amp2, ls = hyper
    if pend.shape[0] == 0:
        m, v, _, _ = predict(kind, hyper, comp, cand, vals)
        return _ei_from_moments(np.min(vals), m, np.sqrt(v))
    cp, Lj, fant, bests = fantasies(kind, hyper, comp, pend, vals, normals)
    Kx = cov(kind, amp2, ls, cp, cand)
    alpha = spla.cho_solve((Lj, True), fant - mean)
    beta = spla.solve_triangular(Lj, Kx, lower=True)
    m = np.dot(Kx.T, alpha) + mean                       # (M,F)
    v = amp2 * (1 + JITTER) - np.sum(beta ** 2, axis=0)   # (M,)
    s = np.sqrt(v[:, None])
    return np.mean(_ei_from_moments(bests[None, :], m, s), axis=1)


def ei_over_hypers(kind, hyper_samples, comp, pend, cand, vals, normals=None):
    """(M,S) matrix, one column per hyper-sample (OPT:331-341)."""
    out = np.zeros((cand.shape[0], len(hyper_samples)))
    for s, h in enumerate(hyper_samples):
        out[:, s] = compute_ei(kind, h, comp, pend, cand, vals, normals)
    return out


def select(overall_ei, grid_subset=None):
    """mean over samples then argmax (OPT:294) or top-k ascending (OPT:270)."""
    mean_ei = np.mean(overall_ei, axis=1)
    if grid_subset is None:
        return int(np.argmax(mean_ei))
    return np.argsort(mean_ei)[-grid_subset:]


# ----------------------------------------------------------------------------- EI per second
def time_mean(kind, time_hyper, comp, cand, durs_log):
    """exp of the time-GP predictive mean, no variance, no TRSM (PSEC:442-459)."""
    tmean, tnoise, tamp2, tls = time_hyper
    n = comp.shape[0]
    L = spla.cholesky(cov(kind, tamp2, tls, comp) + tnoise * np.eye(n), lower=True)
    ta = spla.cho_solve((L, True), durs_log - tmean)
    return np.exp(np.dot(cov(kind, tamp2, tls, comp, cand).T, ta) + tmean)


def compute_ei_per_s(kind, hyper, time_hyper, comp, pend, cand, vals, durs_log, normals=None):
    """GPEIperSecChooser.compute_ei_per_s (PSEC:437-548): EI / exp(predicted log-duration)."""
    return compute_ei(kind, hyper, comp, pend, cand, vals, normals) / \
        time_mean(kind, time_hyper, comp, cand, durs_log)


def ei_over_hypers_per_s(kind, hyper_samples, time_hyper_samples, comp, pend, cand, vals,
                         durs_log, normals=None, mcmc_iters=None):
    """Reproduces the reference's early ``return`` (PSEC:302): only column 0 is ever filled."""
    S = len(hyper_samples) if mcmc_iters is None else mcmc_iters
    out = np.zeros((cand.shape[0], S))
    out[:, 0] = compute_ei_per_s(kind, hyper_samples[0], time_hyper_samples[0], comp, pend, cand,
                                 vals, durs_log, normals)
    return out


# ----------------------------------------------------------------------------- slice-sampler log-probabilities
def gp_logprob(kind, mean, noise, amp2, ls, comp, vals):
    """-sum log diag(L) - 0.5 (y-mu)' K^-1 (y-mu)   (OPT:635-640, 658-661, 689-692)."""
    n = comp.shape[0]
    L = spla.cholesky(cov(kind, amp2, ls, comp) + noise * np.eye(n), lower=True)
    r = vals - mean
    return -np.sum(np.log(np.diag(L))) - 0.5 * np.dot(r, spla.cho_solve((L, True), r))


def logprob_ls(kind, ls, mean, noise, amp2, comp, vals, max_ls=2.0):
    """Length-scale conditional with the top-hat prior (OPT:631-641)."""
    if np.any(ls < 0) or np.any(ls > max_ls):
        return -np.inf
    return gp_logprob(kind, mean, noise, amp2, ls, comp, vals)


def logprob_noisy(kind, hypers, ls, comp, vals, noise_scale=0.1, amp2_scale=1.0, amp2_prior="sqrt"):
    """Joint (mean, amp2, noise) conditional (OPT:646-670). ``amp2_prior='plain'`` is PSEC:614."""
    mean, amp2, noise = hypers
    if mean > np.max(vals) or mean < np.min(vals) or amp2 < 0 or noise < 0:
        return -np.inf
    lp = gp_logprob(kind, mean, noise, amp2, ls, comp, vals)
    lp += np.log(np.log(1 + (noise_scale / noise) ** 2))
    la = np.log(np.sqrt(amp2)) if amp2_prior == "sqrt" else np.log(amp2)
    return lp - 0.5 * (la / amp2_scale) ** 2


def logprob_noiseless(kind, hypers, ls, comp, vals, amp2_scale=1.0, amp2_prior="sqrt"):
    """(mean, amp2) conditional with noise pinned at 1e-3 (OPT:679-700)."""
    mean, amp2 = hypers[0], hypers[1]
    if mean > np.max(vals) or mean < np.min(vals) or amp2 < 0:
        return -np.inf
    lp = gp_logprob(kind, mean, 1e-3, amp2, ls, comp, vals)
    la = np.log(np.sqrt(amp2)) if amp2_prior == "sqrt" else np.log(amp2)
    return lp - 0.5 * (la / amp2_scale) ** 2


# ----------------------------------------------------------------------------- EI value + gradient (L-BFGS refinement)
def grad_optimize_ei(kind, hyper, cand, comp, pend, vals, normals=None):
    """(f, g) for one point and one hyper-sample exactly as the reference returns it (OPT:391-525),

    including the reference's 0.5*amp2 prefactor (OPT:437, 521): g is one half of d(-EI)/dx.
    """
    mean, noise, amp2, ls = hyper
    cand = np.reshape(cand, (-1, comp.shape[1]))
    if pend.shape[0] == 0:
        base, fvals, best = comp, (vals - mean)[:, None], np.array([np.min(vals)])
        L = spla.cholesky(cov(kind, amp2, ls, comp) + noise * np.eye(comp.shape[0]), lower=True)
    else:
        base, L, fant, best = fantasies(kind, hyper, comp, pend, vals, normals)
        fvals = fant - mean
    Kx = cov(kind, amp2, ls, base, cand)                      # (Nb,1)
    gK = np.squeeze(grad_kernel(kind, ls, base, cand), axis=1)  # (Nb,D)
    alpha = spla.cho_solve((L, True), fvals)                  # (Nb,F)
    beta = spla.solve_triangular(L, Kx, lower=True)
    m = np.dot(Kx.T, alpha) + mean                            # (1,F)
    v = amp2 * (1 + JITTER) - np.sum(beta ** 2, axis=0)       # (1,)
    s = np.sqrt(v)[:, None]
    u = (best[None, :] - m) / s
    cdf, pdf = sps.norm.cdf(u), sps.norm.pdf(u)
    ei = s * (u * cdf + pdf)                                  # (1,F)
    g_m = -cdf                                                # dEI/dm
    g_s2 = 0.5 * pdf / s                                      # dEI/dv
    gx_m = np.dot(alpha.T, gK)                                # (F,D)
    gx_v = np.dot(-2 * spla.cho_solve((L, True), Kx).T, gK)   # (1,D)
    g = 0.5 * amp2 * (gx_m * g_m.T + gx_v * g_s2.T)           # (F,D)
    if pend.shape[0] == 0:
        return -np.sum(ei), g.flatten()
    return -np.mean(ei, axis=1), np.mean(g, axis=0).flatten()


def grad_optimize_ei_over_hypers(kind, hyper_samples, cand, comp, pend, vals, normals=None):
    """Sum of (f, g) over hyper-samples (OPT:360-388)."""
    f, g = 0.0, np.zeros(np.size(cand))
    for h in hyper_samples:
        fi, gi = grad_optimize_ei(kind, h, cand, comp, pend, vals, normals)
        f, g = f + fi, g + gi
    return f, g


# ----------------------------------------------------------------------------- EI per second: value + gradient
def grad_optimize_ei_per_s(kind, hyper, time_hyper, cand, comp, vals, durs_log):
    """(f, g) of GPEIperSecChooser.grad_optimize_ei for one point / one sample pair (PSEC:351-435).

    Pending points are ignored by the reference on this path; the 0.5*amp2 prefactors (PSEC:431-432) are kept."""
    mean, noise, amp2, ls = hyper
    tmean, tnoise, tamp2, tls = time_hyper
    n = comp.shape[0]
    cand = np.reshape(cand, (-1, comp.shape[1]))
    best = np.min(vals)
    Lt = spla.cholesky(cov(kind, tamp2, tls, comp) + tnoise * np.eye(n), lower=True)
    ta = spla.cho_solve((Lt, True), durs_log - tmean)
    ftm = np.exp(np.dot(cov(kind, tamp2, tls, comp, cand).T, ta) + tmean)      # (1,)
    gKt = np.squeeze(grad_kernel(kind, tls, comp, cand), axis=1)                # (N,D)
    L = spla.cholesky(cov(kind, amp2, ls, comp) + noise * np.eye(n), lower=True)
    Kx = cov(kind, amp2, ls, comp, cand)
    gK = np.squeeze(grad_kernel(kind, ls, comp, cand), axis=1)
    alpha = spla.cho_solve((L, True), vals - mean)
    beta = spla.solve_triangular(L, Kx, lower=True)
    m = np.dot(Kx.T, alpha) + mean
    v = amp2 * (1 + JITTER) - np.sum(beta ** 2, axis=0)
    s = np.sqrt(v)
    u = (best - m) / s
    cdf, pdf = sps.norm.cdf(u), sps.norm.pdf(u)
    ei = s * (u * cdf + pdf)
    f = -np.sum(ei / ftm)
    gtm = np.dot(ta.T, gKt)
    gx_m = np.dot(alpha.T, gK)
    gx_v = np.dot(-2 * spla.cho_solve((L, True), Kx).T, gK)
    g = 0.5 * amp2 * (gx_m * (-cdf) + gx_v * (0.5 * pdf / s))
    gtm = 0.5 * tamp2 * gtm * ftm
    g = (ftm * g - ei * gtm) / (ftm ** 2)
    return f, g.flatten()


def grad_optimize_ei_per_s_over_hypers(kind, hyper_samples, time_hyper_samples, cand, comp, vals, durs_log):
    """Sum over sample pairs i = 0..len(hyper_samples)-1 (PSEC:321-349; time samples indexed from the OLDEST)."""
    f, g = 0.0, np.zeros(np.size(cand))
    for h, th in zip(hyper_samples, time_hyper_samples):
        fi, gi = grad_optimize_ei_per_s(kind, h, th, cand, comp, vals, durs_log)
        f, g = f + fi, g + gi
    return f, g


# ----------------------------------------------------------------------------- ML-II hyper-parameters (GP.optimize_hypers)
def jitter_chol(covmat):
    """GP.optimize_hypers' jitter_chol (GP:187-203): lower Cholesky of covmat + jitter I, jitter = 1e-8 grown by 1.1x
    until it factors; past 1e5 the factor of the identity.  Returns (chol, jitter_used)."""
    jitter = 1e-8
    while True:
        if jitter > 100000:
            return np.eye(covmat.shape[0]), jitter
        try:
            return spla.cholesky(covmat + jitter * np.eye(covmat.shape[0]), lower=True), jitter
        except (ValueError, np.linalg.LinAlgError):
            jitter = jitter * 1.1


def mll_value_grad(kind, hypers, comp, vals, mean):
    """(nlogprob, grad_nlogprob) of GP.optimize_hypers at log-hypers = [log amp2, log noise, log ls...] (GP:222-264),
    INCLUDING the reference's length-scale 'gradient'  -amp2 * grad_corr[:, :, d] * comp[:, d, None]  (GP:258-259: the
    exp(ls) factors cancel; it is not the derivative of the likelihood, but it is what L-BFGS-B is given)."""
    amp2, noise, ls = np.exp(hypers[0]), np.exp(hypers[1]), np.exp(hypers[2:])
    n, D = comp.shape
    diffs = vals - mean
    corr = kernel(kind, ls, comp)
    grad_corr = grad_kernel(kind, ls, comp, comp)
    covmat = amp2 * (corr + 1e-6 * np.eye(n)) + noise * np.eye(n)
    chol, _ = jitter_chol(covmat)
    solve = spla.cho_solve((chol, True), diffs)
    f = -(-np.sum(np.log(np.diag(chol))) - 0.5 * np.dot(diffs, solve))
    inv_cov = spla.cho_solve((chol, True), np.eye(n))
    jac = np.outer(solve, solve) - inv_cov
    g = np.zeros(D + 2)
    g[0] = 0.5 * np.trace(np.dot(jac, corr + 1e-6 * np.eye(n))) * amp2
    g[1] = 0.5 * np.trace(np.dot(jac, np.eye(n))) * noise
    for d in range(D):
        g[d + 2] = np.trace(np.dot(jac, -amp2 * grad_corr[:, :, d] * comp[:, d][:, None] / np.exp(ls[d]))) * np.exp(ls[d])
    return f, -g


def gp_optimize_hypers(kind, comp, vals):
    """GP.optimize_hypers (GP:181-292): mean = mean(vals); L-BFGS-B over [log amp2, log noise, log ls] from
    (std(vals), 1e-3, ones) within [-10, 10] x [-10, 10] x [-10, 5]^D.  Returns the hyper-sample tuple
    (mean, noise, amp2, ls)."""
    import scipy.optimize as spo
    D = comp.shape[1]
    mean = np.mean(vals)
    x0 = np.zeros(D + 2)
    x0[0], x0[1] = np.log(np.std(vals)), np.log(1e-3)
    b = [(-10, 10), (-10, 10)] + [(-10, 5)] * D
    res = spo.fmin_l_bfgs_b(lambda h: mll_value_grad(kind, h, comp, vals, mean)[0], x0,
                            lambda h: mll_value_grad(kind, h, comp, vals, mean)[1], args=(), bounds=b)
    h = res[0]
    return mean, float(np.exp(h[1])), float(np.exp(h[0])), np.exp(h[2:])
