"""CPU oracle for the latent-variable GP (GaussianProcesses.jl's GPA)  --  TEST INFRASTRUCTURE ONLY.

A numpy restatement of the reference's GPA target and gradient, built on oracle/gp_oracle.py's kernels and means.  It
is the checker for the device path (gpb200_unwhiten / gpb200_gpa_grad) and for the host mirror gpb200/gpa.py.

Reference lines restated (paths relative to a GaussianProcesses.jl checkout):
  src/GPA.jl:111-114, src/GPE.jl:169-175   update_cK!: K + exp(2 * -20) I, Cholesky
  src/GPA.jl:118-128, 261-266              update_ll! / update_target!: f = L v + mu, target = ll - (v'v + N log 2pi)/2
  src/GPA.jl:130-143                       get_L_bar!: tril(dl_df v'), chol_unblocked_rev!
  src/GPA.jl:164-173                       dll_kern!: diagonal doubled, then dmll_kern! (src/GPE.jl:219-241)
  src/GPA.jl:183-228, 268-272, 383-399     update_dll! / update_dtarget!: [v; lik; mean; kernel], prior gradient -v
  src/chol_utils.jl:3-39                   level2partition, chol_unblocked_rev! (Murray 2016, arXiv:1602.07527)
  src/likelihoods/*.jl                     log_dens, dlog_dens_df, dlog_dens_dθ of the six likelihoods

Likelihood spec (neutral tuple form): ("Bern",) ("Bin", n) ("Exp",) ("Gauss", lσ) ("Pois",) ("StuT", ν, lσ).
"""
import math

import numpy as np
from scipy.special import gammaln, ndtr

from oracle import gp_oracle as orc

LOG2PI = math.log(2.0 * math.pi)
GPA_LOG_NOISE = -20.0                       # GPA.jl:112


def _phi(f):
    return np.exp(-0.5 * f * f) / math.sqrt(2.0 * math.pi)


def lik_num_params(lspec):
    return 1 if lspec[0] in ("Gauss", "StuT") else 0


def log_dens(lspec, f, y):
    name = lspec[0]
    if name == "Bern":                                          # bernoulli.jl:12-14
        return np.array([math.log(ndtr(fi)) if yi else math.log(1.0 - ndtr(fi)) for fi, yi in zip(f, y)])
    if name == "Bin":                                           # binomial.jl:16-19
        n = lspec[1]
        th = np.exp(f) / (1 + np.exp(f))
        return np.array([gammaln(n + 1.0) - gammaln(yi + 1.0) - gammaln(n - yi + 1.0) + yi * math.log(ti) + (n - yi) * math.log(1 - ti)
                         for ti, yi in zip(th, y)])
    if name == "Exp":                                           # exponential.jl:13-16
        return np.array([-fi - math.exp(-fi) * yi for fi, yi in zip(f, y)])
    if name == "Gauss":                                         # gaussian.jl:26-28
        s = math.exp(lspec[1])
        return (-0.5 * math.log(2 * math.pi) - math.log(s)) - 0.5 * ((y - f) / s) ** 2
    if name == "Pois":                                          # poisson.jl:13-16
        return y * f - np.exp(f) - gammaln(1.0 + y)
    if name == "StuT":                                          # studentT.jl:29-34
        nu, s = lspec[1], math.exp(lspec[2])
        c = gammaln(0.5 * (nu + 1)) - gammaln(0.5 * nu) - 0.5 * math.log(math.pi * nu) - math.log(s)
        return np.array([c - (0.5 * (nu + 1)) * math.log(1 + (1 / nu) * ((yi - fi) / s) ** 2) for fi, yi in zip(f, y)])
    raise ValueError(lspec)


def dlog_dens_df(lspec, f, y):
    name = lspec[0]
    if name == "Bern":                                          # bernoulli.jl:16-18
        return np.array([_phi(fi) / ndtr(fi) if yi else -_phi(fi) / (1.0 - ndtr(fi)) for fi, yi in zip(f, y)])
    if name == "Bin":                                           # binomial.jl:21-23
        n = lspec[1]
        return np.array([yi / (1.0 + math.exp(fi)) - (n - yi) * math.exp(fi) / (1 + math.exp(fi)) for fi, yi in zip(f, y)])
    if name == "Exp":                                           # exponential.jl:19-21
        return np.array([yi * math.exp(-fi) - 1 for fi, yi in zip(f, y)])
    if name == "Gauss":                                         # gaussian.jl:31-33
        s = math.exp(lspec[1])
        return np.array([(yi - fi) / s ** 2 for fi, yi in zip(f, y)])
    if name == "Pois":                                          # poisson.jl:19-21
        return y - np.exp(f)
    if name == "StuT":                                          # studentT.jl:37-41
        nu, s = lspec[1], math.exp(lspec[2])
        return np.array([(nu + 1) * (yi - fi) / (nu * s ** 2 + (yi - fi) ** 2) for fi, yi in zip(f, y)])
    raise ValueError(lspec)


def dlog_dens_dtheta(lspec, f, y):
    """N x num_params (gaussian.jl:36-38, studentT.jl:44-48)"""
    name = lspec[0]
    if name == "Gauss":
        s = math.exp(lspec[1])
        return (s * np.array([-1 / s + 1 / s ** 3 * (yi - fi) ** 2 for fi, yi in zip(f, y)]))[:, None]
    if name == "StuT":
        nu, s = lspec[1], math.exp(lspec[2])
        return (s * np.array([-1 / s + (nu + 1) * (yi - fi) ** 2 / (nu * s ** 3 + s * (yi - fi) ** 2) for fi, yi in zip(f, y)]))[:, None]
    return np.zeros((len(f), 0))


def chol_factor(spec, X, log_noise=GPA_LOG_NOISE):
    """lower L with K + exp(2 logNoise) I = L L' (GPA.jl:111-114)"""
    return orc._potrf_upper(orc.gram(spec, X, log_noise)).T.copy()


def chol_unblocked_rev(L, A_bar):
    """chol_utils.jl:15-39, literally (0-based j; A_bar is overwritten and returned)"""
    N = A_bar.shape[0]
    for j in range(N - 1, -1, -1):
        r, d = L[j, :j], L[j, j]                               # level2partition, chol_utils.jl:3-12
        B, c = L[j + 1:, :j], L[j + 1:, j]
        r_bar, B_bar, c_bar = A_bar[j, :j], A_bar[j + 1:, :j], A_bar[j + 1:, j]   # views
        A_bar[j, j] -= c_bar @ c / d
        A_bar[j, j] /= d
        c_bar /= d
        r_bar -= A_bar[j, j] * r
        r_bar -= B.T @ c_bar                                    # gemv!('T', -1.0, B, c_bar, 1.0, r_bar)
        B_bar -= np.outer(c_bar, r)                             # ger!(-1.0, c_bar, r, B_bar)
        A_bar[j, j] /= 2
    return A_bar


def dll_kern_literal(spec, X, L, v, dl_df):
    """dll_kern! (GPA.jl:164-173): get_L_bar!, diagonal doubled, dmll_kern!'s lower-triangle contraction (GPE.jl:219-241)"""
    L_bar = np.tril(np.outer(dl_df, v))                         # GPA.jl:131-133
    chol_unblocked_rev(L, L_bar)
    L_bar[np.diag_indices_from(L_bar)] *= 2                     # GPA.jl:168-170
    _, grads = orc.cov_and_grads(spec, X, None, want_grad=True)
    lo = np.tril(L_bar, -1)
    dg = np.diag(L_bar)
    return np.array([np.sum(lo * G) + 0.5 * np.sum(dg * np.diag(G)) for G in grads]), L_bar


def chol_bar_closed_form(L, v, dl_df):
    """P + P' with P = W' Phi(w v') W, W = L^-1, w = L' dl_df, Phi = lower triangle with the diagonal halved"""
    n = L.shape[0]
    W = np.linalg.solve(L, np.eye(n))
    w = L.T @ dl_df
    Phi = np.tril(np.outer(w, v))
    Phi[np.diag_indices(n)] *= 0.5
    P = W.T @ Phi @ W
    return P + P.T


def dll_kern_closed_form(spec, X, L, v, dl_df):
    """1/2 sum_ij (P + P')_ij dK_ij/dθ_p"""
    S = chol_bar_closed_form(L, v, dl_df)
    _, grads = orc.cov_and_grads(spec, X, None, want_grad=True)
    return np.array([0.5 * np.sum(S * G) for G in grads])


def gpa_target(spec, X, y, v, lspec, mspec=("MeanZero",), log_noise=GPA_LOG_NOISE):
    """update_target! (GPA.jl:118-128, 261-266; no priors)"""
    L = chol_factor(spec, X, log_noise)
    mu, _ = orc.mean_and_grads(mspec, X)
    f = L @ v + mu
    ll = float(np.sum(log_dens(lspec, f, y)))
    return ll - (v @ v + LOG2PI * X.shape[0]) / 2.0


def gpa_dtarget(spec, X, y, v, lspec, mspec=("MeanZero",), process=True, lik=True, domean=True, kern=True,
                log_noise=GPA_LOG_NOISE):
    """update_dtarget! (GPA.jl:183-228, 268-272, 383-399): dll + prior gradient (-v for the process block, 0 elsewhere)"""
    L = chol_factor(spec, X, log_noise)
    mu, MG = orc.mean_and_grads(mspec, X)
    f = L @ v + mu
    g = dlog_dens_df(lspec, f, y)
    out = []
    if process:
        out.extend(L.T @ g - v)                                 # GPA.jl:200 (U = L') ; prior -v, GPA.jl:385
    if lik and lik_num_params(lspec) > 0:
        out.extend(np.sum(dlog_dens_dtheta(lspec, f, y), axis=0))        # GPA.jl:203-209
    if domean and MG.shape[1] > 0:
        out.extend(MG.T @ g)                                    # dmll_mean!, GPA.jl:174-176
    if kern:
        out.extend(dll_kern_literal(spec, X, L, v, g)[0])
    return np.array(out, dtype=np.float64)
