"""Likelihoods of the latent-variable GP (src/likelihoods/*.jl) -- O(N) host work next to the device's O(N^3) part.

Same names and methods as the reference: log_dens, dlog_dens_df, dlog_dens_dθ (here `dlog_dens_dtheta`, an N x
num_params array), mean_lik, var_lik, get_params / set_params / num_params, and predict_obs (20-node Gauss-Hermite,
likelihoods.jl:16-31, with the closed forms BernLik and GaussLik define)."""
import math

import numpy as np
from scipy.special import gammaln, ndtr


def _phi(f):
    return np.exp(-0.5 * f * f) / math.sqrt(2.0 * math.pi)


class Likelihood:
    def get_params(self):
        return []

    def set_params(self, hyp):
        if len(hyp) != 0:
            raise ValueError("%s has no free parameters" % type(self).__name__)

    def num_params(self):
        return len(self.get_params())

    def dlog_dens_dtheta(self, f, y):
        return np.zeros((np.size(f), 0))

    def predict_obs(self, fmean, fvar):
        """predictive mean and variance of y for f ~ N(fmean, fvar), by quadrature (likelihoods.jl:16-31)"""
        nodes, weights = np.polynomial.hermite.hermgauss(20)
        weights = weights / math.sqrt(math.pi)
        fmean, fvar = np.asarray(fmean, dtype=np.float64), np.asarray(fvar, dtype=np.float64)
        f = fmean[:, None] + np.sqrt(2.0 * fvar)[:, None] * nodes[None, :]
        m = np.stack([self.mean_lik(f[:, i]) for i in range(nodes.size)], axis=1)
        v = np.stack([self.var_lik(f[:, i]) for i in range(nodes.size)], axis=1)
        mu = m @ weights
        return mu, (v + m ** 2) @ weights - mu ** 2


class BernLik(Likelihood):
    """y in {0, 1}, P(y = 1) = Φ(f) (bernoulli.jl)"""

    def log_dens(self, f, y):
        p = ndtr(f)
        return np.where(np.asarray(y, dtype=bool), np.log(p), np.log(1.0 - p))

    def dlog_dens_df(self, f, y):
        p = ndtr(f)
        return np.where(np.asarray(y, dtype=bool), _phi(f) / p, -_phi(f) / (1.0 - p))

    def mean_lik(self, f):
        return ndtr(f)

    def var_lik(self, f):
        p = ndtr(f)
        return p * (1 - p)

    def predict_obs(self, fmean, fvar):                  # bernoulli.jl:29-32
        p = ndtr(np.asarray(fmean) / np.sqrt(1 + np.asarray(fvar)))
        return p, p - p * p


class BinLik(Likelihood):
    """y successes out of n trials, θ = logistic(f) (binomial.jl)"""

    def __init__(self, n):
        self.n = int(n)

    def log_dens(self, f, y):
        n, y = self.n, np.asarray(y, dtype=np.float64)
        th = np.exp(f) / (1 + np.exp(f))
        return gammaln(n + 1.0) - gammaln(y + 1.0) - gammaln(n - y + 1.0) + y * np.log(th) + (n - y) * np.log(1 - th)

    def dlog_dens_df(self, f, y):
        y = np.asarray(y, dtype=np.float64)
        return y / (1.0 + np.exp(f)) - (self.n - y) * np.exp(f) / (1 + np.exp(f))

    def mean_lik(self, f):
        return self.n * np.exp(f) / (1.0 + np.exp(f))

    def var_lik(self, f):
        return self.n * (np.exp(f) / (1.0 + np.exp(f))) * (1.0 / (1.0 + np.exp(f)))


class ExpLik(Likelihood):
    """y ~ Exponential with rate exp(-f) (exponential.jl)"""

    def log_dens(self, f, y):
        return -f - np.exp(-f) * y

    def dlog_dens_df(self, f, y):
        return y * np.exp(-f) - 1

    def mean_lik(self, f):
        return np.exp(f)

    def var_lik(self, f):
        return np.exp(f) ** 2


class GaussLik(Likelihood):
    """y ~ N(f, σ²), σ = exp(lσ) (gaussian.jl)"""

    def __init__(self, lsigma):
        self.sigma = math.exp(float(lsigma))

    def get_params(self):
        return [math.log(self.sigma)]

    def set_params(self, hyp):
        if len(hyp) != 1:
            raise ValueError("Gaussian/Normal likelihood has only one free parameter")
        self.sigma = math.exp(float(hyp[0]))

    def log_dens(self, f, y):
        s = self.sigma
        return (-0.5 * math.log(2 * math.pi) - math.log(s)) - 0.5 * ((y - f) / s) ** 2

    def dlog_dens_df(self, f, y):
        return (y - f) / self.sigma ** 2

    def dlog_dens_dtheta(self, f, y):
        s = self.sigma
        return (s * (-1 / s + 1 / s ** 3 * (y - f) ** 2))[:, None]

    def mean_lik(self, f):
        return np.asarray(f, dtype=np.float64)

    def var_lik(self, f):
        return np.full(np.size(f), self.sigma ** 2)

    def predict_obs(self, fmean, fvar):                  # gaussian.jl:55-57
        return np.asarray(fmean), np.asarray(fvar) + self.sigma ** 2


class PoisLik(Likelihood):
    """y ~ Poisson(exp(f)) (poisson.jl)"""

    def log_dens(self, f, y):
        y = np.asarray(y, dtype=np.float64)
        return y * f - np.exp(f) - gammaln(1.0 + y)

    def dlog_dens_df(self, f, y):
        return y - np.exp(f)

    def mean_lik(self, f):
        return np.exp(f)

    def var_lik(self, f):
        return np.exp(f)


class StuTLik(Likelihood):
    """y - f ~ σ t_ν, σ = exp(lσ) (studentT.jl)"""

    def __init__(self, nu, lsigma):
        self.nu = int(nu)
        self.sigma = math.exp(float(lsigma))

    def get_params(self):
        return [math.log(self.sigma)]

    def set_params(self, hyp):
        if len(hyp) != 1:
            raise ValueError("Student-t likelihood has only one free parameter")
        self.sigma = math.exp(float(hyp[0]))

    def log_dens(self, f, y):
        nu, s = self.nu, self.sigma
        c = gammaln(0.5 * (nu + 1)) - gammaln(0.5 * nu) - 0.5 * math.log(math.pi * nu) - math.log(s)
        return c - (0.5 * (nu + 1)) * np.log(1 + (1 / nu) * ((y - f) / s) ** 2)

    def dlog_dens_df(self, f, y):
        nu, s = self.nu, self.sigma
        return (nu + 1) * (y - f) / (nu * s ** 2 + (y - f) ** 2)

    def dlog_dens_dtheta(self, f, y):
        nu, s = self.nu, self.sigma
        return (s * (-1 / s + (nu + 1) * (y - f) ** 2 / (nu * s ** 3 + s * (y - f) ** 2)))[:, None]

    def mean_lik(self, f):
        return np.asarray(f, dtype=np.float64)

    def var_lik(self, f):
        return self.sigma ** 2 * (self.nu / (self.nu - 2.0)) * np.ones(np.size(f))
