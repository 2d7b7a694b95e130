"""GPA -- host-side mirror of the reference's latent-variable GP (src/GPA.jl) over the B200 engine.

The latent values are whitened, f = L v + mean(x) with L L' = K + exp(2 * -20) I.  The device keeps the factor and does
every O(N^3) and O(N^2) step: the Gram build and Cholesky (update_cK!), f = L v (unwhiten), and the gradient's
reverse-mode Cholesky contracted with dK/dθ (gpb200_gpa_grad).  The likelihood and mean terms are O(N) host work, as
in the reference.  Same field names (x, y, mean, kernel, lik, dim, nobs, v, μ as `mu`, ll, dll, target, dtarget), same
parameter order [v; lik; mean; kernel] (GPA.jl:336-381) and the same `process/lik/domean/kern` flags; parameter priors
are not modelled (as in GPE), so dtarget = dll + [-v; 0...] (GPA.jl:383-399)."""
import math

import numpy as np

from . import capi
from .gpe import _as_dxn
from .kernels import Kernel, flatten
from .likelihoods import Likelihood
from .means import Mean, MeanZero

LOG2PI = math.log(2.0 * math.pi)
GPA_LOG_NOISE = -20.0                        # update_cK!'s nugget, GPA.jl:111-114
INIT_LOG_NOISE = 0.5 * math.log(1e-6)        # initialise_ll! factorises Σ + 1e-6 I, GPA.jl:105


class GPA:
    def __init__(self, x, y, mean, kernel, lik, device=0, engine=None):
        if kernel is None or not isinstance(kernel, Kernel):
            raise ValueError("GPA needs a kernel")
        self.mean = mean if mean is not None else MeanZero()
        if not isinstance(self.mean, Mean):
            raise ValueError("mean must be a Mean")
        if not isinstance(lik, Likelihood):
            raise ValueError("GPA needs a likelihood")
        self.kernel, self.lik = kernel, lik
        self._eng = engine if engine is not None else capi.Engine(device)
        x = _as_dxn(x)
        y = np.asarray(y).ravel()
        if x.shape[1] != y.size:
            raise ValueError("Input and output observations must have consistent dimensions.")   # GPA.jl:45
        self.x, self.y = x, y
        self.dim, self.nobs = x.shape
        self._xpm = np.ascontiguousarray(x.T)
        self._eng.set_data(self._xpm)
        ops, dims, theta, self._exposed = flatten(self.kernel, self.dim)
        self._eng.set_kernel(ops, dims, theta.size)
        self.v = np.zeros(self.nobs)
        self.mu = None
        self.ll = self.target = float("nan")
        self.dll = self.dtarget = None
        self.initialise_target()

    # ---- log target ----------------------------------------------------------------------
    def update_cK(self, log_noise=GPA_LOG_NOISE):
        """update_cK!(gp) (GPA.jl:111-114): Gram + nugget + Cholesky on the device"""
        self._eng.factorize(flatten(self.kernel, self.dim)[2], log_noise)

    def _latent(self):
        self.mu = self.mean.mean(self._xpm)
        return self._eng.unwhiten(self.v) + self.mu

    def initialise_target(self):                                   # GPA.jl:101-109, 245-250
        self.update_cK(INIT_LOG_NOISE)
        self.ll = float(np.sum(self.lik.log_dens(self._latent(), self.y)))
        self.target = self.ll - (self.v @ self.v + LOG2PI * self.nobs) / 2.0
        return self

    def update_ll(self, process=True, lik=True, domean=True, kern=True):        # GPA.jl:118-128
        if kern:
            self.update_cK()
        self.ll = float(np.sum(self.lik.log_dens(self._latent(), self.y)))
        return self

    def update_target(self, process=True, lik=True, domean=True, kern=True):    # GPA.jl:261-266
        self.update_ll(process=process, lik=lik, domean=domean, kern=kern)
        self.target = self.ll - (self.v @ self.v + LOG2PI * self.nobs) / 2.0
        return self

    def update_dll(self, process=True, lik=True, domean=True, kern=True):       # GPA.jl:183-228
        f = self._latent()                                          # precompute!, GPA.jl:158-163
        dl_df = self.lik.dlog_dens_df(f, self.y)
        dv = dk = None
        if process or kern:
            dv, dk = self._eng.gpa_grad(self.v, dl_df)
        out = []
        if process:
            out.extend(dv)                                          # U * dl_df, GPA.jl:200
        if lik and self.lik.num_params() > 0:
            out.extend(np.sum(self.lik.dlog_dens_dtheta(f, self.y), axis=0))
        if domean and self.mean.num_params() > 0:
            out.extend(self.mean.grad_stack(self._xpm).T @ dl_df)   # dll_mean!, GPA.jl:174-176
        if kern:
            out.extend(dk[self._exposed])
        self.dll = np.array(out, dtype=np.float64)
        return self

    def prior_gradlogpdf(self, process=True, lik=True, domean=True, kern=True):  # GPA.jl:383-399, no parameter priors
        n = (self.lik.num_params() if lik else 0) + (self.mean.num_params() if domean else 0) + \
            (self.kernel.num_params() if kern else 0)
        return np.concatenate([-self.v if process else np.zeros(0), np.zeros(n)])

    def update_dtarget(self, **kw):                                 # GPA.jl:268-272
        self.update_dll(**kw)
        self.dtarget = self.dll + self.prior_gradlogpdf(**kw)
        return self

    def update_target_and_dtarget(self, **kw):                      # GPA.jl:283-291
        self.update_target(**kw)
        return self.update_dtarget(**kw)

    # ---- parameters ----------------------------------------------------------------------
    def get_params(self, lik=True, domean=True, kern=True):         # GPA.jl:336-349
        p = list(self.v)
        if lik and self.lik.num_params() > 0:
            p.extend(self.lik.get_params())
        if domean and self.mean.num_params() > 0:
            p.extend(self.mean.get_params())
        if kern:
            p.extend(self.kernel.get_params())
        return np.array(p, dtype=np.float64)

    def num_params(self, lik=True, domean=True, kern=True):         # GPA.jl:351-357
        return self.get_params(lik=lik, domean=domean, kern=kern).size

    def set_params(self, hyp, process=True, lik=True, domean=True, kern=True):   # GPA.jl:359-381
        hyp = np.asarray(hyp, dtype=np.float64)
        i = 0
        if process:
            self.v = hyp[:self.nobs].copy()
            i += self.nobs
        n = self.lik.num_params()
        if lik and n > 0:
            self.lik.set_params(list(hyp[i:i + n]))
            i += n
        n = self.mean.num_params()
        if domean and n > 0:
            self.mean.set_params(list(hyp[i:i + n]))
            i += n
        if kern:
            n = self.kernel.num_params()
            self.kernel.set_params(list(hyp[i:i + n]))
            i += n
        if i != hyp.size:
            raise ValueError("wrong number of parameters")
        return self

    # ---- prediction ----------------------------------------------------------------------
    def predict_f(self, x, full_cov=False):
        """predict_f via predictMVN with alpha = cK \\ unwhiten(cK, v) (GPA.jl:294), on the current factor"""
        x = _as_dxn(x)
        if x.shape[0] != self.dim:
            raise ValueError("Gaussian Process object and input observations do not have consistent dimensions")
        xs = np.ascontiguousarray(x.T)
        alpha = self._eng.solve(self._eng.unwhiten(self.v))
        mu, var, cov = self._eng.predict(xs, alpha, want_var=not full_cov, full_cov=full_cov)
        mu = mu + self.mean.mean(xs)
        if full_cov:
            return mu, cov
        return mu, np.maximum(var, 0.0)                             # GP.jl:75

    def predict_y(self, x, full_cov=False):                         # GPA.jl:303-306
        mu, s2 = self.predict_f(x, full_cov=full_cov)
        return self.lik.predict_obs(mu, s2)
