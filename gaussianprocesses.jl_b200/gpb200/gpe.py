"""GPE -- host-side mirror of the reference's exact GP object (src/GPE.jl:3-567) driving the
B200 engine through the C ABI.  Same field names (x, y, mean, kernel, logNoise, dim, nobs, alpha,
mll, target, dmll, dtarget), same method names minus Julia's `!`, same gradient order
[noise; mean; kernel] (src/GPE.jl:298-324) and the same error behaviour (PosDefException /
ValueError where the reference throws PosDefException / ArgumentError).

This is the Python twin of julia/GPB200.jl's `B200Covariance <: CovarianceStrategy` methods: each
call below is one of the shim's overloads (update_cK!, \\, logdet, precompute!, dmll_kern!,
dmll_noise, predictMVN, predict_f).  x follows the reference layout: shape (dim, nobs), one
observation per column."""
import math

import numpy as np

from . import capi
from .kernels import Kernel, flatten
from .means import Mean, MeanZero


def _as_dxn(x):
    x = np.asarray(x, dtype=np.float64)
    if x.ndim == 1:                       # GPE(x::AbstractVector, ...) = GPE(x', ...)  (src/GPE.jl:96-97)
        x = x[None, :]
    if x.ndim != 2:
        raise ValueError("x must be a dim x nobs matrix")
    return x


class _RejectedStep(Exception):
    """optimize(): a trial point outside the domain (non-finite hyper-parameter)."""


class GPE:
    def __init__(self, x, y, mean=None, kernel=None, logNoise=-2.0, device=0, engine=None, capacity=0, stepsize=1000):
        if kernel is None or not isinstance(kernel, Kernel):
            raise ValueError("GPE needs a kernel")
        self.mean = mean if mean is not None else MeanZero()
        if not isinstance(self.mean, Mean):
            raise ValueError("mean must be a Mean")
        self.kernel = kernel
        self.logNoise = float(logNoise) if np.ndim(logNoise) == 0 else np.asarray(logNoise, dtype=np.float64).copy()
        self._eng = engine if engine is not None else capi.Engine(device)
        self._capacity, self._stepsize = int(capacity), int(stepsize)       # ElasticGPE(...; capacity, stepsize), GPEelastic.jl:55-66
        if self._capacity:
            self._eng.set_option("capacity", self._capacity)
        self.alpha = None
        self.mll = float("nan")
        self.target = float("nan")
        self.dmll = None
        self.dtarget = None
        self._factored_key = None
        self.fit(x, y)

    # ---- data ----------------------------------------------------------------------------
    def fit(self, x, y):
        """fit!(gp, x, y) (src/GPE.jl:128-136): replace the data, rebuild the device state."""
        x = _as_dxn(x)
        y = np.asarray(y, dtype=np.float64).ravel()
        if x.shape[1] != y.size:
            raise ValueError("Input and output observations must have consistent dimensions.")   # GPE.jl:41
        self.x, self.y = x, y
        self.dim, self.nobs = x.shape
        self._xpm = np.ascontiguousarray(x.T)            # (nobs, dim): Julia's memory layout
        self._eng.set_data(self._xpm)
        if getattr(self, "_world", 1) > 1 and getattr(self, "_p2p", False):
            from .dist import exchange_ipc                # buffers may have been reallocated: re-map the peers
            exchange_ipc(self._eng)
        self._sync_kernel()
        self.initialise_target()
        return self

    def push(self, x, y):
        """push!(gp, x, y) (src/GPE.jl:530-539): append observations and refit (the device state is rebuilt, exactly
        like the reference rebuilds data / cK wholesale)."""
        x = _as_dxn(x)
        if x.shape[0] != self.dim:
            raise ValueError("Input observations must have the same dimension as the GP")
        y = np.atleast_1d(np.asarray(y, dtype=np.float64)).ravel()
        return self.fit(np.concatenate([self.x, x], axis=1), np.concatenate([self.y, y]))

    def append(self, x, y):
        """append!(gp::ElasticGPE, x, y) (src/GPEelastic.jl:13-22): add observations keeping the hyper-parameters; the device
        extends its Cholesky factor in place (O(k N^2)) and update_target!(gp, kern=false, noise=false) refreshes alpha / mll.
        Needs a GPE built with `capacity=` (ElasticGPE(...; capacity, stepsize)); beyond the capacity the data is refitted with
        `stepsize` more rows reserved, which is what ElasticPDMats' resize! amounts to."""
        x = _as_dxn(x)
        if x.shape[0] != self.dim:
            raise ValueError("Input observations must have the same dimension as the GP")
        y = np.atleast_1d(np.asarray(y, dtype=np.float64)).ravel()
        if x.shape[1] != y.size:
            raise ValueError("%d observations, but %d targets." % (x.shape[1], y.size))        # GPEelastic.jl:15
        if np.ndim(self.logNoise) or self.nobs + y.size > getattr(self, "_capacity", 0):
            self._capacity = self.nobs + y.size + getattr(self, "_stepsize", 1000)
            self._eng.set_option("capacity", self._capacity)
            return self.fit(np.concatenate([self.x, x], axis=1), np.concatenate([self.y, y]))
        self._eng.append(np.ascontiguousarray(x.T))
        self.x = np.concatenate([self.x, x], axis=1)
        self.y = np.concatenate([self.y, y])
        self.nobs = self.y.size
        self._xpm = np.ascontiguousarray(self.x.T)
        return self.update_target(kern=False, noise=False)                                  # GPEelastic.jl:21

    def reload_data(self, x, y):
        """Re-upload (x, y) of unchanged shape to the device without re-evaluating the target
        (one host->device copy of the inputs; the next update_mll! uses them)."""
        x = _as_dxn(x)
        y = np.asarray(y, dtype=np.float64).ravel()
        if x.shape != (self.dim, self.nobs) or y.size != self.nobs:
            raise ValueError("reload_data: shape changed; use fit")
        self.x, self.y = x, y
        self._xpm = np.ascontiguousarray(x.T)
        self._eng.set_data(self._xpm)
        return self

    def init_distributed(self, p2p=None):
        """Multi-GPU: join this rank's engine into the NCCL communicator of the torch.distributed
        default group (one process per GPU).  Every later update_*/predict call is collective."""
        import os
        from .dist import init_engine_comm
        if p2p is None:
            # fused peer-memory panel push: measured faster than the NCCL broadcast at 2 and 4 GPUs, slower at 8 (the
            # owner sends one unicast copy per peer; NCCL rides the NVSwitch) -> default on up to 4 ranks
            import torch.distributed as tdist
            env = os.environ.get("GPB200_P2P")
            p2p = (env != "0") if env is not None else (tdist.is_initialized() and tdist.get_world_size() <= 4)
        world, rank = init_engine_comm(self._eng, p2p=p2p)
        self._world, self._p2p = world, bool(p2p)
        if world > 1:
            self.update_target()
        return world, rank

    def _sync_kernel(self):
        ops, dims, theta, exposed = flatten(self.kernel, self.dim)
        self._exposed = exposed
        self._eng.set_kernel(ops, dims, theta.size)
        self._factored_key = None

    def _theta_full(self):
        return flatten(self.kernel, self.dim)[2]

    # ---- log target ----------------------------------------------------------------------
    def noise_variance(self):                             # GPE.jl:269-271
        return np.exp(2.0 * np.asarray(self.logNoise)) if np.ndim(self.logNoise) else math.exp(2.0 * self.logNoise)

    def update_cK(self):
        """update_cK!(gp) (src/GPE.jl:169-195): Gram + noise + Cholesky on the device."""
        self._eng.factorize(self._theta_full(), self.logNoise)

    def update_mll(self, noise=True, domean=True, kern=True):
        """update_mll!(gp) (src/GPE.jl:202-212)."""
        if kern or noise:
            self.update_cK()
        mu = self.mean.mean(self._xpm)
        self.alpha, self.mll = self._eng.mll(self.y - mu)
        return self

    def update_dmll(self, noise=True, domean=True, kern=True):
        """update_dmll!(gp, precomp) (src/GPE.jl:298-324)."""
        gk_full, trA = None, None
        if noise or kern:                                         # mean-only gradient needs neither K^-1 nor the trace
            self._eng.grad_prepare()                              # precompute! -> get_ααinvcKI!
            gk_full, trA = self._eng.grad_kernel()                # dmll_kern! + tr(A)
        out = []
        if noise:
            if np.ndim(self.logNoise):
                raise AssertionError("num_params(gp.logNoise) == 1")        # GPE.jl:310
            out.append(math.exp(2.0 * self.logNoise) * trA)        # dmll_noise, GPE.jl:273-275
        if domean and self.mean.num_params() > 0:
            out.extend(self.mean.grad_stack(self._xpm).T @ self.alpha)      # dmll_mean!, GPE.jl:282-288
        if kern:
            out.extend(gk_full[self._exposed])                     # FixedKernel selection, fixed_kernel.jl:64-66
        self.dmll = np.array(out, dtype=np.float64)
        return self

    def update_mll_and_dmll(self, **kw):                           # GPE.jl:332-335
        self.update_mll(**kw)
        self.update_dmll(**kw)
        return self

    def initialise_target(self):                                   # GPE.jl:346-349 (no priors in this mirror)
        self.update_mll()
        self.target = self.mll
        return self

    def update_target(self, **kw):                                 # GPE.jl:356-360
        self.update_mll(**kw)
        self.target = self.mll
        return self

    def update_target_and_dtarget(self, **kw):                     # GPE.jl:387-392
        self.update_mll_and_dmll(**kw)
        self.target = self.mll
        self.dtarget = self.dmll.copy()
        return self

    # ---- prediction ----------------------------------------------------------------------
    def predict_f(self, x, full_cov=False, partition=False):
        """predict_f(gp, x; full_cov) (src/GP.jl:64-79), batched on the device.
        partition=True (multi-GPU, replicated storage): every rank holds the whole factor, so the test points are split
        over the ranks -- each engine predicts its contiguous slice, independent of the others -- and the O(M) results are
        all-gathered; every rank returns the full vectors.  (Row-sharded storage predicts collectively instead: the
        triangular solve itself is distributed, see shard_predict_solve.)"""
        x = _as_dxn(x)
        if x.shape[0] != self.dim:
            raise ValueError("Gaussian Process object and input observations do not have consistent dimensions")
        xs = np.ascontiguousarray(x.T)
        if partition and getattr(self, "_world", 1) > 1:
            return self._predict_f_partitioned(xs, full_cov)
        mu, var, cov = self._eng.predict(xs, None, want_var=not full_cov, full_cov=full_cov)
        mu = mu + self.mean.mean(xs)
        if full_cov:
            return mu, cov
        return mu, np.maximum(var, 0.0)                            # GP.jl:75

    def _predict_f_partitioned(self, xs, full_cov):
        import torch.distributed as tdist
        from .dist import partition_bounds, allgather_concat
        if full_cov:
            raise ValueError("predict_f(partition=True): the full covariance couples all test points; use partition=False")
        if self._eng.storage_info()["sharded"]:
            raise ValueError("predict_f(partition=True) needs replicated storage; the row-sharded predict is collective")
        world, rank = tdist.get_world_size(), tdist.get_rank()
        b = partition_bounds(xs.shape[0], world)
        counts = [b[r + 1] - b[r] for r in range(world)]
        if counts[rank]:
            mu, var, _ = self._eng.predict(xs[b[rank]:b[rank + 1]], None, want_var=True, full_cov=False)
        else:
            mu, var = np.empty(0), np.empty(0)
        mu = allgather_concat(mu, counts) + self.mean.mean(xs)
        return mu, np.maximum(allgather_concat(var, counts), 0.0)                # GP.jl:75

    def predict_y(self, x, full_cov=False):                        # GPE.jl:408-416
        mu, s2 = self.predict_f(x, full_cov=full_cov)
        nv = self.noise_variance()
        if full_cov:
            return mu, s2 + nv * np.eye(s2.shape[0])
        return mu, s2 + nv

    def predict_LOO(self):
        """predict_LOO(gp) (src/crossvalidation.jl:8-36): leave-one-out means / variances from diag(K_y^-1) and alpha."""
        self._eng.grad_prepare()
        s2 = 1.0 / self._eng.inverse_diag()
        return -self.alpha * s2 + self.y, s2

    def logp_LOO(self):
        """logp_LOO(gp) (src/crossvalidation.jl:37-49): sum of Normal log-pdfs of y_i under the LOO predictions."""
        mu, s2 = self.predict_LOO()
        return float(np.sum(-0.5 * np.log(2.0 * np.pi * s2) - 0.5 * (self.y - mu) ** 2 / s2))

    # ---- cross-validation on the device's resident K_y^-1 (src/crossvalidation.jl) ------------------------------------
    def _loo_component(self, Zja, ZjSinv, s2, mu):
        """body of dlogpdθ_LOO_kern! / dlogpdσ2_LOO for one parameter (crossvalidation.jl:94-107, 130-140), before the -1/2"""
        ds2 = ZjSinv * s2 ** 2
        dmu = Zja * s2 - self.alpha * ds2
        y = self.y
        return float(-np.sum(2.0 * (y - mu) / s2 * dmu) - np.sum((y - mu) ** 2 * ZjSinv) + np.sum(ZjSinv * s2))

    def dlogp_LOO(self, noise=True, domean=False, kern=True):
        """dlogpdθ_LOO(gp; noise, domean, kern) (src/crossvalidation.jl:150-178): gradient of the leave-one-out criterion.
        Per parameter the device forms inv(Σ) dK_j and its product with inv(Σ) (two N^3 GEMMs on the resident inverse) and
        returns Z_j α and diag(Z_j inv(Σ)); the O(N) assembly below follows the reference line by line."""
        if domean and self.mean.num_params() > 0:
            raise NotImplementedError("I don't know how to do means yet")          # crossvalidation.jl:168
        mu, s2 = self.predict_LOO()
        out = []
        if noise:
            Zja, ZjS = self._eng.cv_param(-1)
            out.append(-self._loo_component(Zja, ZjS, s2, mu) / 2.0 * 2.0 * math.exp(2.0 * self.logNoise))
        if kern:
            for j in self._exposed:
                Zja, ZjS = self._eng.cv_param(int(j))
                out.append(-0.5 * self._loo_component(Zja, ZjS, s2, mu))
        return np.array(out)

    def predict_CVfold(self, folds):
        """predict_CVfold(gp, folds) (src/crossvalidation.jl:180-218): per fold V the predictive mean / covariance of y_V given
        the other observations, from the principal sub-block inv(Σ)[V,V] read off the device."""
        self._eng.grad_prepare()
        mus, Sigs = [], []
        for V in folds:
            V = np.asarray(V, dtype=np.int64)
            SVT = np.linalg.inv(self._eng.cv_block(0, V))
            mus.append(self.y[V] - SVT @ self.alpha[V])
            Sigs.append(SVT)
        return mus, Sigs

    def logp_CVfold(self, folds):
        """logp_CVfold(gp, folds) (src/crossvalidation.jl:225-237)."""
        mus, Sigs = self.predict_CVfold(folds)
        cv = 0.0
        for mu, S, V in zip(mus, Sigs, folds):
            V = np.asarray(V, dtype=np.int64)
            L = np.linalg.cholesky(S + 1e-10 * np.eye(V.size))                    # make_posdef!(ΣVT; nugget=1e-10)
            z = np.linalg.solve(L, self.y[V] - mu)
            cv += -0.5 * (z @ z) - np.sum(np.log(np.diag(L))) - 0.5 * V.size * math.log(2.0 * math.pi)
        return float(cv)

    def _fold_component(self, Zja, folds, inv_blocks):
        comp = 0.0
        for V, SVTinv in zip(folds, inv_blocks):                                   # gradient_fold, crossvalidation.jl:248-262
            V = np.asarray(V, dtype=np.int64)
            ZVV = self._eng.cv_block(1, V)
            SVTa = np.linalg.solve(SVTinv, self.alpha[V])
            comp += -2.0 * (SVTa @ Zja[V]) + SVTa @ (ZVV @ SVTa) + np.trace(np.linalg.solve(SVTinv, ZVV))
        return comp

    def dlogp_CVfold(self, folds, noise=True, domean=False, kern=True):
        """dlogpdθ_CVfold(gp, folds; noise, domean, kern) (src/crossvalidation.jl:264-341)."""
        if domean and self.mean.num_params() > 0:
            raise NotImplementedError("I don't know how to do means yet")          # crossvalidation.jl:330
        self._eng.grad_prepare()
        inv_blocks = [self._eng.cv_block(0, np.asarray(V, dtype=np.int64)) for V in folds]
        out = []
        if noise:
            Zja, _ = self._eng.cv_param(-1)
            out.append(-self._fold_component(Zja, folds, inv_blocks) / 2.0 * 2.0 * math.exp(2.0 * self.logNoise))
        if kern:
            for j in self._exposed:
                Zja, _ = self._eng.cv_param(int(j))
                out.append(-0.5 * self._fold_component(Zja, folds, inv_blocks))
        return np.array(out)

    def rand(self, x, n=1, nugget=1e-10, rng=None):
        """rand(gp, X, n) (src/GP.jl:120-146): n posterior draws at the columns of x, computed on the device (predictive
        covariance, make_posdef!(Σ; nugget) Cholesky, unwhiten!); only the standard-normal draws come from the host RNG,
        like the reference's randn(nobs, n_sample).  Returns a (npred, n) array."""
        rng = np.random.default_rng() if rng is None else rng
        x = _as_dxn(x)
        if x.shape[0] != self.dim:
            raise ValueError("Gaussian Process object and input observations do not have consistent dimensions")
        xs = np.ascontiguousarray(x.T)
        z = rng.standard_normal((int(n), xs.shape[0]))
        _, draws = self._eng.rand(xs, z, nugget=nugget)
        return (draws + self.mean.mean(xs)[None, :]).T

    # ---- parameters ----------------------------------------------------------------------
    def get_params(self, noise=True, domean=True, kern=True):      # GPE.jl:447-458
        p = []
        if noise:
            p.extend(np.atleast_1d(self.logNoise))
        if domean:
            p.extend(self.mean.get_params())
        if kern:
            p.extend(self.kernel.get_params())
        return np.array(p, dtype=np.float64)

    def num_params(self, **kw):
        return self.get_params(**kw).size

    def set_params(self, hyp, noise=True, domean=True, kern=True):  # GPE.jl:492-510
        hyp = np.asarray(hyp, dtype=np.float64)
        i = 0
        if noise:
            n = np.size(self.logNoise)
            self.logNoise = float(hyp[0]) if np.ndim(self.logNoise) == 0 else hyp[:n].copy()
            i += n
        if domean:
            n = self.mean.num_params()
            self.mean.set_params(hyp[i:i + n])
            i += n
        if kern:
            n = self.kernel.num_params()
            self.kernel.set_params(list(hyp[i:i + n]))
            i += n
        if i != hyp.size:
            raise ValueError("wrong number of hyper-parameters")
        return self

    # ---- optimisation (src/optimize.jl:19-97) ----------------------------------------------
    def optimize(self, noise=True, domean=True, kern=True, maxiter=100, **kw):
        """optimize!(gp): L-BFGS on -target with the reference's exception filter (PosDefException / ArgumentError ->
        rejected step, parameters rolled back, optimize.jl:46-87).  Optim.jl's line search backs off from the
        reference's `Inf`; scipy's L-BFGS-B stops on it, so a large finite penalty plays that role here."""
        from scipy.optimize import minimize

        flags = dict(noise=noise, domean=domean, kern=kern)
        best = {"f": None}

        def fg(hyp):
            prev = self.get_params(**flags)
            try:
                if not np.all(np.isfinite(hyp)):
                    raise _RejectedStep("non-finite hyper-parameter")
                self.set_params(hyp, **flags)
                self.update_target_and_dtarget(**flags)
                best["f"] = -self.target if best["f"] is None else min(best["f"], -self.target)
                return -self.target, -self.dtarget
            except (np.linalg.LinAlgError, _RejectedStep):            # PosDefException subclasses LinAlgError
                # only the reference's filtered exceptions (PosDefException / non-finite parameters, optimize.jl:46-87)
                # reject a step; call-order / shape errors (ValueError from the engine) propagate.  The penalty's
                # gradient points back to the last accepted point so that the line search retreats.
                self.set_params(prev, **flags)
                return 1e10 + 1e6 * abs(best["f"] or 0.0), np.asarray(hyp, dtype=np.float64) - prev

        res = minimize(fg, self.get_params(**flags), jac=True, method="L-BFGS-B", options=dict(maxiter=maxiter), **kw)
        self.set_params(res.x, **flags)
        self.update_target()
        return res


def GP(x, y, mean, kernel, logNoise=-2.0, **kw):                   # GPE.jl:119
    """GP(x, y, mean, kernel, logNoise) builds a GPE; GP(x, y, mean, kernel, lik) with a Likelihood builds a GPA
    (GPA.jl:93-94)."""
    from .likelihoods import Likelihood
    if isinstance(logNoise, Likelihood):
        from .gpa import GPA
        return GPA(x, y, mean, kernel, logNoise, **kw)
    return GPE(x, y, mean, kernel, logNoise, **kw)


def ElasticGPE(x, y, mean=None, kernel=None, logNoise=-2.0, capacity=1000, stepsize=1000, **kw):
    """ElasticGPE(x, y, mean, kernel, logNoise; capacity, stepsize) (src/GPEelastic.jl:55-66): a GPE whose device buffers
    reserve `capacity` observations so that append! extends the factor in place."""
    return GPE(x, y, mean, kernel, logNoise, capacity=max(int(capacity), np.asarray(y).size), stepsize=stepsize, **kw)
