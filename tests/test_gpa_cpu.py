"""CPU (-m "not gpu"): the latent-variable GP (GPA).  The numpy oracle's gradient against finite differences for the six
likelihoods (the setup of the reference's test/gpa.jl), the closed-form reverse-mode Cholesky the device implements
against the literal chol_unblocked_rev!, the likelihood mirror against scipy.stats and quadrature, and the host
plumbing of gpb200.GPA over a stand-in engine backed by the oracle."""
import itertools
import math
import types

import numpy as np
import pytest
import scipy.linalg as sl
from scipy import integrate, stats
from scipy.special import expit, ndtr
from threadpoolctl import threadpool_limits

import gpb200
import gpa_oracle as go
from oracle import gp_oracle as orc


@pytest.fixture(autouse=True)
def _single_threaded_blas():
    """the oracle's BLAS stays on one thread: OpenBLAS's thread pool hangs in a process that has already run the
    torch.multiprocessing workers of tests/test_dist_cpu.py"""
    with threadpool_limits(1):
        yield


def gpa_jl_data(n=20, d=3, seed=1):
    """test/gpa.jl:8-24 with a seeded numpy RNG: inputs, and one y per likelihood"""
    rng = np.random.default_rng(seed)
    X = 2 * np.pi * rng.random((n, d))
    f = np.sin(X).sum(axis=1) / d
    ys = dict(Bern=rng.random(n) < np.abs(f),
              Bin=rng.binomial(n, expit(f)),
              Exp=rng.exponential(f ** 2),
              Gauss=f.copy(),
              Pois=rng.poisson(np.exp(f)),
              StuT=f + rng.standard_t(3, n))
    return X, ys, rng


LSPECS = [("Bern",), ("Bin", 20), ("Exp",), ("Gauss", -1.0), ("Pois",), ("StuT", 3, 0.1)]


def host_lik(lspec):
    name = lspec[0]
    return dict(Bern=lambda: gpb200.BernLik(), Bin=lambda: gpb200.BinLik(lspec[1]), Exp=lambda: gpb200.ExpLik(),
                Gauss=lambda: gpb200.GaussLik(lspec[1]), Pois=lambda: gpb200.PoisLik(),
                StuT=lambda: gpb200.StuTLik(lspec[1], lspec[2]))[name]()


def _unpack(params, n, lspec):
    """[v; lik; kernel] of test/gpa.jl (MeanZero, SE(0,0))"""
    v = params[:n]
    nl = go.lik_num_params(lspec)
    ls = lspec[:-1] + (params[n],) if nl else lspec
    return v, ls, ("SEIso", list(params[n + nl:]))


@pytest.mark.parametrize("lspec", LSPECS, ids=[l[0] for l in LSPECS])
def test_oracle_dtarget_matches_finite_differences(lspec):
    X, ys, rng = gpa_jl_data()
    y, n = ys[lspec[0]], X.shape[0]
    params = 0.5 * rng.standard_normal(n + go.lik_num_params(lspec) + 2)

    def target(p):
        v, ls, spec = _unpack(p, n, lspec)
        return go.gpa_target(spec, X, y, v, ls)

    v, ls, spec = _unpack(params, n, lspec)
    exact = go.gpa_dtarget(spec, X, y, v, ls)
    h = 1e-6
    num = np.array([(target(params + h * e) - target(params - h * e)) / (2 * h) for e in np.eye(params.size)])
    np.testing.assert_allclose(exact, num, rtol=1e-5, atol=1e-5 * np.max(np.abs(num)))


def test_closed_form_matches_literal_reverse_mode_cholesky():
    rng = np.random.default_rng(3)
    n = 203
    X = rng.standard_normal((n, 3))
    spec = ("Sum", ("Mat32Iso", [0.3, 0.1]), ("RQIso", [0.2, -0.1, 0.3]))
    L = go.chol_factor(spec, X, -2.0)
    v, g = rng.standard_normal(n), rng.standard_normal(n)
    lit, L_bar = go.dll_kern_literal(spec, X, L, v, g)
    cf = go.dll_kern_closed_form(spec, X, L, v, g)
    assert np.max(np.abs(cf - lit)) <= 1e-12 * np.max(np.abs(lit))
    S = go.chol_bar_closed_form(L, v, g)
    lo = np.tril(L_bar, -1)
    S_lit = lo + lo.T + np.diag(np.diag(L_bar))       # the doubled-diagonal L_bar of GPA.jl:168-170, symmetrised
    assert np.max(np.abs(S - S_lit)) <= 1e-12 * np.max(np.abs(S_lit))


def test_chol_unblocked_rev_is_the_adjoint_of_cholesky():
    """<L_bar, dL> = <A_bar, dA> for a symmetric perturbation dA, i.e. chol_unblocked_rev! is the reverse mode of chol"""
    rng = np.random.default_rng(4)
    n = 12
    B = rng.standard_normal((n, n))
    A = B @ B.T + n * np.eye(n)
    dA = rng.standard_normal((n, n)); dA = dA + dA.T
    L = np.linalg.cholesky(A)
    L_bar = np.tril(rng.standard_normal((n, n)))
    A_bar = go.chol_unblocked_rev(L, L_bar.copy())
    h = 1e-6
    dL = (np.linalg.cholesky(A + h * dA) - np.linalg.cholesky(A - h * dA)) / (2 * h)
    lhs = np.sum(L_bar * dL)
    rhs = np.sum(np.tril(A_bar, -1) * dA) + np.sum(np.diag(A_bar) * np.diag(dA))
    assert abs(lhs - rhs) <= 1e-7 * abs(lhs)


# ---- the likelihood mirror ------------------------------------------------------------------------------------------
def _lik_cases():
    rng = np.random.default_rng(5)
    n = 40
    f = 0.8 * rng.standard_normal(n)
    return f, [
        (gpb200.BernLik(), rng.random(n) < 0.5, lambda f, y, L: stats.bernoulli.logpmf(y, ndtr(f))),
        (gpb200.BinLik(7), rng.integers(0, 8, n), lambda f, y, L: stats.binom.logpmf(y, 7, expit(f))),
        (gpb200.ExpLik(), rng.exponential(1.0, n), lambda f, y, L: stats.expon.logpdf(y, scale=np.exp(f))),
        (gpb200.GaussLik(-0.7), rng.standard_normal(n), lambda f, y, L: stats.norm.logpdf(y, f, L.sigma)),
        (gpb200.PoisLik(), rng.poisson(1.5, n), lambda f, y, L: stats.poisson.logpmf(y, np.exp(f))),
        (gpb200.StuTLik(4, 0.2), rng.standard_normal(n), lambda f, y, L: stats.t.logpdf(y, 4, loc=f, scale=L.sigma)),
    ]


def test_likelihood_log_densities_match_scipy_and_oracle():
    f, cases = _lik_cases()
    for (lik, y, ref), ls in zip(cases, [("Bern",), ("Bin", 7), ("Exp",), ("Gauss", -0.7), ("Pois",), ("StuT", 4, 0.2)]):
        np.testing.assert_allclose(lik.log_dens(f, y), ref(f, y, lik), rtol=1e-12, atol=1e-12, err_msg=type(lik).__name__)
        np.testing.assert_allclose(lik.log_dens(f, y), go.log_dens(ls, f, y), rtol=1e-13, atol=1e-13)
        np.testing.assert_allclose(lik.dlog_dens_df(f, y), go.dlog_dens_df(ls, f, y), rtol=1e-13, atol=1e-13)
        np.testing.assert_allclose(lik.dlog_dens_dtheta(f, y), go.dlog_dens_dtheta(ls, f, y), rtol=1e-13, atol=1e-13)


def test_likelihood_derivatives_match_finite_differences():
    f, cases = _lik_cases()
    h = 1e-6
    for lik, y, _ in cases:
        num = (lik.log_dens(f + h, y) - lik.log_dens(f - h, y)) / (2 * h)
        np.testing.assert_allclose(lik.dlog_dens_df(f, y), num, rtol=1e-6, atol=1e-7, err_msg=type(lik).__name__)
        p = np.array(lik.get_params(), dtype=np.float64)
        assert lik.num_params() == p.size
        for j in range(p.size):
            e = np.zeros(p.size); e[j] = h
            lik.set_params(list(p + e)); up = lik.log_dens(f, y)
            lik.set_params(list(p - e)); dn = lik.log_dens(f, y)
            lik.set_params(list(p))
            np.testing.assert_allclose(lik.dlog_dens_dtheta(f, y)[:, j], (up - dn) / (2 * h), rtol=1e-6, atol=1e-7)


def test_predict_obs_matches_direct_quadrature():
    fm, fv = np.array([-0.4, 0.1, 0.6]), np.array([0.05, 0.3, 0.8])
    _, cases = _lik_cases()
    for lik, _, _ in cases:
        mu, s2 = lik.predict_obs(fm, fv)
        for i in range(fm.size):
            dens = stats.norm(fm[i], math.sqrt(fv[i])).pdf
            lo, hi = fm[i] - 12 * math.sqrt(fv[i]), fm[i] + 12 * math.sqrt(fv[i])
            m = integrate.quad(lambda t: lik.mean_lik(np.array([t]))[0] * dens(t), lo, hi, epsabs=1e-13, epsrel=1e-12)[0]
            m2 = integrate.quad(lambda t: (lik.var_lik(np.array([t]))[0] + lik.mean_lik(np.array([t]))[0] ** 2) * dens(t),
                                lo, hi, epsabs=1e-13, epsrel=1e-12)[0]
            assert mu[i] == pytest.approx(m, rel=1e-7, abs=1e-10), type(lik).__name__
            assert s2[i] == pytest.approx(m2 - m * m, rel=1e-6, abs=1e-9), type(lik).__name__


# ---- host plumbing over a stand-in engine ---------------------------------------------------------------------------
class OracleGPAEngine:
    """Stand-in with the Engine interface, backed by the CPU oracle -- TEST ONLY, to exercise the GPA host plumbing
    without a GPU (the kernels used here have no fixed parameters, so the full and exposed parameter vectors agree)."""

    def __init__(self):
        self.n_theta = 0
        self.calls = []

    def bind(self, gp):
        self.gp = gp

    def set_data(self, x):
        self.X = np.array(x); self.N, self.d = x.shape

    def set_kernel(self, ops, dims, n_theta):
        self.n_theta = n_theta

    def factorize(self, theta, ln, extra_nugget=0.0):
        self.calls.append(("factorize", float(ln)))
        self.spec = self.gp.kernel.spec()
        self.L = go.chol_factor(self.spec, self.X, float(ln))

    def unwhiten(self, v):
        return self.L @ v

    def gpa_grad(self, v, g):
        self.calls.append(("gpa_grad",))
        return self.L.T @ g, go.dll_kern_literal(self.spec, self.X, self.L, v, g)[0]

    def solve(self, r):
        return sl.cho_solve((self.L, True), r)

    def predict(self, xs, alpha=None, want_var=True, full_cov=False):
        mu, var = orc.predict_f(self.spec, self.X, dict(U=self.L.T, alpha=alpha), xs, full_cov=full_cov)
        return (mu, None, var) if full_cov else (mu, var, None)


def _gpa(X, y, mean, kernel, lik):
    eng = OracleGPAEngine()
    gp = gpb200.GPA.__new__(gpb200.GPA)
    eng.bind(gp)
    gpb200.GPA.__init__(gp, X.T, y, mean, kernel, lik, engine=eng)
    return gp, eng


def _model(seed=6, n=30):
    rng = np.random.default_rng(seed)
    X = rng.standard_normal((n, 2))
    y = np.sin(X.sum(axis=1)) + 0.3 * rng.standard_normal(n)
    k = gpb200.SEIso(-0.3, 0.1) + gpb200.RQIso(0.2, -0.4, 0.3)
    spec = ("Sum", ("SEIso", [-0.3, 0.1]), ("RQIso", [0.2, -0.4, 0.3]))
    return X, y, k, spec, rng


def test_gpa_parameter_order_and_round_trip():
    X, y, k, _, rng = _model()
    gp, eng = _gpa(X, y, gpb200.MeanConst(0.2), k, gpb200.StuTLik(3, 0.1))
    assert eng.calls == [("factorize", pytest.approx(0.5 * math.log(1e-6)))]       # initialise_ll!'s 1e-6 nugget
    n = X.shape[0]
    assert np.all(gp.v == 0) and gp.num_params() == n + 1 + 1 + 5
    p = gp.get_params()
    assert p[n:].tolist() == pytest.approx([0.1, 0.2, -0.3, 0.1, 0.2, -0.4, 0.3])        # [v; lik; mean; kernel]
    q = rng.standard_normal(p.size)
    gp.set_params(q)
    np.testing.assert_allclose(gp.get_params(), q, rtol=1e-15, atol=1e-15)      # lσ goes through exp / log
    assert gp.get_params(lik=False, domean=False).size == n + 5
    gp.set_params(q[n:n + 1], process=False, domean=False, kern=False)
    assert gp.lik.get_params() == pytest.approx([q[n]])
    with pytest.raises(ValueError):
        gp.set_params(q[:-1])


@pytest.mark.parametrize("flags", list(itertools.product([True, False], repeat=4)))
def test_gpa_dtarget_assembly_under_flags(flags):
    process, lik, domean, kern = flags
    X, y, k, spec, rng = _model()
    gp, eng = _gpa(X, y, gpb200.MeanConst(0.2), k, gpb200.GaussLik(-0.5))
    gp.set_params(np.concatenate([0.5 * rng.standard_normal(X.shape[0]), [-0.4, 0.3], gp.get_params()[-5:]]))
    kw = dict(process=process, lik=lik, domean=domean, kern=kern)
    gp.update_target()                       # cK with update_cK!'s nugget; kern=False below keeps it (GPA.jl:119-123)
    n0 = len(eng.calls)
    gp.update_target_and_dtarget(**kw)
    assert eng.calls[n0:] == [("factorize", -20.0)] * kern + [("gpa_grad",)] * (process or kern)
    ref = go.gpa_dtarget(spec, X, y, gp.v, ("Gauss", -0.4), ("MeanConst", 0.3), **kw)
    np.testing.assert_allclose(gp.dtarget, ref, rtol=1e-12, atol=1e-12)
    assert gp.target == pytest.approx(go.gpa_target(spec, X, y, gp.v, ("Gauss", -0.4), ("MeanConst", 0.3)), rel=1e-13)


def test_gp_with_likelihood_dispatches_to_gpa_and_predicts():
    X, y, k, spec, rng = _model()
    yb = y > 0
    eng = OracleGPAEngine()
    eng.gp = types.SimpleNamespace(kernel=k)
    out = gpb200.GP(X.T, yb, gpb200.MeanZero(), k, gpb200.BernLik(), engine=eng)
    assert isinstance(out, gpb200.GPA) and not isinstance(out, gpb200.GPE)
    out.set_params(np.concatenate([0.5 * rng.standard_normal(X.shape[0]), out.get_params()[-5:]]))
    out.update_target()
    Xs = rng.standard_normal((7, 2))
    L = go.chol_factor(spec, X)
    alpha = sl.cho_solve((L, True), L @ out.v)                 # cK \ unwhiten(cK, v), GPA.jl:294
    mo, vo = orc.predict_f(spec, X, dict(U=L.T, alpha=alpha), Xs)
    mu, s2 = out.predict_f(Xs.T)
    np.testing.assert_allclose(mu, mo, rtol=1e-12, atol=1e-12)
    np.testing.assert_allclose(s2, vo, rtol=1e-12, atol=1e-12)
    p, pv = out.predict_y(Xs.T)
    np.testing.assert_allclose(p, ndtr(mo / np.sqrt(1 + vo)), rtol=1e-12)
    np.testing.assert_allclose(pv, p - p * p, rtol=1e-12)
    with pytest.raises(ValueError):
        gpb200.GPA(X.T, y, gpb200.MeanZero(), k, "not a likelihood", engine=OracleGPAEngine())
