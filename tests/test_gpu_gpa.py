"""GPU: the latent-variable GP (GPA) on the device -- f = L v, the closed-form reverse-mode Cholesky gradient and the
handle state it leaves, against the CPU oracle (tests/gpa_oracle.py)."""
import math

import numpy as np
import pytest
import scipy.linalg as sl
from scipy.special import expit
from threadpoolctl import threadpool_limits

import gpa_oracle as go
from oracle import gp_oracle as orc

pytestmark = pytest.mark.gpu


@pytest.fixture(autouse=True)
def _single_threaded_blas():
    """the oracle's BLAS stays on one thread: OpenBLAS's thread pool hangs in a process that has already run the
    torch.multiprocessing workers of tests/test_dist_cpu.py"""
    with threadpool_limits(1):
        yield


def _data(n, d, seed):
    rng = np.random.default_rng(seed)
    X = rng.standard_normal((n, d))
    f = np.sin(X).sum(axis=1) / d
    ys = dict(Bern=rng.random(n) < np.abs(f), Bin=rng.binomial(20, expit(f)), Exp=rng.exponential(f ** 2 + 0.1),
              Gauss=f.copy(), Pois=rng.poisson(np.exp(f)), StuT=f + rng.standard_t(3, n))
    return X, ys, rng


def _lik(lspec):
    import gpb200 as g
    return dict(Bern=lambda: g.BernLik(), Bin=lambda: g.BinLik(lspec[1]), Exp=lambda: g.ExpLik(), Gauss=lambda: g.GaussLik(lspec[1]),
                Pois=lambda: g.PoisLik(), StuT=lambda: g.StuTLik(lspec[1], lspec[2]))[lspec[0]]()


LSPECS = [("Bern",), ("Bin", 20), ("Exp",), ("Gauss", -1.0), ("Pois",), ("StuT", 3, 0.1)]


def _kernels():
    import gpb200 as g
    # short length-scales keep K + exp(-40) I well conditioned (GPA factorises with update_cK!'s tiny nugget)
    return {"SEIso": (lambda: g.SEIso(math.log(0.4), 0.1), ("SEIso", [math.log(0.4), 0.1])),
            "Mat32+RQ": (lambda: g.Mat32Iso(math.log(0.3), 0.0) + g.RQIso(math.log(0.3), -0.5, 0.2),
                         ("Sum", ("Mat32Iso", [math.log(0.3), 0.0]), ("RQIso", [math.log(0.3), -0.5, 0.2])))}


@pytest.mark.parametrize("n", [20, 700, 3000])
def test_unwhiten_matches_oracle(n):
    import gpb200
    X, _, rng = _data(n, 3, n)
    eng = gpb200.Engine(0)
    eng.set_data(X)
    ops, dims, theta, _ = gpb200.flatten(gpb200.Mat32Iso(0.2, 0.1), 3)
    eng.set_kernel(ops, dims, theta.size)
    eng.factorize(theta, -1.0)
    v = rng.standard_normal(n)
    ref = go.chol_factor(("Mat32Iso", [0.2, 0.1]), X, -1.0) @ v
    f = eng.unwhiten(v)
    assert np.max(np.abs(f - ref)) <= 1e-12 * np.max(np.abs(ref))
    eng.close()


@pytest.mark.parametrize("kname", ["SEIso", "Mat32+RQ"])
@pytest.mark.parametrize("lspec", LSPECS, ids=[l[0] for l in LSPECS])
def test_target_and_dtarget_match_oracle(lspec, kname):
    import gpb200
    n = 300
    X, ys, rng = _data(n, 3, 17)
    y = ys[lspec[0]]
    kmake, spec = _kernels()[kname]
    gp = gpb200.GP(X.T, y, gpb200.MeanConst(0.1), kmake(), _lik(lspec))
    assert isinstance(gp, gpb200.GPA)
    p = gp.get_params()
    p[:n] = 0.5 * rng.standard_normal(n)
    gp.set_params(p)
    gp.update_target_and_dtarget()
    ls = lspec[:-1] + (gp.lik.get_params()[0],) if gp.lik.num_params() else lspec
    t = go.gpa_target(spec, X, y, gp.v, ls, ("MeanConst", 0.1))
    dt = go.gpa_dtarget(spec, X, y, gp.v, ls, ("MeanConst", 0.1))
    assert abs(gp.target - t) <= 1e-10 * abs(t)
    np.testing.assert_allclose(gp.dtarget, dt, rtol=1e-8, atol=1e-10 * np.max(np.abs(dt)))
    if kname == "SEIso" and lspec[0] == "Bern":
        # predict_f = predictMVN with alpha = cK \ (L v) (GPA.jl:294), on the factor the gradient left intact
        Xs = rng.standard_normal((9, 3))
        L = go.chol_factor(spec, X)
        mo, vo = orc.predict_f(spec, X, dict(U=L.T, alpha=sl.cho_solve((L, True), L @ gp.v)), Xs, ("MeanConst", 0.1))
        mu, s2 = gp.predict_f(Xs.T)
        assert np.max(np.abs(mu - mo)) <= 1e-9 * np.max(np.abs(mo))
        assert np.max(np.abs(s2 - vo)) <= 1e-9 * np.max(np.abs(vo)) + 1e-13


def test_chol_bar_matches_literal_reverse_mode():
    import gpb200
    n = 300
    X, _, rng = _data(n, 3, 5)
    kmake, spec = _kernels()["Mat32+RQ"]
    eng = gpb200.Engine(0)
    eng.set_data(X)
    ops, dims, theta, _ = gpb200.flatten(kmake(), 3)
    eng.set_kernel(ops, dims, theta.size)
    eng.factorize(theta, -20.0)
    v, g = rng.standard_normal(n), rng.standard_normal(n)
    dv, dk = eng.gpa_grad(v, g)
    L = go.chol_factor(spec, X)
    lit, L_bar = go.dll_kern_literal(spec, X, L, v, g)
    lo = np.tril(L_bar, -1)
    S_lit = lo + lo.T + np.diag(np.diag(L_bar))
    S = eng.chol_bar()
    assert np.max(np.abs(S - S_lit)) <= 1e-9 * np.max(np.abs(S_lit))
    np.testing.assert_allclose(dk, lit, rtol=1e-8, atol=1e-10 * np.max(np.abs(lit)))
    assert np.max(np.abs(dv - L.T @ g)) <= 1e-12 * np.max(np.abs(L.T @ g))
    eng.close()


def _directional_fd(gp, direction, h):
    p0 = gp.get_params()
    vals = []
    for s in (1, -1):
        gp.set_params(p0 + s * h * direction)
        gp.update_target()
        vals.append(gp.target)
    gp.set_params(p0)
    return (vals[0] - vals[1]) / (2 * h)


def test_device_target_finite_differences_n2000():
    import gpb200
    n = 2000
    X, ys, rng = _data(n, 3, 23)
    gp = gpb200.GPA(X.T, ys["Pois"], gpb200.MeanZero(), gpb200.Mat32Iso(math.log(0.5), 0.0) + gpb200.Noise(-1.0), gpb200.PoisLik())
    p = gp.get_params()
    p[:n] = 0.3 * rng.standard_normal(n)
    gp.set_params(p)
    gp.update_target_and_dtarget()
    g = gp.dtarget.copy()
    for which in (slice(0, n), slice(n, None)):                   # latent block, then kernel block
        d = np.zeros(p.size)
        d[which] = rng.standard_normal(d[which].size)
        num = _directional_fd(gp, d, 1e-5)
        assert num == pytest.approx(g @ d, rel=1e-5), which


def test_gram_fast_paths_agree():
    import gpb200
    n = 500
    X, ys, rng = _data(n, 3, 29)
    out = []
    for fast in (0, 1):
        eng = gpb200.Engine(0)
        eng.set_option("gram_fast", fast)
        gp = gpb200.GPA(X.T, ys["Bern"], gpb200.MeanZero(), gpb200.SEIso(math.log(0.4), 0.1), gpb200.BernLik(), engine=eng)
        gp.set_params(np.concatenate([0.5 * np.random.default_rng(1).standard_normal(n), gp.get_params()[n:]]))
        gp.update_target_and_dtarget()
        out.append((gp.target, gp.dtarget.copy()))
        eng.close()
    assert out[0][0] == pytest.approx(out[1][0], rel=1e-10)
    np.testing.assert_allclose(out[0][1], out[1][1], rtol=1e-8, atol=1e-10 * np.max(np.abs(out[0][1])))


def test_gpa_grad_leaves_the_factor_and_invalidates_the_inverse():
    import gpb200
    n = 600
    X, _, rng = _data(n, 3, 31)
    y = np.sin(X.sum(axis=1))
    Xs = rng.standard_normal((11, 3))
    ops, dims, theta, _ = gpb200.flatten(gpb200.SEIso(0.1, 0.2), 3)

    def fresh():
        e = gpb200.Engine(0)
        e.set_data(X)
        e.set_kernel(ops, dims, theta.size)
        e.factorize(theta, -1.0)
        return e

    ref = fresh()
    alpha_ref, mll_ref = ref.mll(y)
    ref.grad_prepare()
    gk_ref, tr_ref = ref.grad_kernel()
    mu_ref, var_ref, _ = ref.predict(Xs)

    eng = fresh()
    eng.mll(y)
    eng.grad_prepare()
    eng.gpa_grad(rng.standard_normal(n), rng.standard_normal(n))
    for call in (lambda: eng.grad_kernel(alpha_ref), eng.inverse, eng.inverse_diag, lambda: eng.cv_param(0, alpha_ref)):
        with pytest.raises(ValueError, match="grad_prepare first"):
            call()
    with pytest.raises(ValueError):                                # the resident alpha is gone too
        eng.predict(Xs)
    mu, var, _ = eng.predict(Xs, alpha_ref)                       # the factor is intact
    np.testing.assert_array_equal(mu, mu_ref)
    np.testing.assert_array_equal(var, var_ref)
    np.testing.assert_array_equal(eng.solve(y), ref.solve(y))
    alpha, mll = eng.mll(y)
    eng.grad_prepare()
    gk, tr = eng.grad_kernel()
    assert mll == mll_ref and tr == tr_ref
    np.testing.assert_array_equal(alpha, alpha_ref)
    np.testing.assert_array_equal(gk, gk_ref)
    eng.close(); ref.close()


def test_multi_rank_handle_is_rejected():
    import gpb200
    X, ys, _ = _data(300, 3, 37)
    grp = gpb200.LocalGroupEngine(2, rb=1)
    with pytest.raises(ValueError, match="single-GPU"):
        gpb200.GPA(X.T, ys["Bern"], gpb200.MeanZero(), gpb200.SEIso(0.0, 0.0), gpb200.BernLik(), engine=grp)
    with pytest.raises(ValueError, match="single-GPU"):
        grp.gpa_grad(np.zeros(300), np.zeros(300))
    grp.close()


def test_full_size_bernoulli_n32768():
    """N = 32768, d = 8: the adjoint identity v'(L'g) = (Lv)'g and a directional finite difference of the kernel gradient"""
    import gpb200
    n, d = 32768, 8
    rng = np.random.default_rng(41)
    X = rng.standard_normal((n, d))
    y = rng.random(n) < expit(np.sin(X).sum(axis=1))
    gp = gpb200.GPA(X.T, y, gpb200.MeanZero(), gpb200.SEIso(0.0, 0.0) + gpb200.Noise(-2.0), gpb200.BernLik())
    p = gp.get_params()
    p[:n] = 0.5 * rng.standard_normal(n)
    gp.set_params(p)
    gp.update_target_and_dtarget()
    dl_df = gp.lik.dlog_dens_df(gp._eng.unwhiten(gp.v), gp.y)
    Lv = gp._eng.unwhiten(gp.v)
    Ltg, _ = gp._eng.gpa_grad(gp.v, dl_df)
    assert gp.v @ Ltg == pytest.approx(Lv @ dl_df, rel=1e-12)
    dirn = np.zeros(p.size)
    dirn[n:] = rng.standard_normal(p.size - n)
    num = _directional_fd(gp, dirn, 1e-4)
    assert num == pytest.approx(gp.dtarget @ dirn, rel=1e-5)
