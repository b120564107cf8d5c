"""The oracle's generic L-BFGS-B against the installed SciPy on problems that are NOT the
planner's (mixed bound types, consistent gradients, ring wrap, maxiter/maxfun stops), so the
restatement is pinned beyond the regimes the reference gradient reaches (SURVEY App. B)."""
import numpy as np
import pytest

scipy_optimize = pytest.importorskip("scipy.optimize")


def _run_both(oracle_mod, fg, x0, lo, hi, nbd, **opt):
    m = opt.get("m", 10)
    ftol = opt.get("ftol", 2.2e-9)
    gtol = opt.get("gtol", 1e-5)
    maxiter = opt.get("maxiter", 200)
    maxfun = opt.get("maxfun", 15000)
    maxls = opt.get("maxls", 20)
    bounds = []
    for l, h, b in zip(lo, hi, nbd):
        bounds.append((l if b in (1, 2) else None, h if b in (2, 3) else None))
    res = scipy_optimize.minimize(lambda x: fg(x), x0, jac=True, method="L-BFGS-B", bounds=bounds,
                                  options=dict(maxcor=m, ftol=ftol, gtol=gtol, maxiter=maxiter,
                                               maxfun=maxfun, maxls=maxls))
    eps = np.finfo(float).eps
    x, st = oracle_mod.lbfgsb(fg, x0, lo, hi, nbd, m=m, factr=ftol / eps, pgtol=gtol,
                              maxiter=maxiter, maxfun=maxfun, maxls=maxls)
    return res, x, st


@pytest.mark.parametrize("seed", range(12))
def test_bounded_quadratic(oracle_mod, seed):
    rng = np.random.default_rng(seed)
    n = int(rng.integers(5, 40))
    A = rng.normal(size=(n, n))
    H = A @ A.T / n + np.diag(rng.uniform(0.1, 2.0, n))
    c = rng.normal(size=n) * 3

    def fg(x):
        return 0.5 * x @ H @ x - c @ x, H @ x - c

    lo = rng.uniform(-2, -0.1, n)
    hi = rng.uniform(0.1, 2, n)
    nbd = rng.integers(0, 4, n).astype(np.int32)
    x0 = rng.uniform(-3, 3, n)
    res, x, st = _run_both(oracle_mod, fg, x0, lo, hi, nbd, m=int(rng.integers(3, 11)))
    assert (st.nit, st.nfev, st.status) == (res.nit, res.nfev, res.status)
    np.testing.assert_allclose(x, res.x, atol=1e-9)
    assert st.f == pytest.approx(res.fun, rel=1e-10, abs=1e-10)


def _rosenbrock(x):
    f = np.sum(100 * (x[1:] - x[:-1] ** 2) ** 2 + (1 - x[:-1]) ** 2)
    g = np.zeros_like(x)
    g[:-1] = -400 * x[:-1] * (x[1:] - x[:-1] ** 2) - 2 * (1 - x[:-1])
    g[1:] += 200 * (x[1:] - x[:-1] ** 2)
    return f, g


def _rosenbrock_problem(n):
    x0 = np.full(n, -1.2)
    x0[1::2] = 1.0
    lo = np.full(n, -1.5)
    hi = np.full(n, 0.8)          # the optimum (1,..,1) is outside: bounds active
    return x0, lo, hi, np.full(n, 2, np.int32)


@pytest.mark.parametrize("n,m", [(10, 5), (30, 4), (20, 10)])
def test_rosenbrock_ring_wrap(oracle_mod, n, m):
    x0, lo, hi, nbd = _rosenbrock_problem(n)
    res, x, st = _run_both(oracle_mod, _rosenbrock, x0, lo, hi, nbd, m=m, maxiter=400)
    assert res.nit > 2 * m        # the correction ring wrapped
    assert (st.nit, st.nfev, st.status) == (res.nit, res.nfev, res.status)
    np.testing.assert_allclose(x, res.x, atol=1e-8)


def test_stops(oracle_mod):
    def fg(x):
        return float(np.sum(x ** 4 + x ** 2 - 3 * x)), 4 * x ** 3 + 2 * x - 3

    n = 12
    x0 = np.linspace(-2, 2, n)
    lo, hi, nbd = np.full(n, -5.0), np.full(n, 5.0), np.full(n, 2, np.int32)
    res, x, st = _run_both(oracle_mod, fg, x0, lo, hi, nbd, maxiter=3)
    assert res.status == 1 and (st.nit, st.nfev, st.status) == (res.nit, res.nfev, res.status)
    np.testing.assert_allclose(x, res.x, atol=1e-12)
    res, x, st = _run_both(oracle_mod, fg, x0, lo, hi, nbd, maxfun=4)
    assert (st.nit, st.nfev, st.status) == (res.nit, res.nfev, res.status)
    np.testing.assert_allclose(x, res.x, atol=1e-12)


# The solver options away from their defaults: one or two correction pairs (the ring wraps at every
# or every other pair), line searches of one to three trial points, few evaluations, no iteration.
OPTION_CASES = [dict(m=m, maxls=ls) for m in (1, 2) for ls in (1, 2, 3, 20)] + \
    [dict(m=m, maxls=2, maxfun=f) for m in (1, 2) for f in (3, 5, 8)] + \
    [dict(m=1, maxiter=0), dict(m=10, maxiter=0), dict(m=1, maxls=1, maxiter=0)]


def _option_id(o):
    return "-".join(f"{k}{v}" for k, v in o.items())


@pytest.mark.parametrize("opt", OPTION_CASES, ids=[_option_id(o) for o in OPTION_CASES])
@pytest.mark.parametrize("seed", range(3))
def test_bounded_quadratic_options(oracle_mod, seed, opt):
    rng = np.random.default_rng(100 + seed)
    n = int(rng.integers(8, 30))
    A = rng.normal(size=(n, n))
    H = A @ A.T / n + np.diag(rng.uniform(0.01, 2.0, n))
    c = rng.normal(size=n) * 3

    def fg(x):
        return 0.5 * x @ H @ x - c @ x, H @ x - c

    lo, hi = rng.uniform(-2, -0.1, n), rng.uniform(0.1, 2, n)
    nbd = rng.integers(0, 4, n).astype(np.int32)
    x0 = rng.uniform(-3, 3, n)
    res, x, st = _run_both(oracle_mod, fg, x0, lo, hi, nbd, **opt)
    assert (st.nit, st.nfev, st.status) == (res.nit, res.nfev, res.status)
    np.testing.assert_allclose(x, res.x, atol=1e-9)
    if opt.get("maxiter") == 0:
        assert res.status == 1 and res.nit == 1


@pytest.mark.parametrize("opt", OPTION_CASES, ids=[_option_id(o) for o in OPTION_CASES])
def test_rosenbrock_options(oracle_mod, opt):
    x0, lo, hi, nbd = _rosenbrock_problem(12)
    res, x, st = _run_both(oracle_mod, _rosenbrock, x0, lo, hi, nbd, **dict(dict(maxiter=400), **opt))
    assert (st.nit, st.nfev, st.status) == (res.nit, res.nfev, res.status)
    np.testing.assert_allclose(x, res.x, atol=1e-8)
    if opt.get("maxls") == 1:
        assert "ABNORMAL" in res.message                           # the one-point line search failed
    elif "maxfun" in opt:
        assert res.status == 1 and res.nfev > opt["maxfun"]       # the evaluation budget stopped it
    elif opt.get("maxiter") == 0:
        assert res.status == 1 and res.nit == 1
    else:
        assert res.nit > 2 * opt["m"]                              # the ring wrapped
