"""Randomised (fixed seeds) comparison of the product's host logic with the unmodified reference on small problems
that mix the corner cases of the CCSA loop: fixed variables (lb == ub), infinite bounds, infeasible starts (capped
multipliers), vector constraints, maximisation, non-default parameters.  Short runs (<= 18 evaluations) so that the
rounding-level differences between the two summation orders (DESIGN.md section 4) cannot be amplified yet:
same return code, same evaluation count, f to 1e-6 relative and x to 1e-5 (measured differences are <= 1e-7: the
dual problem is solved to ftol_rel = 1e-14, but its flat maximum turns last-bit differences of the sums into
~1e-8 differences of y and x, SURVEY.md 8(c))."""
import numpy as np
import pytest

import nlopt_b200 as nl


def make_problem(seed):
    rng = np.random.default_rng(seed)
    n = int(rng.integers(2, 24))
    m_scalar = int(rng.integers(0, 4))
    vec_dim = int(rng.integers(0, 3))                    # one vector constraint of this dimension (0: none)
    A = rng.normal(size=(n, n)) / np.sqrt(n)
    Q = A @ A.T + 0.2 * np.eye(n)                        # convex quadratic objective
    b = rng.normal(size=n)
    W = rng.normal(size=(m_scalar + vec_dim, n))
    off = rng.normal(size=m_scalar + vec_dim) * 0.3 + (0.4 if rng.random() < 0.5 else -0.4)   # some start infeasible
    curv = rng.random(m_scalar + vec_dim) * 0.5
    lb = -1.0 - rng.random(n)
    ub = 1.0 + rng.random(n)
    for j in rng.choice(n, size=max(1, n // 6), replace=False):
        k = rng.integers(0, 4)
        if k == 0:
            lb[j] = ub[j] = 0.25                           # fixed variable: sigma = 0
        elif k == 1:
            lb[j] = -np.inf
        elif k == 2:
            ub[j] = np.inf
        else:
            lb[j], ub[j] = -np.inf, np.inf
    x0 = np.clip(rng.normal(size=n) * 0.5, np.where(np.isinf(lb), -3, lb), np.where(np.isinf(ub), 3, ub))

    def f(x, grad):
        if grad.size:
            grad[:] = Q @ x + b
        return float(0.5 * x @ Q @ x + b @ x)

    def con(i):
        def c(x, grad):
            if grad.size:
                grad[:] = W[i] + 2 * curv[i] * x
            return float(W[i] @ x + curv[i] * (x @ x) - off[i] - 1.0)
        return c

    def vcon(result, x, grad):
        for k in range(vec_dim):
            i = m_scalar + k
            result[k] = W[i] @ x + curv[i] * (x @ x) - off[i] - 1.0
            if grad.size:
                grad[k, :] = W[i] + 2 * curv[i] * x

    opts = {}
    r = rng.random()
    if r < 0.15:
        opts["inner_maxeval"] = 2
    elif r < 0.3:
        opts["always_improve"] = 0
    elif r < 0.45:
        opts["inner_gradients"] = 0
    elif r < 0.6:
        opts["rho_init"] = 5.0
    elif r < 0.7:
        opts["sigma_min"] = 0.05
    return dict(n=n, f=f, cons=[con(i) for i in range(m_scalar)], vec=(vcon, vec_dim) if vec_dim else None, lb=lb, ub=ub,
                x0=x0, opts=opts, maximize=bool(rng.random() < 0.15), alg=nl.LD_MMA if rng.random() < 0.5 else nl.LD_CCSAQ,
                maxeval=int(rng.integers(6, 19)))


def run(lib, p):
    o = nl.opt(p["alg"], p["n"], library=lib)
    o.set_lower_bounds(p["lb"]); o.set_upper_bounds(p["ub"])
    if p["maximize"]:
        o.set_max_objective(lambda x, g: -p["f"](x, g) if g.size == 0 else _neg(p["f"], x, g))
    else:
        o.set_min_objective(p["f"])
    for c in p["cons"]:
        o.add_inequality_constraint(c, 1e-8)
    if p["vec"]:
        o.add_inequality_mconstraint(p["vec"][0], [1e-8] * p["vec"][1])
    for k, v in p["opts"].items():
        o.set_param(k, v)
    o.set_maxeval(p["maxeval"])
    x = o.optimize(p["x0"].copy())
    return o.last_optimize_result(), o.get_numevals(), o.last_optimum_value(), x


def _neg(f, x, g):
    v = f(x, g)
    g[:] = -g
    return -v


@pytest.mark.parametrize("seed", range(48))
def test_random_small_problems_match_reference(hosttest_lib, reference, seed):
    p = make_problem(1000 + seed)
    b = reference(f"host_fuzz/small/{1000 + seed}", lambda lib: run(lib, p))
    a = run(hosttest_lib, p)
    assert a[0] == b[0] and a[1] == b[1], (a[:3], b[:3])
    assert abs(a[2] - b[2]) <= 1e-6 * max(1.0, abs(b[2])), (a[2], b[2])
    assert np.max(np.abs(a[3] - b[3])) <= 1e-5


@pytest.mark.parametrize("seed", range(16))
@pytest.mark.parametrize("stop", ["xtol_rel", "ftol_rel", "xtol_abs"])
def test_random_small_problems_converge_to_the_reference_optimum(hosttest_lib, reference, seed, stop):
    """The same generator run to convergence under each stopping rule (stop.c:81-108): the result class must be a
    success in both libraries and the optimum must agree (which rule fires first may legitimately differ at ties)."""
    p = make_problem(5000 + seed)

    def solve(lib):
        o = nl.opt(p["alg"], p["n"], library=lib)
        o.set_lower_bounds(p["lb"]); o.set_upper_bounds(p["ub"])
        o.set_min_objective(p["f"])
        for c in p["cons"]:
            o.add_inequality_constraint(c, 1e-8)
        if p["vec"]:
            o.add_inequality_mconstraint(p["vec"][0], [1e-8] * p["vec"][1])
        if stop == "xtol_rel":
            o.set_xtol_rel(1e-9)
        elif stop == "ftol_rel":
            o.set_ftol_rel(1e-12)
        else:
            o.set_xtol_abs(np.full(p["n"], 1e-9))
        o.set_maxeval(4000)
        o.optimize(p["x0"].copy())
        return o.last_optimize_result(), o.last_optimum_value()
    rb, fb = reference(f"host_fuzz/converge/{5000 + seed}/{stop}", solve)
    ra, fa = solve(hosttest_lib)
    assert ra > 0 and rb > 0
    if ra != nl.MAXEVAL_REACHED and rb != nl.MAXEVAL_REACHED:
        assert abs(fa - fb) <= 1e-5 * max(1.0, abs(fb)), (ra, rb, fa, fb)       # slow CCSAQ tails stop a few 1e-6 apart


@pytest.mark.parametrize("alg", [nl.LD_MMA, nl.LD_CCSAQ])
@pytest.mark.parametrize("poison", ["nan_objective_once", "inf_objective_region", "nan_constraint_late"])
def test_non_finite_callback_values_are_handled_like_the_reference(hosttest_lib, reference, alg, poison):
    """Comparisons against NaN / inf decide acceptance and conservativeness (mma.c:302-392); whatever the reference
    does with a non-finite callback value, the host logic must do the same (same code, evaluations and point)."""
    n = 6
    lb, ub, x0 = np.full(n, -2.0), np.full(n, 2.0), np.full(n, 0.7)

    def solve(lib):
        calls = [0]

        def f(x, grad, calls=calls):
            calls[0] += 1
            if grad.size:
                grad[:] = 2 * (x - 0.3)
            v = float(np.sum((x - 0.3) ** 2))
            if poison == "nan_objective_once" and calls[0] == 4:
                return float("nan")
            if poison == "inf_objective_region" and x[0] < 0.45:
                return float("inf")
            return v

        ccalls = [0]

        def c(x, grad, ccalls=ccalls):
            ccalls[0] += 1
            if grad.size:
                grad[:] = 1.0
            if poison == "nan_constraint_late" and ccalls[0] >= 5:
                return float("nan")
            return float(np.sum(x) - 2.5)

        o = nl.opt(alg, n, library=lib)
        o.set_lower_bounds(lb); o.set_upper_bounds(ub)
        o.set_min_objective(f)
        o.add_inequality_constraint(c, 1e-8)
        o.set_xtol_rel(1e-6); o.set_maxeval(60)
        try:
            x = o.optimize(x0.copy())
        except Exception:
            x = np.full(n, np.nan)
        return o.last_optimize_result(), o.get_numevals(), o.last_optimum_value(), x
    b = reference(f"host_fuzz/non_finite/{alg}/{poison}", solve)
    a = solve(hosttest_lib)
    assert a[0] == b[0] and abs(a[1] - b[1]) <= 1, (a[:3], b[:3])      # the xtol test at f* = 0 may fire one iteration apart
    assert (np.isnan(a[2]) and np.isnan(b[2])) or a[2] == b[2] or abs(a[2] - b[2]) <= 1e-7 * max(1.0, abs(b[2]))
    assert np.allclose(a[3], b[3], atol=1e-6, equal_nan=True)


@pytest.mark.gpu
@pytest.mark.parametrize("seed", range(48))
def test_random_small_problems_on_gpu_match_reference(built, reference, seed):
    """The fixed-seed generator above through the product library (CUDA path)."""
    p = make_problem(1000 + seed)
    b = reference(f"host_fuzz/small/{1000 + seed}", lambda lib: run(lib, p))
    a = run(None, p)
    assert a[0] == b[0] and a[1] == b[1], (a[:3], b[:3])
    assert abs(a[2] - b[2]) <= 1e-6 * max(1.0, abs(b[2])), (a[2], b[2])
    assert np.max(np.abs(a[3] - b[3])) <= 1e-5
