"""The oracle is pinned here: the plain-C port (oracle/ccsa_port.c) against
 (a) the known-answer vectors measured from the reference build (SURVEY.md Appendix B), and
 (b) the unmodified reference itself, compiled into oracle/_ref -- bit for bit (its results are stored in
     tests/golden/reference_runs.npz, tests/reference_runs.py; arrays as a SHA-256 of their bits)."""
import hashlib
import os

import numpy as np
import pytest

import oracle_bindings as ob
import problems as P
import synth

KA = dict(n=5, m=2, x=np.array([0.1, -0.3, 0.5, 1.0, 0.0]), lb=np.array([-1, -1, -1, 1, -np.inf]),
          ub=np.array([1, 1, 1, 1, np.inf]), sigma=np.array([1, 0.5, 0.25, 0, 1.0]),
          grad_f=np.array([0.3, -1.2, 2.0, 5.0, -0.7]),
          grad_c=np.array([[1, 0.5, -0.25, 3, 0.2], [-0.4, 0.9, 1.5, -2, 0]]),
          c0=np.array([0.2, -0.1]), rhoc=np.array([1.0, 2.0]), y=np.array([0.7, 1.3]), f0=1.5, rho=0.8)

KA_EXPECT = {
    ob.MMA: dict(ret=-1.3904823680888407, g0=1.3812742479888385, w=0.020018262900815334,
                 gc=[0.18433922561058258, -0.092176413713388472],
                 xcur=[0.03246650263757983, -0.31173666859306337, 0.46077130862355642, 1, 0.097812752129466884]),
    ob.CCSAQ: dict(ret=-1.3319190167682924, g0=1.3123389723378938, w=0.043434386154074967,
                   gc=[0.15830862395895301, -0.070181532569898869],
                   xcur=[-0.017073170731707318, -0.31951219512195123, 0.44245426829268292, 1, 0.13658536585365855]),
}


@pytest.mark.parametrize("variant", [ob.MMA, ob.CCSAQ])
def test_known_answer_dual(built, variant):
    r = ob.port_dual(variant, KA)
    e = KA_EXPECT[variant]
    assert r["ret"] == e["ret"] and r["g0"] == e["g0"] and r["w"] == e["w"]
    assert list(r["gc"]) == e["gc"]
    assert list(r["xcur"]) == e["xcur"]
    assert list(r["grad"]) == [-v for v in e["gc"]]


def _sha256(x):
    """digest of an array's bits; every NaN counts as the same NaN and -0.0 as 0.0, as np.array_equal(equal_nan=True) does"""
    x = np.asarray(x, dtype=np.float64)
    return hashlib.sha256(np.where(np.isnan(x), np.nan, x + 0.0).tobytes()).hexdigest()


def _digest(r):
    return dict(ret=r["ret"], g0=r["g0"], w=r["w"], gc=r["gc"], xcur_sha256=_sha256(r["xcur"]))


def _same(a, b):
    for k in ("ret", "g0", "w"):
        assert a[k] == b[k] or (np.isnan(a[k]) and np.isnan(b[k])), k
    assert np.array_equal(a["gc"], b["gc"], equal_nan=True)
    assert a["xcur_sha256"] == b["xcur_sha256"]


@pytest.mark.parametrize("n,m", [(1, 0), (2, 2), (7, 1), (1000, 1), (4097, 3), (100000, 4), (20000, 16)])
@pytest.mark.parametrize("variant", [ob.MMA, ob.CCSAQ])
def test_port_dual_bitwise_vs_reference(built, reference, variant, n, m):
    inst = synth.kernel_instance(n, m)
    rng = np.random.default_rng(n + 31 * m)
    # the instance's own multipliers, then others, including zeros and huge ones
    ys = [None] + [rng.choice([0.0, 1e-3, 1.0, 50.0, 1e40], size=m) * rng.random(m) for _ in range(3)]
    for i, y in enumerate(ys):
        want = reference(f"oracle_port/dual/{variant}/n={n}/m={m}/y{i}", lambda lib: _digest(ob.ref_dual(variant, inst, y)))
        _same(_digest(ob.port_dual(variant, inst, y)), want)


def test_port_dual_nan_constraint_switches_off_mma(built, reference):
    """mma.c:78,103,126: a NaN constraint value removes that constraint from the MMA dual."""
    inst = synth.kernel_instance(5000, 3)
    inst["c0"] = np.array([-0.1, np.nan, 0.2])
    a = ob.port_dual(ob.MMA, inst)
    _same(_digest(a), reference("oracle_port/dual_nan_constraint", lambda lib: _digest(ob.ref_dual(ob.MMA, inst))))
    drop = dict(inst, m=2, grad_c=inst["grad_c"][[0, 2]], c0=inst["c0"][[0, 2]], rhoc=inst["rhoc"][[0, 2]],
                y=inst["y"][[0, 2]])
    b = ob.port_dual(ob.MMA, drop)
    assert np.array_equal(a["xcur"], b["xcur"]) and a["ret"] == b["ret"]
    assert a["gc"][1] == 0.0


# ---- full solver: tutorial problem, every setting of SURVEY.md Appendix B -------------------------------
GOLD = [  # (variant, setting, ret, evals, x0, x1, f)
    (ob.MMA, "s1", 4, 11, 0.33333333482477717, 0.29629628914423661, 0.54433104738223104),
    (ob.CCSAQ, "s1", 4, 22, 0.33333333559482431, 0.29629629249427253, 0.54433105045943553),
    (ob.MMA, "s2", 2, 10, 0.33333339461697409, 0.29632159814805525, 0.5443542946905584),
    (ob.CCSAQ, "s2", 2, 20, 0.33332808736843805, 0.29631100381513564, 0.54434456350287508),
    (ob.MMA, "s3", 4, 11, 0.33333333459224374, 0.29629628904448441, 0.54433104729060278),
    (ob.CCSAQ, "s3", 4, 22, 0.33333333565210099, 0.29629629282503789, 0.54433105076326294),
    (ob.MMA, "s4", 4, 24, 0.33333333337243021, 0.29629629165122456, 0.54433104968504653),
    (ob.CCSAQ, "s4", 4, 56, 0.33333334245161117, 0.29629627976215528, 0.54433103876423883),
    (ob.MMA, "s5", 2, 23, 0.33333333617988786, 0.29629710643768237, 0.54433179811368948),
    (ob.CCSAQ, "s5", 2, 51, 0.33305261429836952, 0.29682398256407033, 0.54481554912104913),
]
SETTINGS = {
    "s1": dict(lb=[-np.inf, 0.0], ub=[np.inf, np.inf], xtol_rel=1e-4),
    "s2": dict(lb=[-np.inf, 0.0], ub=[np.inf, np.inf], stopval=P.TUT_FSTAR + 1e-3),
    "s3": dict(lb=[-np.inf, 1e-6], ub=[np.inf, np.inf], xtol_rel=1e-4),
    "s4": dict(lb=[-np.inf, 1e-6], ub=[np.inf, np.inf], xtol_rel=1e-4, inner_maxeval=123, rho_init=0.5,
               sigma_init=[0.1, 0.1]),
    "s5": dict(lb=[1e-6, 1e-6], ub=[10.0, 10.0], stopval=P.TUT_FSTAR + 1e-3, inner_maxeval=123, rho_init=0.5,
               sigma_init=[0.1, 0.1]),
}


@pytest.mark.parametrize("variant,setting,ret,evals,x0,x1,f", GOLD)
def test_port_solver_matches_reference_goldens(built, variant, setting, ret, evals, x0, x1, f):
    s = dict(SETTINGS[setting])
    lb, ub = s.pop("lb"), s.pop("ub")
    r = ob.port_minimize(variant, P.tut_f, [P.tut_c(2, 0), P.tut_c(-1, 1)], [1e-8, 1e-8], lb, ub, P.TUT_X0, **s)
    assert (r["ret"], r["numevals"]) == (ret, evals)
    assert r["x"][0] == x0 and r["x"][1] == x1 and r["minf"] == f      # bit-identical to the reference build


def test_port_dual_eval_counts_match_reference_verbosity(built):
    """SURVEY.md Appendix B: dual evaluations per inner iteration printed by verbosity=1."""
    s = dict(SETTINGS["s1"]); lb, ub = s.pop("lb"), s.pop("ub")
    r = ob.port_minimize(ob.MMA, P.tut_f, [P.tut_c(2, 0), P.tut_c(-1, 1)], [1e-8, 1e-8], lb, ub, P.TUT_X0, **s)
    assert r["dual_count_log"][:10] == [136, 18, 32, 39, 22, 26, 37, 40, 52, 32]
    r = ob.port_minimize(ob.CCSAQ, P.tut_f, [P.tut_c(2, 0), P.tut_c(-1, 1)], [1e-8, 1e-8], lb, ub, P.TUT_X0, **s)
    assert r["dual_count_log"][:12] == [101, 95, 19, 18, 15, 19, 16, 17, 17, 2374, 39, 42]


def _run_lib(lib, alg, n, f, cons, tols, lb, ub, x0, **kw):
    import nlopt_b200 as nl
    o = nl.opt(alg, n, library=lib)
    o.set_lower_bounds(lb); o.set_upper_bounds(ub)
    o.set_min_objective(f)
    for c, t in zip(cons, tols):
        o.add_inequality_constraint(c, t)
    for k, v in kw.items():
        if k in ("xtol_rel", "ftol_rel", "maxeval", "stopval"):
            getattr(o, "set_" + k)(v)
        else:
            o.set_param(k, v)
    x = o.optimize(x0)
    return dict(ret=o.last_optimize_result(), x_sha256=_sha256(x), minf=o.last_optimum_value(), numevals=o.get_numevals())


@pytest.mark.parametrize("variant", [ob.MMA, ob.CCSAQ])
def test_port_solver_bitwise_vs_reference_rosenbrock(built, reference, variant):
    """chained Rosenbrock + 4 dense linear constraints (the BASELINE config-3 instance, small n)."""
    import nlopt_b200 as nl
    n, m = 500, 4
    cons = [P.lin_constraint(k, n) for k in range(m)]
    lb, ub = np.full(n, -2.0), np.full(n, 2.0)
    alg = nl.LD_MMA if variant == ob.MMA else nl.LD_CCSAQ
    b = reference(f"oracle_port/solver_rosenbrock/{variant}",
                  lambda lib: _run_lib(lib, alg, n, P.rosen_f, cons, [1e-8] * m, lb, ub, P.rosen_x0(n), maxeval=25))
    a = ob.port_minimize(variant, P.rosen_f, cons, [1e-8] * m, lb, ub, P.rosen_x0(n), maxeval=25)
    assert a["ret"] == b["ret"] and a["numevals"] == b["numevals"]
    assert a["minf"] == b["minf"] and _sha256(a["x"]) == b["x_sha256"]


@pytest.mark.parametrize("variant", [ob.MMA, ob.CCSAQ])
@pytest.mark.parametrize("x0v", [-0.5, 0.5])
def test_port_solver_bitwise_vs_reference_quadratic(built, reference, variant, x0v):
    """separable quadratic + mean constraint (config-2 shape); x0=+0.5 starts infeasible (dual_ub = 1e40 path)."""
    import nlopt_b200 as nl
    n = 2000
    f, c = P.quad_problem(n)
    lb, ub = np.full(n, -1.0), np.full(n, 1.0)
    alg = nl.LD_MMA if variant == ob.MMA else nl.LD_CCSAQ
    b = reference(f"oracle_port/solver_quadratic/{variant}/x0={x0v}",
                  lambda lib: _run_lib(lib, alg, n, f, [c], [0.0], lb, ub, np.full(n, x0v), xtol_rel=1e-6, maxeval=200))
    a = ob.port_minimize(variant, f, [c], [0.0], lb, ub, np.full(n, x0v), xtol_rel=1e-6, maxeval=200)
    assert a["ret"] == b["ret"] and a["numevals"] == b["numevals"]
    assert a["minf"] == b["minf"] and _sha256(a["x"]) == b["x_sha256"]


def test_port_sigma_and_stop_helpers(built):
    L = ob.port()
    n = 9
    lb = np.array([-1, -np.inf, 0, 0, 1, -2, -2, -2, 5.0]); ub = np.array([1, 1, np.inf, 0, 3, 2, 2, 2, 5.0])
    s = np.zeros(n)
    L.port_sigma_init(n, ob._p(lb), ob._p(ub), None, 0.0, ob._p(s))
    assert list(s) == [1.0, 1.0, 1.0, 0.0, 1.0, 2.0, 2.0, 2.0, 0.0]
    si = np.array([0.1, -1, 0, 0.2, 0.3, 0, 0, 0, 0.0])
    L.port_sigma_init(n, ob._p(lb), ob._p(ub), ob._p(si), 0.25, ob._p(s))
    assert list(s) == [0.25, 1.0, 1.0, 0.25, 0.3, 2.0, 2.0, 2.0, 0.25]
    assert L.port_relstop(1.0, 1.0, 1e-4, 0.0) == 1 and L.port_relstop(np.inf, 1.0, 1.0, 1.0) == 0
    assert L.port_relstop(0.0, 0.0, 0.0, 0.0) == 0
