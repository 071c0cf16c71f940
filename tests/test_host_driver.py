"""Host-side logic of the product (nlopt_api.cpp, ccsa_driver.cpp, dual_mma.hpp) on a machine without
a GPU: the same sources are linked against the oracle-backed CPU backend (tests/cpp/oracle_backend.cpp)
and driven through the C ABI.  The O(n) kernels are NOT exercised here -- test_gpu_parity.py does that.

Tolerance: the driver adds the O(m) constants after the n-term sums (like the GPU path), so results
differ from the reference by rounding that the flat dual optimum amplifies (SURVEY.md 8(c)):
|f - f_ref| <= 1e-6, |x - x_ref| <= 1e-5, evaluation counts within a few."""
import os
import subprocess

import numpy as np
import pytest

import nlopt_b200 as nl
import oracle_bindings as ob
import problems as P
import refsrc
from test_oracle_port import GOLD, SETTINGS

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run(lib, alg, n, f, cons, tols, lb, ub, x0, maximize=False, **kw):
    o = nl.opt(alg, n, library=lib)
    o.set_lower_bounds(lb); o.set_upper_bounds(ub)
    (o.set_max_objective if maximize else o.set_min_objective)(f)
    for c, t in zip(cons, tols):
        o.add_inequality_constraint(c, t)
    for k, v in kw.items():
        if k in ("xtol_rel", "ftol_rel", "ftol_abs", "maxeval", "stopval", "maxtime"):
            getattr(o, "set_" + k)(v)
        elif k == "initial_step":
            o.set_initial_step(v)
        elif k == "xtol_abs":
            o.set_xtol_abs(v)
        else:
            o.set_param(k, v)
    x = o.optimize(x0)
    return dict(ret=o.last_optimize_result(), x=x, minf=o.last_optimum_value(), numevals=o.get_numevals(), opt=o)


def plain(r, fields=("ret", "numevals", "minf", "x")):
    """the part of a run() result that is compared (and stored for the reference, tests/reference_runs.py)"""
    return {k: r[k] for k in fields}


def okey(opts):
    return ",".join(f"{k}={v}" for k, v in sorted(opts.items())) or "defaults"


@pytest.mark.parametrize("variant,setting,ret,evals,x0,x1,f", GOLD)
def test_tutorial_goldens(hosttest_lib, variant, setting, ret, evals, x0, x1, f):
    s = dict(SETTINGS[setting])
    lb, ub = s.pop("lb"), s.pop("ub")
    if "sigma_init" in s:
        s["initial_step"] = s.pop("sigma_init")
    alg = nl.LD_MMA if variant == ob.MMA else nl.LD_CCSAQ
    r = run(hosttest_lib, alg, 2, P.tut_f, [P.tut_c(2, 0), P.tut_c(-1, 1)], [1e-8, 1e-8], lb, ub, P.TUT_X0, **s)
    assert r["ret"] == ret
    assert abs(r["numevals"] - evals) <= 2
    assert abs(r["minf"] - f) <= 1e-6 and abs(r["x"][0] - x0) <= 1e-5 and abs(r["x"][1] - x1) <= 1e-5
    st_ok = hosttest_lib.nlopt_get_numevals(r["opt"]._h) == r["numevals"]
    assert st_ok


@pytest.mark.parametrize("alg", [nl.LD_MMA, nl.LD_CCSAQ])
def test_rosenbrock_vs_reference(hosttest_lib, reference, alg):
    n, m = 400, 4
    cons = [P.lin_constraint(k, n) for k in range(m)]
    lb, ub = np.full(n, -2.0), np.full(n, 2.0)
    b = reference(f"host_driver/rosenbrock/{alg}",
                  lambda lib: plain(run(lib, alg, n, P.rosen_f, cons, [1e-8] * m, lb, ub, P.rosen_x0(n), maxeval=25)))
    a = run(hosttest_lib, alg, n, P.rosen_f, cons, [1e-8] * m, lb, ub, P.rosen_x0(n), maxeval=25)
    assert a["ret"] == b["ret"] == nl.MAXEVAL_REACHED and a["numevals"] == b["numevals"] == 25
    assert abs(a["minf"] - b["minf"]) <= 1e-6 * abs(b["minf"])
    assert np.max(np.abs(a["x"] - b["x"])) <= 1e-5


@pytest.mark.parametrize("alg", [nl.LD_MMA, nl.LD_CCSAQ])
@pytest.mark.parametrize("opts", [dict(), dict(inner_gradients=0), dict(always_improve=0), dict(sigma_min=0.05),
                                  dict(inner_maxeval=2), dict(rho_init=10.0)])
def test_algorithm_parameters_vs_reference(hosttest_lib, reference, alg, opts):
    """Every MMA/CCSAQ parameter of optimize.c:798-803 against the reference: (a) the first 20
    evaluations must track the reference to rounding (same counts, f to 1e-8, x to 1e-7); (b) run to
    convergence the result class and optimum must agree (rounding differences are amplified by the
    flat dual optimum, so the paths -- and evaluation counts -- may legitimately differ late in the run)."""
    n = 300
    f, c = P.quad_problem(n)
    lb, ub = np.full(n, -1.0), np.full(n, 1.0)
    kw = dict(xtol_rel=1e-7, dual_ftol_rel=1e-8, **opts)
    key = f"host_driver/algorithm_parameters/{alg}/{okey(opts)}"
    b = reference(key + "/maxeval=20", lambda lib: plain(run(lib, alg, n, f, [c], [0.0], lb, ub, np.full(n, -0.5), maxeval=20, **kw)))
    a = run(hosttest_lib, alg, n, f, [c], [0.0], lb, ub, np.full(n, -0.5), maxeval=20, **kw)
    assert a["ret"] == b["ret"] and a["numevals"] == b["numevals"] == 20
    assert abs(a["minf"] - b["minf"]) <= 1e-8 * max(1.0, abs(b["minf"]))
    assert np.max(np.abs(a["x"] - b["x"])) <= 1e-7
    b = reference(key + "/maxeval=150", lambda lib: plain(run(lib, alg, n, f, [c], [0.0], lb, ub, np.full(n, -0.5), maxeval=150, **kw),
                                                          ("ret", "minf")))
    a = run(hosttest_lib, alg, n, f, [c], [0.0], lb, ub, np.full(n, -0.5), maxeval=150, **kw)
    assert a["ret"] == b["ret"]
    assert abs(a["minf"] - b["minf"]) <= 1e-5 * max(1.0, abs(b["minf"]))


@pytest.mark.parametrize("alg", [nl.LD_MMA, nl.LD_CCSAQ])
def test_default_dual_tolerance_agrees_loosely(hosttest_lib, reference, alg):
    n = 300
    f, c = P.quad_problem(n)
    lb, ub = np.full(n, -1.0), np.full(n, 1.0)
    b = reference(f"host_driver/default_dual_tolerance/{alg}",
                  lambda lib: plain(run(lib, alg, n, f, [c], [0.0], lb, ub, np.full(n, -0.5), xtol_rel=1e-7, maxeval=150)))
    a = run(hosttest_lib, alg, n, f, [c], [0.0], lb, ub, np.full(n, -0.5), xtol_rel=1e-7, maxeval=150)
    assert a["ret"] == b["ret"] == nl.XTOL_REACHED
    assert abs(a["minf"] - b["minf"]) <= 5e-6 * max(1.0, abs(b["minf"]))
    assert np.max(np.abs(a["x"] - b["x"])) <= 2e-4


def test_infeasible_start_uses_capped_multipliers(hosttest_lib, reference):
    """x0 violates the constraint: dual_ub = 1e40 until a feasible point is accepted (mma.c:245-246, :384-388)."""
    n = 300
    f, c = P.quad_problem(n)
    lb, ub = np.full(n, -1.0), np.full(n, 1.0)
    b = reference("host_driver/infeasible_start",
                  lambda lib: plain(run(lib, nl.LD_MMA, n, f, [c], [0.0], lb, ub, np.full(n, 0.5), xtol_rel=1e-7, maxeval=200),
                                    ("ret", "minf")))
    a = run(hosttest_lib, nl.LD_MMA, n, f, [c], [0.0], lb, ub, np.full(n, 0.5), xtol_rel=1e-7, maxeval=200)
    assert a["ret"] == b["ret"] == nl.XTOL_REACHED
    assert abs(a["minf"] - b["minf"]) <= 1e-6 * abs(b["minf"])


def test_unconstrained_m0(hosttest_lib, reference):
    """reference test/cpp_functor.cxx shape: LD_MMA, no constraints, no bounds (sigma0 = 1)."""
    A = np.array([[4.0, 1, 0], [1, 3, 1], [0, 1, 2]]); b = np.array([1.0, -2.0, 0.5])

    def f(x, g):
        if g.size:
            g[:] = A @ x - b
        return float(0.5 * x @ A @ x - b @ x)
    inf = np.full(3, np.inf)
    r = reference("host_driver/unconstrained_m0",
                  lambda lib: plain(run(lib, nl.LD_MMA, 3, f, [], [], -inf, inf, np.zeros(3), xtol_rel=1e-4, maxeval=1000)))
    a = run(hosttest_lib, nl.LD_MMA, 3, f, [], [], -inf, inf, np.zeros(3), xtol_rel=1e-4, maxeval=1000)
    assert a["ret"] == r["ret"] and a["numevals"] == r["numevals"]
    assert abs(a["minf"] - r["minf"]) <= 1e-12 and np.max(np.abs(a["x"] - r["x"])) <= 1e-10


def test_vector_constraint_equals_scalar_constraints(hosttest_lib):
    lb, ub = [-np.inf, 0.0], [np.inf, np.inf]
    a = run(hosttest_lib, nl.LD_MMA, 2, P.tut_f, [P.tut_c(2, 0), P.tut_c(-1, 1)], [1e-8, 1e-8], lb, ub, P.TUT_X0,
            xtol_rel=1e-4)
    o = nl.opt(nl.LD_MMA, 2, library=hosttest_lib)
    o.set_lower_bounds(lb); o.set_min_objective(P.tut_f); o.set_xtol_rel(1e-4)
    c0, c1 = P.tut_c(2, 0), P.tut_c(-1, 1)

    def both(result, x, grad):
        result[0] = c0(x, grad[0] if grad.size else grad)
        result[1] = c1(x, grad[1] if grad.size else grad)
    o.add_inequality_mconstraint(both, [1e-8, 1e-8])
    x = o.optimize(P.TUT_X0)
    assert o.last_optimize_result() == a["ret"] and o.get_numevals() == a["numevals"]
    assert np.array_equal(x, a["x"]) and o.last_optimum_value() == a["minf"]


def test_optimize_inplace_is_the_c_call_on_the_callers_buffer(hosttest_lib):
    """opt.optimize_inplace(x): nlopt_optimize(opt, x, &minf) on the caller's own array -- same run as opt.optimize(),
    the solution left in the array, nothing copied; anything but a contiguous float64 array of the right size is refused."""
    lb = [-np.inf, 0.0]
    a = run(hosttest_lib, nl.LD_CCSAQ, 2, P.tut_f, [P.tut_c(2, 0), P.tut_c(-1, 1)], [1e-8, 1e-8], lb, [np.inf, np.inf], P.TUT_X0,
            xtol_rel=1e-4)
    o = nl.opt(nl.LD_CCSAQ, 2, library=hosttest_lib)
    o.set_lower_bounds(lb); o.set_min_objective(P.tut_f); o.set_xtol_rel(1e-4)
    o.add_inequality_constraint(P.tut_c(2, 0), 1e-8); o.add_inequality_constraint(P.tut_c(-1, 1), 1e-8)
    x = np.array(P.TUT_X0, dtype=np.float64)
    ret = o.optimize_inplace(x)
    assert ret == a["ret"] == o.last_optimize_result() and o.get_numevals() == a["numevals"]
    assert np.array_equal(x, a["x"]) and o.last_optimum_value() == a["minf"]
    for bad in ([1.0, 2.0], np.zeros(3), np.zeros(2, dtype=np.float32), np.zeros(4)[::2]):
        with pytest.raises(ValueError):
            o.optimize_inplace(bad)


def test_maximize_flips_sign(hosttest_lib):
    lb, ub = [-np.inf, 0.0], [np.inf, np.inf]
    a = run(hosttest_lib, nl.LD_CCSAQ, 2, P.tut_f, [P.tut_c(2, 0), P.tut_c(-1, 1)], [1e-8, 1e-8], lb, ub, P.TUT_X0,
            xtol_rel=1e-4)

    def negf(x, g):
        v = P.tut_f(x, g)
        if g.size:
            g[:] = -g
        return -v
    b = run(hosttest_lib, nl.LD_CCSAQ, 2, negf, [P.tut_c(2, 0), P.tut_c(-1, 1)], [1e-8, 1e-8], lb, ub, P.TUT_X0,
            maximize=True, xtol_rel=1e-4)
    assert b["ret"] == a["ret"] and np.array_equal(a["x"], b["x"]) and b["minf"] == -a["minf"]


def test_stopping_and_forced_stop(hosttest_lib):
    lb, ub = [-np.inf, 0.0], [np.inf, np.inf]
    cons, tols = [P.tut_c(2, 0), P.tut_c(-1, 1)], [1e-8, 1e-8]
    r = run(hosttest_lib, nl.LD_MMA, 2, P.tut_f, cons, tols, lb, ub, P.TUT_X0, maxeval=5)
    assert r["ret"] == nl.MAXEVAL_REACHED and r["numevals"] == 5
    r = run(hosttest_lib, nl.LD_MMA, 2, P.tut_f, cons, tols, lb, ub, P.TUT_X0, ftol_rel=1e-3)
    assert r["ret"] == nl.FTOL_REACHED
    r = run(hosttest_lib, nl.LD_MMA, 2, P.tut_f, cons, tols, lb, ub, P.TUT_X0, xtol_abs=1e-3)
    assert r["ret"] == nl.XTOL_REACHED
    # an exception inside the objective becomes a forced stop and is re-raised (nlopt.hpp:149-166)
    calls = [0]

    def boom(x, g):
        calls[0] += 1
        if calls[0] == 3:
            raise KeyError("stop here")
        return P.tut_f(x, g)
    o = nl.opt(nl.LD_MMA, 2, library=hosttest_lib)
    o.set_lower_bounds(lb); o.set_min_objective(boom)
    for c in cons:
        o.add_inequality_constraint(c, 1e-8)
    with pytest.raises(KeyError):
        o.optimize(P.TUT_X0)
    assert o.last_optimize_result() == nl.FORCED_STOP


def test_nan_constraint_is_ignored_by_mma(hosttest_lib, reference):
    """mma.c:141-143 hidden feature: a constraint that returns NaN is inactive."""
    def nanc(x, g):
        if g.size:
            g[:] = 0.0
        return float("nan")
    lb, ub = [-np.inf, 0.0], [np.inf, np.inf]
    cons, tols = [P.tut_c(2, 0), nanc, P.tut_c(-1, 1)], [1e-8, 0.0, 1e-8]
    b = reference("host_driver/nan_constraint",
                  lambda lib: plain(run(lib, nl.LD_MMA, 2, P.tut_f, cons, tols, lb, ub, P.TUT_X0, xtol_rel=1e-4), ("ret", "minf")))
    a = run(hosttest_lib, nl.LD_MMA, 2, P.tut_f, cons, tols, lb, ub, P.TUT_X0, xtol_rel=1e-4)
    assert a["ret"] == b["ret"] and abs(a["minf"] - b["minf"]) <= 1e-6


def test_local_optimizer_supplies_dual_tolerances(hosttest_lib, reference):
    """optimize.c:817-826: ftol/maxeval of a local optimiser configure the dual solve (same outcome as
    the reference, including its premature stop with these loose settings)."""
    def solve(lib):
        o = nl.opt(nl.LD_MMA, 2, library=lib)
        lo = nl.opt(nl.LD_MMA, 2, library=lib)
        lo.set_ftol_rel(1e-6); lo.set_maxeval(50)
        o.set_local_optimizer(lo)
        o.set_lower_bounds([-np.inf, 1e-6]); o.set_min_objective(P.tut_f); o.set_xtol_rel(1e-4)
        o.add_inequality_constraint(P.tut_c(2, 0), 1e-8); o.add_inequality_constraint(P.tut_c(-1, 1), 1e-8)
        x = o.optimize(P.TUT_X0)
        return o.last_optimize_result(), o.get_numevals(), x, o.last_optimum_value()
    ref = reference("host_driver/local_optimizer_dual_tolerances", solve)
    out = [solve(hosttest_lib), ref]
    assert out[0][0] == out[1][0] and out[0][1] == out[1][1]
    assert np.allclose(out[0][2], out[1][2], atol=1e-9) and abs(out[0][3] - out[1][3]) <= 1e-9
    bad = nl.opt(nl.LD_SLSQP, 2, library=hosttest_lib)
    o2 = nl.opt(nl.LD_MMA, 2, library=hosttest_lib)
    o2.set_local_optimizer(bad)
    o2.set_min_objective(P.tut_f)
    with pytest.raises(ValueError):
        o2.optimize([1.0, 1.0])
    assert "dual_algorithm" in o2.get_errmsg()


@pytest.mark.skipif(not refsrc.built(), reason=refsrc.NOT_BUILT)
@pytest.mark.parametrize("use_our_header", [False, True])
@pytest.mark.parametrize("arg", [None, "24", "41", "31"])      # 31 = LD_AUGLAG over the default MMA (ctest t_tutorial_31)
def test_reference_t_tutorial_links_and_passes(hosttest_lib, use_our_header, arg):
    """BASELINE config 1: the reference's own test/t_tutorial.cxx, unmodified, compiled against the
    reference-generated nlopt.hpp and linked with OUR object API + CCSA driver."""
    out = os.path.join(ROOT, "tests", "_build", "refinc")
    exe = refsrc.reference_test("t_tutorial", hosttest_lib.path, out, use_our_header)
    r = subprocess.run([exe] + ([arg] if arg else []), capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "found minimum" in r.stdout


@pytest.mark.skipif(not refsrc.built(), reason=refsrc.NOT_BUILT)
def test_reference_cpp_functor_links_and_runs(hosttest_lib):
    out = os.path.join(ROOT, "tests", "_build", "refinc")
    exe = refsrc.reference_test("cpp_functor", hosttest_lib.path, out, False)
    r = subprocess.run([exe], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr


def test_deprecated_one_call_api_matches_reference(hosttest_lib, reference):
    """nlopt_minimize_constrained / nlopt_minimize_econstrained / nlopt_minimize and the process-wide local-search
    settings (reference src/api/deprecated.c, nlopt.h:305-343): same results as the reference through the same call."""
    import ctypes as C
    OLD = C.CFUNCTYPE(C.c_double, C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_double), C.c_void_p)

    class CD(C.Structure):
        _fields_ = [("a", C.c_double), ("b", C.c_double)]

    def f_old(n, x, grad, _d):
        if grad:
            grad[0], grad[1] = 0.0, 0.5 / np.sqrt(x[1])
        return float(np.sqrt(x[1]))

    def c_old(n, x, grad, d):
        cd = CD.from_address(d)
        t = cd.a * x[0] + cd.b
        if grad:
            grad[0], grad[1] = 3 * cd.a * t * t, -1.0
        return float(t ** 3 - x[1])

    fo, co = OLD(f_old), OLD(c_old)
    data = (CD * 2)(CD(2.0, 0.0), CD(-1.0, 1.0))

    def one_call(lib):
        L = lib.dll
        L.nlopt_minimize_constrained.restype = C.c_int
        L.nlopt_minimize_constrained.argtypes = [C.c_int, C.c_int, OLD, C.c_void_p, C.c_int, OLD, C.c_void_p, C.c_ssize_t,
                                                 C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_double),
                                                 C.POINTER(C.c_double), C.c_double, C.c_double, C.c_double, C.c_double,
                                                 C.POINTER(C.c_double), C.c_int, C.c_double]
        lb, ub = (C.c_double * 2)(-np.inf, 1e-6), (C.c_double * 2)(np.inf, np.inf)
        x, minf = (C.c_double * 2)(1.234, 5.678), C.c_double(0)
        ret = L.nlopt_minimize_constrained(nl.LD_MMA, 2, fo, None, 2, co, C.cast(data, C.c_void_p), C.sizeof(CD), lb, ub, x, C.byref(minf),
                                           -1e300, 0.0, 0.0, 1e-6, None, 500, 0.0)
        result = (ret, minf.value, x[0], x[1])
        L.nlopt_get_local_search_algorithm.argtypes = [C.POINTER(C.c_int)] * 3
        d, nd, me = C.c_int(), C.c_int(), C.c_int()
        L.nlopt_get_local_search_algorithm(C.byref(d), C.byref(nd), C.byref(me))
        assert (d.value, nd.value, me.value) == (nl.LD_MMA, nl.LN_COBYLA, -1)
        L.nlopt_set_stochastic_population(7)
        assert L.nlopt_get_stochastic_population() == 7
        L.nlopt_set_stochastic_population(-3)
        assert L.nlopt_get_stochastic_population() == 0
        return result
    out = {"ref": reference("host_driver/deprecated_one_call_api", one_call), "ours": one_call(hosttest_lib)}
    assert out["ours"][0] == out["ref"][0] == nl.XTOL_REACHED
    assert abs(out["ours"][1] - out["ref"][1]) <= 1e-6 and abs(out["ours"][1] - P.TUT_FSTAR) <= 1e-3
    assert abs(out["ours"][2] - out["ref"][2]) <= 1e-5 and abs(out["ours"][3] - out["ref"][3]) <= 1e-5


@pytest.mark.skipif(not refsrc.built(), reason=refsrc.NOT_BUILT)
@pytest.mark.parametrize("alg", [24, 41])
@pytest.mark.parametrize("obj", [0, 1])
def test_reference_testopt_runs_against_our_library(hosttest_lib, reflib, alg, obj):
    """ctest's `testopt_algo24_obj{0,1}` (test/CMakeLists.txt:39-60): the reference's own benchmark driver, compiled
    unmodified against our library, must behave like the same driver linked with the reference: identical printed
    optimum for a short run from the deterministic start (-c), success and the same optimum to 1e-3 for a long one."""
    out = os.path.join(ROOT, "tests", "_build")
    ours = refsrc.reference_testopt(hosttest_lib.path, out)
    ref = refsrc.reference_testopt(reflib.path, out)

    def run(exe, evals):
        r = subprocess.run([exe, "-c", "-e", str(evals), "-a", str(alg), "-o", str(obj)], stdout=subprocess.PIPE,
                           stderr=subprocess.STDOUT, text=True, timeout=120)
        assert r.returncode == 0, r.stdout
        lines = [l for l in r.stdout.splitlines() if l.startswith(("return code", "Found minimum", "Minimum at"))]
        return lines

    assert run(ours, 25) == run(ref, 25)
    a, b = run(ours, 3000), run(ref, 3000)
    fa = float(a[1].split("f = ")[1].split()[0])
    fb = float(b[1].split("f = ")[1].split()[0])
    assert a[0] == b[0] and abs(fa - fb) <= 1e-3 * max(1.0, abs(fb))


@pytest.mark.skipif(not refsrc.available(), reason="reference tree not mounted")
@pytest.mark.parametrize("arg", [None, "24", "41", "31"])
def test_reference_t_python_runs_on_the_shim(hosttest_lib, arg):
    """The reference's own test/t_python.py (ctest t_python*), unmodified, with `import nlopt` resolved by
    nlopt_b200/shim and the library pointed at the CPU-backed build of our host logic."""
    env = dict(os.environ, PYTHONPATH=os.path.join(ROOT, "nlopt_b200", "shim"), NLOPT_B200_LIBRARY_PATH=hosttest_lib.path)
    r = subprocess.run([os.sys.executable, os.path.join(refsrc.REF, "test", "t_python.py")] + ([arg] if arg else []),
                       capture_output=True, text=True, env=env, timeout=120)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "minimum value: 0.5443" in r.stdout


def test_distinct_objects_on_distinct_threads(hosttest_lib):
    """SURVEY.md 8(b) threading contract: an nlopt_opt must not be shared, but distinct objects may run on distinct
    threads.  Eight threads, each with its own object and problem size; results must equal the sequential ones."""
    import threading

    def solve(n):
        f, c = P.quad_problem(n)
        r = run(hosttest_lib, nl.LD_MMA if n % 2 else nl.LD_CCSAQ, n, f, [c], [0.0], np.full(n, -1.0), np.full(n, 1.0),
                np.full(n, -0.5), xtol_rel=1e-7, maxeval=80)
        return r["ret"], r["numevals"], r["minf"], r["x"].tobytes()

    sizes = [40 + 7 * k for k in range(8)]
    want = [solve(n) for n in sizes]
    got = [None] * len(sizes)

    def worker(i):
        got[i] = solve(sizes[i])

    ts = [threading.Thread(target=worker, args=(i,)) for i in range(len(sizes))]
    for t in ts:
        t.start()
    for t in ts:
        t.join()
    assert got == want


def precond_problem(n, seed=3):
    """f(x) = 1/2 x^T A x - b^T x with A = tridiag(-1, d_j, -1) SPD, preconditioner H = A (the exact Hessian); one linear
    constraint with the zero preconditioner (its model is then the plain separable one)."""
    rng = np.random.default_rng(seed)
    d = 2.5 + rng.random(n)
    b = rng.standard_normal(n)

    def A(v):
        out = d * v
        out[:-1] -= v[1:]
        out[1:] -= v[:-1]
        return out

    def f(x, g):
        Ax = A(x)
        if g.size:
            g[:] = Ax - b
        return float(0.5 * x @ Ax - b @ x)

    def pre(x, v, vpre):
        vpre[:] = A(v)

    w = (1.0 + 0.5 * np.sin(0.37 * np.arange(n))) / n

    def c(x, g):
        if g.size:
            g[:] = w
        return float(w @ x) + 0.05
    return f, pre, c, A, b


def run_precond(lib, n, with_constraint_pre=False, **kw):
    f, pre, c, A, b = precond_problem(n)
    o = nl.opt(nl.LD_CCSAQ, n, library=lib)
    o.set_lower_bounds(np.full(n, -2.0)); o.set_upper_bounds(np.full(n, 2.0))
    o.set_precond_min_objective(f, pre)
    if with_constraint_pre:
        o.add_precond_inequality_constraint(c, lambda x, v, vpre: vpre.__setitem__(slice(None), 0.0), 1e-8)
    else:
        o.add_inequality_constraint(c, 1e-8)
    for k, v in kw.items():
        if k in ("xtol_rel", "ftol_rel", "maxeval"):
            getattr(o, "set_" + k)(v)
        else:
            o.set_param(k, v)
    x = o.optimize(np.zeros(n))
    return dict(ret=o.last_optimize_result(), x=x, minf=o.last_optimum_value(), numevals=o.get_numevals())


@pytest.mark.parametrize("with_constraint_pre", [False, True])
def test_preconditioned_ccsaq_converges_to_the_reference_optimum(hosttest_lib, reference, with_constraint_pre):
    """SURVEY.md 8(f)-2, ccsa_quadratic.c:153-206, :299-324, :415-441.  With the exact Hessian as preconditioner the
    model is exact, so every inner iteration is conservative and both libraries walk to the constrained optimum of the
    quadratic; trajectories are not comparable step by step (the reference reads an uninitialised dd.wval on this
    branch, DESIGN.md), the optimum is: f* to 1e-7 relative, x* to 1e-5, and the KKT residual of the returned point."""
    n = 60
    b = reference(f"host_driver/preconditioned_ccsaq/constraint_pre={with_constraint_pre}",
                  lambda lib: run_precond(lib, n, with_constraint_pre, xtol_rel=1e-9, maxeval=60, dual_ftol_rel=1e-12))
    a = run_precond(hosttest_lib, n, with_constraint_pre, xtol_rel=1e-9, maxeval=60, dual_ftol_rel=1e-12)
    assert a["ret"] > 0 and b["ret"] > 0
    assert abs(a["minf"] - b["minf"]) <= 1e-7 * max(1.0, abs(b["minf"]))
    assert np.max(np.abs(a["x"] - b["x"])) <= 1e-5
    f, pre, c, A, bb = precond_problem(n)
    g = A(a["x"]) - bb
    w = (1.0 + 0.5 * np.sin(0.37 * np.arange(n))) / n
    lam = -float(g @ w) / float(w @ w)        # multiplier of the active linear constraint (interior of the box here)
    assert lam > 0 and np.max(np.abs(g + lam * w)) <= 1e-4
