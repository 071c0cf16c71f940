"""The comparisons of tests/test_host_driver.py -- every MMA/CCSAQ parameter of optimize.c:798-826, the dual
tolerances supplied by a local optimiser, infeasible starts, NaN constraints, vector constraints, maximisation,
stopping rules, threads -- run through the PRODUCT library (CUDA kernels, fused dual solve) instead of the
CPU-backed build of the host logic.  Same assertions, same tolerances; the unmodified reference's stored results
(tests/reference_runs.py) are the other side of each comparison."""
import numpy as np
import pytest

import nlopt_b200 as nl
import oracle_bindings as ob
import test_host_driver as H
from test_oracle_port import GOLD

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def gpulib(built):
    from nlopt_b200._capi import default_library
    return default_library()


@pytest.mark.parametrize("alg", [nl.LD_MMA, nl.LD_CCSAQ])
def test_rosenbrock_vs_reference(gpulib, reference, alg):
    H.test_rosenbrock_vs_reference(gpulib, reference, alg)


@pytest.mark.parametrize("alg", [nl.LD_MMA, nl.LD_CCSAQ])
@pytest.mark.parametrize("opts", [dict(), dict(inner_gradients=0), dict(always_improve=0), dict(sigma_min=0.05),
                                  dict(inner_maxeval=2), dict(rho_init=10.0)])
def test_algorithm_parameters_vs_reference(gpulib, reference, alg, opts):
    H.test_algorithm_parameters_vs_reference(gpulib, reference, alg, opts)


@pytest.mark.parametrize("alg", [nl.LD_MMA, nl.LD_CCSAQ])
@pytest.mark.parametrize("opts", [dict(dual_ftol_rel=1e-6), dict(dual_xtol_rel=1e-6), dict(dual_maxeval=5),
                                  dict(dual_ftol_abs=1e-10), dict(dual_xtol_abs=1e-9, dual_ftol_rel=0.0)])
def test_dual_tolerances_vs_reference(gpulib, reference, alg, opts):
    """dual_* parameters (optimize.c:822-826) through the persistent solve kernel against the reference over the first 20
    evaluations.  Tolerance: a dual solve that stops on a loose rule stops at a y that depends on the last bits of the
    n-term sums (tree order here, sequential in the reference), so the two runs separate by ~1e-7 relative in f and
    ~1e-5 in x (measured: 1.4e-7 / 1.3e-5 with dual_xtol_abs = 1e-9); the default rule (1e-14) tracks to 1e-8."""
    n = 300
    f, c = H.P.quad_problem(n)
    lb, ub = np.full(n, -1.0), np.full(n, 1.0)
    kw = dict(xtol_rel=1e-7, **opts)
    b = reference(f"host_driver_gpu/dual_tolerances/{alg}/{H.okey(opts)}",
                  lambda lib: H.plain(H.run(lib, alg, n, f, [c], [0.0], lb, ub, np.full(n, -0.5), maxeval=20, **kw)))
    a = H.run(gpulib, alg, n, f, [c], [0.0], lb, ub, np.full(n, -0.5), maxeval=20, **kw)
    assert a["ret"] == b["ret"] and a["numevals"] == b["numevals"]
    assert abs(a["minf"] - b["minf"]) <= 1e-6 * max(1.0, abs(b["minf"]))
    assert np.max(np.abs(a["x"] - b["x"])) <= 1e-4


@pytest.mark.parametrize("alg", [nl.LD_MMA, nl.LD_CCSAQ])
def test_default_dual_tolerance_agrees_loosely(gpulib, reference, alg):
    H.test_default_dual_tolerance_agrees_loosely(gpulib, reference, alg)


def test_infeasible_start_uses_capped_multipliers(gpulib, reference):
    H.test_infeasible_start_uses_capped_multipliers(gpulib, reference)


def test_unconstrained_m0(gpulib, reference):
    H.test_unconstrained_m0(gpulib, reference)


def test_vector_constraint_equals_scalar_constraints(gpulib):
    H.test_vector_constraint_equals_scalar_constraints(gpulib)


def test_maximize_flips_sign(gpulib):
    H.test_maximize_flips_sign(gpulib)


def test_stopping_and_forced_stop(gpulib):
    H.test_stopping_and_forced_stop(gpulib)


def test_nan_constraint_is_ignored_by_mma(gpulib, reference):
    H.test_nan_constraint_is_ignored_by_mma(gpulib, reference)


def test_local_optimizer_supplies_dual_tolerances(gpulib, reference):
    H.test_local_optimizer_supplies_dual_tolerances(gpulib, reference)


def test_deprecated_one_call_api_matches_reference(gpulib, reference):
    H.test_deprecated_one_call_api_matches_reference(gpulib, reference)


def test_distinct_objects_on_distinct_threads(gpulib):
    H.test_distinct_objects_on_distinct_threads(gpulib)


@pytest.mark.parametrize("variant,setting,ret,evals,x0,x1,f", GOLD)
def test_tutorial_goldens(gpulib, variant, setting, ret, evals, x0, x1, f):
    H.test_tutorial_goldens(gpulib, variant, setting, ret, evals, x0, x1, f)


def test_maxtime_returns_maxtime(gpulib):
    """nlopt_set_maxtime through the fused solve (in-kernel %globaltimer test) and the driver's polls."""
    import time
    n = 200000
    f, c = H.P.quad_problem(n)
    t0 = time.perf_counter()
    r = H.run(gpulib, nl.LD_MMA, n, f, [c], [0.0], np.full(n, -1.0), np.full(n, 1.0), np.full(n, -0.5), maxtime=0.05,
              xtol_rel=1e-15, maxeval=100000)
    assert r["ret"] == nl.MAXTIME_REACHED
    assert time.perf_counter() - t0 < 5.0


@pytest.mark.parametrize("with_constraint_pre", [False, True])
def test_preconditioned_ccsaq_converges_to_the_reference_optimum(gpulib, reference, with_constraint_pre):
    H.test_preconditioned_ccsaq_converges_to_the_reference_optimum(gpulib, reference, with_constraint_pre)
