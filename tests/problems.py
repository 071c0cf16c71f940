"""Test problems shared by the parity tests (host-callback form: f(x, grad) -> float)."""
import math

import numpy as np


# ---- the NLopt tutorial problem (reference test/t_tutorial.cxx:11-34, doc NLopt_Tutorial.md) ----
def tut_f(x, grad):
    if grad.size > 0:
        grad[0] = 0.0
        grad[1] = 0.5 / math.sqrt(x[1])
    return math.sqrt(x[1])


def tut_c(a, b):
    def c(x, grad):
        t = a * x[0] + b
        if grad.size > 0:
            grad[0] = 3 * a * t * t
            grad[1] = -1.0
        return t * t * t - x[1]
    return c


TUT_X0 = [1.234, 5.678]
TUT_FSTAR = 0.544331053951817355154952   # sqrt(8/27)


# ---- chained Rosenbrock (formula of reference test/testfuncs.c:124-139) + m dense linear constraints ----
def rosen_f(x, grad):
    d = x[1:] - x[:-1] ** 2
    e = 1.0 - x[:-1]
    if grad.size > 0:
        grad[:] = 0.0
        grad[:-1] += -400.0 * x[:-1] * d - 2.0 * e
        grad[1:] += 200.0 * d
    return float(np.sum(100.0 * d * d + e * e))


def lin_constraint(k, n):
    j = np.arange(n, dtype=np.float64)
    w = (1.0 + 0.5 * np.sin(0.37 * (k + 1) * j)) / n
    b = 0.5 + 0.1 * k

    def c(x, grad):
        if grad.size > 0:
            grad[:] = w
        # numpy's pairwise sum, not np.dot: BLAS splits a long dot product over its threads, so its last bits depend on
        # the host's core count, and the stored reference results are compared bit for bit
        return float(np.sum(w * x)) - b
    return c


def rosen_x0(n):
    return -1.2 + 0.001 * (np.arange(n) % 7)


# ---- separable quadratic + mean constraint (BASELINE config 2 shape) ----
def quad_problem(n, seed=0x5EED0000):
    from synth import u01
    a = 1.0 + u01(0, n, seed)
    b = 2.0 * u01(1, n, seed) - 1.0

    def f(x, grad):
        d = x - b
        if grad.size > 0:
            grad[:] = a * d
        return float(0.5 * np.sum(a * d * d))

    def c(x, grad):
        if grad.size > 0:
            grad[:] = 1.0 / n
        return float(np.sum(x) / n + 0.1)
    return f, c


# ---- synthetic SIMP compliance + volume constraint (BASELINE config 4 shape) ----
def simp_problem(n, seed=0x5EED0000, eps=1e-3, vol=0.4):
    from synth import u01
    a = 0.5 + u01(0, n, seed)

    def f(x, grad):
        d = eps + (1.0 - eps) * x ** 3
        if grad.size > 0:
            grad[:] = -a * (1.0 - eps) * 3.0 * x * x / (d * d)
        return float(np.sum(a / d))

    def c(x, grad):
        if grad.size > 0:
            grad[:] = 1.0 / n
        return float(np.sum(x) / n - vol)
    return f, c
