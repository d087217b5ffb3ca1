"""CPU oracle of the compactly supported WSINDy test functions — TEST INFRASTRUCTURE ONLY.

The family of WSINDyWrapper(test_func_family='poly') has no counterpart in the reference, so this restatement is its
definition (as the oracle is for the degree-4/5 libraries): NumPy fp64, built row by row from the formula and
independently of the product's table code. The library Θ comes from `oracle.sindy_oracle`. Imported by the tests and
by `__graft_entry__.smoke()`; the product never imports it.
"""
import math

import numpy as np

from oracle import sindy_oracle as O


def wsindy_local_test_functions(T, dt, n_test, support=None, degree=None, rounded=True):
    """Dense V, V' (n_test × T) of the compactly supported polynomial family (no reference: the definition of
    WSINDyWrapper(test_func_family='poly')), built row by row in fp64 from the formula
      φ(u) = (4u(1−u))^p on u = q/(L−1), q = 0..L−1,  V[j, s_j+q] = dt·c·φ(u_q),  V'[j, s_j+q] = dt·c·dφ/dt(u_q),
      c = 1/sqrt(dt·Σ_q φ(u_q)²),  s_j = ⌊j·(T−L)/(n_test−1)⌋,
    defaults L = min(T, 2·⌊T/(n_test+1)⌋ + 1), p = 6; rounded to fp32 unless rounded=False."""
    L = min(T, 2 * (T // (n_test + 1)) + 1) if support is None else support
    p = 6 if degree is None else degree
    V = np.zeros((n_test, T))
    Vd = np.zeros((n_test, T))
    for j in range(n_test):
        s = 0 if n_test == 1 else (j * (T - L)) // (n_test - 1)
        for q in range(L):
            u = q / (L - 1)
            V[j, s + q] = (4.0 * u * (1.0 - u)) ** p
            # d/dt of (4u(1−u))^p with u = (t − t_s)/((L−1)·dt)
            Vd[j, s + q] = p * (4.0 * u * (1.0 - u)) ** (p - 1) * (4.0 - 8.0 * u) / ((L - 1) * dt)
        c = 1.0 / math.sqrt(dt * np.sum(V[j, s:s + L] ** 2))
        V[j] *= dt * c
        Vd[j] *= dt * c
    if rounded:
        return V.astype(np.float32), Vd.astype(np.float32)
    return V, Vd


def wsindy_local_integrals(x, dt, p, sine=False, exp=False, n_test=50, support=None, degree=None):
    """G = VΘ(x), b = −V'x with the compactly supported family, fp64 contraction of the fp32 factors (the convention of
    `wsindy_integrals`); x of shape (T, d) or (n_traj, T, d)."""
    x = np.asarray(x, dtype=np.float32)
    V, Vd = wsindy_local_test_functions(x.shape[-2], dt, n_test, support, degree)
    th = O.theta(x, p, sine, exp).astype(np.float64)
    return V.astype(np.float64) @ th, -(Vd.astype(np.float64) @ x.astype(np.float64))
