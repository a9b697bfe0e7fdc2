"""CPU emulation of the two bookkeeping orders of k_cg_strip (csrc/piso_b200.cu): cg_impl 13 updates the iterate between
the <p,Ap> and <r,r> reductions and stores every improving iterate as the best one; cg_impl 11 (LAZY) defers x += alpha p into
the next direction update (same p_old, same operands), stores the best iterate only on the first non-improving iteration after
an improving run (the registers are not advanced yet then) and applies the pending update on every exit that leaves with the
current iterate.  Both orders are run here in float32 with the same expressions (oracle/krylov_eval.py, which the GPU tests
also run in float64 as the reference of the kernels), including the residual reset, the 100-rising-steps cut-off and the
iteration cap: solution, iteration count, criterion and best iterate must be bit-identical.
(The GPU check of the kernels themselves: tests/test_gpu_cg_strip_lazy.py.)"""
import numpy as np
import pytest
import scipy.sparse as sp

import krylov_eval as ke

f32 = np.float32


def _poisson(n, seed, consistent=True):
    rng = np.random.default_rng(seed)
    k = (0.5 + rng.random(n)).astype(f32)
    main = np.zeros(n, f32)
    off = np.zeros(n - 1, f32)
    off[:] = -(k[:-1] + k[1:]) * f32(0.5)
    main[:-1] -= off
    main[1:] -= off
    jump = -(rng.random(n - 7).astype(f32))                                # a second, wider coupling: 5 entries per row
    main[:-7] -= jump
    main[7:] -= jump
    A = sp.diags([main, off, off, jump, jump], [0, 1, -1, 7, -7], format="csr", dtype=f32)
    b = rng.standard_normal(n).astype(f32)
    # singular like the pressure matrix; consistent = right-hand side of zero mean (else the residual cannot vanish)
    return A, ((b - b.mean()) if consistent else b).astype(f32)


def strip_cg_eager(A, f, x0, tol, reset_steps, maxit):
    """statement order of k_cg_strip<..., LAZY = false> (cg_impl 13), mean kept"""
    r = ke.cg(A, f, x0, tol, reset_steps, maxit, dtype=f32, flags=2)
    return r.x, r.used, f32(r.fin), r.best


def strip_cg_lazy(A, f, x0, tol, reset_steps, maxit):
    """statement order of k_cg_strip<..., LAZY = true> (cg_impl 11), mean kept"""
    r = ke.cg(A, f, x0, tol, reset_steps, maxit, dtype=f32, flags=2, lazy=True)
    return r.x, r.used, f32(r.fin), r.best


def _history(A, f, x0, reset_steps, maxit):
    """criterion of every iteration of an uncapped, unconverging run (both orders share the recurrence)"""
    return ke.cg_history(A, f, x0, reset_steps, maxit, dtype=f32)[0]


def _x0(n, warm, seed):
    return (np.random.default_rng(seed).standard_normal(n) * 0.3).astype(f32) if warm else np.zeros(n, f32)


def _same(A, f, x0, tol, reset_steps, maxit):
    xe, ue, fe, be = strip_cg_eager(A, f, x0, f32(tol), reset_steps, maxit)
    xl, ul, fl, bl = strip_cg_lazy(A, f, x0, f32(tol), reset_steps, maxit)
    assert ue == ul and fe == fl
    assert np.array_equal(xe, xl) and np.array_equal(be, bl)
    return ue, fe


@pytest.mark.parametrize("warm", [False, True])
@pytest.mark.parametrize("reset_steps", [0, 7, 100])
@pytest.mark.parametrize("n", [257, 400])
def test_converged_solve_is_bit_identical(n, reset_steps, warm):
    A, f = _poisson(n, seed=n)
    used, fin = _same(A, f, _x0(n, warm, n + 1), 1e-5, reset_steps, 5000)
    assert 20 < used < 4999 and fin < f32(1e-5)


@pytest.mark.parametrize("warm", [False, True])
@pytest.mark.parametrize("reset_steps", [0, 7, 100])
def test_iteration_cap_is_bit_identical(reset_steps, warm):
    """cap on an improving iteration (the best iterate is the pending one) and on a non-improving one (an older best iterate
    from the scratch store)"""
    n = 400
    A, f = _poisson(n, seed=3)
    x0 = _x0(n, warm, 4)
    c = _history(A, f, x0, reset_steps, 120)
    best = np.minimum.accumulate(c)
    improving = [i for i in range(1, c.size) if c[i] < best[i - 1]]
    rising = [i for i in range(2, c.size) if c[i] >= best[i - 1] and c[i - 1] < best[i - 2]]
    assert improving and rising
    for cap_at, older in ((improving[-1], False), (rising[len(rising) // 2], True), (rising[-1], True)):
        used, fin = _same(A, f, x0, 0.0, reset_steps, cap_at + 1)
        assert (used < cap_at) == older and fin == best[cap_at]


@pytest.mark.parametrize("reset_steps", [0, 7])
def test_rising_steps_cut_off_is_bit_identical(reset_steps):
    """tol 0 on an inconsistent singular system: the residual stalls at its null-space part and the criterion stops falling,
    until 100 iterations in a row have not fallen below their predecessor"""
    n = 257
    A, f = _poisson(n, seed=11, consistent=False)
    for warm in (False, True):
        used, _ = _same(A, f, _x0(n, warm, 12), 0.0, reset_steps, 5000)
        assert used < 4899
