"""CPU emulation of the two bookkeeping orders of k_cg_strip (csrc/piso_b200.cu): cg_impl 13 updates the iterate between
the <p,Ap> and <r,r> reductions and stores every improving iterate as the best one; cg_impl 11 (LAZY) defers x += alpha p into
the next direction update (same p_old, same operands), stores the best iterate only on the first non-improving iteration after
an improving run (the registers are not advanced yet then) and applies the pending update on every exit that leaves with the
current iterate.  Both orders are written here in float32 numpy with the same expressions, including the residual reset, the
100-rising-steps cut-off and the iteration cap: solution, iteration count, criterion and best iterate must be bit-identical.
(The GPU check of the kernels themselves: tests/test_gpu_cg_strip_lazy.py.)"""
import numpy as np
import pytest
import scipy.sparse as sp

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


def _crit(rr, n):
    return f32(np.sqrt(rr)) * f32(1.0 / np.sqrt(f32(n)))


def _start(A, f, x0):
    x = x0.copy()
    r = f.copy() if not x.any() else (f - A @ x).astype(f32)
    return x, r, x.copy(), np.dot(r, r), r.copy()                          # x, r, best (x0 stored), rho, p


def strip_cg_eager(A, f, x0, tol, reset_steps, maxit):
    """statement order of k_cg_strip<..., LAZY = false> (cg_impl 13)"""
    n = f.size
    x, r, best, rho, p = _start(A, f, x0)
    bestc = lastc = f32(0); best_it, rising, used, fin = -1, 0, -1, f32(0)
    take_best = False
    until_reset = reset_steps - 1 if reset_steps > 0 else -1
    for i in range(maxit):
        if until_reset == 0:
            until_reset = reset_steps
            r = (f - A @ x).astype(f32); rho = np.dot(r, r); p = r.copy()
        until_reset -= 1
        ap = (A @ p).astype(f32)
        alpha = f32(rho / np.dot(p, ap))
        x = (x + alpha * p).astype(f32)
        r = (r - alpha * ap).astype(f32)
        rr = np.dot(r, r)
        crit = _crit(rr, n)
        stop = 0 if np.isfinite(crit) else 1
        used, fin = i, crit
        if not stop:
            if i == 0 or crit < bestc:
                bestc, best_it, best = crit, i, x.copy()
            rising = rising + 1 if (i > 0 and crit >= lastc) else 0
            lastc = crit
            if crit < tol:
                stop = 1
            elif i == maxit - 1 or rising >= 100:
                stop = 2
        if stop:
            take_best = stop == 2
            break
        beta = f32(rr / rho); rho = rr
        p = (r + beta * p).astype(f32)
    if take_best:
        x = best.copy(); used, fin = best_it, bestc
    return x, used, fin, best


def strip_cg_lazy(A, f, x0, tol, reset_steps, maxit):
    """statement order of k_cg_strip<..., LAZY = true> (cg_impl 11)"""
    n = f.size
    x, r, best, rho, p = _start(A, f, x0)
    bestc = lastc = f32(0); best_it, rising, used, fin = -1, 0, -1, f32(0)
    take_best = pending = advance = False
    alpha = f32(0)
    until_reset = reset_steps - 1 if reset_steps > 0 else -1
    for i in range(maxit):
        if until_reset == 0:
            until_reset = reset_steps
            r = (f - A @ x).astype(f32); rho = np.dot(r, r); p = r.copy()
        until_reset -= 1
        ap = (A @ p).astype(f32)
        alpha = f32(rho / np.dot(p, ap))
        r = (r - alpha * ap).astype(f32)                                   # x waits for the direction update
        rr = np.dot(r, r)
        crit = _crit(rr, n)
        stop = 0 if np.isfinite(crit) else 1
        used, fin = i, crit
        if not stop:
            if i == 0 or crit < bestc:
                bestc, best_it = crit, i
                pending = True
            elif pending:                                                  # x is still the iterate of best_it
                pending = False
                best = x.copy()
            rising = rising + 1 if (i > 0 and crit >= lastc) else 0
            lastc = crit
            if crit < tol:
                stop = 1
            elif i == maxit - 1 or rising >= 100:
                stop = 2
        if stop:
            take_best = stop == 2 and not pending
            advance = not take_best
            break
        beta = f32(rr / rho); rho = rr
        p_old = p
        p = (r + beta * p_old).astype(f32)
        x = (x + alpha * p_old).astype(f32)
    if take_best:
        x = best.copy(); used, fin = best_it, bestc
    elif advance:
        x = (x + alpha * p).astype(f32)
    return x, used, fin, (x if pending else best)


def _history(A, f, x0, reset_steps, maxit):
    """criterion of every iteration of an uncapped, unconverging run (both orders share the recurrence)"""
    crits = []
    n = f.size
    x, r, _, rho, p = _start(A, f, x0)
    until_reset = reset_steps - 1 if reset_steps > 0 else -1
    for _ in range(maxit):
        if until_reset == 0:
            until_reset = reset_steps
            r = (f - A @ x).astype(f32); rho = np.dot(r, r); p = r.copy()
        until_reset -= 1
        ap = (A @ p).astype(f32)
        alpha = f32(rho / np.dot(p, ap))
        x = (x + alpha * p).astype(f32)
        r = (r - alpha * ap).astype(f32)
        rr = np.dot(r, r)
        crits.append(_crit(rr, n))
        beta = f32(rr / rho); rho = rr
        p = (r + beta * p).astype(f32)
    return np.array(crits)


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
