"""TEST INFRASTRUCTURE ONLY -- the recurrences of the 2-D Krylov kernels (csrc/piso_b200.cu), in a dtype of the caller's choice.

``cg`` states the pressure CG of ``k_cg`` / ``k_cg_cluster*`` / ``k_cg_smem`` / ``k_cg_strip*`` statement by statement (CG.cu:225-446):
zero or warm start, the all-zero right-hand side shortcut (exact zeros, ``used = -1``, ``fin = 0``), the residual reset when
``(i + 1) % reset_steps == 0``, the absolute criterion ``sqrt(<r,r>) / sqrt(N)``, best-iterate tracking (the solve leaves with the
stored best iterate at the iteration cap or after 100 rising steps, with the current one on a non-finite criterion) and the mean
removal the kernels report in ``pmean``.  ``flags`` are the kernels' flags: bit 0 solves with the transposed operator (what the
kernels build through ``tables.rev``), bit 1 keeps the mean.  ``lazy`` selects the bookkeeping order of ``k_cg_strip<..., LAZY = true>``
(cg_impl 11): the iterate update is deferred into the next direction update and the best iterate is stored on the first
non-improving iteration after an improving run.  Both orders perform the same operations on the same values, so in any dtype their
results are bit-identical (tests/test_cg_strip_bookkeeping_cpu.py).

``bicgstab`` states ``k_bicgstab`` / ``k_bicgstab_cluster`` (BICG.cu:237-376, no preconditioner) for NC right-hand sides in lock
step: every component stops on its own, at the half step (``used = i``) or at the full step (``used = i + 1``).

Run in float32 these are the kernels' arithmetic up to the summation order of the dot products; run in float64 they are the
reference of the same operation that the GPU tests compare the kernels with (tests/test_gpu_krylov_instantiations.py).
"""
from __future__ import annotations

from typing import NamedTuple

import numpy as np
import scipy.sparse as sp


class CGResult(NamedTuple):
    x: np.ndarray          # returned iterate, mean removed unless flags bit 1 (the kernels' p_out)
    mean: float            # removed mean (the kernels' pmean; 0 with flags bit 1)
    used: int              # iteration the result belongs to (-1: no iteration ran)
    fin: float             # its criterion sqrt(<r,r>) / sqrt(N)
    best: np.ndarray       # best iterate as stored when the solve ended (before mean removal)


class BiCGStabResult(NamedTuple):
    x: np.ndarray          # [NC, N]
    used: np.ndarray       # [NC]
    fin: np.ndarray        # [NC]


def _operator(A, dtype, flags):
    A = sp.csr_matrix(A)
    return (A.T if flags & 1 else A).astype(dtype).tocsr()


def _crit(rr, n, dt):
    return dt.type(np.sqrt(rr)) * dt.type(1.0 / np.sqrt(dt.type(n)))


def cg(A, f, x0=None, tol=1e-5, reset_steps=100, maxit=5000, dtype=np.float64, flags=0, lazy=False) -> CGResult:
    """One pressure CG solve of A x = f (A: any scipy sparse matrix; x0 None = zero start)."""
    dt = np.dtype(dtype)
    A = _operator(A, dt, flags)
    f = np.asarray(f).astype(dt)
    n = f.size
    x = np.zeros(n, dt) if x0 is None else np.asarray(x0).astype(dt)
    if not f.any():
        z = np.zeros(n, dt)
        return CGResult(z, 0.0, -1, 0.0, z.copy())
    x, used, fin, best = (_cg_lazy if lazy else _cg_eager)(A, f, x, dt.type(tol), reset_steps, maxit, dt)
    mean = dt.type(0) if flags & 2 else x.mean(dtype=dt)
    return CGResult((x - mean).astype(dt), float(mean), int(used), float(fin), best)


def _start(A, f, x0, dt):
    x = x0.copy()
    r = f.copy() if not x.any() else (f - A @ x).astype(dt)
    return x, r, x.copy(), np.dot(r, r), r.copy()                          # x, r, best (x0 stored), rho, p


def _cg_eager(A, f, x0, tol, reset_steps, maxit, dt):
    """statement order of k_cg, k_cg_cluster_mb and k_cg_strip<..., LAZY = false> (cg_impl 13)"""
    n = f.size
    x, r, best, rho, p = _start(A, f, x0, dt)
    bestc = lastc = dt.type(0); best_it, rising, used, fin = -1, 0, -1, dt.type(0)
    take_best = False
    until_reset = reset_steps - 1 if reset_steps > 0 else -1
    for i in range(maxit):
        if until_reset == 0:
            until_reset = reset_steps
            r = (f - A @ x).astype(dt); rho = np.dot(r, r); p = r.copy()
        until_reset -= 1
        ap = (A @ p).astype(dt)
        alpha = dt.type(rho / np.dot(p, ap))
        x = (x + alpha * p).astype(dt)
        r = (r - alpha * ap).astype(dt)
        rr = np.dot(r, r)
        crit = _crit(rr, n, dt)
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
        beta = dt.type(rr / rho); rho = rr
        p = (r + beta * p).astype(dt)
    if take_best:
        x = best.copy(); used, fin = best_it, bestc
    return x, used, fin, best


def _cg_lazy(A, f, x0, tol, reset_steps, maxit, dt):
    """statement order of k_cg_strip<..., LAZY = true> (cg_impl 11)"""
    n = f.size
    x, r, best, rho, p = _start(A, f, x0, dt)
    bestc = lastc = dt.type(0); best_it, rising, used, fin = -1, 0, -1, dt.type(0)
    take_best = pending = advance = False
    alpha = dt.type(0)
    until_reset = reset_steps - 1 if reset_steps > 0 else -1
    for i in range(maxit):
        if until_reset == 0:
            until_reset = reset_steps
            r = (f - A @ x).astype(dt); rho = np.dot(r, r); p = r.copy()
        until_reset -= 1
        ap = (A @ p).astype(dt)
        alpha = dt.type(rho / np.dot(p, ap))
        r = (r - alpha * ap).astype(dt)                                    # x waits for the direction update
        rr = np.dot(r, r)
        crit = _crit(rr, n, dt)
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
        beta = dt.type(rr / rho); rho = rr
        p_old = p
        p = (r + beta * p_old).astype(dt)
        x = (x + alpha * p_old).astype(dt)
    if take_best:
        x = best.copy(); used, fin = best_it, bestc
    elif advance:
        x = (x + alpha * p).astype(dt)
    return x, used, fin, (x if pending else best)


def cg_history(A, f, x0=None, reset_steps=100, maxit=100, dtype=np.float64, flags=0):
    """(criteria, iterates) of the first ``maxit`` iterations of an uncapped run that never stops: what a solve capped at
    m + 1 iterations chooses its best iterate from"""
    dt = np.dtype(dtype)
    A = _operator(A, dt, flags)
    f = np.asarray(f).astype(dt)
    n = f.size
    x, r, _, rho, p = _start(A, f, np.zeros(n, dt) if x0 is None else np.asarray(x0).astype(dt), dt)
    crits, xs = [], []
    until_reset = reset_steps - 1 if reset_steps > 0 else -1
    for _ in range(maxit):
        if until_reset == 0:
            until_reset = reset_steps
            r = (f - A @ x).astype(dt); rho = np.dot(r, r); p = r.copy()
        until_reset -= 1
        ap = (A @ p).astype(dt)
        alpha = dt.type(rho / np.dot(p, ap))
        x = (x + alpha * p).astype(dt)
        r = (r - alpha * ap).astype(dt)
        rr = np.dot(r, r)
        crits.append(_crit(rr, n, dt))
        xs.append(x.copy())
        beta = dt.type(rr / rho); rho = rr
        p = (r + beta * p).astype(dt)
    return np.array(crits), xs


def bicgstab(A, F, X0=None, tol=1e-5, maxit=5000, dtype=np.float64, flags=0) -> BiCGStabResult:
    """BiCGStab of A x_c = F[c] for the NC rows of F in lock step (X0 None = zero start)."""
    dt = np.dtype(dtype)
    A = _operator(A, dt, flags)
    F = np.atleast_2d(np.asarray(F)).astype(dt)
    NC, n = F.shape
    X = np.zeros((NC, n), dt) if X0 is None else np.atleast_2d(np.asarray(X0)).astype(dt).copy()
    R = np.stack([F[c] if not X[c].any() else (F[c] - A @ X[c]).astype(dt) for c in range(NC)])
    RW, P = R.copy(), R.copy()
    V, TT = np.zeros_like(R), np.zeros_like(R)
    fin = np.array([_crit(np.dot(R[c], R[c]), n, dt) for c in range(NC)], dtype=dt)
    used = np.full(NC, -1)
    done = fin < dt.type(tol)
    rho = np.ones(NC, dt); alpha = np.ones(NC, dt); omega = np.ones(NC, dt)
    tol = dt.type(tol)
    for i in range(maxit):
        if done.all():
            break
        for c in range(NC):
            if done[c]:
                continue
            rhop, rho[c] = rho[c], np.dot(RW[c], R[c])
            if i > 0:
                beta = dt.type((rho[c] / rhop) * (alpha[c] / omega[c]))
                P[c] = (R[c] + beta * (P[c] - omega[c] * V[c])).astype(dt)
            V[c] = (A @ P[c]).astype(dt)
            alpha[c] = dt.type(rho[c] / np.dot(RW[c], V[c]))
            R[c] = (R[c] - alpha[c] * V[c]).astype(dt)
            X[c] = (X[c] + alpha[c] * P[c]).astype(dt)
            nr = _crit(np.dot(R[c], R[c]), n, dt)
            used[c], fin[c] = i, nr
            if not np.isfinite(nr) or nr < tol:                             # half step
                done[c] = True
                continue
            TT[c] = (A @ R[c]).astype(dt)
            omega[c] = dt.type(np.dot(TT[c], R[c]) / np.dot(TT[c], TT[c]))
            X[c] = (X[c] + omega[c] * R[c]).astype(dt)
            R[c] = (R[c] - omega[c] * TT[c]).astype(dt)
            nr = _crit(np.dot(R[c], R[c]), n, dt)
            fin[c] = nr
            if nr < tol:                                                   # full step
                done[c] = True
                used[c] = i + 1
    return BiCGStabResult(X, used, fin.astype(np.float64))


# ---- systems in the kernels' layout: off [4, N] (coefficient of the neighbour across face f of cell g), diag [N] --------------
def ell_matrix(nbr, off, diag):
    """scipy CSR (float64) of the kernels' stencil layout; coefficients of faces without a neighbour are not part of it"""
    nbr = np.asarray(nbr)
    N = nbr.shape[1]
    rows, cols, vals = [np.arange(N)], [np.arange(N)], [np.asarray(diag, np.float64)]
    for f in range(4):
        g = np.nonzero(nbr[f] >= 0)[0]
        rows.append(g); cols.append(nbr[f][g]); vals.append(np.asarray(off[f], np.float64)[g])
    return sp.csr_matrix((np.concatenate(vals), (np.concatenate(rows), np.concatenate(cols))), shape=(N, N))


def synthetic_spd(nbr, rev, seed, shift=0.05):
    """SPD system on the domain's own stencil: positive edge weights, made symmetric through rev (the face of the neighbour that
    points back), a diagonal shift of ``shift`` times the mean row weight; NaN in the slots of faces without a neighbour (a kernel
    that reads them poisons its result).  Returns float32 (off [4, N], diag [N])."""
    nbr, rev = np.asarray(nbr), np.asarray(rev)
    N = nbr.shape[1]
    w = 0.5 + np.random.default_rng(seed).random((4, N))
    for f in range(4):
        g = np.nonzero(nbr[f] >= 0)[0]
        nb, fb = nbr[f][g], rev[f][g]
        assert (nbr[fb, nb] == g).all(), "rev does not invert nbr"
        lo = g < nb
        w[fb[lo], nb[lo]] = w[f][g[lo]]
    w = np.where(nbr >= 0, w, 0.0).astype(np.float32)
    rowsum = w.sum(0)
    diag = (rowsum + np.float32(shift) * rowsum.mean()).astype(np.float32)
    return np.where(nbr >= 0, -w, np.nan).astype(np.float32), diag


def synthetic_nonsym(nbr, seed, dominance=1.25):
    """Non-symmetric, diagonally dominant system on the domain's stencil (independent coefficients per cell and face, some of
    them positive like an upwinded convection term); NaN where a face has no neighbour.  Returns float32 (off [4, N], diag [N])."""
    nbr = np.asarray(nbr)
    rng = np.random.default_rng(seed)
    w = np.where(nbr >= 0, -(0.2 + rng.random(nbr.shape)) * np.where(rng.random(nbr.shape) < 0.15, -0.5, 1.0), 0.0)
    diag = (dominance * np.abs(w).sum(0) + 0.05).astype(np.float32)
    return np.where(nbr >= 0, w, np.nan).astype(np.float32), diag
