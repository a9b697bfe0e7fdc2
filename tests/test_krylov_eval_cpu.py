"""oracle/krylov_eval.py, the recurrences the GPU Krylov tests take as their float64 reference, pinned on the CPU:

* in float32 it is the C oracle's CG / BiCGStab (oracle/piso_oracle.c) up to the summation order of the dot products (the oracle
  accumulates them in double): same iteration counts, iterates equal within float32 rounding;
* in float64, on the reference's own pressure system of the cylinder-24 trace, it lands inside the tolerance ball of the reference's
  pressure and needs the reference's iteration count (2 % + 2, the band the GPU parity tests allow the kernels);
* the kernels' conventions: zero right-hand side, mean removal, transposed operator, per-component stopping of BiCGStab."""
import os

import numpy as np
import pytest
import scipy.sparse as sp

import krylov_eval as ke
from conftest import GOLDEN, rel_l2

f32 = np.float32


@pytest.fixture(scope="module")
def cyl8():
    from fluidgym_b200.envs.cylinder_domain import make_cylinder_domain
    return make_cylinder_domain(8).prepare()


def _ell(cd, off, diag):
    """the C oracle's ELL(5) rows: diagonal first, then the four faces (index -1 where a face has no neighbour)"""
    nbr = np.asarray(cd.nbr)
    val = np.concatenate([diag[:, None], np.where(nbr >= 0, off, 0).T], axis=1).astype(f32)
    idx = np.concatenate([np.arange(cd.N)[:, None], np.where(nbr >= 0, nbr, -1).T], axis=1).astype(np.int32)
    return val, idx


@pytest.mark.parametrize("warm", [False, True])
@pytest.mark.parametrize("reset_steps", [0, 7, 100])
@pytest.mark.parametrize("maxit", [5, 21, 5000])
def test_float32_cg_is_the_c_oracle(cyl8, warm, reset_steps, maxit):
    from oracle import Oracle
    off, diag = ke.synthetic_spd(cyl8.nbr, cyl8.rev, seed=1)
    P = ke.ell_matrix(cyl8.nbr, off, diag)
    rng = np.random.default_rng(2)
    f = rng.standard_normal(cyl8.N).astype(f32)
    x0 = rng.standard_normal(cyl8.N).astype(f32) if warm else None
    ours = ke.cg(P, f, x0, 1e-5, reset_steps, maxit, dtype=f32, flags=2)
    orc = Oracle.from_compiled(cyl8)
    x, used, fin, conv = orc.cg(*_ell(cyl8, off, diag), f, x0=x0, maxit=maxit, tol=1e-5, reset=reset_steps)
    assert ours.used == used and conv == (maxit == 5000)
    # a converged criterion is small enough to carry the float32 rounding of every update of the recurrence residual
    assert abs(ours.fin - fin) <= 5e-3 * fin
    assert rel_l2(ours.x, x) < 1e-5


def test_float32_bicgstab_is_the_c_oracle(cyl8):
    from oracle import Oracle
    off, diag = ke.synthetic_nonsym(cyl8.nbr, seed=3)
    C = ke.ell_matrix(cyl8.nbr, off, diag)
    F = np.random.default_rng(4).standard_normal((2, cyl8.N)).astype(f32)
    F[1] *= f32(1e-3)                                      # absolute criterion: the scaled component finishes much earlier
    ours = ke.bicgstab(C, F, None, 1e-5, 5000, dtype=f32)
    orc = Oracle.from_compiled(cyl8)
    val, idx = _ell(cyl8, off, diag)
    for c in range(2):
        x, used, fin, conv = orc.bicgstab(val, idx, F[c], maxit=5000, tol=1e-5)
        assert conv and ours.used[c] == used and abs(ours.fin[c] - fin) <= 5e-3 * fin
        assert rel_l2(ours.x[c], x) < 1e-5
    assert ours.used[1] < ours.used[0]
    # a cap reports used = i of the last half step; the iterate includes the full step that followed
    capped = ke.bicgstab(C, F, None, 1e-5, 3, dtype=f32)
    for c in range(2):
        x, used, fin, conv = orc.bicgstab(val, idx, F[c], maxit=3, tol=1e-5)
        assert capped.used[c] == used and rel_l2(capped.x[c], x) < 1e-5


def test_float64_cg_on_the_reference_pressure_system():
    fx = np.load(os.path.join(GOLDEN, "cyl24_substep1.npz"))
    N = fx["div0"].size
    P = sp.csr_matrix((fx["P_value"], fx["P_index"], fx["P_row"]), shape=(N, N))
    res = ke.cg(P, fx["div0"], None, 1e-5, 100, 5000, dtype=np.float64)
    ref = int(fx["cg_iters"][0])
    assert abs(res.used - ref) <= 0.02 * ref + 2 and res.fin < 1e-5
    assert rel_l2(res.x, fx["p0"]) < 5e-4
    assert abs(res.x.mean()) < 1e-12 * np.abs(res.x).max() and res.mean != 0.0


def test_conventions(cyl8):
    off, diag = ke.synthetic_spd(cyl8.nbr, cyl8.rev, seed=5)
    P = ke.ell_matrix(cyl8.nbr, off, diag)
    zero = ke.cg(P, np.zeros(cyl8.N, f32), np.ones(cyl8.N, f32))
    assert zero.used == -1 and zero.fin == 0.0 and zero.mean == 0.0 and not zero.x.any()
    f = np.random.default_rng(6).standard_normal(cyl8.N)
    kept, removed = ke.cg(P, f, flags=2), ke.cg(P, f)
    assert kept.mean == 0.0 and np.allclose(kept.x - kept.x.mean(), removed.x, rtol=0, atol=1e-12)
    assert np.isclose(removed.mean, kept.x.mean(), rtol=1e-14)
    # the transposed solve of a non-symmetric system is the solve with the transpose
    offn, diagn = ke.synthetic_nonsym(cyl8.nbr, seed=7)
    C = ke.ell_matrix(cyl8.nbr, offn, diagn)
    a, b = ke.cg(C, f, flags=1 | 2, maxit=9), ke.cg(C.T.tocsr(), f, flags=2, maxit=9)
    assert np.array_equal(a.x, b.x) and a.used == b.used
    # tol 0: every iteration runs, the cap returns the best iterate of the history
    crit, xs = ke.cg_history(P, f, None, 7, 12)
    capped = ke.cg(P, f, None, 0.0, 7, 12, flags=2)
    assert capped.used == int(np.argmin(crit)) and np.array_equal(capped.x, xs[capped.used])
    # the lazy order is the eager one
    for m in (3, 12, 5000):
        e, l = ke.cg(P, f, None, 1e-5, 7, m), ke.cg(P, f, None, 1e-5, 7, m, lazy=True)
        assert e.used == l.used and np.array_equal(e.x, l.x)
