"""GPU tests of BK_SPARSE contexts (a caller-assembled sparse Jacobian): k_spmv against scipy, the SH2d Jacobian as a matrix
against the named stencil, complex contexts and J', GMRES / Jacobi / grid preconditioners, bordered solvers, shift-invert
eigenvalues, the PALC drop-in, the Mittelmann branch with bifurcation detection, the Brusselator Hopf point, and the errors."""
import numpy as np
import pytest
import scipy.sparse as sp

import __graft_entry__ as g
from oracle import problems, krylov, bls as obls, palc as opalc, precond as oprecond
from tests import sparse_problems as S
from tests.test_codim2_curves_cpu import NumpyProblem2
from tests.test_host_logic_cpu import BlsAdapter

pytestmark = pytest.mark.gpu
LX, LY = 8 * np.pi, 4 * np.pi / np.sqrt(3)


@pytest.fixture(scope="module")
def bk():
    return g.load_package()


def _rel(a, b):
    return np.linalg.norm(np.asarray(a) - np.asarray(b)) / max(np.linalg.norm(b), 1e-300)


def _irregular(n=3000, seed=0):
    """rows of 0, 1, 3, 7, 20, 60 entries, one of 12000 and one of 1500 (CTA rows), random (unsorted, duplicate) columns:
    raw CSR arrays, raw CSC arrays of the same entries (random order within a column), and the scipy matrix (duplicates summed)"""
    rng = np.random.default_rng(seed)
    lens = rng.choice([0, 0, 1, 1, 3, 7, 20, 60], n)
    lens[17], lens[2500] = 12000, 1500
    rows = np.repeat(np.arange(n), lens)
    cols = rng.integers(0, n, len(rows))
    cols[:5] = cols[0]  # explicit duplicates
    vals = rng.standard_normal(len(rows))
    indptr = np.concatenate([[0], np.cumsum(lens)])
    order = np.lexsort((rng.random(len(rows)), cols))
    colptr = np.concatenate([[0], np.cumsum(np.bincount(cols, minlength=n))])
    ref = sp.coo_matrix((vals, (rows, cols)), shape=(n, n)).tocsr()
    return (indptr, cols, vals), (colptr, rows[order], vals[order]), ref


@pytest.mark.parametrize("fmt,base", [("csr", 0), ("csr", 1), ("csc", 0), ("csc", 1)])
def test_spmv_irregular_against_scipy(bk, fmt, base):
    (rp, ci, rv), (cp, ri, cv), ref = _irregular()
    n = ref.shape[0]
    ctx = bk.Context(bk.BK_SPARSE, (n,), krylov_m=4)
    ptr, idx, vals = (rp, ci, rv) if fmt == "csr" else (cp, ri, cv)
    ctx.sparse_pattern((fmt, base, ptr + base, idx + base))
    ctx.sparse_values(vals)
    x = np.random.default_rng(1).standard_normal(n)
    for a0, a1 in ((0.0, 1.0), (0.7, -1.3), (2.0, 0.0)):
        y = ctx.jvp(x, a0=a0, a1=a1)
        assert _rel(y, a0 * x + a1 * (ref @ x)) < 1e-13
    y1 = ctx.jvp(x, a0=0.7, a1=-1.3)
    y2 = ctx.jvp(ctx.to_device(x), a0=0.7, a1=-1.3).numpy()
    y3 = ctx.jvp(x, a0=0.7, a1=-1.3)
    assert np.array_equal(y1, y2) and np.array_equal(y1, y3)          # host / device pointers, two applies: same bits
    ctx.sparse_values(ctx.to_device(vals))                             # values from a device pointer
    assert np.array_equal(ctx.jvp(x, a0=0.7, a1=-1.3), y1)
    ctx.set_transpose(True)
    assert _rel(ctx.jvp(x, a0=0.3, a1=2.0), 0.3 * x + 2.0 * (ref.T @ x)) < 1e-13
    ctx.sparse_values(2.0 * vals)                                      # new values refresh J' as well
    assert _rel(ctx.jvp(x), 2.0 * (ref.T @ x)) < 1e-13
    ctx.set_transpose(False)
    assert _rel(ctx.jvp(x), 2.0 * (ref @ x)) < 1e-13


@pytest.mark.parametrize("dims", [(64, 32), (1024, 1024)])
def test_sh2d_jacobian_as_matrix_equals_named_stencil(bk, dims):
    sh = problems.SwiftHohenberg(dims, (LX, LY), l=-0.1, nu=1.3)
    u = problems.sh2d_sol0(*dims, LX, LY)
    v = np.random.default_rng(2).standard_normal(sh.N)
    named = bk.Context(bk.BK_SH2D, dims, (LX, LY), krylov_m=4, params=(-0.1, 1.3))
    named.jacobian(u)
    ctx = bk.Context(bk.BK_SPARSE, dims, (LX, LY), krylov_m=4)
    ctx.sparse_load(sh.jac_sparse(u))   # CSC, as SparseMatrixCSC
    for a0, a1 in ((0.0, 1.0), (2.0, -1.0)):
        assert _rel(ctx.jvp(v, a0=a0, a1=a1), named.jvp(v, a0=a0, a1=a1)) < 1e-12


def test_transpose_on_brusselator(bk):
    par = list(S.BRU_PAR)
    x = S.bru_steady(par) + 0.1 * np.random.default_rng(3).standard_normal(2 * S.BRU_N)
    J = S.bru_J(x, par)
    ctx = bk.Context(bk.BK_SPARSE, (2 * S.BRU_N,), krylov_m=4)
    ctx.sparse_load(J)
    v = np.random.default_rng(4).standard_normal(ctx.N)
    assert _rel(ctx.jvp(v), J @ v) < 1e-13
    ctx.set_transpose(True)
    assert _rel(ctx.jvp(v), J.T @ v) < 1e-13 and _rel(J.T @ v, J @ v) > 1e-5   # J' != J (the coupling blocks)


def test_complex_context_shift_and_adjoint(bk):
    par = list(S.BRU_PAR)
    n = 100
    x = S.bru_steady(par, n) + 0.1 * np.random.default_rng(5).standard_normal(2 * n)
    J = S.bru_J(x, par)
    M = J.toarray()
    cctx = bk.Context(bk.BK_SPARSE, (2 * n,), krylov_m=420, complex=True)
    cctx.sparse_load(J)
    rng = np.random.default_rng(6)
    z = rng.standard_normal(2 * n) + 1j * rng.standard_normal(2 * n)
    a0 = 0.4 - 1.7j
    for tr, A in ((False, M), (True, M.T)):
        cctx.set_transpose(tr)
        cctx.set_shift_imag(a0.imag)
        out = bk.core.cjoin(cctx.jvp(bk.core.csplit(z), a0=a0.real, a1=-0.5))
        cctx.set_shift_imag(0.0)
        assert _rel(out, a0 * z - 0.5 * (A @ z)) < 1e-12
        Jc = cctx.cjacobian(x, transpose=tr)
        cctx.sparse_load(J)
        cls = bk.ComplexGMRESB200(reltol=1e-12, restart=420, maxiter=840, orth="cgs2")
        y, cv, it = cls(Jc, z, a0=2.0j)
        assert cv and _rel(y, np.linalg.solve(2.0j * np.eye(2 * n) + A, z)) < 1e-8


def test_gmres_unpreconditioned_and_dct_on_sparse_sh2d(bk):
    """100 un-preconditioned iterations reach the named context's residual norm (1e-6, as test_config2); Pr = SH_DCT on the
    grid-shaped sparse context gives the named solution to 1e-8 with iteration counts +-2"""
    import bench
    n = 512
    L = bench.domain(n)
    sh = problems.SwiftHohenberg((n, n), L, l=-0.1, nu=1.3)
    u = bench.sol0(n)
    rhs = np.random.default_rng(1234).standard_normal(sh.N)
    named = bk.Context(bk.BK_SH2D, (n, n), L, krylov_m=100, params=(-0.1, 1.3))
    ctx = bk.Context(bk.BK_SPARSE, (n, n), L, krylov_m=100)
    Jn = named.jacobian(named.to_device(u))
    ctx.sparse_load(sh.jac_sparse(u))
    Js = bk.Jacobian(ctx)
    res = []
    for c, J in ((named, Jn), (ctx, Js)):
        ls = bk.GMRESB200(reltol=1e-14, restart=100, maxiter=100, orth="cgs2")
        x, ok, it = ls(J, c.to_device(rhs), a0=50.0, a1=-1.0)
        assert not ok and it == 100
        x = x.numpy()
        res.append(np.linalg.norm(rhs - (50.0 * x - sh.dF(u, x))))
    assert abs(res[0] - res[1]) < 1e-6 * res[0], res
    sols = []
    for c, J in ((named, Jn), (ctx, Js)):
        c.precond_setup(bk.BK_PC_SH_DCT, 1.0)
        x, ok, it = bk.GMRESB200(reltol=1e-8, restart=100, maxiter=100, Pr=True)(J, c.to_device(rhs), a0=2.0, a1=-1.0)
        assert ok
        sols.append((x.numpy(), it))
    assert _rel(sols[1][0], sols[0][0]) < 1e-8 and abs(sols[1][1] - sols[0][1]) <= 2, (sols[0][1], sols[1][1])


def test_jacobi_gmres_on_mittelmann_against_oracle(bk):
    mit = S.Mittelmann()
    u = 0.05 * np.random.default_rng(7).standard_normal(S.MIT_N ** 2)
    J = mit.J(u, [0.05])
    d = J.diagonal()
    rhs = np.random.default_rng(8).standard_normal(J.shape[0])
    xo, oko, ito = krylov.GMRESIterativeSolvers(reltol=1e-10, restart=300, maxiter=3000, Pl=lambda r: r / d)(lambda v: J @ v, rhs)
    ctx = bk.Context(bk.BK_SPARSE, (S.MIT_N, S.MIT_N), (S.MIT_L, S.MIT_L), krylov_m=300)
    ctx.sparse_load(J)
    ctx.precond_setup(bk.BK_PC_JACOBI, 0.0, 1.0)
    assert _rel(ctx.precond_apply(rhs), rhs / d) < 1e-15
    x, ok, it = bk.GMRESB200(reltol=1e-10, restart=300, maxiter=3000, Pl=True)(bk.Jacobian(ctx), rhs)
    assert ok and oko and _rel(x, xo) < 1e-8 and abs(it - ito) <= 2, (it, ito, _rel(x, xo))


def test_bordered_solvers_and_eigenvalues_brusselator(bk):
    n = 100
    par = list(S.BRU_PAR)
    par[S.BRU_LENS_L] = 0.6
    x = S.bru_steady(par, n) + 0.05 * np.random.default_rng(9).standard_normal(2 * n)
    J = S.bru_J(x, par)
    M, N = J.toarray(), 2 * n
    ctx = bk.Context(bk.BK_SPARSE, (N,), krylov_m=N + 20)
    ctx.sparse_load(J)
    Jd = bk.Jacobian(ctx)
    ls = bk.GMRESB200(reltol=1e-13, restart=N + 20, maxiter=4 * N, orth="cgs2")
    rng = np.random.default_rng(10)
    dR, dzu, R = rng.standard_normal(N), rng.standard_normal(N), rng.standard_normal(N)
    dzp, nr, xiu, xip, shift, ds = 0.8, -0.4, 0.5, 0.5, 0.3, 1.0 / N
    A = np.block([[M + shift * np.eye(N), dR[:, None]], [xiu * ds * dzu[None, :], np.array([[xip * dzp]])]])
    ex = np.linalg.solve(A, np.concatenate([R, [nr]]))
    for bls in (bk.BorderingBLSB200(ls, check_precision=False), bk.MatrixFreeBLSB200(ls)):
        dX, dl, cv, _ = bls(Jd, dR, dzu, dzp, R, nr, xiu, xip, shift=shift, dotscale=ds)
        assert cv and _rel(dX, ex[:-1]) < 1e-8 and abs(dl - ex[-1]) < 1e-8 * max(1, abs(ex[-1]))
    # block borders, m = 2
    a, b = (rng.standard_normal(N), rng.standard_normal(N)), (rng.standard_normal(N), rng.standard_normal(N))
    c = np.array([[0.3, -0.2], [0.1, 0.9]])
    rhsb = np.array([0.5, -1.5])
    B = np.block([[M + shift * np.eye(N), np.column_stack(a)], [np.vstack(b), c]])
    exb = np.linalg.solve(B, np.concatenate([R, rhsb]))
    u, p, cv, _ = bk.BorderingBLSB200(ls).solve_block(Jd, a, b, c, R, rhsb, shift=shift)
    assert cv and _rel(u, exb[:N]) < 1e-8 and np.allclose(p, exb[N:], rtol=1e-8, atol=1e-10)
    u, p, cv, _ = bk.MatrixFreeBLSB200(ls).solve_block(Jd, a, b, c, R, rhsb, shift=shift)
    assert cv and _rel(u, exb[:N]) < 1e-8 and np.allclose(p, exb[N:], rtol=1e-8, atol=1e-10)
    # shift-invert eigenvalues near the imaginary axis against the dense spectrum
    vals, _, cv, _ = bk.ShiftInvertB200(0.5, ls, krylovdim=40, tol=1e-12, maxrestart=40)(Jd, 6)
    dense = np.linalg.eigvals(M)
    assert cv
    for lam in vals:
        assert np.min(np.abs(dense - lam)) < 1e-7 * max(1.0, abs(lam)), lam
    near = dense[np.argsort(np.abs(dense - 0.5))[:6]]
    assert np.allclose(np.sort_complex(np.round(near, 6)), np.sort_complex(np.round(vals, 6)))


def test_palc_drop_in_sh2d_sparse(bk):
    """test_newton_hexagons_and_palc_branch with F = the oracle's host residual and J = jac_sparse on a sparse context"""
    P = bk.palc
    dims = (128, 64)
    sh = problems.SwiftHohenberg(dims, (LX, LY), l=-0.1, nu=1.3)
    Pinv = oprecond.dct_precond(dims, (LX, LY), 1.0)
    ols = krylov.GMRESIterativeSolvers(reltol=1e-8, restart=100, maxiter=100, N=sh.N, Pl=Pinv)
    oprob = lambda u0: opalc.Problem(F=lambda u, l: sh.F(u, l), J=lambda u, l: (lambda v: sh.dF(u, v, l)), u0=u0, p0=-0.1)
    u0 = problems.sh2d_sol0(*dims, LX, LY)
    osol = opalc.newton(oprob(u0), u0, -0.1, opalc.NewtonPar(tol=1e-8, max_iterations=20, linsolver=ols), opalc.norminf)
    front = problems.sh2d_front_guess(osol.u, *dims, LX, LY)
    ofront = opalc.newton(oprob(front), front, -0.1, opalc.NewtonPar(tol=1e-8, max_iterations=30, linsolver=ols), opalc.norminf)
    assert ofront.converged
    cpo = opalc.ContinuationPar(dsmin=1e-4, dsmax=5e-3, ds=-1e-3, p_min=-1.0, p_max=0.0, max_steps=8,
                                newton_options=opalc.NewtonPar(tol=1e-9, max_iterations=15, linsolver=ols))
    orows, _ = opalc.continuation(oprob(ofront.u), opalc.PALC(bls=obls.BorderingBLS(ols, check_precision=False)), cpo,
                                  normC=opalc.norminf)
    ctx = bk.Context(bk.BK_SPARSE, dims, (LX, LY), krylov_m=100)
    ctx.precond_setup(bk.BK_PC_SH_DCT, 1.0)
    ls = bk.GMRESB200(reltol=1e-8, restart=100, maxiter=100, N=sh.N, Pl=True)
    prob = P.SparseProblemB200(ctx, lambda u, q: sh.F(u, q[0]), lambda u, q: sh.jac_sparse(u, q[0]), np.array(ofront.u),
                               [-0.1, 1.3], lens=0)
    cp = P.ContinuationPar(dsmin=1e-4, dsmax=5e-3, ds=-1e-3, p_min=-1.0, p_max=0.0, max_steps=8,
                           newton_options=P.NewtonPar(tol=1e-9, max_iterations=15, linsolver=ls))
    rows, _ = P.continuation(prob, P.PALC(bls=bk.BorderingBLSB200(ls, check_precision=False)), cp, normC=P.norminf)
    assert len(rows) == len(orows) == 9
    for r, o in zip(rows, orows):
        assert abs(r["param"] - o["param"]) < 1e-7 and abs(r["x"] - o["x"]) < 1e-6 * o["x"], (r, o)
        assert r["itnewton"] == o["itnewton"]


def test_mittelmann_branch_with_bifurcation_detection(bk):
    """examples/mittleman.jl at 30 x 30: NumPy F, scipy J, Jacobi-preconditioned GMRES, detect_bifurcation = 3 through
    ShiftInvertB200 on the sparse context; rows and unstable-eigenvalue counts equal the host run with the oracle's solvers"""
    P, E = bk.palc, bk.events
    mit = S.Mittelmann()
    N = S.MIT_N ** 2
    kw = dict(dsmin=1e-4, dsmax=0.04, ds=0.01, p_min=0.0, p_max=0.5, max_steps=30, nev=8, detect_bifurcation=3, n_inversion=4,
              max_bisection_steps=20, tol_stability=1e-8)
    hls = krylov.DefaultLS()
    hprob = NumpyProblem2(mit.F, mit.J, np.zeros(N), [0.01], 0)
    hopts = P.NewtonPar(tol=1e-9, max_iterations=20, linsolver=hls, eigsolver=lambda J, nev: krylov.ShiftInvert(0.5, hls, krylovdim=40, tol=1e-10)(J, nev))
    hbr = E.continuation(hprob, P.PALC(bls=BlsAdapter(obls.BorderingBLS(hls, check_precision=False))),
                         P.ContinuationPar(newton_options=hopts, **kw), normC=P.norminf)
    ctx = bk.Context(bk.BK_SPARSE, (S.MIT_N, S.MIT_N), (S.MIT_L, S.MIT_L), krylov_m=300)
    ctx.sparse_load(mit.J(np.zeros(N), [0.01]))
    ctx.precond_setup(bk.BK_PC_JACOBI, 0.0, 1.0)
    ls = bk.GMRESB200(reltol=1e-12, restart=300, maxiter=3000, Pl=True)
    eig = bk.ShiftInvertB200(0.5, bk.GMRESB200(reltol=1e-12, restart=300, maxiter=3000, orth="cgs2"), krylovdim=40, tol=1e-10)
    dopts = P.NewtonPar(tol=1e-9, max_iterations=20, linsolver=ls, eigsolver=eig)
    prob = P.SparseProblemB200(ctx, mit.F, mit.J, np.zeros(N), [0.01], lens=0)
    br = E.continuation(prob, P.PALC(bls=bk.BorderingBLSB200(ls, check_precision=False)), P.ContinuationPar(newton_options=dopts, **kw),
                        normC=P.norminf)
    assert len(br.rows) == len(hbr.rows) > 5
    for r, o in zip(br.rows, hbr.rows):
        assert abs(r["param"] - o["param"]) < 1e-7 and abs(r["x"] - o["x"]) < 1e-6 * max(1.0, o["x"]), (r, o)
        assert r["n_unstable"] == o["n_unstable"], (r, o)
    assert [s.type for s in br.specialpoint] == [s.type for s in hbr.specialpoint]


def _bru_device(bk, complex_ctx):
    N = 2 * S.BRU_N
    ctx = bk.Context(bk.BK_SPARSE, (N,), krylov_m=1024, complex=complex_ctx)
    return ctx


def test_brusselator_hopf_on_device(bk):
    """newton_hopf on sparse real and complex contexts gives the closed-form l_H, omega to 1e-7; a short continuation_hopf in
    beta stays on the closed-form curve l_H(beta), omega(beta) to 1e-6.  Only Jacobi preconditioning exists for this problem, so
    every solve is a near-full GMRES(1024) on 1000 / 2000 unknowns: the slowest test of the file (minutes)"""
    C2, P = bk.codim2, bk.palc
    par = list(S.BRU_PAR)
    l0 = 1.02 * S.BRU_LH
    par[S.BRU_LENS_L] = l0
    x0 = S.bru_steady(par)
    rctx, cctx = _bru_device(bk, False), _bru_device(bk, True)
    prob = P.SparseProblemB200(rctx, S.bru_F, S.bru_J, x0, par, lens=S.BRU_LENS_L)
    cprob = C2.ComplexSparseProblemB200(cctx, S.bru_J, par, lens=S.BRU_LENS_L)
    for c in (rctx, cctx):
        c.sparse_load(S.bru_J(x0, par))
        c.precond_setup(bk.BK_PC_JACOBI, 0.0, 1.0)
    ls = bk.GMRESB200(reltol=1e-12, restart=1024, maxiter=4096, Pl=True, orth="cgs2")
    cls = bk.ComplexGMRESB200(reltol=1e-10, restart=1024, maxiter=8192, Pl=True, orth="cgs2")
    ev, v, w = S.bru_eigvecs(S.bru_J(x0, par))
    hp = C2.newton_hopf(prob, cprob, x0, l0, ev.imag, v, w, P.NewtonPar(tol=1e-9, max_iterations=15, linsolver=ls), ls, cls)
    assert hp.converged, hp.residuals
    assert abs(hp.p - S.BRU_LH) < 1e-7 and abs(hp.omega - S.BRU_OMEGA) < 1e-7, (hp.p - S.BRU_LH, hp.omega - S.BRU_OMEGA)
    # Hopf curve in (l, beta), beta from 5.45 upwards
    cp = P.ContinuationPar(dsmin=1e-4, dsmax=0.2, ds=0.1, p_min=5.1, p_max=10.5, max_steps=2,
                           newton_options=P.NewtonPar(tol=1e-9, max_iterations=10, linsolver=ls))
    hpar = list(par)
    hpar[S.BRU_LENS_L] = hp.p
    prob.params, cprob.params = list(hpar), list(hpar)
    ev, v, w = S.bru_eigvecs(S.bru_J(hp.u, hpar))
    curve = C2.continuation_hopf(prob, cprob, hp.u, hp.p, hp.omega, S.BRU_LENS_BETA, v, w, cp, ls, cls)
    assert len(curve.p1) >= 3
    for l, b, om in zip(curve.p1, curve.p2, curve.omega):
        lh, omh = S.bru_hopf(beta=b)
        assert abs(l - lh) < 1e-6 and abs(om - omh) < 1e-6, (b, l - lh, om - omh)


def test_errors_are_reported_not_faults(bk):
    n = 10
    ctx = bk.Context(bk.BK_SPARSE, (n,), krylov_m=4)
    with pytest.raises(bk.BK200Error, match="set_pattern"):
        ctx.jvp(np.ones(n))
    with pytest.raises(bk.BK200Error, match="residual"):
        ctx.residual(np.ones(n))
    ok = sp.identity(n, format="csr")
    bad = [("csr", 0, np.arange(n + 1) + 1, np.arange(n)),                               # ptr[0] != base
           ("csr", 0, np.r_[0, 2, 1, np.arange(3, n + 1)], np.arange(n)),               # not monotone
           ("csr", 0, np.arange(n + 1), np.r_[np.arange(n - 1), n]),                    # index out of range
           ("csc", 1, np.arange(n + 1) + 1, np.arange(n)),                              # 0 is out of range in base 1
           ("csr", 0, np.arange(n + 1), np.arange(n + 1))]                              # ptr[N] != nnz
    for A in bad:
        with pytest.raises(bk.BK200Error, match="bk_sparse_set_pattern"):
            ctx.sparse_pattern(A)
    ctx.sparse_load(ok)
    assert np.array_equal(ctx.jvp(np.arange(n, dtype=float)), np.arange(n, dtype=float))
    with pytest.raises(bk.BK200Error, match="zero pivot"):
        ctx.precond_setup(bk.BK_PC_JACOBI, 1.0, -1.0)
    ctx.precond_setup(bk.BK_PC_JACOBI, 0.0, 1.0)
    ctx.sparse_values(np.r_[0.0, np.ones(n - 1)])
    with pytest.raises(bk.BK200Error, match="zero pivot"):
        ctx.precond_apply(np.ones(n))
    with pytest.raises(bk.BK200Error, match="grid"):
        ctx.precond_setup(bk.BK_PC_SH_DCT, 1.0)
    named = bk.Context(bk.BK_SH2D, (16, 16), (1.0, 1.0), krylov_m=4, params=(-0.1, 1.3))
    with pytest.raises(bk.BK200Error, match="BK_SPARSE"):
        named.precond_setup(bk.BK_PC_JACOBI, 0.0, 1.0)
    with pytest.raises(bk.BK200Error, match="BK_SPARSE"):
        named.sparse_pattern(ok)
    # the native loop needs the library's own residual
    P = bk.palc
    ls = bk.GMRESB200(reltol=1e-8, restart=4, maxiter=4)
    prob = P.SparseProblemB200(ctx, lambda x, q: x, lambda x, q: ok, np.ones(n), [0.0], lens=0)
    with pytest.raises(bk.BK200Error, match="bk_palc_run"):
        P.continuation_native(prob, P.PALC(bls=bk.BorderingBLSB200(ls)), P.ContinuationPar(newton_options=P.NewtonPar(linsolver=ls)))
    ctx.sparse_values(np.ones(n))
    assert np.array_equal(ctx.jvp(np.ones(n)), np.ones(n))   # the context is still usable
