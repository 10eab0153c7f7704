"""Host side of the hot path: Newton, newton_palc and the PALC continuation loop, driving the device
kernels through the plugin mirror in core.py.  In the reference this layer is Julia and stays Julia
(src/Newton.jl:66-114, src/continuation/Palc.jl:112-305, src/Continuation.jl:349-504, 506-601,
src/continuation/Contbase.jl:69-102, src/continuation/Tangents.jl:8-42,71-104,
src/continuation/Natural.jl:36-58); it is restated here because no Julia toolchain exists in this image
(julia/BK200.jl is the adapter a maintainer would load instead).

The state vector is either a ``DeviceVec`` (device-resident, "option B") or a NumPy array (host
buffers crossing the C ABI on every call, "option A"): the loop below is written against the small
vector interface ``V`` and never touches elements.
"""
from dataclasses import dataclass, field
import math

import numpy as np

from scipy.linalg import blas as _blas

from .core import DeviceVec, Jacobian

SQRT_EPS = math.sqrt(np.finfo(np.float64).eps)  # src/Problems.jl:69


def _obj(x):
    """vectors that carry their own method set (DeviceVec; codim2.BorderedVec = BorderedArray(u, p)) vs plain ndarrays"""
    return not isinstance(x, np.ndarray)


class V:
    """VectorInterface subset (src/BorderedArrays.jl:86-217) for DeviceVec, BorderedVec and ndarray."""
    host_alloc = None  # optional n -> ndarray factory (e.g. Context.pinned_empty) for host-resident state

    @staticmethod
    def copy(x):
        if _obj(x) or V.host_alloc is None:
            return x.copy()
        y = V.host_alloc(len(x))
        y[...] = x
        return y

    @staticmethod
    def copyto(dst, src):
        if _obj(dst):
            dst.copyto(src)
        else:
            dst[...] = src
        return dst

    @staticmethod
    def axpby(y, a, x, b=1.0):
        """y <- a x + b y (VI.add!)"""
        if _obj(y):
            return y.axpby_(a, x, b)
        if b != 1.0:
            _blas.dscal(b, y)
        _blas.daxpy(x, y, a=a)  # in place (threaded BLAS-1, no temporaries)
        return y

    @staticmethod
    def scale(x, a):
        """x <- a x (VI.scale!)"""
        if _obj(x):
            return x.scale_(a)
        _blas.dscal(a, x)
        return x

    @staticmethod
    def dot(x, y):
        return x.dot(y) if _obj(x) else float(np.dot(x, y))

    _scratch = {}  # host path: one reusable buffer per vector length (an 8 MB temporary per call costs ~1 ms of page faults)

    @staticmethod
    def diffdot(x, x0, tau):
        if _obj(x):
            return x.diffdot(x0, tau)
        buf = V._scratch.get(len(x))
        if buf is None:
            buf = V._scratch[len(x)] = np.empty(len(x))
        return float(np.dot(np.subtract(x, x0, out=buf), tau))

    @staticmethod
    def norm2(x):
        return x.norm() if _obj(x) else float(np.linalg.norm(x))

    @staticmethod
    def norminf(x):
        if _obj(x):
            return x.norminf()  # NaN-propagating on the device (k_reduce MODE 1)
        return nanmax2(float(np.max(x)), -float(np.min(x)))  # = max|x|, no temporary; NaN if any entry is NaN

    @staticmethod
    def zeros_like(x):
        if _obj(x):
            return x.copy().zero_()
        if V.host_alloc is None:
            return np.zeros_like(x)
        y = V.host_alloc(len(x))
        y[...] = 0.0
        return y


def nanmax2(a, b):
    """max that propagates NaN like Julia's norm(x, Inf) / max: Python's max(0.0, nan) is 0.0, which would let a NaN
    iterate pass `res < tol` as converged (the reference rejects the step, src/continuation/Palc.jl:228-231)."""
    return max(a, b) if (a == a and b == b) else math.nan


norminf = V.norminf
norm2 = V.norm2


@dataclass
class NewtonPar:
    """src/Newton.jl:17-33"""
    tol: float = 1e-10
    max_iterations: int = 25
    linsolver: object = None
    eigsolver: object = None


@dataclass
class ContinuationPar:
    """src/ContParameters.jl:44-100 (fields the hot path reads)"""
    dsmin: float = 1e-4
    dsmax: float = 1e-1
    ds: float = 1e-2
    a: float = 0.5
    p_min: float = -1.0
    p_max: float = 1.0
    max_steps: int = 400
    newton_options: NewtonPar = field(default_factory=NewtonPar)
    eta: float = 150.0
    nev: int = 3
    detect_bifurcation: int = 0
    tol_stability: float = 1e-10
    # events.py (SURVEY 8f.2): fold detection by parameter monotony and bisection on the number of unstable eigenvalues
    detect_fold: bool = True
    n_inversion: int = 2
    max_bisection_steps: int = 25
    dsmin_bisection: float = 1e-16
    tol_bisection_eigenvalue: float = 1e-16


@dataclass
class PALC:
    """src/continuation/Palc.jl:70-84"""
    tangent: str = "secant"
    theta: float = 0.5
    bls: object = None


class BifurcationProblemB200:
    """BifurcationProblem whose F and J are the context's device kernels; `lens` = index of the
    continuation parameter inside the context's parameter tuple (the @optic of the reference)."""

    def __init__(self, ctx, u0, params, lens=0, record=None, delta=SQRT_EPS):
        self.ctx, self.u0, self.params, self.lens, self.delta = ctx, u0, list(params), lens, delta
        self.p0 = float(params[lens])
        self.record = record or V.norm2  # record_from_solution default = norm(x) (src/Problems.jl:286)

    def _set(self, p):
        q = list(self.params)
        q[self.lens] = p
        self.ctx.set_params(q)

    def F(self, x, p, out=None):
        self._set(p)
        return self.ctx.residual(x, out)

    def J(self, x, p):
        self._set(p)
        return self.ctx.jacobian(x)


def _host(x):
    """a state as a NumPy array (the user functions of SparseProblemB200 are host code)"""
    return x.numpy() if isinstance(x, DeviceVec) else x


class SparseProblemB200(BifurcationProblemB200):
    """BifurcationProblem(F, u0, params, lens; J) of a user's own problem on a BK_SPARSE context (examples/brusselator.jl:86-93,
    J = Jbru_sp): F(x, par) -> residual and J(x, par) -> scipy CSR / CSC matrix (or the values of the pattern already loaded), both
    host functions of a NumPy state and the parameter list `par` (params with par[lens] = p).  J uploads the values and returns
    the context's Jacobian, so GMRESB200, the bordered solvers and ShiftInvertB200 run on the device SpMV; the pattern is re-set
    when it changes (indptr / indices compared on every call unless check_pattern is False, then only the first is loaded)."""

    def __init__(self, ctx, F, J, u0, params, lens=0, record=None, delta=SQRT_EPS, check_pattern=True):
        super().__init__(ctx, u0, params, lens, record, delta)
        self.F_, self.J_, self.check_pattern = F, J, check_pattern

    def _par(self, p):
        q = list(self.params)
        q[self.lens] = p
        return q

    def F(self, x, p, out=None):
        r = np.ascontiguousarray(self.F_(_host(x), self._par(p)), dtype=np.float64)
        if out is None:
            return self.ctx.to_device(r) if isinstance(x, DeviceVec) else r
        if isinstance(out, DeviceVec):
            out.copyto(self.ctx.to_device(r))
        else:
            out[...] = r
        return out

    def J(self, x, p):
        self._set(p)
        self.ctx.sparse_load(self.J_(_host(x), self._par(p)), self.check_pattern)
        return Jacobian(self.ctx)


@dataclass
class NonLinearSolution:
    u: object
    p: float
    residuals: list
    converged: bool
    itnewton: int
    itlineartot: int


def newton(prob, x0, p, opts, normN=V.norm2):
    """src/Newton.jl:66-114"""
    x = V.copy(x0)
    fx = prob.F(x, p)
    res = normN(fx)
    residuals = [res]
    step = itlin = 0
    while step < opts.max_iterations and res > opts.tol:
        J = prob.J(x, p)
        u, cv, it = opts.linsolver(J, fx)
        itlin += int(np.sum(it))
        V.axpby(x, -1.0, u, 1.0)  # minus!!(x, u)
        fx = prob.F(x, p, out=fx)
        res = normN(fx)
        residuals.append(res)
        step += 1
    return NonLinearSolution(x, p, residuals, residuals[-1] < opts.tol, step, itlin)


def _dot_theta(u1, u2, p1, p2, theta):
    return V.dot(u1, u2) / len(u1) * theta + p1 * p2 * (1.0 - theta)


def solve_bls_palc(bls, theta, tau_u, tau_p, J, dR, R, n):
    """src/LinearBorderSolver.jl:16-36: xiu = theta, xip = 1 - theta, dotp = dot / N"""
    return bls(J, dR, tau_u, tau_p, R, n, theta, 1.0 - theta, shift=None, dotscale=1.0 / len(R))


def newton_palc(prob, z0u, z0p, tau_u, tau_p, zpred_u, zpred_p, ds, theta, contpar, bls, normN=V.norm2):
    """src/continuation/Palc.jl:187-305 (linesearch = false)."""
    opts = contpar.newton_options
    eps = prob.delta
    N = len(z0u)

    def Nfun(u, p):  # arc_length_eq, Palc.jl:44-56
        return theta * V.diffdot(u, z0u, tau_u) / N + (1.0 - theta) * (p - z0p) * tau_p - ds

    x = V.copy(zpred_u)
    p = zpred_p
    res_f = prob.F(x, p)
    res_n = Nfun(x, p)
    dFdp = V.zeros_like(x)
    res = nanmax2(normN(res_f), abs(res_n))
    residuals = [res]
    step = itlin = 0
    while step < opts.max_iterations and res > opts.tol:
        dFdp = prob.F(x, p + eps, out=dFdp)
        V.axpby(dFdp, -1.0 / eps, res_f, 1.0 / eps)  # (F(x,p+eps) - F(x,p)) / eps
        J = prob.J(x, p)
        u, up, flag, it = solve_bls_palc(bls, theta, tau_u, tau_p, J, dFdp, res_f, res_n)
        itlin += int(np.sum(it))
        V.axpby(x, -1.0, u, 1.0)
        p = min(max(p - up, contpar.p_min), contpar.p_max)
        res_f = prob.F(x, p, out=res_f)
        res_n = Nfun(x, p)
        res = nanmax2(normN(res_f), abs(res_n))
        residuals.append(res)
        step += 1
    return NonLinearSolution(x, p, residuals, residuals[-1] < opts.tol, step, itlin)


def step_size_control(ds, converged, itnewton, contpar):
    """src/continuation/Contbase.jl:77-102"""
    if not converged:
        if abs(ds) <= contpar.dsmin:
            return ds, True
        dsnew = math.copysign(max(abs(ds) / 2, contpar.dsmin), ds)
    else:
        Nmax = contpar.newton_options.max_iterations
        factor = (Nmax - itnewton) / Nmax
        dsnew = ds * (1 + contpar.a * (factor * factor))  # factor^2 is a literal power in Julia: x * x
    dsnew = math.copysign(min(max(abs(dsnew), contpar.dsmin), contpar.dsmax), dsnew)
    return dsnew, False


@dataclass
class ContState:
    z_u: object
    z_p: float
    zold_u: object
    zold_p: float
    tau_u: object
    tau_p: float
    zpred_u: object
    zpred_p: float
    ds: float
    step: int = 0
    converged: bool = True
    itnewton: int = 0
    itlinear: int = 0
    stop: bool = False
    n_unstable: tuple = (-1, -1)
    eigvals: object = None
    nfail: int = 0
    work_newton: int = 0
    work_linear: int = 0
    n_imag: tuple = (-1, -1)       # events.py: unstable eigenvalues with nonzero imaginary part (current, previous)
    stepsizecontrol: bool = True   # events.py: switched off inside the bisection
    in_bisection: bool = False


def _secant(st, theta):
    """src/continuation/Tangents.jl:28-42: tau = (z - z_old) * sign(ds) / ||.||_theta (in place)"""
    V.copyto(st.tau_u, st.z_u)
    V.axpby(st.tau_u, -1.0, st.zold_u, 1.0)
    st.tau_p = st.z_p - st.zold_p
    alpha = math.copysign(1.0, st.ds) / math.sqrt(_dot_theta(st.tau_u, st.tau_u, st.tau_p, st.tau_p, theta))
    V.scale(st.tau_u, alpha)
    st.tau_p *= alpha


def _bordered_tangent(prob, st, theta, bls):
    """src/continuation/Tangents.jl:71-104"""
    eps = prob.delta
    dFdl = prob.F(st.z_u, st.z_p + eps)
    f0 = prob.F(st.z_u, st.z_p)
    V.axpby(dFdl, -1.0 / eps, f0, 1.0 / eps)
    J = prob.J(st.z_u, st.z_p)
    tu, tp, flag, it = solve_bls_palc(bls, theta, st.tau_u, st.tau_p, J, dFdl, V.zeros_like(st.z_u), 1.0)
    alpha = 1.0 / math.sqrt(_dot_theta(tu, tu, tp, tp, theta))
    alpha *= math.copysign(1.0, _dot_theta(st.tau_u, tu, st.tau_p, tp, theta))
    V.copyto(st.tau_u, tu)
    V.scale(st.tau_u, alpha)
    st.tau_p = tp * alpha


def _predict(st):
    """addtangent! (src/continuation/Tangents.jl:8-15): z_pred = z + ds * tau"""
    V.copyto(st.zpred_u, st.z_u)
    V.axpby(st.zpred_u, st.ds, st.tau_u, 1.0)
    st.zpred_p = st.z_p + st.ds * st.tau_p


def continuation(prob, alg, contpar, normC=V.norm2, u1=None, p1=None, verbose=False, callback=None):
    """src/Continuation.jl:349-504,506-601.  Returns (rows, state); rows mirror ContResult.branch
    (param, x = record_from_solution, itnewton, itlinear, ds, step, n_unstable; src/Continuation.jl:259-272).
    With (u1, p1) the branch starts from two points (iterate_from_two_points, :408-456) -- used to seed
    branch segments on other GPUs."""
    opts = contpar.newton_options
    theta, bls = alg.theta, alg.bls
    p0 = prob.p0
    if u1 is None:
        assert contpar.p_min <= p0 <= contpar.p_max
        sol0 = newton(prob, prob.u0, p0, opts, normC)
        if not sol0.converged:
            raise RuntimeError(f"Newton failed to converge for the initial guess: {sol0.residuals}")
        p1 = p0 + contpar.ds / contpar.eta
        sol1 = newton(prob, sol0.u, p1, opts, normC)
        if not sol1.converged:
            raise RuntimeError("Newton failed to converge for the initial tangent")
        u0, u1 = sol0.u, sol1.u
    else:
        u0 = V.copy(prob.u0)
    # state.z = z1, z_old = z0 -> secant tangent; then z <- z0 (initialize!, Palc.jl:112-123)
    st = ContState(z_u=u1, z_p=p1, zold_u=u0, zold_p=p0, tau_u=V.zeros_like(u0), tau_p=0.0,
                   zpred_u=V.zeros_like(u0), zpred_p=0.0, ds=contpar.ds)
    _secant(st, theta)
    st.z_u, st.z_p = V.copy(u0), p0
    _predict(st)
    rows = []

    def eig_update():
        if contpar.detect_bifurcation > 0 and opts.eigsolver is not None:
            nprev = st.n_unstable[1]
            nev_ = max(nprev + 5, contpar.nev) if nprev >= 0 else contpar.nev  # src/Utils.jl:78-79
            J = prob.J(st.z_u, st.z_p)
            vals = opts.eigsolver(J, nev_)[0]
            nun = int(np.sum(np.real(vals) > contpar.tol_stability))  # src/Bifurcations.jl:5-18
            st.n_unstable = (nun, st.n_unstable[0])
            st.eigvals = vals

    def save():
        rows.append(dict(param=st.z_p, x=prob.record(st.z_u), itnewton=st.itnewton, itlinear=st.itlinear,
                         ds=st.ds, step=st.step, n_unstable=st.n_unstable[0]))

    eig_update()
    save()
    if callback is not None and callback(st) is False:  # step 0 (lets callers mark the start of the continuation! loop)
        st.stop = True

    def done():  # src/Continuation.jl:254-257
        return (st.step <= contpar.max_steps) and ((contpar.p_min < st.z_p < contpar.p_max) or st.step == 0) and not st.stop

    first = True
    while True:
        if not first and st.converged and st.step <= contpar.max_steps and st.step > 0:
            save()
            if callback is not None and callback(st) is False:
                st.stop = True
        first = False
        if not done():
            break
        if st.zpred_p <= contpar.p_min or st.zpred_p >= contpar.p_max:  # Palc.jl:157-160 -> Natural corrector
            st.zpred_p = min(max(st.zpred_p, contpar.p_min), contpar.p_max)
            sol = newton(prob, st.zpred_u, st.zpred_p, opts, normC)
            sol.p = st.zpred_p
        else:
            sol = newton_palc(prob, st.z_u, st.z_p, st.tau_u, st.tau_p, st.zpred_u, st.zpred_p, st.ds, theta, contpar,
                              bls, normC)
        st.converged, st.itnewton, st.itlinear = sol.converged, sol.itnewton, sol.itlineartot
        st.work_newton += sol.itnewton      # all corrector work, including rejected attempts
        st.work_linear += sol.itlineartot
        st.nfail += 0 if sol.converged else 1
        if sol.converged:
            st.zold_u, st.z_u = st.z_u, st.zold_u  # swap buffers: z_old <- z
            st.zold_p = st.z_p
            V.copyto(st.z_u, sol.u)
            st.z_p = sol.p
            eig_update()
            st.step += 1
        if verbose:
            print(f"step {st.step} p={st.z_p:.6e} ds={st.ds:.3e} conv={st.converged} itn={st.itnewton} itl={st.itlinear}",
                  flush=True)
        if not st.stop:
            st.ds, st.stop = step_size_control(st.ds, st.converged, st.itnewton, contpar)
        if st.converged:
            if alg.tangent == "secant":
                _secant(st, theta)
            else:
                _bordered_tangent(prob, st, theta, bls)
        _predict(st)
    return rows, st


def continuation_native(prob, alg, contpar, normC=V.norm2, u1=None, p1=None, callback=None, max_rows=None):
    """The same branch through ONE C-ABI call: bk_palc_run (include/bk200.h; the loop above restated as host C++ inside
    libbk200.so, csrc/bk_palc_loop.hpp) -- same kernels in the same order, so the rows are bit-identical to `continuation`
    with a device-resident state; what disappears is the host-language dispatch between the kernels (a dozen ABI crossings and
    a few allocations per Newton iteration).  `prob.u0` / `u1` may be NumPy arrays (uploaded once) or DeviceVecs.
    detect_bifurcation = 0 only.  `callback(step, row_dict, z_u_device_pointer, z_p)` -> False stops the run.
    Returns (rows, info): rows as `continuation`, info = dict(steps, nfail, stopped, work_newton, work_linear, p, ds, u)."""
    import ctypes as C
    from . import lib as _l
    from .core import _chk, BorderingBLSB200, MatrixFreeBLSB200
    ctx = prob.ctx
    assert contpar.detect_bifurcation == 0 or contpar.newton_options.eigsolver is None, "bk_palc_run: no eigen-solve per step"
    assert normC in (V.norm2, V.norminf), "bk_palc_run: normC is norm or norminf"
    bls = alg.bls
    assert isinstance(bls, (BorderingBLSB200, MatrixFreeBLSB200)), "bk_palc_run: bls must be one of the library's bordered solvers"
    ls = contpar.newton_options.linsolver
    bord = isinstance(bls, BorderingBLSB200)
    po = _l.PalcOpts(ds=contpar.ds, dsmin=contpar.dsmin, dsmax=contpar.dsmax, a=contpar.a, p_min=contpar.p_min, p_max=contpar.p_max,
                     theta=alg.theta, eta=contpar.eta, newton_tol=contpar.newton_options.tol, fd_eps=prob.delta,
                     bls_tol=bls.tol if bord else 0.0, max_steps=contpar.max_steps, newton_maxit=contpar.newton_options.max_iterations,
                     lens=prob.lens, tangent=0 if alg.tangent == "secant" else 1, bls=1 if bord else 0,
                     bls_check_precision=int(bls.check_precision) if bord else 0, bls_k=bls.k if bord else 1,
                     normc=1 if normC is V.norminf else 0)
    go = (bls.solver or ls).opts()  # PALC hands the Newton linear solver to a bordered solver built without one (Palc.jl:100-110)
    go_newton = ls.opts()
    assert bytes(go) == bytes(go_newton), "bk_palc_run: one linear solver for the start-up Newton solves and the bordered solver"
    ctx.set_params(prob.params)
    max_rows = max_rows or contpar.max_steps + 8
    rows = np.zeros((max_rows, _l.BK_PALC_ROW))
    res = _l.PalcResult()
    uf = DeviceVec(ctx, ctx.N)
    as_row = lambda r: dict(param=r[0], x=r[1], itnewton=int(r[2]), itlinear=int(r[3]), ds=r[4], step=int(r[5]), n_unstable=-1)

    def thunk(user, step, row, z_u, z_p):
        r = np.ctypeslib.as_array(row, shape=(_l.BK_PALC_ROW,))
        return 0 if callback(step, as_row(r), z_u, z_p) is False else 1

    cb = _l.PalcCallback(thunk) if callback is not None else _l.PalcCallback()  # no-argument form = NULL
    st = ctx.lib.bk_palc_run(ctx.handle, C.byref(po), C.byref(go), _l.ptr(prob.u0), float(prob.p0), _l.ptr(u1),
                             0.0 if p1 is None else float(p1), rows.ctypes.data_as(C.POINTER(C.c_double)), max_rows, cb, None,
                             uf.dptr, C.byref(res))
    if st == -3:  # BK_ERR_STATE: the reference throws here (src/Continuation.jl:375-393)
        raise RuntimeError("bk_palc_run: " + ctx.lib.bk_last_error(ctx.handle).decode())
    _chk(ctx, st)
    info = dict(steps=res.steps, nfail=res.nfail, stopped=res.stopped, work_newton=res.work_newton, work_linear=res.work_linear,
                p=res.p_final, ds=res.ds_final, u=uf)
    return [as_row(r) for r in rows[: res.nrows]], info
