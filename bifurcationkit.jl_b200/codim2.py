"""SURVEY section 8f.3: Fold and Hopf points by the minimally augmented (MA) formulation, as host orchestration over the
same C ABI -- every linear solve is a (bordered) solve through `bk_bls_*` / `bk_gmres`, every operator application a `bk_jvp`.

Mirror of src/codim2/MinAugFold.jl:
  FoldMinAug.residual      <->  (F::FoldMinimallyAugmentedFormulation)(x, p, params)            :15-39
  FoldMinAug.bordered_terms <-> _compute_bordered_vectors / _get_bordered_terms                   :55-104
  FoldMinAug.solve         <->  foldMALinearSolver, finite-difference branch (usehessian = false) :122-146
  newton_fold              <->  newton_fold(prob, foldpointguess, par, eigenvec, eigenvec_ad, options; bdlinsolver)  :201-222
Swift-Hohenberg is self-adjoint (is_symmetric = true, examples/SH3d.jl:123), so J' = J and no adjoint kernel is needed (for
the Chan problem J' = J only up to the two boundary rows: the left null vector, hence sigma_x and sigma_p, are then approximate
and Newton on the MA system degrades to a quasi-Newton iteration that still converges to the same fold).

Mirror of src/codim2/MinAugHopf.jl:
  HopfMinAug.residual       <->  (H::HopfMinimallyAugmentedFormulation)(x, p, omega, params)      :19-40
  HopfMinAug.bordered_terms <->  __compute_bordered_vectors / _get_bordered_terms                 :59-104
  HopfMinAug.solve          <->  _hopf_MA_linear_solver, finite-difference branch                 :122-188
  newton_hopf               <->  newton_hopf(prob, hopfpointguess, par, eigenvec, eigenvec_ad, options)  :258-283
The complex shifts (J - i omega, (J - i omega)^H = J' + i omega) are solved on a BK_COMPLEX context (include/bk200.h): split
complex vectors, GMRES on the real-equivalent system, J' from bk_jac_set_transpose.  The complex bordered systems
[A a; b^H 0] are eliminated by bordering on the host (one complex solve each, since their right-hand side is (0, 1));
complex vectors are NumPy arrays (a Hopf refinement is a handful of solves, not a hot loop), real ones keep their container.
"""
from dataclasses import dataclass
import math

import numpy as np

from .palc import V


def _apply(J, v):
    """apply(J, v) (src/Utils.jl:192): J may be a callable Jacobian object or a matrix"""
    return J(v) if callable(J) else J @ v


@dataclass
class FoldSolution:
    u: object
    p: float
    residuals: list
    converged: bool
    itnewton: int
    itlinear: int
    sigma: float


class FoldMinAug:
    """[F(x, p); sigma(x, p)] with sigma from  [J a; b' 0] [v; sigma] = [0; 1]  (Govaerts 2000: a ~ left, b ~ right null vector)."""

    def __init__(self, prob, a, b, bls, symmetric=True, norm=V.norm2):
        assert symmetric or hasattr(prob, "Jt"), "non-symmetric problem: prob.Jt(x, p) (jacobian_adjoint) is required"
        self.prob, self.a, self.b, self.bls, self.symmetric, self.norm = prob, V.copy(a), V.copy(b), bls, symmetric, norm
        self.zero = V.zeros_like(a)
        self.itlinear = 0
        self.BT, self.CP = 1.0, 1.0  # test functions of the Bogdanov-Takens / cusp events (MinAugFold.jl:421-423, 551-575)

    def _Jt(self, x, p):
        """jacobian_adjoint(prob, x, p) (has_adjoint) -- J itself for a self-adjoint problem (is_symmetric, MinAugFold.jl:96-100)"""
        return self.prob.J(x, p) if self.symmetric else self.prob.Jt(x, p)

    def _border(self, J, a, b):
        """linbdsolver(J, a, b, 0, zero, 1) -> (v, sigma): J v + a sigma = 0, <b, v> = 1"""
        v, sig, cv, it = self.bls(J, a, b, 0.0, self.zero, 1.0)
        self.itlinear += int(np.sum(it))
        return v, sig

    def residual(self, x, p):
        J = self.prob.J(x, p)
        _, sigma = self._border(J, self.a, self.b)
        return self.prob.F(x, p), sigma

    def bordered_terms(self, x, p):
        prob = self.prob
        eps = prob.delta
        J = prob.J(x, p)
        v, _ = self._border(J, self.a, self.b)
        w, _ = self._border(J if self.symmetric else self._Jt(x, p), self.b, self.a)   # adjoint system J' w + b sigma2 = 0, <a, w> = 1
        # d_p F and sigma_p = -<w, d_p(J v)> by centred differences (MinAugFold.jl:92-101)
        dpF = prob.F(x, p + eps)
        V.axpby(dpF, -1.0 / (2 * eps), prob.F(x, p - eps), 1.0 / (2 * eps))
        jp = _apply(prob.J(x, p + eps), v)
        jm = _apply(prob.J(x, p - eps), v)
        V.axpby(jp, -1.0 / (2 * eps), jm, 1.0 / (2 * eps))
        sigma_p = -V.dot(w, jp)
        return v, w, dpF, sigma_p

    def solve(self, x, p, rhsu, rhsp, cache=None):
        """foldMALinearSolver: [J d_pF; sigma_x' sigma_p] [dX; dp] = [rhsu; rhsp] with
        sigma_x = (J'(x) w - J'(x + eps v) w) / eps  (MinAugFold.jl:135-141).  `cache`: an object whose `.terms` keeps
        (d_pF, sigma_x, sigma_p) between the right-hand sides solved at the same (x, p)."""
        prob = self.prob
        eps = prob.delta
        if cache is not None and cache.terms is not None:
            dpF, sigma_x, sigma_p = cache.terms
        else:
            v, w, dpF, sigma_p = self.bordered_terms(x, p)
            xs = V.copy(x)
            V.axpby(xs, eps, v, 1.0)
            u1 = _apply(self._Jt(xs, p), w)
            sigma_x = _apply(self._Jt(x, p), w)
            V.axpby(sigma_x, -1.0 / eps, u1, 1.0 / eps)  # (u2 - u1) / eps
            if cache is not None:
                cache.terms = (dpF, sigma_x, sigma_p)
        J = prob.J(x, p)                                 # back to the linearisation at x (one state per context)
        dX, dp, cv, it = self.bls(J, dpF, sigma_x, sigma_p, rhsu, rhsp)
        self.itlinear += int(np.sum(it))
        return dX, dp, cv

    def update(self, x, p, keep_borders=False):
        """update!(probma, iter, state) (MinAugFold.jl:276-309) and test_bt_cusp (:551-575): after an accepted step the border
        vectors follow the null vectors, a <- w / ||w||, b <- v / ||v||; BT = <w / ||w||, v / ||v||>.  keep_borders: only the
        test function (inside an event bisection the reference leaves a, b alone, :287-289)."""
        J = self.prob.J(x, p)
        v, _ = self._border(J, self.a, self.b)
        w, _ = self._border(J if self.symmetric else self._Jt(x, p), self.b, self.a)
        V.scale(v, 1.0 / self.norm(v))
        V.scale(w, 1.0 / self.norm(w))
        if not keep_borders:
            V.copyto(self.a, w)
            V.copyto(self.b, v)
        self.BT = V.dot(w, v)
        return self.BT


def newton_fold(prob, x0, p0, eigenvec, eigenvec_ad, opts, bls, normN=V.norm2, symmetric=True):
    """Newton on the MA system from the guess (x0, p0) with guesses for the right / left null vectors
    (newton_fold, MinAugFold.jl:201-222 + src/Newton.jl:66-114 on the bordered state)."""
    ma = FoldMinAug(prob, eigenvec_ad, eigenvec, bls, symmetric=symmetric)
    x, p = V.copy(x0), float(p0)
    F, sigma = ma.residual(x, p)
    res = math.hypot(normN(F), abs(sigma))
    residuals = [res]
    step = 0
    while step < opts.max_iterations and res > opts.tol:
        dX, dp, _ = ma.solve(x, p, F, sigma)
        V.axpby(x, -1.0, dX, 1.0)
        p -= dp
        F, sigma = ma.residual(x, p)
        res = math.hypot(normN(F), abs(sigma))
        residuals.append(res)
        step += 1
    return FoldSolution(x, p, residuals, residuals[-1] < opts.tol, step, ma.itlinear, sigma)


# ------------------------------------------------------------------------------------------------ Fold curves in two parameters
class BorderedVec:
    """BorderedArray(u, p) (src/BorderedArrays.jl:23-70, 86-217) with the method set of a DeviceVec, so that the PALC host
    loop (palc.py) runs on the state of a minimally augmented problem unchanged: (x, p1) for Folds, (x, [p1, omega]) for Hopf
    points (hopf_point, MinAugHopf.jl:13).  u is a DeviceVec or an ndarray, p a float or a short ndarray."""

    def __init__(self, u, p):
        self.u = u
        self.p = float(p) if np.ndim(p) == 0 else np.array(p, dtype=np.float64)

    def __len__(self):                 # Base.length(b) = length(b.u) + length(b.p)   (:49-50)
        return len(self.u) + int(np.size(self.p))

    def copy(self):
        return BorderedVec(V.copy(self.u), self.p)

    def copyto(self, src):
        V.copyto(self.u, src.u)
        self.p = src.p if np.ndim(src.p) == 0 else src.p.copy()
        return self

    def zero_(self):                   # VI.zerovector!: exact zeros (0 * NaN would stay NaN)
        if hasattr(self.u, "zero_"):
            self.u.zero_()
        else:
            self.u[...] = 0.0
        self.p = 0.0 if np.ndim(self.p) == 0 else np.zeros_like(self.p)
        return self

    def scale_(self, a):
        V.scale(self.u, a)
        self.p = self.p * a
        return self

    def axpby_(self, a, x, b=1.0):     # VI.add!(y, x, a, b)
        V.axpby(self.u, a, x.u, b)
        self.p = a * x.p + b * self.p
        return self

    def dot(self, y):                  # VI.inner(a, b) = inner(a.u, b.u) + inner(a.p, b.p)   (:53)
        return V.dot(self.u, y.u) + float(np.sum(self.p * y.p))

    def norm(self):                    # :55-58
        return math.sqrt(V.norm2(self.u) ** 2 + float(np.sum(self.p * self.p)))

    def norminf(self):                 # :62
        from .palc import nanmax2
        return nanmax2(V.norminf(self.u), float(np.max(np.abs(self.p))))

    def diffdot(self, x0, tau):
        return V.diffdot(self.u, x0.u, tau.u) + float(np.sum((self.p - x0.p) * tau.p))


class _FoldMAJacobian:
    """jacobian(FoldMAProblem{MinAug}, z, p2): a handle on (x, p1, p2); the bordered terms are computed once per handle and
    shared by the right-hand sides BorderingBLS solves with it (the reference recomputes them per right-hand side)."""

    def __init__(self, pb, z, p2):
        self.pb, self.z, self.p2, self.terms = pb, z, p2, None


class FoldLinearSolverMinAug:
    """(foldl::FoldLinearSolverMinAug)(Jfold, rhs) -> (sol, converged, iters)   (MinAugFold.jl:148-163)"""

    def __call__(self, Jma, rhs):
        pb, ma = Jma.pb, Jma.pb.ma
        pb._set2(Jma.p2)
        it0 = ma.itlinear
        dX, dp, cv = ma.solve(Jma.z.u, Jma.z.p, rhs.u, rhs.p, cache=Jma)
        return BorderedVec(dX, dp), cv, ma.itlinear - it0


class FoldMAProblem:
    """FoldMAProblem: the minimally augmented Fold system [F(x, p1, p2); sigma(x, p1, p2)] as a problem in the state
    z = (x, p1) with continuation parameter p2 = params[lens2] (continuation_fold, MinAugFold.jl:366-452)."""

    def __init__(self, ma, lens2, z0, record=None):
        assert lens2 != ma.prob.lens, "Please choose 2 different parameters."
        self.ma, self.lens2, self.u0 = ma, lens2, z0
        self.p0 = float(ma.prob.params[lens2])
        self.delta = ma.prob.delta
        self.record = record or (lambda z: z.p)   # record_from_solution of the Fold curve: (p1, p2) -- p2 is the row's param

    def _set2(self, p2):
        self.ma.prob.params[self.lens2] = p2

    def F(self, z, p2, out=None):
        self._set2(p2)
        Fu, sigma = self.ma.residual(z.u, z.p)
        if out is None:
            return BorderedVec(Fu, sigma)
        V.copyto(out.u, Fu)
        out.p = sigma
        return out

    def J(self, z, p2):
        return _FoldMAJacobian(self, z, p2)


class BorderingBLSHost:
    """BorderingBLS with check_precision = false (BEC, src/LinearBorderSolver.jl:125-144) over ANY linear solver and any vectors
    of the V interface: the `linear_algo` continuation_fold hands to PALC (MinAugFold.jl:446)."""

    def __init__(self, solver):
        self.solver = solver

    def __call__(self, J, dR, dzu, dzp, R, n, xiu=1.0, xip=1.0, shift=None, dotscale=1.0):
        assert shift is None
        x1, cv1, it1 = self.solver(J, R)
        dx, cv2, it2 = self.solver(J, dR)
        dl = (n - dotscale * V.dot(dzu, x1) * xiu) / (dzp * xip - dotscale * V.dot(dzu, dx) * xiu)
        V.axpby(x1, -dl, dx, 1.0)
        return x1, dl, bool(cv1 and cv2), (it1, it2)


@dataclass
class Codim2Point:
    """an entry of br.specialpoint on a codim-2 curve: type "bt" | "cusp", param = p2, p1, and the state of the located point"""
    type: str
    param: float
    p1: float
    step: int
    status: str      # converged | guess | guessL (locate_event!)
    interval: tuple
    x: object


def locate_event(it, _st, values_at, labels, indicator=None):
    """locate_event!(event, iter, state) (src/events/EventDetection.jl:28-235) for a ContinuousEvent whose indicator is the number of
    positive test functions (nb_signs): bisection on ds from the state `_st` just AFTER the event -- first half a step back, then
    halving, reversing at every change of the indicator -- until contpar.n_inversion reversals (or max_bisection_steps /
    dsmin_bisection).  On return `_st` holds the located state (just after the event for an even number of reversals) and its
    predictor.  values_at(st) -> tuple of test-function values at a state.  Returns (status, interval, label)."""
    from . import events as E
    from .palc import _predict
    cp = it.contpar
    nb = indicator or (lambda vals: sum(1 for v in vals if v > 0))   # nb_signs: ContinuousEvent -> number of positive values;
    if abs(_st.ds) < cp.dsmin:                                         # DiscreteEvent -> the value itself (EventDetection.jl:2-3)
        return "none", (0.0, 0.0), None
    v_after = values_at(_st)
    after, st, before = E.copy_state(_st), E.copy_state(_st), E.copy_state(_st)
    st.in_bisection = True
    before.zold_p, before.z_p = before.z_p, before.zold_p
    st.ds *= -1
    st.step = 0
    st.stepsizecontrol = False
    nsigns = [nb(v_after)]
    interval = list(E.getinterval(st.z_p, st.zold_p))
    indinterval = 0 if interval[0] == st.z_p else 1
    n_inversion, alive, vals = 0, True, v_after
    changed = None
    while True:
        if not st.converged or not alive:
            break
        prev, vals = vals, values_at(st)      # update_event!: on the first pass this is the state the bisection starts from
        nsigns.append(nb(vals))
        if nsigns[-1] == nsigns[-2]:
            st.ds /= 2                        # the event is still ahead of the current state
        else:
            st.ds /= -2                       # passed it: reverse
            n_inversion += 1
            indinterval = 1 - indinterval
            changed = [k for k, (a_, b_) in enumerate(zip(prev, vals)) if ((a_ > 0) != (b_ > 0) if indicator is None else a_ != b_)]
        _predict(st)
        E.copyto_state(after if n_inversion % 2 == 0 else before, st)
        if st.step > 0:
            interval[indinterval] = st.z_p
        if not (abs(st.ds) >= cp.dsmin_bisection and st.step < cp.max_bisection_steps and n_inversion < cp.n_inversion):
            break
        alive = it.iterate(st)
    if n_inversion % 2 == 0:
        status, src, interval = ("converged" if n_inversion >= cp.n_inversion else "guess"), st, (st.z_p, before.z_p)
    else:
        status, src, interval = "guessL", after, (st.z_p, after.z_p)
    for k in ("z_u", "zold_u", "tau_u", "zpred_u"):
        V.copyto(getattr(_st, k), getattr(src, k))
    _st.z_p, _st.zold_p, _st.tau_p, _st.zpred_p = src.z_p, src.zold_p, src.tau_p, src.zpred_p
    _st.work_newton, _st.work_linear = st.work_newton, st.work_linear
    _predict(_st)                             # update_predictor!(_state, iter) with the outer ds
    return status, E.getinterval(*interval), (labels[min(changed[0], len(labels) - 1)] if changed else None)


@dataclass
class FoldCurve:
    rows: list      # palc rows: param = p2, x = record (default p1), itnewton, itlinear, ds, step
    p1: list        # the Fold curve (p1[k], p2[k])
    p2: list
    BT: list        # test function <w / ||w||, v / ||v||> at every point: zero at a Bogdanov-Takens point (test_bt_cusp)
    CP: list        # p2-component of the tangent, getp(state.tau) (test_bt_cusp): changes sign at a cusp, where p2 is extremal along the curve
    ma: object
    state: object
    specialpoint: list = None   # Codim2Point entries (detect_event > 0)


def test_zh(eigvals, tol_stability):
    """test_zh (MinAugFold.jl:533-543): Zero-Hopf test function on a Fold curve -- the number of eigenvalues of J(x, p) to the right
    of the (numerically) zero one with a positive imaginary part; a change between two points is a "zh" event"""
    if eigvals is None:
        return 1
    ev = np.asarray(eigvals)
    rho = float(np.min(np.abs(ev.real)))
    return int(np.sum((ev.real > rho) & (ev.imag > tol_stability)))


def continuation_fold(prob, x0, p1_0, lens2, eigenvec, eigenvec_ad, contpar, bls, alg=None, normC=V.norminf, symmetric=True,
                      update_minaug_every_step=1, record=None, callback=None, detect_event=0, eigsolver=None):
    """Codim-2 continuation of a Fold point in the parameters (p1 = params[prob.lens], p2 = params[lens2]):
    continuation_fold(prob, alg, foldpointguess, par, lens1, lens2, eigenvec, eigenvec_ad, options_cont; jacobian_ma = MinAug())
    (MinAugFold.jl:366-452).  PALC on the minimally augmented system, Newton linear solver = FoldLinearSolverMinAug over the
    bordered solver `bls` (bdlinsolver: MatrixFreeBLSB200 / BorderingBLSB200 on the device), outer bordered solver =
    BorderingBLS(that solver, check_precision = false), border vectors updated after every accepted step (update!), the
    Bogdanov-Takens and cusp test functions recorded along the curve.  detect_event = 1: a change of sign of a test function
    between two points is recorded as a special point ("bt" / "cusp", the event of :428-431); = 2: it is located by the reference's
    bisection (locate_event) with contpar.n_inversion / max_bisection_steps / dsmin_bisection, and the curve goes on from the
    located state, as in the reference.  eigsolver (J, nev) -> (eigenvalues, ...): eigenvalues of J along the curve (FoldEig, :577-590;
    contpar.nev of them) for the Zero-Hopf event "zh" (DiscreteEvent(1, test_zh), :431; recorded at the point after the change)."""
    from . import palc as P
    ma = FoldMinAug(prob, eigenvec_ad, eigenvec, bls, symmetric=symmetric, norm=normC)
    z0 = BorderedVec(V.copy(x0), p1_0)
    pb = FoldMAProblem(ma, lens2, z0, record)
    fls = FoldLinearSolverMinAug()
    no = contpar.newton_options
    cp = P.ContinuationPar(**{**contpar.__dict__, "newton_options": P.NewtonPar(tol=no.tol, max_iterations=no.max_iterations, linsolver=fls),
                              "detect_bifurcation": 0})
    alg = alg or P.PALC()
    alg = P.PALC(tangent=alg.tangent, theta=alg.theta, bls=BorderingBLSHost(fls))
    curve = FoldCurve([], [], [], [], [], ma, None, [])
    from . import events as E
    it = E._Iter(pb, alg, cp, normC)
    zh_hist = []

    def values_at(s):   # test_bt_cusp at a state, the border vectors untouched
        pb._set2(s.z_p)
        return (ma.update(s.z_u.u, s.z_u.p, keep_borders=True), s.tau_p)

    def cb(st):
        pb._set2(st.z_p)
        if st.step % update_minaug_every_step == 0:
            ma.update(st.z_u.u, st.z_u.p)
        else:
            ma.update(st.z_u.u, st.z_u.p, keep_borders=True)
        vals = (ma.BT, st.tau_p)
        if eigsolver is not None:
            zh = test_zh(eigsolver(prob.J(st.z_u.u, st.z_u.p), contpar.nev)[0], contpar.tol_stability)
            if detect_event > 0 and zh_hist and st.step > 0 and zh != zh_hist[-1]:
                curve.specialpoint.append(Codim2Point("zh", st.z_p, st.z_u.p, st.step, "guess", tuple(E.getinterval(curve.p2[-1], st.z_p)),
                                                      V.copy(st.z_u.u)))
            zh_hist.append(zh)
        if detect_event > 0 and curve.BT and st.step > 0:
            prev = (curve.BT[-1], curve.CP[-1])
            flips = [k for k in range(2) if (prev[k] > 0) != (vals[k] > 0)]
            if flips:
                status, interval, label = "guess", E.getinterval(curve.p2[-1], st.z_p), ("bt", "cusp")[flips[0]]
                if detect_event > 1:
                    status, interval, lab = locate_event(it, st, values_at, ("bt", "cusp"))
                    label = lab or label
                    pb._set2(st.z_p)
                    vals = (ma.update(st.z_u.u, st.z_u.p, keep_borders=True), st.tau_p)
                if status != "none":
                    curve.specialpoint.append(Codim2Point(label, st.z_p, st.z_u.p, st.step, status, tuple(interval), V.copy(st.z_u.u)))
        curve.p1.append(st.z_u.p)
        curve.p2.append(st.z_p)
        curve.BT.append(vals[0])
        curve.CP.append(vals[1])
        return True if callback is None else callback(st)

    p2_0 = prob.params[lens2]
    try:
        curve.rows, curve.state = P.continuation(pb, alg, cp, normC=normC, callback=cb)
    finally:
        prob.params[lens2] = p2_0  # the caller's parameter tuple is left as it was
    return curve


# ------------------------------------------------------------------------------------------------ Hopf
def _np(x):
    return x.numpy() if hasattr(x, "numpy") else np.asarray(x)


def _shifted(x, eps, d):
    """x + eps d for a real state x (NumPy array or DeviceVec) and a real NumPy direction d"""
    if hasattr(x, "ctx"):
        t = x.copy()
        t.axpby_(eps, x.ctx.to_device(d), 1.0)
        return t
    return x + eps * d


class ComplexProblemB200:
    """Complexified twin of a BifurcationProblemB200: the same stencil, grid and parameters on a BK_COMPLEX context.
    J(x, p, transpose) -> callable on complex vectors, consumable by ComplexGMRESB200."""

    def __init__(self, cctx, params, lens=0):
        assert cctx.complex
        self.ctx, self.params, self.lens = cctx, list(params), lens

    def J(self, x, p, transpose=False):
        q = list(self.params)
        q[self.lens] = p
        self.ctx.set_params(q)
        return self.ctx.cjacobian(x, transpose)


class ComplexSparseProblemB200:
    """Complexified twin of a palc.SparseProblemB200 on a BK_SPARSE | BK_COMPLEX context: the same user J(x, par) (scipy CSR / CSC
    matrix or pattern values), loaded on the complex context; J(x, p, transpose) -> callable on complex vectors, consumable by
    ComplexGMRESB200, which sets the transpose flag (J') per call."""

    def __init__(self, cctx, J, params, lens=0, check_pattern=True):
        assert cctx.complex
        self.ctx, self.J_, self.params, self.lens, self.check_pattern = cctx, J, list(params), lens, check_pattern

    def J(self, x, p, transpose=False):
        from .core import ComplexJacobian
        q = list(self.params)
        q[self.lens] = p
        self.ctx.sparse_load(self.J_(_np(x), q), self.check_pattern)
        return ComplexJacobian(self.ctx, transpose)


@dataclass
class HopfSolution:
    u: object
    p: float
    omega: float
    residuals: list
    converged: bool
    itnewton: int
    itlinear: int


class HopfMinAug:
    """[F(x, p); Re sigma; Im sigma](x, p, omega) with  [J - i omega, a; b^H, 0] [v; sigma] = [0; 1]
    (a ~ null vector of (J - i omega)^H, b ~ null vector of J - i omega)."""

    def __init__(self, prob, cprob, a, b, ls, cls, cbls=None):
        self.prob, self.cprob, self.ls, self.cls, self.cbls = prob, cprob, ls, cls, cbls
        self.a, self.b = np.array(a, dtype=complex), np.array(b, dtype=complex)
        self.itlinear = 0

    def _border(self, Jc, shift, a, b):
        """(Jc + shift) v + a sigma = 0, <b, v> = 1 (linbdsolver(J, a, b, 0, zero, 1; shift), MinAugHopf.jl:17).  With a complex
        bordered solver `cbls(Jc, a, b, shift) -> (v, sigma, converged, iters)` (the reference's MatrixBLS / BorderingBLS on the
        bordered matrix, regular AT the Hopf point) that is one call; otherwise by bordering: y = (Jc + shift)^-1 a,
        sigma = -1 / <b, y>, v = -sigma y -- fine for an iterative solver next to the point, singular exactly on it."""
        if self.cbls is not None:
            v, sigma, cv, it = self.cbls(Jc, a, b, shift)
            self.itlinear += int(np.sum(it))
            return v, sigma
        y, cv, it = self.cls(Jc, a, a0=shift)
        self.itlinear += int(np.sum(it))
        sigma = -1.0 / np.vdot(b, y)
        return -sigma * y, sigma

    def residual(self, x, p, om):
        _, sigma = self._border(self.cprob.J(x, p), complex(0.0, -om), self.a, self.b)
        return self.prob.F(x, p), sigma.real, sigma.imag

    def bordered_terms(self, x, p, om):
        prob, cprob = self.prob, self.cprob
        eps = prob.delta
        v, _ = self._border(cprob.J(x, p), complex(0.0, -om), self.a, self.b)
        w, _ = self._border(cprob.J(x, p, transpose=True), complex(0.0, om), self.b, self.a)
        dpF = prob.F(x, p + eps)
        V.axpby(dpF, -1.0 / (2 * eps), prob.F(x, p - eps), 1.0 / (2 * eps))
        dpJv = (cprob.J(x, p + eps)(v) - cprob.J(x, p - eps)(v)) / (2 * eps)
        sigma_p = -np.vdot(w, dpJv)
        sigma_om = 1j * np.vdot(w, v)
        return v, w, dpF, sigma_p, sigma_om

    def solve(self, x, p, om, duu, dup, duom):
        """_hopf_MA_linear_solver: [J dpF 0; sigma_x sigma_p sigma_om] [dX; dp; dom] = [duu; dup; duom]"""
        prob, cprob = self.prob, self.cprob
        eps = prob.delta
        v, w, dpF, sigma_p, sigma_om = self.bordered_terms(x, p, om)
        x1, x2, cv, it = self.ls(prob.J(x, p), duu, dpF)
        self.itlinear += int(np.sum(it))
        cw = np.conj(w)
        u1r = cprob.J(_shifted(x, eps, np.ascontiguousarray(v.real)), p, transpose=True)(cw)
        u1i = cprob.J(_shifted(x, eps, np.ascontiguousarray(v.imag)), p, transpose=True)(cw)
        u2 = cprob.J(x, p, transpose=True)(cw)
        sigma_x = -(u1r - u2) / eps + 1j * (-(u1i - u2) / eps)
        sxx1 = np.vdot(sigma_x, _np(x1))
        sxx2 = np.vdot(sigma_x, _np(x2))
        # the inner product conjugates its first argument: hence + Im(sxx2) and + Im(sxx1) (MinAugHopf.jl:180-186)
        LS = np.array([[(sigma_p - sxx2).real, sigma_om.real], [(sigma_p + sxx2).imag, sigma_om.imag]])
        rhs = np.array([dup - sxx1.real, duom + sxx1.imag])
        dp, dom = np.linalg.solve(LS, rhs)
        V.axpby(x1, -dp, x2, 1.0)
        return x1, float(dp), float(dom), cv


def newton_hopf(prob, cprob, x0, p0, omega0, eigenvec, eigenvec_ad, opts, ls, cls, normN=V.norm2, cbls=None):
    """Newton on the Hopf MA system from (x0, p0, omega0) with guesses for the i omega eigenvector and its adjoint
    (newton_hopf, MinAugHopf.jl:258-283 + src/Newton.jl:66-114 on the state (x, [p, omega]))."""
    ma = HopfMinAug(prob, cprob, eigenvec_ad, eigenvec, ls, cls, cbls)
    x, p, om = V.copy(x0), float(p0), float(omega0)
    F, sr, si = ma.residual(x, p, om)
    res = math.sqrt(normN(F) ** 2 + sr * sr + si * si)
    residuals = [res]
    step = 0
    while step < opts.max_iterations and res > opts.tol:
        dX, dp, dom, _ = ma.solve(x, p, om, F, sr, si)
        V.axpby(x, -1.0, dX, 1.0)
        p -= dp
        om -= dom
        F, sr, si = ma.residual(x, p, om)
        res = math.sqrt(normN(F) ** 2 + sr * sr + si * si)
        residuals.append(res)
        step += 1
    return HopfSolution(x, p, om, residuals, residuals[-1] < opts.tol, step, ma.itlinear)


# ------------------------------------------------------------------------------------------------ Hopf curves in two parameters
class _HopfMAJacobian:
    def __init__(self, pb, z, p2):
        self.pb, self.z, self.p2 = pb, z, p2


class HopfLinearSolverMinAug:
    """(hopfl::HopfLinearSolverMinAug)(Jhopf, rhs) -> (sol, converged, iters)   (MinAugHopf.jl:190-205)"""

    def __call__(self, Jma, rhs):
        pb, ma = Jma.pb, Jma.pb.ma
        pb._set2(Jma.p2)
        it0 = ma.itlinear
        z = Jma.z
        dX, dp, dom, cv = ma.solve(z.u, float(z.p[0]), float(z.p[1]), V.copy(rhs.u), float(rhs.p[0]), float(rhs.p[1]))
        return BorderedVec(dX, [dp, dom]), cv, ma.itlinear - it0


class HopfMAProblem:
    """HopfMAProblem: [F(x, p1, p2); Re sigma; Im sigma] in the state z = (x, [p1, omega]) with continuation parameter
    p2 = params[lens2] (continuation_hopf, MinAugHopf.jl:425-522)."""

    def __init__(self, ma, lens2, z0, record=None):
        assert lens2 != ma.prob.lens, "Please choose 2 different parameters."
        self.ma, self.lens2, self.u0 = ma, lens2, z0
        self.p0 = float(ma.prob.params[lens2])
        self.delta = ma.prob.delta
        self.record = record or (lambda z: float(z.p[0]))

    def _set2(self, p2):
        self.ma.prob.params[self.lens2] = p2
        self.ma.cprob.params[self.lens2] = p2

    def F(self, z, p2, out=None):
        self._set2(p2)
        Fu, sr, si = self.ma.residual(z.u, float(z.p[0]), float(z.p[1]))
        if out is None:
            return BorderedVec(Fu, [sr, si])
        V.copyto(out.u, Fu)
        out.p = np.array([sr, si])
        return out

    def J(self, z, p2):
        return _HopfMAJacobian(self, z, p2)


@dataclass
class HopfCurve:
    rows: list
    p1: list        # the Hopf curve (p1[k], p2[k]) with the frequency omega[k]
    p2: list
    omega: list
    ma: object
    state: object
    stopped_at_bt: bool = False
    specialpoint: list = None   # Codim2Point entries: "zh" / "hh" (detect_event > 0 with an eigsolver)


def continuation_hopf(prob, cprob, x0, p1_0, omega0, lens2, eigenvec, eigenvec_ad, contpar, ls, cls, alg=None, normC=V.norminf,
                      update_minaug_every_step=1, record=None, callback=None, cbls=None, detect_event=0, eigsolver=None):
    """Codim-2 continuation of a Hopf point in (p1 = params[prob.lens], p2 = params[lens2]): continuation_hopf(prob, alg,
    hopfpointguess, par, lens1, lens2, eigenvec, eigenvec_ad, options_cont; jacobian_ma = MinAug()) (MinAugHopf.jl:425-522).
    PALC on the minimally augmented system in the state (x, [p1, omega]); Newton linear solver = HopfLinearSolverMinAug (one
    two-right-hand-side real solve + four complex shifted solves on the BK_COMPLEX twin `cprob`), outer bordered solver =
    BorderingBLS(that solver, check_precision = false); after every accepted step a <- w / ||w||, b <- v / ||v|| (update!,
    :323-367); the curve stops where omega -> 0 (Bogdanov-Takens, |omega| < 100 Newton tol).  With eigsolver (J, nev) -> (eigenvalues,
    ...) and detect_event > 0 the number of unstable eigenvalues of J along the curve is the reference's BifDetectEvent (:489-500,
    src/events/BifurcationDetection.jl:57-70; tol_stability raised to 10 x the Newton tolerance so that the Hopf pair itself does not
    count): a change is a Zero-Hopf ("zh", one real eigenvalue) or Hopf-Hopf ("hh", a second pair) point, recorded (1) or located by
    the event bisection (2).  The Bautin test function (first Lyapunov coefficient) needs normal forms and is not evaluated."""
    from . import palc as P
    ma = HopfMinAug(prob, cprob, eigenvec_ad, eigenvec, ls, cls, cbls)
    z0 = BorderedVec(V.copy(x0), [p1_0, omega0])
    pb = HopfMAProblem(ma, lens2, z0, record)
    hls = HopfLinearSolverMinAug()
    no = contpar.newton_options
    cp = P.ContinuationPar(**{**contpar.__dict__, "newton_options": P.NewtonPar(tol=no.tol, max_iterations=no.max_iterations, linsolver=hls),
                              "detect_bifurcation": 0})
    alg = alg or P.PALC()
    alg = P.PALC(tangent=alg.tangent, theta=alg.theta, bls=BorderingBLSHost(hls))
    curve = HopfCurve([], [], [], [], ma, None)
    curve.specialpoint = []
    cnorm = lambda z: float(np.max(np.abs(z)))
    from . import events as E
    it = E._Iter(pb, alg, cp, normC)
    tol_st = max(10 * no.tol, contpar.tol_stability)
    nhist = []

    def unstable_at(s):   # (n_unstable, n_imag) of J at the Hopf point of state s (is_stable, src/Bifurcations.jl:5-18)
        pb._set2(s.z_p)
        ev = np.asarray(eigsolver(prob.J(s.z_u.u, float(s.z_u.p[0])), contpar.nev)[0])
        un = ev.real > tol_st
        return (int(np.sum(un)), int(np.sum(un & (np.abs(ev.imag) > tol_st))))

    def cb(st):
        pb._set2(st.z_p)
        x, p1, om = st.z_u.u, float(st.z_u.p[0]), float(st.z_u.p[1])
        if eigsolver is not None:
            nu = unstable_at(st)
            if detect_event > 0 and nhist and st.step > 0 and nu[0] != nhist[-1][0]:
                prev, status, interval = nhist[-1], "guess", E.getinterval(curve.p2[-1], st.z_p)
                if detect_event > 1:
                    status, interval, _ = locate_event(it, st, lambda s: (unstable_at(s)[0],), ("hh",), indicator=lambda v: v[0])
                    pb._set2(st.z_p)
                    nu = unstable_at(st)
                    x, p1, om = st.z_u.u, float(st.z_u.p[0]), float(st.z_u.p[1])
                if status != "none":
                    dn, di = abs(nu[0] - prev[0]), abs(nu[1] - prev[1])
                    curve.specialpoint.append(Codim2Point("zh" if dn == 1 else ("hh" if di == 2 else "nd"), st.z_p, p1, st.step, status, tuple(interval), V.copy(x)))
            nhist.append(nu)
        if st.step % update_minaug_every_step == 0:
            v, _ = ma._border(cprob.J(x, p1), complex(0.0, -om), ma.a, ma.b)
            w, _ = ma._border(cprob.J(x, p1, transpose=True), complex(0.0, om), ma.b, ma.a)
            ma.a, ma.b = w / cnorm(w), v / cnorm(v)
        curve.p1.append(p1)
        curve.p2.append(st.z_p)
        curve.omega.append(om)
        if abs(om) < 100 * no.tol:  # the frequency is null: not a Hopf point any more, the curve ends on a Bogdanov-Takens point
            curve.stopped_at_bt = True
            return False
        return True if callback is None else callback(st)

    p2_0, c2_0 = prob.params[lens2], cprob.params[lens2]
    try:
        curve.rows, curve.state = P.continuation(pb, alg, cp, normC=normC, callback=cb)
    finally:
        prob.params[lens2], cprob.params[lens2] = p2_0, c2_0
    return curve
