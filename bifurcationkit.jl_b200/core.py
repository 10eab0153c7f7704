"""Host-side mirror of the reference's plugin surfaces over libbk200.so.

Names, argument meaning and return tuples follow the reference so that parity tests read
like the reference's own tests:

* ``GMRESB200``       <-> ``GMRESIterativeSolvers`` (src/LinearSolver.jl:149-206):
                           ``ls(J, rhs; a0, a1) -> (x, converged, iters)``; two-rhs form
                           (src/LinearSolver.jl:15-19) ``-> (x1, x2, ok, (it1, it2))``.
* ``BorderingBLSB200`` / ``MatrixFreeBLSB200`` <-> src/LinearBorderSolver.jl:59-166 / :404-437:
                           ``bls(J, dR, dzu, dzp, R, n, xiu, xip; shift, dotp) -> (dX, dl, ok, iters)``.
* ``ShiftInvertB200`` <-> ``ShiftInvert`` (src/EigSolver.jl:246-266):
                           ``eig(J, nev) -> (vals, vecs, converged, niter)``, vals sorted by decreasing real part.
* ``Jacobian``        <-> the "any user struct" form of ``prob.VF.J(x, p)`` (src/Problems.jl:98-101,
                           pattern of examples/SH2d-fronts-cuda.jl:31-37): callable ``J(dx)`` so that
                           ``apply(J, dx)`` (src/Utils.jl:192) works with stock solvers too.
* ``DeviceVec``       <-> a state vector type implementing the VectorInterface subset the
                           reference needs (src/BorderedArrays.jl:17-35, examples/chan-af.jl:7-16).

Vectors may be NumPy arrays (host buffers: every call copies H2D/D2H inside the C ABI -- "option A")
or ``DeviceVec`` (device-resident, zero copies -- "option B").  Results have the container type of
the right-hand side, as the reference requires (Newton does ``minus!!(x, u)``, src/Newton.jl:97).
"""
import ctypes as C

import numpy as np

from . import lib as _l


def _chk(ctx, status):
    if status < 0:
        msg = _l.load().bk_last_error(ctx.handle)
        raise _l.BK200Error(f"libbk200 error {status}: {msg.decode() if msg else ''}")
    return status


class Context:
    """One per GPU: owns the CUDA stream, Krylov workspace and the problem description."""

    def __init__(self, kind, dims, lengths=(1.0, 1.0, 1.0), krylov_m=100, device=0, params=None, complex=False):
        self.lib = _l.load()
        if complex:
            kind |= _l.BK_COMPLEX  # vectors [re; im] of length 2 N0, shifts a0 + i a0_imag (include/bk200.h)
        d = (C.c_int64 * 3)(*(list(dims) + [1, 1, 1])[:3])
        L = (C.c_double * 3)(*(list(lengths) + [1.0, 1.0, 1.0])[:3])
        h = C.c_void_p()
        st = self.lib.bk_ctx_create(device, kind, d, L, krylov_m, C.byref(h))
        self.handle = h
        if st < 0:
            msg = self.lib.bk_last_error(h) if h else b"context allocation failed"
            raise _l.BK200Error(f"bk_ctx_create failed ({st}): {msg.decode()}")
        self.kind, self.dims, self.lengths, self.krylov_m = kind, tuple(dims), tuple(lengths), krylov_m
        self.N = int(self.lib.bk_problem_size(h))
        self.N0 = int(self.lib.bk_state_size(h))
        self.complex = bool(complex)
        self.params = None
        if params is not None:
            self.set_params(params)

    def close(self):
        if getattr(self, "handle", None):
            self.lib.bk_ctx_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- parameters / problem ----
    def set_params(self, params):
        p = np.ascontiguousarray(params, dtype=np.float64)
        _chk(self, self.lib.bk_set_params(self.handle, p.ctypes.data_as(C.POINTER(C.c_double)), len(p)))
        self.params = tuple(float(x) for x in p)

    def stats(self):
        s = _l.Stats()
        _chk(self, self.lib.bk_get_stats(self.handle, C.byref(s)))
        return {k: getattr(s, k) for k, _ in s._fields_}

    def set_timing(self, on):
        _chk(self, self.lib.bk_set_timing(self.handle, int(on)))  # True / 1: every solve; k > 1: every k-th solve

    def sync(self):
        _chk(self, self.lib.bk_sync(self.handle))

    # ---- vectors ----
    def zeros(self, n=None):
        return DeviceVec(self, self.N if n is None else n)

    def to_device(self, a):
        a = np.ascontiguousarray(a, dtype=np.float64)
        v = DeviceVec(self, a.shape[0])
        _chk(self, self.lib.bk_vec_upload(self.handle, v.dptr, a.ctypes.data, a.shape[0]))
        return v

    def _like(self, x, n=None):
        n = len(x) if n is None else n
        if isinstance(x, DeviceVec):
            return DeviceVec(self, n)
        return self.pinned_empty(n) if self.pin_host else np.empty(n)

    # ---- pinned host arrays (option A callers): pooled cudaHostAlloc buffers exposed as NumPy arrays
    pin_host = False

    def pinned_empty(self, n):
        import weakref
        pool = self.__dict__.setdefault("_pin_pool", {})
        free = pool.setdefault(n, [])
        if free:
            addr = free.pop()
        else:
            p = C.c_void_p()
            _chk(self, self.lib.bk_host_alloc(self.handle, n, C.byref(p)))
            addr = p.value
        buf = (C.c_double * n).from_address(addr)
        arr = np.frombuffer(buf, dtype=np.float64)
        weakref.finalize(buf, free.append, addr)  # recycled when the last view dies; freed with the process
        return arr

    def pinned_array(self, a):
        out = self.pinned_empty(len(a))
        out[...] = a
        return out

    # ---- K1 / K2 ----
    def residual(self, u, out=None):
        out = self._like(u) if out is None else out
        _chk(self, self.lib.bk_residual(self.handle, _l.ptr(u), _l.ptr(out)))
        return out

    def jacobian(self, u):
        """J = jacobian(prob, u, params): snapshot of (u, current params) inside the context."""
        _chk(self, self.lib.bk_jac_set_state(self.handle, _l.ptr(u)))
        return Jacobian(self)

    def cjacobian(self, u, transpose=False):
        """BK_COMPLEX contexts: J (or J') at the real state u, acting on complex vectors."""
        assert self.complex
        _chk(self, self.lib.bk_jac_set_state(self.handle, _l.ptr(u)))
        return ComplexJacobian(self, transpose)

    def set_shift_imag(self, a0_imag):
        _chk(self, self.lib.bk_jac_set_shift_imag(self.handle, float(a0_imag)))

    def set_transpose(self, on):
        _chk(self, self.lib.bk_jac_set_transpose(self.handle, 1 if on else 0))

    def jvp(self, v, out=None, a0=0.0, a1=1.0):
        out = self._like(v) if out is None else out
        _chk(self, self.lib.bk_jvp(self.handle, _l.ptr(v), _l.ptr(out), a0, a1))
        return out

    def precond_setup(self, kind, a0=1.0, a1=1.0):
        _chk(self, self.lib.bk_precond_setup(self.handle, kind, a0, a1))

    def precond_apply(self, x, out=None):
        out = self._like(x) if out is None else out
        _chk(self, self.lib.bk_precond_apply(self.handle, _l.ptr(x), _l.ptr(out)))
        return out

    def potrap_set_section(self, phi, xpi=None):
        _chk(self, self.lib.bk_potrap_set_section(self.handle, _l.ptr(phi), _l.ptr(xpi)))

    # ---- BK_SPARSE: the Jacobian as a sparse matrix assembled by the caller ----
    _sp_key = None  # (format, base, indptr, indices) of the pattern loaded last
    nnz = None

    def sparse_pattern(self, A):
        """bk_sparse_set_pattern from a scipy CSR / CSC matrix or raw (format, base, ptr, idx) (see sparse_pattern_args)"""
        fmt, base, nnz, ptr, idx = sparse_pattern_args(A)
        i64p = C.POINTER(C.c_int64)
        _chk(self, self.lib.bk_sparse_set_pattern(self.handle, fmt, base, nnz, ptr.ctypes.data_as(i64p), idx.ctypes.data_as(i64p)))
        self._sp_key, self.nnz = (fmt, base, ptr, idx), nnz

    def sparse_values(self, vals):
        """bk_sparse_set_values: nnz values in the pattern's order -- a NumPy array, a DeviceVec, or a scipy matrix (its .data)"""
        assert self.nnz is not None, "sparse_pattern must be called first"
        if hasattr(vals, "tocsr"):
            vals = vals.data
        if not hasattr(vals, "dptr"):
            vals = np.ascontiguousarray(vals, dtype=np.float64)
        if len(vals) != self.nnz:
            raise _l.BK200Error(f"sparse_values: {len(vals)} values for a pattern of {self.nnz} entries")
        _chk(self, self.lib.bk_sparse_set_values(self.handle, _l.ptr(vals)))

    def sparse_load(self, A, check_pattern=True):
        """J <- A: a scipy CSR / CSC matrix (its pattern is (re)loaded when it differs from the last one -- compared by indptr /
        indices unless check_pattern is False, then only when none is loaded yet) or the values array of the loaded pattern"""
        if hasattr(A, "tocsr"):
            if self._sp_key is None or (check_pattern and not _same_pattern(self._sp_key, A)):
                self.sparse_pattern(A)
        self.sparse_values(A)


def sparse_pattern_args(A):
    """A scipy CSR / CSC matrix, or raw (format, base, ptr, idx) with format BK_SPARSE_CSR / BK_SPARSE_CSC (or "csr" / "csc") and
    base 0 or 1 (Julia's colptr / rowval as they are: ("csc", 1, colptr, rowval)) -> the arguments (format, base, nnz, ptr, idx) of
    bk_sparse_set_pattern, ptr and idx as contiguous int64 arrays"""
    if isinstance(A, tuple):
        fmt, base, ptr, idx = A
        fmt = {"csr": _l.BK_SPARSE_CSR, "csc": _l.BK_SPARSE_CSC}.get(fmt, fmt)
    else:
        f = getattr(A, "format", None)
        if f not in ("csr", "csc"):
            raise _l.BK200Error(f"sparse pattern: a CSR or CSC matrix is needed, got {type(A).__name__} ({f})")
        fmt, base, ptr, idx = (_l.BK_SPARSE_CSR if f == "csr" else _l.BK_SPARSE_CSC), 0, A.indptr, A.indices
    if fmt not in (_l.BK_SPARSE_CSR, _l.BK_SPARSE_CSC) or base not in (0, 1):
        raise _l.BK200Error(f"sparse pattern: bad format {fmt!r} or index base {base!r}")
    ptr = np.ascontiguousarray(ptr, dtype=np.int64)
    idx = np.ascontiguousarray(idx, dtype=np.int64)
    return int(fmt), int(base), int(len(idx)), ptr, idx


def _same_pattern(key, A):
    fmt, base, ptr, idx = key
    return (base == 0 and fmt == (_l.BK_SPARSE_CSR if A.format == "csr" else _l.BK_SPARSE_CSC)
            and np.array_equal(ptr, A.indptr) and np.array_equal(idx, A.indices))


class DeviceVec:
    """Device-resident fp64 vector with the VectorInterface subset used by the continuation host loop."""

    def __init__(self, ctx, n):
        self.ctx, self.n = ctx, int(n)
        p = C.c_void_p()
        _chk(ctx, ctx.lib.bk_vec_alloc(ctx.handle, self.n, C.byref(p)))
        self.dptr = p.value

    def __del__(self):
        try:
            if self.dptr and self.ctx.handle:
                self.ctx.lib.bk_vec_free(self.ctx.handle, self.dptr)
        except Exception:
            pass
        self.dptr = None

    def __len__(self):
        return self.n

    def numpy(self):
        out = np.empty(self.n)
        _chk(self.ctx, self.ctx.lib.bk_vec_download(self.ctx.handle, out.ctypes.data, self.dptr, self.n))
        return out

    def copy(self):
        v = DeviceVec(self.ctx, self.n)
        _chk(self.ctx, self.ctx.lib.bk_vec_copy(self.ctx.handle, v.dptr, self.dptr, self.n))
        return v

    def copyto(self, src):  # _copyto!(self, src)
        _chk(self.ctx, self.ctx.lib.bk_vec_copy(self.ctx.handle, self.dptr, src.dptr, self.n))
        return self

    def zero_(self):
        _chk(self.ctx, self.ctx.lib.bk_vec_zero(self.ctx.handle, self.dptr, self.n))
        return self

    def scale_(self, a):  # VI.scale!
        _chk(self.ctx, self.ctx.lib.bk_vec_scale(self.ctx.handle, self.dptr, float(a), self.n))
        return self

    def axpby_(self, a, x, b=1.0):  # VI.add!(self, x, a, b): self = a x + b self
        _chk(self.ctx, self.ctx.lib.bk_vec_axpby(self.ctx.handle, self.dptr, float(a), x.dptr, float(b), self.n))
        return self

    def dot(self, y):  # VI.inner
        out = C.c_double()
        _chk(self.ctx, self.ctx.lib.bk_vec_dot(self.ctx.handle, self.dptr, y.dptr, self.n, C.byref(out)))
        return out.value

    def norm(self):
        out = C.c_double()
        _chk(self.ctx, self.ctx.lib.bk_vec_norm2(self.ctx.handle, self.dptr, self.n, C.byref(out)))
        return out.value

    def norminf(self):
        out = C.c_double()
        _chk(self.ctx, self.ctx.lib.bk_vec_norminf(self.ctx.handle, self.dptr, self.n, C.byref(out)))
        return out.value

    def diffdot(self, x0, tau):  # <self - x0, tau>
        out = C.c_double()
        _chk(self.ctx, self.ctx.lib.bk_vec_diffdot(self.ctx.handle, self.dptr, x0.dptr, tau.dptr, self.n, C.byref(out)))
        return out.value


class Jacobian:
    """Handle on the context's linearisation state.  Only the most recent Jacobian of a context is
    live (the reference recomputes J every Newton iteration, src/Newton.jl:91, Palc.jl:243)."""

    def __init__(self, ctx):
        self.ctx = ctx

    def __call__(self, dx):
        return self.ctx.jvp(dx)


def csplit(z):
    """complex array -> the split layout [re; im] of a BK_COMPLEX context"""
    z = np.asarray(z)
    return np.ascontiguousarray(np.concatenate([z.real, z.imag]), dtype=np.float64)


def cjoin(x):
    n = len(x) // 2
    return x[:n] + 1j * x[n:]


class ComplexJacobian:
    """J or its transpose (apply_jacobian(prob, x, par, dx, true), src/codim2/MinAugHopf.jl:152-155) on complex NumPy vectors;
    handle on a BK_COMPLEX context's linearisation state, like `Jacobian`."""

    def __init__(self, ctx, transpose=False):
        self.ctx, self.transpose = ctx, bool(transpose)

    def __call__(self, z):
        self.ctx.set_transpose(self.transpose)
        self.ctx.set_shift_imag(0.0)
        return cjoin(self.ctx.jvp(csplit(z)))


def make_opts(reltol=1e-8, abstol=0.0, restart=200, maxiter=100, pc_side=_l.BK_SIDE_NONE, orth=_l.BK_ORTH_CGS, fused=True):
    return _l.GmresOpts(reltol, abstol, restart, maxiter, pc_side, orth, int(fused), 0)  # fused: 0 off, 1 auto, 2 force


class GMRESB200:
    """Drop-in for GMRESIterativeSolvers (src/LinearSolver.jl:149-206).  ``Pl`` / ``Pr`` name the
    side on which the context's preconditioner (``Context.precond_setup``) is applied."""

    def __init__(self, reltol=1e-8, abstol=0.0, restart=200, maxiter=100, N=0, Pl=False, Pr=False,
                 orth="cgs", fused=True):
        assert not (Pl and Pr), "one preconditioner per context"
        self.reltol, self.abstol, self.restart, self.maxiter, self.N = reltol, abstol, restart, maxiter, N
        self.Pl, self.Pr, self.orth, self.fused = Pl, Pr, orth, fused

    def opts(self):
        side = _l.BK_SIDE_LEFT if self.Pl else (_l.BK_SIDE_RIGHT if self.Pr else _l.BK_SIDE_NONE)
        return make_opts(self.reltol, self.abstol, self.restart, self.maxiter, side,
                         _l.BK_ORTH_CGS2 if self.orth == "cgs2" else _l.BK_ORTH_CGS, self.fused)

    def __call__(self, J, rhs, rhs2=None, a0=0.0, a1=1.0):
        ctx = J.ctx
        if rhs2 is not None:
            # src/LinearSolver.jl:15-19: ls(J, rhs1, rhs2) -> (x1, x2, flag1 & flag2, (it1, it2)): one ABI crossing (bk_gmres2)
            x1, x2 = ctx._like(rhs), ctx._like(rhs2)
            o = self.opts()
            cv = C.c_int32()
            its = (C.c_int32 * 2)()
            _chk(ctx, ctx.lib.bk_gmres2(ctx.handle, _l.ptr(rhs), _l.ptr(rhs2), _l.ptr(x1), _l.ptr(x2), a0, a1, C.byref(o), C.byref(cv), its))
            return x1, x2, bool(cv.value), (its[0], its[1])
        x = ctx._like(rhs)
        o = self.opts()
        cv, it, rn = C.c_int32(), C.c_int32(), C.c_double()
        _chk(ctx, ctx.lib.bk_gmres(ctx.handle, _l.ptr(rhs), _l.ptr(x), a0, a1, C.byref(o), C.byref(cv), C.byref(it), C.byref(rn)))
        self.last_resnorm = rn.value
        return x, bool(cv.value), it.value


class ComplexGMRESB200(GMRESB200):
    """ls(J, rhs; a0 = complex shift, a1) on a BK_COMPLEX context: (a0 I + a1 J) x = rhs for complex rhs -- the
    `shift = Complex(0, -omega)` solves of the Hopf functional (src/codim2/MinAugHopf.jl:19-40).  GMRES runs on the
    real-equivalent system; the solution, not the iterate sequence, is what parity pins."""

    def __call__(self, J, rhs, a0=0.0, a1=1.0):
        ctx = J.ctx
        a0 = complex(a0)
        ctx.set_transpose(getattr(J, "transpose", False))
        ctx.set_shift_imag(a0.imag)
        try:
            x, cv, it = GMRESB200.__call__(self, J, csplit(rhs), a0=a0.real, a1=a1)
        finally:
            ctx.set_shift_imag(0.0)
        return cjoin(x), cv, it


def _block_args(a, b, c, rhsb):
    """tuples of border vectors -> pointer arrays; c -> m x m column-major (the Julia matrix layout); rhsb -> host doubles"""
    a, b = (a,) if not isinstance(a, (tuple, list)) else tuple(a), (b,) if not isinstance(b, (tuple, list)) else tuple(b)
    m = len(a)
    assert m == len(b) and m in (1, 2), "block borders: one or two border vectors"
    pa = (C.c_void_p * m)(*[_l.ptr(v) for v in a])
    pb = (C.c_void_p * m)(*[_l.ptr(v) for v in b])
    cm = np.asfortranarray(np.atleast_2d(np.asarray(c, dtype=np.float64)))
    assert cm.shape == (m, m), "Linear bordered solver, wrong sizes!"
    rb = None if rhsb is None else np.ascontiguousarray(np.atleast_1d(rhsb), dtype=np.float64)
    return m, pa, pb, cm, rb, (a, b)  # the last entry keeps the vectors alive for the duration of the call


class BorderingBLSB200:
    """src/LinearBorderSolver.jl:59-166."""

    def __init__(self, solver=None, tol=1e-12, check_precision=True, k=1):
        assert k > 0
        self.solver, self.tol, self.check_precision, self.k = solver, tol, check_precision, k

    def __call__(self, J, dR, dzu, dzp, R, n, xiu=1.0, xip=1.0, shift=None, dotscale=1.0):
        ctx = J.ctx
        dX = ctx._like(R)
        o = self.solver.opts()
        dl, cv = C.c_double(), C.c_int32()
        it = (C.c_int32 * 2)()
        _chk(ctx, ctx.lib.bk_bls_bordering(ctx.handle, _l.ptr(dR), _l.ptr(dzu), dzp, _l.ptr(R), n, xiu, xip,
                                           0 if shift is None else 1, 0.0 if shift is None else shift, dotscale,
                                           C.byref(o), 1 if self.check_precision else 0, self.k, self.tol,
                                           _l.ptr(dX), C.byref(dl), C.byref(cv), it))
        return dX, dl.value, bool(cv.value), (it[0], it[1])

    def solve_block(self, J, a, b, c, rhst, rhsb, shift=None):
        """solve_bls_block(lbs::BorderingBLS, J, b, c, d, rhst, rhsb) (src/LinearBorderSolver.jl:173-206):
        a / b tuples of one or two border vectors (columns / rows), c the m x m corner -> (u, p, converged, iters)"""
        ctx = J.ctx
        m, pa, pb, cm, rb, keep = _block_args(a, b, c, rhsb)
        u = ctx._like(rhst)
        sp = np.zeros(m)
        o = self.solver.opts()
        cv = C.c_int32()
        it = (C.c_int32 * 3)()
        dp = C.POINTER(C.c_double)
        _chk(ctx, ctx.lib.bk_bls_block_bordering(ctx.handle, m, pa, pb, cm.ctypes.data_as(dp), _l.ptr(rhst), rb.ctypes.data_as(dp),
                                                 0 if shift is None else 1, 0.0 if shift is None else shift, C.byref(o),
                                                 _l.ptr(u), sp.ctypes.data_as(dp), C.byref(cv), it))
        return u, sp, bool(cv.value), tuple(it[: m + 1])


class MatrixFreeBLSB200:
    """src/LinearBorderSolver.jl:404-437 (rhs = vcat(R, n), one GMRES on the N+1 system)."""

    def __init__(self, solver=None):
        self.solver = solver

    def __call__(self, J, dR, dzu, dzp, R, n, xiu=1.0, xip=1.0, shift=None, dotscale=1.0):
        ctx = J.ctx
        dX = ctx._like(R)
        o = self.solver.opts()
        dl, cv, it = C.c_double(), C.c_int32(), C.c_int32()
        _chk(ctx, ctx.lib.bk_bls_matrixfree(ctx.handle, _l.ptr(dR), _l.ptr(dzu), dzp, _l.ptr(R), n, xiu, xip,
                                            0 if shift is None else 1, 0.0 if shift is None else shift, dotscale,
                                            C.byref(o), _l.ptr(dX), C.byref(dl), C.byref(cv), C.byref(it)))
        return dX, dl.value, bool(cv.value), it.value

    def solve_block(self, J, a, b, c, rhst, rhsb, shift=None, dotscale=1.0):
        """solve_bls_block(lbs::MatrixFreeBLS, J, a, b, c, rhst, rhsb; shift, dotp) (src/LinearBorderSolver.jl:440-450): one GMRES
        on the (N + m) system through the tuple form of MatrixFreeBLSmap (:338-389)"""
        ctx = J.ctx
        m, pa, pb, cm, rb, keep = _block_args(a, b, c, rhsb)
        u = ctx._like(rhst)
        sp = np.zeros(m)
        o = self.solver.opts()
        cv, it = C.c_int32(), C.c_int32()
        dp = C.POINTER(C.c_double)
        _chk(ctx, ctx.lib.bk_bls_block_matrixfree(ctx.handle, m, pa, pb, cm.ctypes.data_as(dp), _l.ptr(rhst), rb.ctypes.data_as(dp),
                                                  0 if shift is None else 1, 0.0 if shift is None else shift, dotscale, C.byref(o),
                                                  _l.ptr(u), sp.ctypes.data_as(dp), C.byref(cv), C.byref(it)))
        return u, sp, bool(cv.value), it.value


def bls_map_block(J, a, b, c, x, shift=None, dotscale=1.0):
    """MatrixFreeBLSmap(J, a::Tuple, b::Tuple, c::Matrix, shift, dot)(x) (src/LinearBorderSolver.jl:366-389), x of length N + m."""
    ctx = J.ctx
    m, pa, pb, cm, _, keep = _block_args(a, b, c, None)
    out = ctx._like(x)
    _chk(ctx, ctx.lib.bk_bls_block_map(ctx.handle, m, pa, pb, cm.ctypes.data_as(C.POINTER(C.c_double)), 0 if shift is None else 1,
                                       0.0 if shift is None else shift, dotscale, _l.ptr(x), _l.ptr(out)))
    return out


def bls_map(J, a, b, c, x, shift=None, dotscale=1.0):
    """MatrixFreeBLSmap(J, a, b, c, shift, dot)(x) (src/LinearBorderSolver.jl:312-325), x of length N+1."""
    ctx = J.ctx
    out = ctx._like(x)
    _chk(ctx, ctx.lib.bk_bls_map(ctx.handle, _l.ptr(a), _l.ptr(b), c, 0 if shift is None else 1,
                                 0.0 if shift is None else shift, dotscale, _l.ptr(x), _l.ptr(out)))
    return out


class ShiftInvertB200:
    """src/EigSolver.jl:246-266 with the inner linear solver = GMRESB200 (a0 = -sigma, a1 = 1)."""

    def __init__(self, sigma, ls, krylovdim=None, tol=1e-10, maxrestart=20):
        self.sigma, self.ls, self.krylovdim, self.tol, self.maxrestart = sigma, ls, krylovdim, tol, maxrestart

    def __call__(self, J, nev, v0=None, want_vectors=False):
        ctx = J.ctx
        kd = self.krylovdim or max(30, nev + 30)
        kd = min(kd, ctx.N)
        nev = min(nev, kd)
        re, im = np.zeros(nev), np.zeros(nev)
        vecs = np.zeros((nev, ctx.N)) if want_vectors else None
        nconv, nops = C.c_int32(), C.c_int32()
        o = self.ls.opts()
        dp = C.POINTER(C.c_double)
        _chk(ctx, ctx.lib.bk_eigs_shift_invert(ctx.handle, self.sigma, nev, kd, self.tol, self.maxrestart, C.byref(o),
                                               _l.ptr(v0), re.ctypes.data_as(dp), im.ctypes.data_as(dp),
                                               _l.ptr(vecs) if want_vectors else None, C.byref(nconv), C.byref(nops)))
        vals = re + 1j * im
        return vals, (vecs.T if want_vectors else None), nconv.value >= nev, nops.value


def hessenberg_eig(H, vectors=True):
    """Host-only: eigenpairs of a real upper-Hessenberg matrix through the library's QR iteration."""
    lib = _l.load()
    H = np.asfortranarray(H, dtype=np.float64)
    n = H.shape[0]
    wr, wi = np.zeros(n), np.zeros(n)
    vr = np.zeros((n, n), order="F")
    vi = np.zeros((n, n), order="F")
    dp = C.POINTER(C.c_double)
    st = lib.bk_hessenberg_eig(H.ctypes.data_as(dp), n, n, wr.ctypes.data_as(dp), wi.ctypes.data_as(dp),
                               vr.ctypes.data_as(dp) if vectors else None, vi.ctypes.data_as(dp) if vectors else None)
    if st != 0:
        raise _l.BK200Error(f"bk_hessenberg_eig failed ({st})")
    return wr + 1j * wi, (vr + 1j * vi) if vectors else None
