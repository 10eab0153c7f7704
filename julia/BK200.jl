# BK200.jl -- Julia-side adapter: the three BifurcationKit plugin surfaces over libbk200.so.
#
# NOT EXECUTED in this repository's CI: the build image has no Julia toolchain (SURVEY.md, "Environment
# facts").  It is the binding a BifurcationKit maintainer would load; every method mirrors the signature of
# the reference method it replaces (file:line cited inline) and forwards to one C-ABI entry point of
# include/bk200.h.  The Python mirror bifurcationkit.jl_b200/core.py implements exactly the same mapping and
# IS exercised by the GPU test-suite.
#
#   using BifurcationKit, BK200
#   ctx  = BK200.Context(:SH2D, (Nx, Ny), (lx, ly); krylov_m = 100)
#   prob = BifurcationProblem((u, p) -> BK200.residual(ctx, u, (p.l, p.ν)), u0, (l = -0.1, ν = 1.3), (@optic _.l);
#                             J = (u, p) -> BK200.Jac(ctx, u, (p.l, p.ν)))
#   BK200.precond!(ctx, :SH_DCT, 1.0)                       # (L1 + I)^-1, cf. examples/SH2d-fronts.jl:121
#   ls   = BK200.GMRESB200(ctx; reltol = 1e-5, Pr = true)
#   opts = ContinuationPar(...; newton_options = NewtonPar(linsolver = ls, eigsolver = BK200.ShiftInvertB200(ctx, 0.1, ls)))
#   br   = continuation(prob, PALC(bls = BK200.BorderingBLSB200(ls)), opts; normC = norminf)
#
# A user problem with an assembled sparse Jacobian (examples/brusselator.jl, J = Jbru_sp) runs on a :SPARSE context:
#   ctx = BK200.Context(:SPARSE, (2n,), (1.0,); krylov_m = 200); BK200.precond!(ctx, :JACOBI, 0.0, 1.0)
#   ls  = BK200.GMRESB200(ctx; Pl = true)          # methods for J::SparseMatrixCSC load J with BK200.sparse!
module BK200

using BifurcationKit, LinearAlgebra, SparseArrays
const BK = BifurcationKit
const VI = BK.VI
const lib = get(ENV, "BK200_LIB", joinpath(@__DIR__, "..", "bifurcationkit.jl_b200", "libbk200.so"))

const KINDS = Dict(:CHAN => 1, :SH2D => 2, :SH3D => 3, :CGL2D => 4, :POTRAP_CGL2D => 5, :SPARSE => 6)
const PCS = Dict(:NONE => 0, :SH_DCT => 1, :CHAN_TRIDIAG => 2, :CGL_DST => 3, :POTRAP_CIRC => 4, :JACOBI => 5)

struct GmresOpts            # == bk_gmres_opts
    reltol::Cdouble; abstol::Cdouble; restart::Int32; maxiter::Int32
    pc_side::Int32; orth::Int32; fused::Int32; reserved::Int32
end

mutable struct Context
    handle::Ptr{Cvoid}
    N::Int
    pattern::Any   # :SPARSE contexts: (colptr, rowval) of the pattern loaded last (sparse!)
    # complex = true: BK_COMPLEX context (include/bk200.h) -- vectors [re; im], complex shifts, for MinAugHopf.jl's solves
    function Context(kind::Symbol, dims, lengths; krylov_m = 100, device = 0, complex = false)
        d = Int64[dims..., 1, 1][1:3]; L = Float64[lengths..., 1.0, 1.0][1:3]
        h = Ref{Ptr{Cvoid}}(C_NULL)
        st = ccall((:bk_ctx_create, lib), Int32, (Int32, Int32, Ptr{Int64}, Ptr{Float64}, Int32, Ptr{Ptr{Cvoid}}),
                   device, KINDS[kind] | (complex ? 0x100 : 0), d, L, krylov_m, h)
        st < 0 && error("bk_ctx_create: " * unsafe_string(ccall((:bk_last_error, lib), Cstring, (Ptr{Cvoid},), h[])))
        c = new(h[], Int(ccall((:bk_problem_size, lib), Int64, (Ptr{Cvoid},), h[])), nothing)
        # bk_ctx_destroy frees every vector still alive (vec_live); the handle is nulled so that DeviceVec finalizers
        # running AFTER this one (finalizer order is unspecified for objects that die together) do not touch a freed ctx
        finalizer(c) do x
            h = x.handle
            x.handle = C_NULL
            h == C_NULL || ccall((:bk_ctx_destroy, lib), Int32, (Ptr{Cvoid},), h)
        end
    end
end
check(c::Context, st) = st < 0 ? error(unsafe_string(ccall((:bk_last_error, lib), Cstring, (Ptr{Cvoid},), c.handle))) : st
setparams!(c::Context, p) = (v = collect(Float64, p); check(c, ccall((:bk_set_params, lib), Int32, (Ptr{Cvoid}, Ptr{Float64}, Int32), c.handle, v, length(v))))
precond!(c::Context, kind::Symbol, a0 = 1.0, a1 = 1.0) = check(c, ccall((:bk_precond_setup, lib), Int32, (Ptr{Cvoid}, Int32, Float64, Float64), c.handle, PCS[kind], a0, a1))

# ---- state vectors ---------------------------------------------------------------------------------------------------
# Option A: plain Vector{Float64} (host pointers cross the ABI; the library copies H2D/D2H inside each call).
# Option B: DeviceVec, a device-resident vector implementing the method set the reference itself needs for a
# foreign state type (examples/chan-af.jl:7-16; src/BorderedArrays.jl:17-35).
mutable struct DeviceVec
    ctx::Context; ptr::Ptr{Float64}; n::Int
    function DeviceVec(ctx::Context, n::Int)
        p = Ref{Ptr{Float64}}(C_NULL)
        check(ctx, ccall((:bk_vec_alloc, lib), Int32, (Ptr{Cvoid}, Int64, Ptr{Ptr{Float64}}), ctx.handle, n, p))
        v = new(ctx, p[], n)
        finalizer(v) do x
            x.ctx.handle == C_NULL || ccall((:bk_vec_free, lib), Int32, (Ptr{Cvoid}, Ptr{Float64}), x.ctx.handle, x.ptr)
        end
    end
end
DeviceVec(ctx::Context, a::Vector{Float64}) = (v = DeviceVec(ctx, length(a)); ccall((:bk_vec_upload, lib), Int32, (Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}, Int64), ctx.handle, v.ptr, a, length(a)); v)
Base.Array(v::DeviceVec) = (a = Vector{Float64}(undef, v.n); ccall((:bk_vec_download, lib), Int32, (Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}, Int64), v.ctx.handle, a, v.ptr, v.n); a)
ptr(a::Vector{Float64}) = pointer(a)
ptr(a::DeviceVec) = a.ptr
like(c::Context, ::Vector{Float64}, n = c.N) = Vector{Float64}(undef, n)
like(c::Context, ::DeviceVec, n = c.N) = DeviceVec(c, n)

Base.length(v::DeviceVec) = v.n
Base.eltype(::Type{DeviceVec}) = Float64
Base.similar(v::DeviceVec) = DeviceVec(v.ctx, v.n)
Base.copy(v::DeviceVec) = copyto!(similar(v), v)
Base.copyto!(d::DeviceVec, s::DeviceVec) = (ccall((:bk_vec_copy, lib), Int32, (Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}, Int64), d.ctx.handle, d.ptr, s.ptr, d.n); d)
function _red(f, v::DeviceVec, args...)
    out = Ref{Float64}(0.0); f(out); out[]
end
LinearAlgebra.dot(x::DeviceVec, y::DeviceVec) = (o = Ref(0.0); ccall((:bk_vec_dot, lib), Int32, (Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}, Int64, Ptr{Float64}), x.ctx.handle, x.ptr, y.ptr, x.n, o); o[])
function LinearAlgebra.norm(x::DeviceVec, p::Real = 2)
    o = Ref(0.0)
    if p == Inf
        ccall((:bk_vec_norminf, lib), Int32, (Ptr{Cvoid}, Ptr{Float64}, Int64, Ptr{Float64}), x.ctx.handle, x.ptr, x.n, o)
    else
        ccall((:bk_vec_norm2, lib), Int32, (Ptr{Cvoid}, Ptr{Float64}, Int64, Ptr{Float64}), x.ctx.handle, x.ptr, x.n, o)
    end
    o[]
end
# VectorInterface methods used by BorderedArray algebra (src/BorderedArrays.jl:86-217)
VI.scalartype(::Type{DeviceVec}) = Float64
VI.zerovector(x::DeviceVec, ::Type{Float64} = Float64) = (z = similar(x); ccall((:bk_vec_zero, lib), Int32, (Ptr{Cvoid}, Ptr{Float64}, Int64), z.ctx.handle, z.ptr, z.n); z)
VI.zerovector!(x::DeviceVec) = (ccall((:bk_vec_zero, lib), Int32, (Ptr{Cvoid}, Ptr{Float64}, Int64), x.ctx.handle, x.ptr, x.n); x)
VI.scale!(x::DeviceVec, a::Number) = (ccall((:bk_vec_scale, lib), Int32, (Ptr{Cvoid}, Ptr{Float64}, Float64, Int64), x.ctx.handle, x.ptr, a, x.n); x)
VI.scale!!(x::DeviceVec, a::Number) = VI.scale!(x, a)
VI.scale(x::DeviceVec, a::Number) = VI.scale!(copy(x), a)
VI.add!(y::DeviceVec, x::DeviceVec, a::Number = 1, b::Number = 1) = (ccall((:bk_vec_axpby, lib), Int32, (Ptr{Cvoid}, Ptr{Float64}, Float64, Ptr{Float64}, Float64, Int64), y.ctx.handle, y.ptr, a, x.ptr, b, y.n); y)
VI.add!!(y::DeviceVec, x::DeviceVec, a::Number = 1, b::Number = 1) = VI.add!(y, x, a, b)
VI.inner(x::DeviceVec, y::DeviceVec) = dot(x, y)
BK._copy(x::DeviceVec) = copy(x)
BK._copyto!(d::DeviceVec, s::DeviceVec) = copyto!(d, s)
BK.minus!!(x::DeviceVec, y::DeviceVec) = VI.add!(x, y, -1, 1)

# ---- F and J ----------------------------------------------------------------------------------------------------------
"F(u; p): prob.VF.F (src/Problems.jl:133)"
function residual(c::Context, u, params)
    setparams!(c, params)
    out = like(c, u)
    check(c, ccall((:bk_residual, lib), Int32, (Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}), c.handle, ptr(u), ptr(out)))
    out
end

"""J = prob.VF.J(u, p): 'any user struct' form (src/Problems.jl:98-101; pattern of examples/SH2d-fronts-cuda.jl:31-37).
Callable so that `apply(J, dx)` (src/Utils.jl:192) also works with stock solvers."""
struct Jac
    ctx::Context
end
function Jac(c::Context, u, params)
    setparams!(c, params)
    check(c, ccall((:bk_jac_set_state, lib), Int32, (Ptr{Cvoid}, Ptr{Float64}), c.handle, ptr(u)))
    Jac(c)
end
function (J::Jac)(dx; a₀ = 0.0, a₁ = 1.0)
    out = like(J.ctx, dx)
    check(J.ctx, ccall((:bk_jvp, lib), Int32, (Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}, Float64, Float64), J.ctx.handle, ptr(dx), ptr(out), a₀, a₁))
    out
end

# ---- :SPARSE contexts: J assembled by the user as a SparseMatrixCSC (J = Jbru_sp, examples/brusselator.jl:50-82) --------------
"""sparse!(ctx, J): load J on a :SPARSE context and return its `Jac`.  The pattern goes over once, as it is (CSC, 1-based
colptr / rowval, bk_sparse_set_pattern), and again only when it changes; the values go over on every call."""
function sparse!(c::Context, J::SparseMatrixCSC{Float64, Int})
    if c.pattern === nothing || c.pattern[1] != J.colptr || c.pattern[2] != J.rowval
        check(c, ccall((:bk_sparse_set_pattern, lib), Int32, (Ptr{Cvoid}, Int32, Int32, Int64, Ptr{Int64}, Ptr{Int64}),
                       c.handle, 1, 1, nnz(J), J.colptr, J.rowval))
        c.pattern = (copy(J.colptr), copy(J.rowval))
    end
    check(c, ccall((:bk_sparse_set_values, lib), Int32, (Ptr{Cvoid}, Ptr{Float64}), c.handle, nonzeros(J)))
    Jac(c)
end

# ---- AbstractIterativeLinearSolver (src/LinearSolver.jl:8-12,149-206) --------------------------------------------------
Base.@kwdef mutable struct GMRESB200 <: BK.AbstractIterativeLinearSolver
    ctx::Context
    abstol::Float64 = 0.0
    reltol::Float64 = 1e-8
    restart::Int64 = 200
    maxiter::Int64 = 100
    N::Int64 = 0
    Pl::Bool = false          # side on which the context's preconditioner (precond!) is applied
    Pr::Bool = false
    orth::Symbol = :cgs       # :cgs (single classical Gram-Schmidt pass) or :cgs2
    fused::Bool = true
end
GMRESB200(ctx::Context; k...) = GMRESB200(; ctx, k...)
opts(l::GMRESB200) = GmresOpts(l.reltol, l.abstol, l.restart, l.maxiter, l.Pl ? 1 : (l.Pr ? 2 : 0), l.orth == :cgs2 ? 1 : 0, l.fused ? 1 : 0, 0)
_num(a) = a === VI.Zero() ? 0.0 : (a === VI.One() ? 1.0 : Float64(a))

# (l::GMRESIterativeSolvers)(J, rhs; a₀, a₁) -> (x, converged, iters)   src/LinearSolver.jl:186-206
function (l::GMRESB200)(J::Jac, rhs; a₀ = VI.Zero(), a₁ = VI.One(), kwargs...)
    c = J.ctx; x = like(c, rhs); o = Ref(opts(l))
    cv = Ref{Int32}(0); it = Ref{Int32}(0); rn = Ref{Float64}(0.0)
    check(c, ccall((:bk_gmres, lib), Int32, (Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}, Float64, Float64, Ptr{GmresOpts}, Ptr{Int32}, Ptr{Int32}, Ptr{Float64}),
                   c.handle, ptr(rhs), ptr(x), _num(a₀), _num(a₁), o, cv, it, rn))
    cv[] == 0 && @debug "bk_gmres iterated maxiter = $(it[]) times without achieving the desired tolerance."
    return x, cv[] != 0, Int(it[])
end
# complex right-hand side / shift on a BK_COMPLEX context: the `shift = Complex(0, -ω)` solves of src/codim2/MinAugHopf.jl:17.
# J.ctx must have been created with complex = true; jacobian_adjoint maps to transpose!(ctx, true).
transpose!(c::Context, on::Bool) = check(c, ccall((:bk_jac_set_transpose, lib), Int32, (Ptr{Cvoid}, Int32), c.handle, on ? 1 : 0))
function (l::GMRESB200)(J::Jac, rhs::AbstractVector{<:Complex}; a₀ = VI.Zero(), a₁ = VI.One(), kwargs...)
    c = J.ctx; s = ComplexF64(a₀ === VI.Zero() ? 0 : (a₀ === VI.One() ? 1 : a₀))
    check(c, ccall((:bk_jac_set_shift_imag, lib), Int32, (Ptr{Cvoid}, Float64), c.handle, imag(s)))
    x, cv, it = try
        l(J, vcat(real(rhs), imag(rhs)); a₀ = real(s), a₁)
    finally
        ccall((:bk_jac_set_shift_imag, lib), Int32, (Ptr{Cvoid}, Float64), c.handle, 0.0)
    end
    n = length(rhs)
    return complex.(x[1:n], x[n+1:2n]), cv, it
end
# two right-hand sides (src/LinearSolver.jl:15-19): one ABI crossing, (x1, x2, flag1 & flag2, (it1, it2))
function (l::GMRESB200)(J::Jac, rhs1, rhs2; a₀ = VI.Zero(), a₁ = VI.One(), kwargs...)
    c = J.ctx; o = Ref(opts(l))
    x1, x2 = like(c, rhs1, length(rhs1)), like(c, rhs2, length(rhs2))
    cv = Ref{Int32}(0); its = zeros(Int32, 2)
    check(c, ccall((:bk_gmres2, lib), Int32, (Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Float64, Float64, Ptr{GmresOpts}, Ptr{Int32}, Ptr{Int32}),
                   c.handle, ptr(rhs1), ptr(rhs2), ptr(x1), ptr(x2), _num(a₀), _num(a₁), o, cv, its))
    return x1, x2, cv[] != 0, (Int(its[1]), Int(its[2]))
end

# ---- AbstractBorderedLinearSolver (src/LinearBorderSolver.jl:1-6) ------------------------------------------------------
Base.@kwdef struct BorderingBLSB200{S} <: BK.AbstractBorderedLinearSolver   # src/LinearBorderSolver.jl:59-166
    solver::S = nothing
    tol::Float64 = 1e-12
    check_precision::Bool = true
    k::Int64 = 1
end
BorderingBLSB200(ls::GMRESB200; k...) = BorderingBLSB200(; solver = ls, k...)   # BorderingBLS(solver; tol, check_precision, k), src/LinearBorderSolver.jl:59-75
BK.update_bls(b::BorderingBLSB200, ls) = BorderingBLSB200(ls, b.tol, b.check_precision, b.k)   # src/LinearBorderSolver.jl:38,490-493

struct MatrixFreeBLSB200{S} <: BK.AbstractBorderedLinearSolver                # src/LinearBorderSolver.jl:404-437
    solver::S
end
MatrixFreeBLSB200() = MatrixFreeBLSB200(nothing)
BK.update_bls(::MatrixFreeBLSB200, ls) = MatrixFreeBLSB200(ls)

# dotp handling: PALC passes dotp(x, y) = dot(x, y) / length(x) (src/continuation/Palc.jl:4, LinearBorderSolver.jl:22);
# the C ABI takes it as the scalar `dotscale`.
_dotscale(dotp, N) = dotp === LinearAlgebra.dot || dotp === VI.inner ? 1.0 : (dotp isa BK.NormalisedDot ? 1.0 / N : error("BK200: unsupported dotp"))

# (lbs)(J, dR, dzu, dzp, R, n, ξu, ξp; shift, dotp, applyξu!) -> (dX, dl, ok, iters)   src/LinearBorderSolver.jl:88-123
function (b::BorderingBLSB200)(J::Jac, dR, dzu, dzp::T, R, n::T, ξu = one(T), ξp = one(T); shift = nothing, dotp = dot, applyξu! = nothing) where {T}
    c = J.ctx; dX = like(c, R); o = Ref(opts(b.solver))
    dl = Ref{Float64}(0.0); cv = Ref{Int32}(0); it = zeros(Int32, 2)
    check(c, ccall((:bk_bls_bordering, lib), Int32,
                   (Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}, Float64, Ptr{Float64}, Float64, Float64, Float64, Int32, Float64, Float64, Ptr{GmresOpts}, Int32, Int32, Float64, Ptr{Float64}, Ptr{Float64}, Ptr{Int32}, Ptr{Int32}),
                   c.handle, ptr(dR), ptr(dzu), dzp, ptr(R), n, ξu, ξp, isnothing(shift) ? 0 : 1, isnothing(shift) ? 0.0 : shift, _dotscale(dotp, c.N), o,
                   b.check_precision ? 1 : 0, b.k, b.tol, ptr(dX), dl, cv, it))
    return dX, dl[], cv[] != 0, (Int(it[1]), Int(it[2]))
end

# (lbs::MatrixFreeBLS)(J, dR, dzu, dzp, R, n, ξu, ξp; shift, dotp) -> (dX, dl, cv, it)   src/LinearBorderSolver.jl:424-437
function (b::MatrixFreeBLSB200)(J::Jac, dR, dzu, dzp::T, R, n::T, ξu = 1, ξp = 1; shift = nothing, dotp = dot, applyξu! = nothing) where {T <: Number}
    c = J.ctx; dX = like(c, R); o = Ref(opts(b.solver))
    dl = Ref{Float64}(0.0); cv = Ref{Int32}(0); it = Ref{Int32}(0)
    check(c, ccall((:bk_bls_matrixfree, lib), Int32,
                   (Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}, Float64, Ptr{Float64}, Float64, Float64, Float64, Int32, Float64, Float64, Ptr{GmresOpts}, Ptr{Float64}, Ptr{Float64}, Ptr{Int32}, Ptr{Int32}),
                   c.handle, ptr(dR), ptr(dzu), dzp, ptr(R), n, ξu, ξp, isnothing(shift) ? 0 : 1, isnothing(shift) ? 0.0 : shift, _dotscale(dotp, c.N), o, ptr(dX), dl, cv, it))
    return dX, dl[], cv[] != 0, Int(it[])
end

# solve_bls_block with one or two borders (src/LinearBorderSolver.jl:173-206 and :440-450): a, b tuples of vectors, c the m x m corner
function BK.solve_bls_block(lbs::BorderingBLSB200, J::Jac, a::NTuple{M}, b::NTuple{M}, c::AbstractMatrix, rhst, rhsb; shift = nothing) where {M}
    (1 <= M <= 2 && size(c) == (M, M)) || error("Linear bordered solver, wrong sizes!")
    ctx = J.ctx; u = like(ctx, rhst); o = Ref(opts(lbs.solver))
    pa = Ptr{Float64}[ptr(v) for v in a]; pb = Ptr{Float64}[ptr(v) for v in b]
    cm = Matrix{Float64}(c); rb = collect(Float64, rhsb); sp = zeros(M); cv = Ref{Int32}(0); it = zeros(Int32, 3)
    GC.@preserve a b check(ctx, ccall((:bk_bls_block_bordering, lib), Int32,
        (Ptr{Cvoid}, Int32, Ptr{Ptr{Float64}}, Ptr{Ptr{Float64}}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Int32, Float64, Ptr{GmresOpts}, Ptr{Float64}, Ptr{Float64}, Ptr{Int32}, Ptr{Int32}),
        ctx.handle, M, pa, pb, cm, ptr(rhst), rb, isnothing(shift) ? 0 : 1, isnothing(shift) ? 0.0 : shift, o, ptr(u), sp, cv, it))
    return u, sp, cv[] != 0, Tuple(Int.(it[1:M+1]))
end
function BK.solve_bls_block(lbs::MatrixFreeBLSB200, J::Jac, a::NTuple{M}, b::NTuple{M}, c::AbstractMatrix, rhst, rhsb; shift = nothing, dotp = dot) where {M}
    (1 <= M <= 2 && size(c) == (M, M)) || error("Linear bordered solver, wrong sizes!")
    ctx = J.ctx; u = like(ctx, rhst); o = Ref(opts(lbs.solver))
    pa = Ptr{Float64}[ptr(v) for v in a]; pb = Ptr{Float64}[ptr(v) for v in b]
    cm = Matrix{Float64}(c); rb = collect(Float64, rhsb); sp = zeros(M); cv = Ref{Int32}(0); it = Ref{Int32}(0)
    GC.@preserve a b check(ctx, ccall((:bk_bls_block_matrixfree, lib), Int32,
        (Ptr{Cvoid}, Int32, Ptr{Ptr{Float64}}, Ptr{Ptr{Float64}}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Int32, Float64, Float64, Ptr{GmresOpts}, Ptr{Float64}, Ptr{Float64}, Ptr{Int32}, Ptr{Int32}),
        ctx.handle, M, pa, pb, cm, ptr(rhst), rb, isnothing(shift) ? 0 : 1, isnothing(shift) ? 0.0 : shift, _dotscale(dotp, ctx.N), o, ptr(u), sp, cv, it))
    return u, sp, cv[] != 0, Int(it[])
end

# ---- AbstractEigenSolver (src/EigSolver.jl:4-8,246-266) ----------------------------------------------------------------
struct ShiftInvertB200 <: BK.AbstractEigenSolver
    ctx::Context
    sigma::Float64
    ls::GMRESB200
    krylovdim::Int
    tol::Float64
    maxrestart::Int
end
ShiftInvertB200(ctx, sigma, ls; krylovdim = 0, tol = 1e-10, maxrestart = 20) = ShiftInvertB200(ctx, sigma, ls, krylovdim, tol, maxrestart)
BK.geteigenvector(::ShiftInvertB200, vecs, n::Union{Int, AbstractVector{Int64}}) = vecs[:, n]        # src/EigSolver.jl:12

# (eig)(J, nev; kwargs...) -> (vals::Vector{Complex}, vecs, converged, niter), vals by decreasing real part (EigSolver.jl:16-19,257-266)
function (e::ShiftInvertB200)(J::Jac, nev; kwargs...)
    c = J.ctx; kd = e.krylovdim > 0 ? e.krylovdim : max(30, nev + 30)    # examples/SH3d.jl:110
    re = zeros(nev); im_ = zeros(nev); vecs = zeros(c.N, nev); o = Ref(opts(e.ls))
    nconv = Ref{Int32}(0); nops = Ref{Int32}(0)
    check(c, ccall((:bk_eigs_shift_invert, lib), Int32,
                   (Ptr{Cvoid}, Float64, Int32, Int32, Float64, Int32, Ptr{GmresOpts}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Int32}, Ptr{Int32}),
                   c.handle, e.sigma, nev, kd, e.tol, e.maxrestart, o, C_NULL, re, im_, vecs, nconv, nops))
    return complex.(re, im_), vecs, nconv[] >= nev, Int(nops[])
end

# ---- the plugin surfaces for J::SparseMatrixCSC (a :SPARSE context; GMRESIterativeSolvers takes any J with mul!,
# src/LinearSolver.jl:186-206): load J with sparse! on the solver's context, then the Jac methods above
(l::GMRESB200)(J::SparseMatrixCSC, rhs; k...) = l(sparse!(l.ctx, J), rhs; k...)
(l::GMRESB200)(J::SparseMatrixCSC, rhs1, rhs2; k...) = l(sparse!(l.ctx, J), rhs1, rhs2; k...)
(b::BorderingBLSB200)(J::SparseMatrixCSC, args...; k...) = b(sparse!(b.solver.ctx, J), args...; k...)
(b::MatrixFreeBLSB200)(J::SparseMatrixCSC, args...; k...) = b(sparse!(b.solver.ctx, J), args...; k...)
BK.solve_bls_block(lbs::BorderingBLSB200, J::SparseMatrixCSC, a::NTuple{M}, b::NTuple{M}, c::AbstractMatrix, rhst, rhsb; k...) where {M} =
    BK.solve_bls_block(lbs, sparse!(lbs.solver.ctx, J), a, b, c, rhst, rhsb; k...)
BK.solve_bls_block(lbs::MatrixFreeBLSB200, J::SparseMatrixCSC, a::NTuple{M}, b::NTuple{M}, c::AbstractMatrix, rhst, rhsb; k...) where {M} =
    BK.solve_bls_block(lbs, sparse!(lbs.solver.ctx, J), a, b, c, rhst, rhsb; k...)
(e::ShiftInvertB200)(J::SparseMatrixCSC, nev; k...) = e(sparse!(e.ctx, J), nev; k...)

# ---- the all-native loop (optional): one ccall per BRANCH instead of a dozen per Newton iteration ------------------------
# bk_palc_run (include/bk200.h) runs continuation(prob, PALC(tangent, bls), opts; normC) of src/Continuation.jl:349-601 for the
# context's own problem inside the library (csrc/bk_palc_loop.hpp): same kernels in the same order as the plugin-surface
# path above, hence the same branch bit for bit.  Use it when no Julia callback is needed between the steps
# (detect_bifurcation = 0); everything else keeps going through continuation(...).
struct PalcOpts             # == bk_palc_opts
    ds::Cdouble; dsmin::Cdouble; dsmax::Cdouble; a::Cdouble; p_min::Cdouble; p_max::Cdouble
    theta::Cdouble; eta::Cdouble; newton_tol::Cdouble; fd_eps::Cdouble; bls_tol::Cdouble
    max_steps::Int32; newton_maxit::Int32; lens::Int32; tangent::Int32; bls::Int32
    bls_check_precision::Int32; bls_k::Int32; normc::Int32
end
struct PalcResult           # == bk_palc_result
    nrows::Int32; steps::Int32; nfail::Int32; stopped::Int32
    work_newton::Int64; work_linear::Int64; p_final::Cdouble; ds_final::Cdouble
end
"""
    continuation_native(ctx, u0, params, lens::Int, alg::PALC, contpar::ContinuationPar; normC = norm, u1 = nothing, p1 = 0.0)

`lens` = 1-based index of the continuation parameter inside `params`.  `alg.bls` is a `BorderingBLSB200` or a `MatrixFreeBLSB200`,
`contpar.newton_options.linsolver` a `GMRESB200`.  Returns `(rows, result)`: `rows[:, k] = (param, ‖u‖, itnewton, itlinear, ds, step)`
like `br.branch` (src/Continuation.jl:259-272), `result::PalcResult`, and the last state in a `DeviceVec`.
"""
function continuation_native(c::Context, u0, params, lens::Int, alg, contpar; normC = norm, u1 = nothing, p1 = 0.0)
    setparams!(c, params)
    ls = contpar.newton_options.linsolver
    b = alg.bls
    bord = b isa BorderingBLSB200
    po = Ref(PalcOpts(contpar.ds, contpar.dsmin, contpar.dsmax, contpar.a, contpar.p_min, contpar.p_max, alg.θ, contpar.η, contpar.newton_options.tol, 0.0,
                      bord ? b.tol : 0.0, contpar.max_steps, contpar.newton_options.max_iterations, lens - 1,
                      alg.tangent isa BK.Bordered ? 1 : 0, bord ? 1 : 0, bord && b.check_precision ? 1 : 0, bord ? b.k : 1,
                      normC === BK.norminf ? 1 : 0))
    o = Ref(opts(ls))
    maxrows = contpar.max_steps + 8
    rows = zeros(6, maxrows); res = Ref(PalcResult(0, 0, 0, 0, 0, 0, 0.0, 0.0)); uf = DeviceVec(c, c.N)
    st = GC.@preserve u0 u1 ccall((:bk_palc_run, lib), Int32,
        (Ptr{Cvoid}, Ptr{PalcOpts}, Ptr{GmresOpts}, Ptr{Float64}, Float64, Ptr{Float64}, Float64, Ptr{Float64}, Int32, Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Float64}, Ptr{PalcResult}),
        c.handle, po, o, ptr(u0), Float64(params[lens]), isnothing(u1) ? Ptr{Float64}(C_NULL) : ptr(u1), p1, rows, maxrows, C_NULL, C_NULL, uf.ptr, res)
    check(c, st)   # BK_ERR_STATE: "Newton failed to converge for the initial guess" (src/Continuation.jl:375-393)
    return rows[:, 1:res[].nrows], res[], uf
end

end # module
