/* bk200.h -- C ABI of libbk200.so: the B200-native Newton-Krylov corrector hot path of
 * BifurcationKit.jl's pseudo-arclength continuation (PALC).
 *
 * Every entry point replaces the arithmetic behind one reference plugin surface; the citation
 * after each prototype is the reference interface (file:line under the BifurcationKit.jl tree)
 * whose work it performs.  The Julia-side binding (ccall stubs + the three plugin structs) is in
 * julia/BK200.jl and INTEGRATION.md; the Python ctypes binding used by the tests and the
 * benchmark is bifurcationkit.jl_b200/lib.py.
 *
 * Conventions
 *   - Every function returns int32 status: 0 ok, >0 non-fatal (BK_NOT_CONVERGED), <0 error;
 *     the message for the last error of a context is bk_last_error(ctx).  Nothing throws or
 *     aborts across the boundary (the reference only logs linear-solver non-convergence,
 *     src/LinearSolver.jl:202-205).
 *   - All vectors are fp64.  A `const double*` / `double*` vector argument may be EITHER a host
 *     pointer (option A: the library stages it through device scratch, H2D/D2H inside the call)
 *     OR a device pointer obtained from bk_vec_alloc (option B: zero copies).  The library tells
 *     them apart with cudaPointerGetAttributes.  The caller owns every pointer; the library never
 *     retains a caller pointer past the call (bk_jac_set_state COPIES u).
 *   - One context per GPU; a context is not thread-safe; calls are synchronous with respect to
 *     host-visible outputs.
 *   - Layout: Julia column-major, x fastest: u[i + j*Nx (+ k*Nx*Ny)], 0-based here.
 */
#ifndef BK200_H
#define BK200_H
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

typedef struct bk_ctx bk_ctx;

enum { BK_OK = 0, BK_NOT_CONVERGED = 1, BK_ERR_ARG = -1, BK_ERR_CUDA = -2, BK_ERR_STATE = -3 };

/* problem kinds = the named PDE stencils (SURVEY.md section 8a, P1-P5) */
enum {
  BK_CHAN = 1,   /* examples/chan.jl:5-19,85-95      params (alpha, beta)            dims (n)        */
  BK_SH2D = 2,   /* examples/SH2d-fronts.jl:13-34,124-127  params (l, nu)           dims (Nx,Ny)    */
  BK_SH3D = 3,   /* examples/SH3d.jl:16-53           params (l, nu)                  dims (Nx,Ny,Nz) */
  BK_CGL2D = 4,  /* examples/cGL2d.jl:6-22,262-318   params (r, mu, nu, c3, c5)      dims (Nx,Ny), N = 2 Nx Ny */
  BK_POTRAP_CGL2D = 5, /* src/periodicorbit/PeriodicOrbitTrapeze.jl:209-330 over BK_CGL2D; dims (Nx,Ny,M), N = 2 Nx Ny M + 1 */
  /* a Jacobian assembled by the caller as a sparse matrix (J = Jbru_sp, examples/brusselator.jl:50-82; JFmit, examples/
   * mittleman.jl:56-63; any J supporting mul!, GMRESIterativeSolvers src/LinearSolver.jl:149-206).  dims (N) or a grid
   * (Nx, Ny[, Nz]) with N = Nx Ny Nz: a grid shape lets BK_PC_SH_DCT / BK_PC_CGL_DST be set up on the context (lengths are only
   * read by them).  The operator is the matrix of bk_sparse_set_pattern + bk_sparse_set_values; bk_jac_set_state stays legal
   * (it snapshots u and the parameters) but the operator does not read u.  F is the caller's: bk_residual and bk_palc_run fail. */
  BK_SPARSE = 6,
  /* OR-ed into one of the kinds above (not BK_POTRAP_CGL2D): a COMPLEXIFIED context for the complex shifts of the Hopf
   * minimally augmented system (src/codim2/MinAugHopf.jl:19-40, shift = Complex(0, -omega)) and complex eigenvector work.
   * Unknowns are z = x + i y stored split, [x; y]: bk_problem_size = 2 N0, with N0 = bk_state_size the size of the real
   * problem.  The operator of bk_jvp / bk_gmres / bk_gmres2 is ((a0 + i a0_imag) I + a1 J) z with the REAL Jacobian J (or its
   * transpose) acting on both halves; a0_imag comes from bk_jac_set_shift_imag.  GMRES runs on the real-equivalent 2 N0 system
   * (inner product Re<.,.>), the preconditioner is applied to both halves.  bk_residual / bk_jac_set_state still take real
   * N0-vectors. */
  BK_COMPLEX = 0x100
};

/* preconditioner kinds (the reference's Pl/Pr contract: src/Preconditioner.jl:11-37; the
 * examples use sparse factorisations: SH2d-fronts.jl:120-122 lu(L1+I), SH3d.jl:88, chan.jl:108-111) */
enum {
  BK_PC_NONE = 0,
  BK_PC_SH_DCT = 1,     /* (L1 + shift I)^-1 by separable DCT-II (exact for the Neumann-closure operator) */
  BK_PC_CHAN_TRIDIAG = 2, /* lu(P), P = tridiagonal Laplacian with identity boundary rows (chan.jl:108-109) */
  BK_PC_CGL_DST = 3,    /* per-component (a0 I + a1 Lap_dirichlet)^-1 by DST-I (block Jacobi over slices) */
  BK_PC_POTRAP_CIRC = 4, /* Trapeze PO Jacobian of cGL linearised at the trivial state: DST-I in space (mixed-radix FFT of the odd extension, bk_fft_gen.cuh),
                           u1 +- i u2, DFT over the M-1 cyclic slices, scalar symbol; a0 = period T.  Stand-in for the ILU
                           of the assembled PO Jacobian (examples/cGL2d.jl:209-213) */
  BK_PC_JACOBI = 5      /* (a0 I + a1 diag(J))^-1 with the current values of a BK_SPARSE context (a structurally missing diagonal
                           entry counts as 0; a zero pivot is an error at setup, or at the first apply after new values).  The diagonal preconditioner a user
                           passes as Pl = Diagonal(...) to GMRESIterativeSolvers (src/LinearSolver.jl:149-182) */
};
/* sparse pattern formats of bk_sparse_set_pattern: CSC is Julia's SparseMatrixCSC (colptr, rowval) */
enum { BK_SPARSE_CSR = 0, BK_SPARSE_CSC = 1 };
enum { BK_SIDE_NONE = 0, BK_SIDE_LEFT = 1, BK_SIDE_RIGHT = 2 };
enum { BK_ORTH_CGS = 0, BK_ORTH_CGS2 = 1 };

/* GMRES options = fields of GMRESIterativeSolvers (src/LinearSolver.jl:149-182) */
typedef struct bk_gmres_opts {
  double reltol;   /* 1e-8 */
  double abstol;   /* 0    */
  int32_t restart; /* 200  */
  int32_t maxiter; /* 100  */
  int32_t pc_side; /* BK_SIDE_*: which of Pl / Pr holds the context's preconditioner */
  int32_t orth;    /* BK_ORTH_CGS (single classical Gram-Schmidt pass) or BK_ORTH_CGS2 */
  int32_t fused;   /* 0: separate kernels; 1: automatic (JVP fused into the Arnoldi dot kernel where that is the fastest
                      arrangement: 2-D SH incl. the bordered map); 2: fused wherever a fused kernel exists (also 3-D SH) */
  int32_t reserved;
} bk_gmres_opts;

/* per-call statistics (all optional outputs may be NULL) */
typedef struct bk_stats {
  int64_t kernel_launches; /* kernels launched by this context since creation */
  int64_t h2d_bytes, d2h_bytes;
  double  last_fused_ms;   /* device time of the fused JVP+Arnoldi kernels in the last bk_gmres call (0 unless timing enabled) */
  int64_t last_fused_bytes;/* algorithmic bytes moved by them, 8N(2j+4) summed over the iterations run */
  int64_t last_fused_launches;
  double  total_fused_ms;     /* cumulative over all solves that ran the FUSED JVP+Arnoldi kernel (timing enabled) */
  int64_t total_fused_bytes;  /* cumulative algorithmic bytes of those launches */
  int64_t total_fused_launches;
  int64_t cgs_fallbacks;      /* solves whose single-pass CGS cycle failed the true-residual check and continued with CGS2 */
  double  total_precond_ms;   /* cumulative device time of preconditioner applications inside bk_gmres (timing enabled) */
  int64_t total_precond_applies;
} bk_stats;

/* ---- context --------------------------------------------------------------------------- */
int32_t bk_ctx_create(int32_t device, int32_t problem_kind, const int64_t dims[3], const double lengths[3],
                      int32_t krylov_m, bk_ctx** out);
int32_t bk_ctx_destroy(bk_ctx* ctx);
const char* bk_last_error(bk_ctx* ctx);
int64_t bk_problem_size(bk_ctx* ctx);                       /* N = number of unknowns of F */
int64_t bk_state_size(bk_ctx* ctx);                         /* N0: length of u in bk_residual / bk_jac_set_state (= N unless BK_COMPLEX) */
int32_t bk_set_params(bk_ctx* ctx, const double* params, int32_t n);
int32_t bk_get_stats(bk_ctx* ctx, bk_stats* out);
int32_t bk_set_timing(bk_ctx* ctx, int32_t on);              /* CUDA-event timing of the fused kernels and the preconditioner: 0 off, 1 every bk_gmres call, k > 1 every k-th call (the event records sit between PDL launches; sampling keeps the overhead small) */
int32_t bk_sync(bk_ctx* ctx);
void*   bk_stream(bk_ctx* ctx);                              /* cudaStream_t the kernels are launched on */

/* ---- S11 device vectors: BorderedArray / VectorInterface algebra (src/BorderedArrays.jl:30-35,53-70,79-217) */
int32_t bk_vec_alloc(bk_ctx* ctx, int64_t n, double** out);
int32_t bk_vec_free(bk_ctx* ctx, double* v);
/* pinned (page-locked) host buffers for callers that keep the state on the host (option A) */
int32_t bk_host_alloc(bk_ctx* ctx, int64_t n, double** out);
int32_t bk_host_free(bk_ctx* ctx, double* p);
int32_t bk_vec_upload(bk_ctx* ctx, double* dst_dev, const double* src_host, int64_t n);
int32_t bk_vec_download(bk_ctx* ctx, double* dst_host, const double* src_dev, int64_t n);
int32_t bk_vec_copy(bk_ctx* ctx, double* dst, const double* src, int64_t n);          /* _copyto! */
int32_t bk_vec_zero(bk_ctx* ctx, double* x, int64_t n);                                 /* zerovector! */
int32_t bk_vec_scale(bk_ctx* ctx, double* x, double a, int64_t n);                      /* VI.scale! */
int32_t bk_vec_axpby(bk_ctx* ctx, double* y, double a, const double* x, double b, int64_t n); /* VI.add!(y,x,a,b): y = a x + b y */
int32_t bk_vec_dot(bk_ctx* ctx, const double* x, const double* y, int64_t n, double* out); /* VI.inner */
int32_t bk_vec_norm2(bk_ctx* ctx, const double* x, int64_t n, double* out);
int32_t bk_vec_norminf(bk_ctx* ctx, const double* x, int64_t n, double* out);           /* normC = norminf, src/LinearSolver.jl:4 */
/* S8: arc_length_eq (src/continuation/Palc.jl:44-56): theta*<x - x0, tau>/N in one fused reduction; out = <x - x0, tau> */
int32_t bk_vec_diffdot(bk_ctx* ctx, const double* x, const double* x0, const double* tau, int64_t n, double* out);

/* ---- K1/K2: the named PDE stencils ------------------------------------------------------- */
int32_t bk_residual(bk_ctx* ctx, const double* u, double* out);        /* F(u; params)  (prob.VF.F, src/Problems.jl:133) */
int32_t bk_jac_set_state(bk_ctx* ctx, const double* u);                /* J = jacobian(prob,u,params): copies u + current params (src/Problems.jl:98-101) */
int32_t bk_jvp(bk_ctx* ctx, const double* v, double* out, double a0, double a1); /* out = a0 v + a1 J v (_axpy_op, src/LinearSolver.jl:46-62) */
/* BK_COMPLEX contexts: imaginary part of the shift a0 of every later operator application (default 0) */
int32_t bk_jac_set_shift_imag(bk_ctx* ctx, double a0_imag);
/* apply J' instead of J from now on: apply_jacobian(prob, x, par, dx, true) / jacobian_adjoint (src/codim2/MinAugHopf.jl:79-81,
 * 152-155).  SH2d / SH3d are self-adjoint (no-op), cGL2d transposes its 2 x 2 reaction block, BK_SPARSE applies the transposed
 * matrix; BK_CHAN / BK_POTRAP_CGL2D: error */
int32_t bk_jac_set_transpose(bk_ctx* ctx, int32_t on);

/* ---- BK_SPARSE contexts: the Jacobian as a caller-assembled sparse matrix (J::SparseMatrixCSC of the examples above; the
 * linear solvers only need mul!, src/LinearSolver.jl:186-206).
 *   bk_sparse_set_pattern: format BK_SPARSE_CSR (ptr = row pointers, idx = column indices) or BK_SPARSE_CSC (ptr = colptr,
 *   idx = rowval, Julia's layout passed unchanged with index_base = 1); HOST arrays, ptr of length N + 1, idx of length nnz.
 *   Checked: ptr monotone from base to nnz + base, every index in range, N and nnz below 2^31 (else BK_ERR_ARG with a message).
 *   Duplicate entries are summed (as scipy and SparseArrays do), indices need not be sorted.  Setting a pattern drops the values.
 *   bk_sparse_set_values: nnz values in the pattern's order, host or device pointer; J is the matrix of the last values given (it
 *   also refreshes the diagonal of BK_PC_JACOBI).  bk_jac_set_transpose(ctx, 1) applies J' (the adjoint of MinAugHopf.jl:79-81). */
int32_t bk_sparse_set_pattern(bk_ctx* ctx, int32_t format, int32_t index_base, int64_t nnz, const int64_t* ptr, const int64_t* idx);
int32_t bk_sparse_set_values(bk_ctx* ctx, const double* vals);

/* ---- K6: preconditioner --------------------------------------------------------------------- */
int32_t bk_precond_setup(bk_ctx* ctx, int32_t kind, double a0, double a1); /* SH_DCT: (L1 + a0 I)^-1; CGL_DST: (a0 I + a1 Lap)^-1 */
int32_t bk_precond_apply(bk_ctx* ctx, const double* in, double* out);  /* ldiv!(out, P, in) (src/Preconditioner.jl:11-37) */

/* ---- S1/S2: GMRES = (l::GMRESIterativeSolvers)(J, rhs; a0, a1) (src/LinearSolver.jl:186-206, 15-19) */
int32_t bk_gmres(bk_ctx* ctx, const double* rhs, double* x, double a0, double a1, const bk_gmres_opts* opts,
                 int32_t* converged, int32_t* iters, double* resnorm);
int32_t bk_gmres2(bk_ctx* ctx, const double* rhs1, const double* rhs2, double* x1, double* x2, double a0, double a1,
                  const bk_gmres_opts* opts, int32_t* converged, int32_t iters[2]);

/* ---- S3/S4/S5: bordered linear solvers (src/LinearBorderSolver.jl:88-166, 299-335, 404-437)
 *   [ shift I + J     dR    ] [dX]   [R]
 *   [ xiu dzu'      xip dzp ] [dl] = [n],     dotp(x,y) = dotscale * <x,y>  (PALC: 1/N, Palc.jl:4)      */
int32_t bk_bls_bordering(bk_ctx* ctx, const double* dR, const double* dzu, double dzp, const double* R, double n,
                         double xiu, double xip, int32_t has_shift, double shift, double dotscale,
                         const bk_gmres_opts* opts, int32_t check_precision, int32_t k, double tol,
                         double* dX, double* dl, int32_t* converged, int32_t iters[2]);
int32_t bk_bls_matrixfree(bk_ctx* ctx, const double* dR, const double* dzu, double dzp, const double* R, double n,
                          double xiu, double xip, int32_t has_shift, double shift, double dotscale,
                          const bk_gmres_opts* opts, double* dX, double* dl, int32_t* converged, int32_t* iters);
/* the bordered map alone: out = MatrixFreeBLSmap(J,a,b,c,shift)(x), x and out of length N+1 (src/LinearBorderSolver.jl:312-325) */
int32_t bk_bls_map(bk_ctx* ctx, const double* a, const double* b, double c, int32_t has_shift, double shift, double dotscale,
                   const double* x, double* out);

/* block / tuple borders, m = 1 or 2 (solve_bls_block, src/LinearBorderSolver.jl:168-206 and :440-450 over the tuple form of
 * MatrixFreeBLSmap :338-389 -- the bordered systems of the Hopf / codim-2 formulations):
 *   [ shift I + J   a[0] .. a[m-1] ] [solu]   [rhst]
 *   [ dotp(b[i], .)       c        ] [solp] = [rhsb],   c is m x m column-major, rhsb / solp are HOST arrays of m doubles,
 * a[i] / b[i] / rhst / solu are host or device vectors of length N.  bordering: m + 1 solves with J and the Schur complement
 * (plain <.,.>, as the reference's VI.inner); matrixfree: one GMRES on the (N + m) system, dotp = dotscale <.,.>. */
int32_t bk_bls_block_bordering(bk_ctx* ctx, int32_t m, const double* const* a, const double* const* b, const double* c,
                               const double* rhst, const double* rhsb, int32_t has_shift, double shift,
                               const bk_gmres_opts* opts, double* solu, double* solp, int32_t* converged, int32_t iters[3]);
int32_t bk_bls_block_matrixfree(bk_ctx* ctx, int32_t m, const double* const* a, const double* const* b, const double* c,
                                const double* rhst, const double* rhsb, int32_t has_shift, double shift, double dotscale,
                                const bk_gmres_opts* opts, double* solu, double* solp, int32_t* converged, int32_t* iters);
int32_t bk_bls_block_map(bk_ctx* ctx, int32_t m, const double* const* a, const double* const* b, const double* c,
                         int32_t has_shift, double shift, double dotscale, const double* x, double* out); /* x, out: N + m */

/* ---- S10: shift-invert Arnoldi (src/EigSolver.jl:246-266; inner solver = bk_gmres with a0=-sigma)
 *   vals sorted by decreasing real part; vecs (N x nev, column-major, real Schur/Ritz vectors; complex pairs
 *   as (re, im) consecutive columns) may be NULL. */
int32_t bk_eigs_shift_invert(bk_ctx* ctx, double sigma, int32_t nev, int32_t krylovdim, double tol, int32_t maxrestart,
                             const bk_gmres_opts* inner, const double* v0, double* vals_re, double* vals_im, double* vecs,
                             int32_t* nconv, int32_t* nops);

/* host-only helper of the eigensolver: eigenpairs of a real upper-Hessenberg matrix (column-major, leading
 * dimension ldh), complex shifted QR + inverse iteration; vec_* are n x n column-major (may be NULL). */
int32_t bk_hessenberg_eig(const double* H, int32_t n, int32_t ldh, double* wr, double* wi, double* vec_re, double* vec_im);

/* ---- P5: trapezoid periodic-orbit functional over the context's vector field
 *   (BK_POTRAP_CGL2D contexts; x = [x_1..x_M; T], src/periodicorbit/PeriodicOrbitTrapeze.jl:249-330) */
int32_t bk_potrap_set_section(bk_ctx* ctx, const double* phi, const double* xpi); /* length N-1 each */

/* ---- the all-native PALC loop (SURVEY.md 8(b), optional entry): continuation(prob, PALC(...), opts; normC) of
 *   src/Continuation.jl:349-504, 506-601 for the context's problem -- two start-up Newton solves (src/Newton.jl:66-114), secant or
 *   Bordered tangent (src/continuation/Tangents.jl:8-42, 71-104), newton_palc corrector (src/continuation/Palc.jl:187-305,
 *   linesearch = false) on bk_bls_matrixfree / bk_bls_bordering, step-size control (src/continuation/Contbase.jl:77-102) -- as host
 *   C++ inside the library (csrc/bk_palc_loop.hpp), the state device-resident, one ABI crossing per BRANCH instead of a dozen per
 *   Newton iteration.  It issues exactly the kernel sequence of the plugin-surface loop (julia/BK200.jl under continuation(...), or
 *   bifurcationkit.jl_b200/palc.py), so the branch is bit-identical to that loop's.  detect_bifurcation = 0 (no eigen-solve per
 *   step; call bk_eigs_shift_invert from the callback if wanted). */
typedef struct bk_palc_opts {
  double ds, dsmin, dsmax, a, p_min, p_max;  /* ContinuationPar (src/ContParameters.jl:44-100) */
  double theta;                              /* PALC.theta (src/continuation/Palc.jl:70-84) */
  double eta;                                /* second start point at p0 + ds / eta (src/Continuation.jl:384) */
  double newton_tol;                         /* NewtonPar.tol */
  double fd_eps;                             /* finite-difference step of dF/dp (Palc.jl:239-240); 0: sqrt(eps) */
  double bls_tol;                            /* BorderingBLS.tol (check_precision) */
  int32_t max_steps, newton_maxit;
  int32_t lens;                              /* index of the continuation parameter in the context's parameter tuple */
  int32_t tangent;                           /* 0 secant, 1 Bordered() */
  int32_t bls;                               /* 0 MatrixFreeBLS, 1 BorderingBLS */
  int32_t bls_check_precision, bls_k;        /* BorderingBLS fields (src/LinearBorderSolver.jl:59-75) */
  int32_t normc;                             /* normC of the Newton residuals: 0 norm (2-norm), 1 norminf */
} bk_palc_opts;
enum { BK_PALC_ROW = 6 };                    /* doubles per row: param, ||u|| (record_from_solution), itnewton, itlinear, ds, step */
typedef struct bk_palc_result {
  int32_t nrows, steps, nfail;               /* rows written, accepted steps, rejected steps */
  int32_t stopped;                           /* 0 max_steps / parameter bound, 1 ds fell to dsmin, 2 callback, 3 row buffer full */
  int64_t work_newton, work_linear;          /* all corrector iterations, rejected attempts included */
  double p_final, ds_final;
} bk_palc_result;
/* called at step 0 and after every accepted step (finalise_solution / callback of the reference); z_u is the DEVICE state;
 * return 0 to stop the run */
typedef int32_t (*bk_palc_callback)(void* user, int32_t step, const double* row, const double* z_u, double z_p);
/* u0: start guess at p0 = params[lens] given by p0 (host or device, N doubles).  u1 != NULL: start from the two points (u0, p0),
 * (u1, p1) without Newton corrections (iterate_from_two_points, src/Continuation.jl:408-456).  rows: HOST array, max_rows x
 * BK_PALC_ROW.  u_final (may be NULL): last state, host or device.  Returns BK_ERR_STATE when a start-up Newton solve fails
 * (the reference throws there, src/Continuation.jl:375-393). */
int32_t bk_palc_run(bk_ctx* ctx, const bk_palc_opts* opts, const bk_gmres_opts* linsolver, const double* u0, double p0,
                    const double* u1, double p1, double* rows, int32_t max_rows, bk_palc_callback cb, void* user,
                    double* u_final, bk_palc_result* result);

/* ---- environment switches read once by the library (tuning / diagnostics; none is needed for normal use)
 *   BK2_E=1..8          tile height of the TMA-ring Arnoldi kernels instead of the heuristic (bk_krylov.cu::plan2)
 *   BK_NO_PDL=1         launch without programmatic dependent launch (plain stream order)
 *   BK_FFT_LOGE=2..5    complex values per thread (2^e) of the power-of-two transform kernels instead of the per-size default
 *   BK_FFT_NO_FAST=1    every transform through the general mixed-radix kernel (bk_fft_gen.cuh)
 *   BK_SH2D_NO_TMA=1    stand-alone SH2d residual / JVP on the first-generation 64 x 32 tile kernel instead of the TMA-staged tile */

#ifdef __cplusplus
}
#endif
#endif
