// bk_common.cuh -- context, operator descriptor and small device helpers shared by the
// libbk200 translation units.  sm_100a only.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdlib.h>
#include <string>
#include <unordered_map>
#include <vector>
#include "../../include/bk200.h"
#include <nvtx3/nvToolsExt.h>   // header-only NVTX v3: ranges around the ABI entry points (visible in nsys / ncu --nvtx)

struct BkRange {  // RAII range
  explicit BkRange(const char* name) { nvtxRangePushA(name); }
  ~BkRange() { nvtxRangePop(); }
};

#define BK_MAX_PAR 8
#define BK_NSM_FALLBACK 148

// Operator descriptor, passed BY VALUE to kernels.  Describes  out = a0*in + a1*J(u)*in  for the
// named PDE stencils, optionally bordered (MatrixFreeBLSmap, src/LinearBorderSolver.jl:299-335).
struct OpDesc {
  int kind;
  int nx, ny, nz;        // grid (potrap: nz = M time slices)
  double cx, cy, cz;     // 1/h^2
  double par[BK_MAX_PAR];
  const double* u;       // linearisation state (device)
  double a0, a1;         // a0 I + a1 J
  long long N;           // unknowns of the un-bordered problem
  // bordered map:  out.u = Op(x.u) + x.p * ba (+ bshift * x.u);  out.p = bscale*<bb, x.u> + bc * x.p
  int bordered;          // number of borders: 0, 1 or 2
  const double* ba;
  const double* bb;
  double bc, bshift, bscale;
  // second border of the block / tuple form (src/LinearBorderSolver.jl:338-389): x.p and out.p have two entries,
  //   out.u += x.p[1] ba2;   out.p = bscale [<bb, x.u>; <bb2, x.u>] + [bc bc01; bc10 bc11] x.p
  const double* ba2;
  const double* bb2;
  double bc01, bc10, bc11;
  // potrap extras
  const double* phi;     // section (length N-1)
  const double* fcache;  // F(x_i) cache, M slices (device)
  // complexified contexts (BK_COMPLEX): N = 2 N0, vectors are [re; im], operator ((a0 + i a0i) I + a1 J) with J real
  int cplx;
  double a0i;
  int transpose;         // J' instead of J (cGL2d: transposed reaction block; SH: self-adjoint)
};

// general-length transform plan (bk_fft_gen.cuh), passed by value to the kernels
namespace bkg {
#define BKG_MAXPASS 16
struct Plan {
  int n;                   // line length
  int L;                   // FFT length: 2n (DCT-II, even extension) or 2n + 2 (DST-I, odd extension)
  int npass;
  int radix[BKG_MAXPASS];  // Stockham radices (prime factors of L, 4 preferred over 2 x 2)
  const double2* wl;       // W_L^t = exp(-2 pi i t / L), t < L
  const double2* ph;       // exp(-i pi k / 2n), k < n (DCT-II pre/post twiddle)
  double dst_scale;        // sqrt(2 / (n + 1)) / 2
};
}  // namespace bkg

// BK_SPARSE: one matrix in CSR form (int32 indices) plus the SpMV work partition built with the pattern (bk_sparse.cu)
struct SpCsr {
  long long n = 0, nnz = 0;
  int* rowptr = nullptr;   // n + 1
  int* col = nullptr;      // nnz
  double* val = nullptr;   // nnz, CSR order
  int* perm = nullptr;     // val[k] = src[perm[k]] (src: the caller's value order, or A's CSR values for A'); nullptr: identity
  int2* blocks = nullptr;  // per CTA: rows [x, y) handled by sub-warps of `width` lanes, or (row, -1): one long row, the whole CTA
  int nblocks = 0;
  int width = 32;
};
struct SparseMat {
  long long nnz = 0;
  SpCsr a;                          // J
  SpCsr at;                         // J', built at the first transposed application
  std::vector<int> h_rowptr, h_col; // host copy of J's CSR pattern (source of J')
  bool have_vals = false;
  bool at_built = false, at_vals = false;
  double* stage = nullptr;          // nnz: the caller's values in the caller's order (gather source when a.perm is set)
  double* diag = nullptr;           // N: diag(J), duplicates summed, 0 where structurally missing
};

struct Precond {
  int kind = BK_PC_NONE;
  double a0 = 0, a1 = 0;
  double* lam[3] = {nullptr, nullptr, nullptr};     // 1-D eigenvalues of the Laplacian factors (natural order)
  int ttype[3] = {0, 0, 0};                         // 0: DCT-II (Neumann), 1: DST-I (Dirichlet)
  // register-resident power-of-two kernels (bk_fft_fast.cuh): log2(n) or 0, and their tables
  int fast[3] = {0, 0, 0};
  double2* ftw[3] = {nullptr, nullptr, nullptr};    // per-pass contiguous FFT twiddles
  double2* fom[3] = {nullptr, nullptr, nullptr};    // w_k = exp(-i pi k / 2n), register-major
  double2* flam2[3] = {nullptr, nullptr, nullptr};  // (lambda[k], lambda[n-k]), register-major
  // general lengths (bk_fft_gen.cuh)
  bkg::Plan gplan[3] = {};
  double2* gwl[3] = {nullptr, nullptr, nullptr};
  double2* gph[3] = {nullptr, nullptr, nullptr};
  double* work = nullptr;                           // scratch vector (N)
  double* work2 = nullptr;
  // chan tridiagonal LU factors
  double* tri = nullptr;
  // potrap circulant preconditioner
  double2* tdft = nullptr;   // exp(-2 pi i j / (M-1))
  double po_r = 0, po_nu = 0, po_T = 0;
  // Jacobi: out = in / (a0 + a1 diag(J)); the pivots are recomputed (and checked for zeros) at the first application after new values
  double* jpiv = nullptr;          // a0 + a1 diag(J)
  unsigned int* jflag = nullptr;
  bool jdirty = false;
};

struct bk_ctx {
  int device = 0;
  int nsm = BK_NSM_FALLBACK;
  cudaStream_t stream = nullptr;
  int kind = 0;
  long long dims[3] = {1, 1, 1};
  double lengths[3] = {1, 1, 1};
  double par[BK_MAX_PAR] = {0};
  long long N = 0;        // unknowns (BK_COMPLEX: 2 N0)
  long long N0 = 0;       // size of the real problem: length of the state u and of F(u)
  bool cplx = false;      // BK_COMPLEX context
  double shift_imag = 0;  // imaginary part of a0 (bk_jac_set_shift_imag)
  bool transpose = false; // bk_jac_set_transpose
  int m = 0;              // Krylov dimension capacity (basis holds m+1 vectors of length N+1)
  long long ld = 0;       // leading dimension of the basis (>= N+1, multiple of 32)
  // Jacobian state
  double* u_state = nullptr;
  double jpar[BK_MAX_PAR] = {0};
  bool have_state = false;
  // potrap
  double* phi = nullptr;
  double* xpi = nullptr;
  double* fcache = nullptr;
  double phi_dot_xpi = 0;
  // Krylov workspace
  double* V = nullptr;        // (m+1) x ld, unnormalised basis vectors v'_i
  double* w = nullptr;        // ld
  double* z = nullptr;        // ld  (preconditioned vector)
  double* r = nullptr;        // ld
  double* scales = nullptr;   // m+2 : s_i = 1/||v'_i||
  double* gcoef = nullptr;    // m+2 : g_i = h_i * s_i (device), also lincomb coefficients
  double* hcols = nullptr;    // (m+1) x (m+4) device H columns
  double* hcols2 = nullptr;   // second-pass (CGS2) corrections
  double* h_pinned = nullptr; // pinned host mirror of hcols (+ hcols2 behind it)
  double* partials = nullptr; // (m+4) x Gmax
  int gmax = 0;
  unsigned int* counters = nullptr; // last-block tickets
  double* red_out = nullptr;  // small device buffer for scalar reductions (16 doubles)
  double* red_pinned = nullptr;
  double* coef_pinned = nullptr; // m+2
  std::vector<cudaEvent_t> events;
  // staging buffers for host-pointer arguments
  std::vector<double*> stage;  // each ld doubles
  double* host_pinned = nullptr; // pinned bounce buffer (ld doubles) for pageable host memory
  // generic temporaries for BLS/eigs
  std::vector<double*> tmp;
  // bk_vec_alloc pool: live allocations (ptr -> padded length) and the recycled free list
  std::unordered_map<double*, size_t> vec_live;
  std::vector<std::pair<size_t, double*>> vec_pool;
  // eigensolver workspace (lazily allocated)
  double* Q = nullptr;       // (qcap+1) x ld Arnoldi basis of the shift-invert operator
  double* Q2 = nullptr;      // second basis buffer for thick restarts
  int q2cap = 0;
  int qcap = 0;
  double* eig_dev = nullptr; // ones (qcap+2) | hcolA (qcap+2) | hcolB (qcap+2) | g (qcap+2) | coef (2*(qcap+2))
  double* eig_pinned = nullptr;
  Precond pc;
  SparseMat* sp = nullptr;  // BK_SPARSE contexts
  bk_stats stats = {};
  bool timing = false;      // bk_set_timing: event pairs around the fused kernels / preconditioner applications
  int timing_every = 1;     // ... of every timing_every-th bk_gmres call only (event records sit between PDL launches: sampling keeps the overhead small)
  long long solve_count = 0;
  bool timing_now = false;  // decided per solve
  cudaEvent_t tev0 = nullptr, tev1 = nullptr;
  std::vector<std::pair<cudaEvent_t, cudaEvent_t>> tpairs;
  std::vector<std::pair<cudaEvent_t, cudaEvent_t>> pc_pairs;  // one pair per preconditioner application (timing enabled)
  size_t pc_pairs_used = 0;
  // dynamic shared memory this context has already asked for, per kernel (first-level filter in front of bk_grant_smem)
  std::unordered_map<const void*, size_t> smem_attr;
  std::string err;
};

// ---- error helpers ---------------------------------------------------------------------------
int bk_fail(bk_ctx* c, int code, const char* what, const char* file, int line);
#define BK_CUDA(c, expr)                                                             \
  do {                                                                               \
    cudaError_t _e = (expr);                                                         \
    if (_e != cudaSuccess) return bk_fail((c), BK_ERR_CUDA, cudaGetErrorString(_e), __FILE__, __LINE__); \
  } while (0)
#define BK_CHECK(c, cond, msg)                                                       \
  do {                                                                               \
    if (!(cond)) return bk_fail((c), BK_ERR_ARG, (msg), __FILE__, __LINE__);         \
  } while (0)
// first statement of every extern "C" entry point: a process may hold contexts on several GPUs (Context(device=...)),
// and kernel launches / cudaFuncSetAttribute / cudaMalloc all act on the CURRENT device
#define BK_ENTER(c)                                 \
  do {                                              \
    if (!(c)) return BK_ERR_ARG;                    \
    if (cudaSetDevice((c)->device) != cudaSuccess)  \
      return bk_fail((c), BK_ERR_CUDA, "cudaSetDevice failed", __FILE__, __LINE__); \
  } while (0)
#define BK_TRY(expr)                 \
  do {                               \
    int _s = (expr);                 \
    if (_s < 0) return _s;           \
  } while (0)

// ---- host-side internal API (cross-TU) ----------------------------------------------------------
bool bk_is_device_ptr(const void* p);
// Returns a device pointer for argument p (n doubles): p itself when device memory, else stage slot `slot`
// filled by H2D (when `in`).  For outputs call bk_stage_out afterwards.
int bk_stage_in(bk_ctx* c, const double* p, long long n, int slot, bool copy_in, double** dev);
int bk_stage_out(bk_ctx* c, double* p, long long n, const double* dev);

OpDesc bk_make_op(bk_ctx* c, double a0, double a1);
OpDesc bk_make_residual_op(bk_ctx* c);
int bk_launch_residual(bk_ctx* c, const double* u_dev, double* out_dev);
// out = a0*in*in_scale + a1*J*(in*in_scale) [+ bordered terms]; in_scale_ptr (device, may be NULL => 1)
int bk_launch_apply(bk_ctx* c, const OpDesc& op, const double* in_dev, const double* in_scale_ptr, double* out_dev);
int bk_potrap_refresh_cache(bk_ctx* c);

// BK_SPARSE (bk_sparse.cu): out = a0 s in + a1 A (s in) on N0 values, A = J or J' (op.transpose)
int bk_sparse_apply(bk_ctx* c, const OpDesc& op, const double* in_dev, const double* in_scale_ptr, double* out_dev);
void bk_sparse_free(bk_ctx* c);
int bk_jacobi_refresh(bk_ctx* c);                                         // pc.jinv from diag(J), pc.a0, pc.a1; zero pivot -> error
int bk_jacobi_apply(bk_ctx* c, const double* in_dev, double* out_dev);    // N0 values

int bk_precond_apply_dev(bk_ctx* c, const double* in_dev, double* out_dev, long long n);
void bk_harvest_pc_timing(bk_ctx* c);

// vector kernels (device pointers)
int bk_dev_axpby(bk_ctx* c, double* y, double a, const double* x, double b, long long n);
int bk_dev_scale(bk_ctx* c, double* x, double a, long long n);
int bk_dev_dot(bk_ctx* c, const double* x, const double* y, long long n, double* out_host);
int bk_dev_norminf(bk_ctx* c, const double* x, long long n, double* out_host);
int bk_dev_copy(bk_ctx* c, double* dst, const double* src, long long n);

// GMRES on device pointers; n = op.N (+1 if bordered)
int bk_gmres_dev(bk_ctx* c, const OpDesc& op, const double* rhs_dev, double* x_dev, const bk_gmres_opts* o,
                 int* converged, int* iters, double* resnorm);
// Arnoldi building blocks (used by the eigensolver): dots h_i = s_i <B_i, w> (also g_i = h_i s_i), update
// vout = w - sum g_i B_i with its norm -> *h_out, 1/norm -> *scale_out, and x = beta x + sum coef_i s_i B_i.
int bk_launch_dots(bk_ctx* c, const double* basis, const double* scales, const double* w, long long n, int j, double* hcol,
                   double* gcoef);
int bk_launch_update(bk_ctx* c, const double* basis, const double* gcoef, const double* w, long long n, int j, double* vout,
                     double* h_out, double* scale_out);
int bk_launch_lincomb(bk_ctx* c, const double* basis, const double* scales, double* x, double beta, long long n, int k,
                      const double* coef_dev);
int bk_tmp(bk_ctx* c, int slot, double** out);  // lazily allocated ld-sized temporaries

// grant `bytes` of dynamic shared memory to `kern` on the context's device.  cudaFuncAttributeMaxDynamicSharedMemorySize is a
// property of (device, kernel), shared by every context of the process: the grant only ever grows (bk_grant_smem keeps the
// process-wide maximum under a mutex -- a context with a smaller Krylov dimension must not shrink what another one needs),
// and the per-context map is just a lock-free first-level filter.
void bk_grant_smem(int device, const void* kern, size_t bytes);
template <typename K>
static inline void bk_ensure_smem(bk_ctx* c, K kern, size_t bytes) {
  size_t& cur = c->smem_attr[(const void*)kern];
  if (bytes > cur) {
    bk_grant_smem(c->device, (const void*)kern, bytes);
    cur = bytes;
  }
}

// ---- programmatic dependent launch (PDL): the next kernel of the stream is launched while this one drains ---------
#ifdef __CUDACC__
template <typename... KArgs, typename... Args>
static inline cudaError_t bk_launch_pdl(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st,
                                        Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at;
  static int no_pdl = -1;  // BK_NO_PDL=1: plain stream order (diagnostics)
  if (no_pdl < 0) no_pdl = getenv("BK_NO_PDL") ? 1 : 0;
  cfg.numAttrs = no_pdl ? 0 : 1;
  return cudaLaunchKernelEx(&cfg, kern, KArgs(args)...);
}
// first statement of every kernel launched through bk_launch_pdl: wait for the previous grid's memory, then let the next
// grid start launching (its CTAs block at their own wait)
__device__ __forceinline__ void bk_pdl_sync() {
  asm volatile("griddepcontrol.wait;" ::: "memory");
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
}
#endif

// ---- device helpers ---------------------------------------------------------------------------
#ifdef __CUDACC__
__device__ __forceinline__ double bk_warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
// NaN-propagating max: fmax() drops NaN, which would turn an all-NaN residual into norminf = 0 ("converged").
// norm(x, Inf) of the reference returns NaN there and the step is rejected (src/continuation/Palc.jl:228-231).
__device__ __forceinline__ double bk_nanmax(double a, double b) { return (a != a) ? a : ((b != b) ? b : fmax(a, b)); }
__device__ __forceinline__ double bk_warp_max(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = bk_nanmax(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
// Grid-wide "last block done" ticket.  Returns true in exactly one block (the last to arrive),
// after all other blocks' prior global writes are visible.  Resets the counter for the next launch.
__device__ __forceinline__ bool bk_last_block(unsigned int* counter, int* s_flag) {
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned int t = atomicAdd(counter, 1u);
    int last = (t == gridDim.x * gridDim.y * gridDim.z - 1);
    if (last) *counter = 0u;
    *s_flag = last;
  }
  __syncthreads();
  bool last = (*s_flag != 0);
  if (last) __threadfence();
  return last;
}
#endif
