// bk_sparse.cu -- BK_SPARSE contexts: the Jacobian as a caller-assembled sparse matrix (Jbru_sp, examples/brusselator.jl:50-82;
// JFmit, examples/mittleman.jl:56-63; GMRESIterativeSolvers takes any J with mul!, src/LinearSolver.jl:149-206).
//   k_spmv         out = a0 s x + a1 A (s x), A = J or J' in CSR form, work partitioned by nnz at bk_sparse_set_pattern
//   k_gather       caller value order -> CSR order (CSC input), J -> J' values
//   k_diag         diag(J), duplicates summed (the Jacobi preconditioner)
//   k_jacobi_*     BK_PC_JACOBI pivots and application
// Every row sum is accumulated in a fixed order (no atomics on data): results are bit-reproducible, as every reduction here.
#include <algorithm>
#include <cstdio>
#include "bk_common.cuh"

#define BK_SP_THREADS 256
#define BK_SP_LONG 1024     // rows with more entries get a CTA of their own (a dense border row must not serialise a warp)
#define BK_SP_BUDGET 2048   // per-CTA work of a short-row block, in entries (a row costs at least one pass of its sub-warp)

// values and indices are streamed once per application: read-only path without L1 allocation (they stay in L2 when they fit)
__device__ __forceinline__ double ld_stream(const double* p) {
  double v;
  asm("ld.global.nc.L1::no_allocate.f64 %0, [%1];" : "=d"(v) : "l"(p));
  return v;
}
__device__ __forceinline__ int ld_stream(const int* p) {
  int v;
  asm("ld.global.nc.L1::no_allocate.s32 %0, [%1];" : "=r"(v) : "l"(p));
  return v;
}

// blocks[b] = (r0, r1): rows r0..r1-1, sub-warp of W lanes per row, rows dealt round-robin to the 256 / W sub-warps;
// blocks[b] = (r, -1): row r alone, all 256 threads (strided partial sums, warp tree, 8 warp sums in order)
template <int W>
static __global__ void __launch_bounds__(BK_SP_THREADS) k_spmv(const int* __restrict__ rowptr, const int* __restrict__ col,
                                                               const double* __restrict__ val, const int2* __restrict__ blocks,
                                                               const double* __restrict__ x, const double* __restrict__ in_scale_ptr,
                                                               double* __restrict__ out, double a0, double a1) {
  bk_pdl_sync();
  __shared__ double s_w[BK_SP_THREADS / 32];
  const int2 b = blocks[blockIdx.x];
  const double s = in_scale_ptr ? __ldg(in_scale_ptr) : 1.0;
  if (b.y < 0) {
    const int row = b.x;
    const int k0 = __ldg(rowptr + row), k1 = __ldg(rowptr + row + 1);
    double acc = 0.0;
    for (int k = k0 + threadIdx.x; k < k1; k += BK_SP_THREADS) acc = fma(ld_stream(val + k), __ldg(x + ld_stream(col + k)), acc);
    acc = bk_warp_sum(acc);
    if ((threadIdx.x & 31) == 0) s_w[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
      double t = 0.0;
      for (int w = 0; w < BK_SP_THREADS / 32; ++w) t += s_w[w];
      out[row] = a0 * (s * __ldg(x + row)) + a1 * (s * t);
    }
    return;
  }
  constexpr int G = BK_SP_THREADS / W;
  const int g = threadIdx.x / W, lane = threadIdx.x % W;
  for (int base = b.x; base < b.y; base += G) {  // uniform trip count: every lane reaches the shuffles
    const int row = base + g;
    double acc = 0.0;
    if (row < b.y) {
      const int k0 = __ldg(rowptr + row), k1 = __ldg(rowptr + row + 1);
      for (int k = k0 + lane; k < k1; k += W) acc = fma(ld_stream(val + k), __ldg(x + ld_stream(col + k)), acc);
    }
#pragma unroll
    for (int o = W / 2; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if (row < b.y && lane == 0) out[row] = a0 * (s * __ldg(x + row)) + a1 * (s * acc);
  }
}

static __global__ void __launch_bounds__(256) k_gather(double* __restrict__ dst, const double* __restrict__ src,
                                                       const int* __restrict__ perm, long long n) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    dst[i] = src[perm[i]];
}

static __global__ void __launch_bounds__(256) k_diag(const int* __restrict__ rowptr, const int* __restrict__ col,
                                                     const double* __restrict__ val, double* __restrict__ diag, long long n) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    double d = 0.0;
    for (int k = rowptr[i]; k < rowptr[i + 1]; ++k)
      if (col[k] == (int)i) d += val[k];
    diag[i] = d;
  }
}

static __global__ void __launch_bounds__(256) k_jacobi_piv(const double* __restrict__ diag, double* __restrict__ piv, double a0,
                                                           double a1, long long n, unsigned int* flag) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const double d = a0 + a1 * diag[i];
    if (d == 0.0) *flag = 1u;
    piv[i] = d;
  }
}

static __global__ void __launch_bounds__(256) k_jacobi_apply(const double* __restrict__ piv, const double* __restrict__ in,
                                                             double* __restrict__ out, long long n) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    out[i] = in[i] / piv[i];
}

// ------------------------------------------------------------------------------------------ host
static inline int sp_grid(bk_ctx* c, long long n) {
  long long g = (n + 255) / 256;
  long long cap = (long long)c->nsm * 8;
  return (int)(g < cap ? (g > 0 ? g : 1) : cap);
}

// (optr, oidx) compressed along one dimension (0-based) -> CSR compressed along the other, stable in the input order:
// CSC -> CSR, and CSR(A) -> CSR(A').  perm[p] = input position of output entry p.
static void recompress(long long n, const int* optr, const int* oidx, std::vector<int>& rp, std::vector<int>& cl,
                       std::vector<int>& perm) {
  const long long nnz = optr[n];
  rp.assign(n + 1, 0);
  cl.resize(nnz);
  perm.resize(nnz);
  for (long long k = 0; k < nnz; ++k) rp[oidx[k] + 1]++;
  for (long long i = 0; i < n; ++i) rp[i + 1] += rp[i];
  std::vector<int> pos(rp.begin(), rp.end() - 1);
  for (long long j = 0; j < n; ++j)
    for (int k = optr[j]; k < optr[j + 1]; ++k) {
      const int p = pos[oidx[k]]++;
      cl[p] = (int)j;
      perm[p] = k;
    }
}

// SpMV partition: long rows alone; runs of short rows in blocks of about BK_SP_BUDGET entries; the sub-warp width is the
// power of two (2..32) just above the mean length of the short rows
static void partition(const std::vector<int>& rp, long long n, std::vector<int2>& blocks, int& width) {
  long long short_rows = 0, short_nnz = 0;
  for (long long i = 0; i < n; ++i) {
    const int len = rp[i + 1] - rp[i];
    if (len <= BK_SP_LONG) {
      short_rows++;
      short_nnz += len;
    }
  }
  const double mean = short_rows ? (double)short_nnz / (double)short_rows : 0.0;
  int w = 2;
  while (w < 32 && w < mean) w <<= 1;
  width = w;
  const long long max_rows = 32LL * (BK_SP_THREADS / w);
  blocks.clear();
  long long i = 0;
  while (i < n) {
    if (rp[i + 1] - rp[i] > BK_SP_LONG) {
      blocks.push_back(make_int2((int)i, -1));
      ++i;
      continue;
    }
    const long long r0 = i;
    long long cost = 0;
    while (i < n) {
      const long long len = rp[i + 1] - rp[i];
      if (len > BK_SP_LONG) break;
      const long long ci = len > w ? len : w;
      if (i > r0 && (cost + ci > BK_SP_BUDGET || i - r0 >= max_rows)) break;
      cost += ci;
      ++i;
    }
    blocks.push_back(make_int2((int)r0, (int)i));
  }
}

template <typename T>
static int upload(bk_ctx* c, T** dst, const T* src, size_t count) {
  BK_CUDA(c, cudaMalloc(dst, sizeof(T) * (count > 0 ? count : 1)));
  if (count) BK_CUDA(c, cudaMemcpy(*dst, src, sizeof(T) * count, cudaMemcpyHostToDevice));
  return BK_OK;
}

static void free_csr(SpCsr& A) {
  void* bufs[] = {A.rowptr, A.col, A.val, A.perm, A.blocks};
  for (void* b : bufs)
    if (b) cudaFree(b);
  A = SpCsr();
}

static int upload_csr(bk_ctx* c, SpCsr& A, long long n, const std::vector<int>& rp, const std::vector<int>& cl,
                      const std::vector<int>* perm) {
  A.n = n;
  A.nnz = rp[n];
  BK_TRY(upload(c, &A.rowptr, rp.data(), (size_t)n + 1));
  BK_TRY(upload(c, &A.col, cl.data(), (size_t)A.nnz));
  BK_CUDA(c, cudaMalloc(&A.val, 8 * (size_t)(A.nnz > 0 ? A.nnz : 1)));
  if (perm) BK_TRY(upload(c, &A.perm, perm->data(), (size_t)A.nnz));
  std::vector<int2> blocks;
  partition(rp, n, blocks, A.width);
  A.nblocks = (int)blocks.size();
  return upload(c, &A.blocks, blocks.data(), blocks.size());
}

void bk_sparse_free(bk_ctx* c) {
  if (!c->sp) return;
  free_csr(c->sp->a);
  free_csr(c->sp->at);
  if (c->sp->stage) cudaFree(c->sp->stage);
  if (c->sp->diag) cudaFree(c->sp->diag);
  delete c->sp;
  c->sp = nullptr;
}

static int gather(bk_ctx* c, double* dst, const double* src, const int* perm, long long n) {
  if (n == 0) return BK_OK;
  k_gather<<<sp_grid(c, n), 256, 0, c->stream>>>(dst, src, perm, n);
  c->stats.kernel_launches++;
  BK_CUDA(c, cudaGetLastError());
  return BK_OK;
}

// J' on first use: its pattern from the host copy of J's, its values gathered from J's whenever they changed
static int ensure_transpose(bk_ctx* c) {
  SparseMat* m = c->sp;
  if (!m->at_built) {
    std::vector<int> rp, cl, perm;
    recompress(c->N0, m->h_rowptr.data(), m->h_col.data(), rp, cl, perm);
    BK_TRY(upload_csr(c, m->at, c->N0, rp, cl, &perm));
    m->at_built = true;
  }
  if (!m->at_vals) {
    BK_TRY(gather(c, m->at.val, m->a.val, m->at.perm, m->nnz));
    m->at_vals = true;
  }
  return BK_OK;
}

int bk_sparse_apply(bk_ctx* c, const OpDesc& op, const double* in, const double* sp, double* out) {
  SparseMat* m = c->sp;
  BK_CHECK(c, m && m->have_vals, "BK_SPARSE: call bk_sparse_set_pattern and bk_sparse_set_values before applying the operator");
  const SpCsr* A = &m->a;
  if (op.transpose) {
    BK_TRY(ensure_transpose(c));
    A = &m->at;
  }
  const dim3 grid(A->nblocks), block(BK_SP_THREADS);
#define BK_SP_GO(WW) \
  BK_CUDA(c, bk_launch_pdl(k_spmv<WW>, grid, block, 0, c->stream, A->rowptr, A->col, A->val, A->blocks, in, sp, out, op.a0, op.a1))
  switch (A->width) {
    case 2: BK_SP_GO(2); break;
    case 4: BK_SP_GO(4); break;
    case 8: BK_SP_GO(8); break;
    case 16: BK_SP_GO(16); break;
    default: BK_SP_GO(32); break;
  }
#undef BK_SP_GO
  return BK_OK;
}

int bk_jacobi_refresh(bk_ctx* c) {
  Precond& pc = c->pc;
  BK_CHECK(c, c->sp && c->sp->have_vals, "BK_PC_JACOBI needs the values of the sparse Jacobian (bk_sparse_set_values)");
  const long long n = c->N0;
  if (!pc.jpiv) BK_CUDA(c, cudaMalloc(&pc.jpiv, 8 * (size_t)n));
  if (!pc.jflag) BK_CUDA(c, cudaMalloc(&pc.jflag, sizeof(unsigned int)));
  BK_CUDA(c, cudaMemsetAsync(pc.jflag, 0, sizeof(unsigned int), c->stream));
  k_jacobi_piv<<<sp_grid(c, n), 256, 0, c->stream>>>(c->sp->diag, pc.jpiv, pc.a0, pc.a1, n, pc.jflag);
  c->stats.kernel_launches++;
  BK_CUDA(c, cudaGetLastError());
  unsigned int zero_pivot = 0;
  BK_CUDA(c, cudaMemcpyAsync(&zero_pivot, pc.jflag, sizeof zero_pivot, cudaMemcpyDeviceToHost, c->stream));
  BK_CUDA(c, cudaStreamSynchronize(c->stream));
  BK_CHECK(c, zero_pivot == 0, "BK_PC_JACOBI: zero pivot, a0 + a1 J_ii = 0 for some i");
  pc.jdirty = false;
  return BK_OK;
}

int bk_jacobi_apply(bk_ctx* c, const double* in, double* out) {
  if (c->pc.jdirty) BK_TRY(bk_jacobi_refresh(c));
  k_jacobi_apply<<<sp_grid(c, c->N0), 256, 0, c->stream>>>(c->pc.jpiv, in, out, c->N0);
  c->stats.kernel_launches++;
  BK_CUDA(c, cudaGetLastError());
  return BK_OK;
}

// ------------------------------------------------------------------------------------------ C ABI
#define BK_SP_FAIL(c, ...)                                    \
  do {                                                        \
    char _m[256];                                             \
    snprintf(_m, sizeof _m, __VA_ARGS__);                     \
    return bk_fail((c), BK_ERR_ARG, _m, __FILE__, __LINE__);  \
  } while (0)

extern "C" int32_t bk_sparse_set_pattern(bk_ctx* c, int32_t format, int32_t base, int64_t nnz, const int64_t* ptr,
                                         const int64_t* idx) {
  BK_ENTER(c);
  BK_CHECK(c, c->kind == BK_SPARSE, "bk_sparse_set_pattern needs a BK_SPARSE context");
  BK_CHECK(c, format == BK_SPARSE_CSR || format == BK_SPARSE_CSC, "bk_sparse_set_pattern: format is BK_SPARSE_CSR or BK_SPARSE_CSC");
  BK_CHECK(c, base == 0 || base == 1, "bk_sparse_set_pattern: index_base is 0 or 1");
  const long long n = c->N0;
  BK_CHECK(c, n < (1LL << 31), "bk_sparse_set_pattern: N must be below 2^31");
  if (nnz < 0 || nnz >= (1LL << 31)) BK_SP_FAIL(c, "bk_sparse_set_pattern: nnz = %lld must be in [0, 2^31)", (long long)nnz);
  BK_CHECK(c, ptr && (idx || nnz == 0), "bk_sparse_set_pattern: null pattern array");
  if (ptr[0] != base) BK_SP_FAIL(c, "bk_sparse_set_pattern: ptr[0] = %lld, expected the index base %d", (long long)ptr[0], base);
  for (long long i = 0; i < n; ++i)
    if (ptr[i + 1] < ptr[i]) BK_SP_FAIL(c, "bk_sparse_set_pattern: ptr is not monotone at entry %lld", i + 1);
  if (ptr[n] != nnz + base)
    BK_SP_FAIL(c, "bk_sparse_set_pattern: ptr[N] = %lld, expected nnz + base = %lld", (long long)ptr[n], (long long)(nnz + base));
  for (long long k = 0; k < nnz; ++k)
    if (idx[k] < base || idx[k] >= n + base)
      BK_SP_FAIL(c, "bk_sparse_set_pattern: index %lld at entry %lld is outside [%d, %lld]", (long long)idx[k], k, base, n - 1 + base);
  std::vector<int> optr(n + 1), oidx(nnz);
  for (long long i = 0; i <= n; ++i) optr[i] = (int)(ptr[i] - base);
  for (long long k = 0; k < nnz; ++k) oidx[k] = (int)(idx[k] - base);
  BK_CUDA(c, cudaStreamSynchronize(c->stream));  // the old matrix may still be in use
  bk_sparse_free(c);
  c->sp = new SparseMat();
  SparseMat* m = c->sp;
  m->nnz = nnz;
  if (format == BK_SPARSE_CSR) {
    m->h_rowptr.swap(optr);
    m->h_col.swap(oidx);
    BK_TRY(upload_csr(c, m->a, n, m->h_rowptr, m->h_col, nullptr));
  } else {
    std::vector<int> perm;
    recompress(n, optr.data(), oidx.data(), m->h_rowptr, m->h_col, perm);
    BK_TRY(upload_csr(c, m->a, n, m->h_rowptr, m->h_col, &perm));
    BK_CUDA(c, cudaMalloc(&m->stage, 8 * (size_t)(nnz > 0 ? nnz : 1)));
  }
  BK_CUDA(c, cudaMalloc(&m->diag, 8 * (size_t)n));
  c->pc.jdirty = true;
  return BK_OK;
}

extern "C" int32_t bk_sparse_set_values(bk_ctx* c, const double* vals) {
  BK_ENTER(c);
  BkRange nvtx_range("bk_sparse_set_values");
  SparseMat* m = c->sp;
  BK_CHECK(c, c->kind == BK_SPARSE && m, "bk_sparse_set_pattern must be called before bk_sparse_set_values");
  BK_CHECK(c, vals || m->nnz == 0, "bk_sparse_set_values: null values");
  SpCsr& A = m->a;
  const bool dev = m->nnz > 0 && bk_is_device_ptr(vals);
  double* dst = A.perm ? m->stage : A.val;
  if (m->nnz) {
    BK_CUDA(c, cudaMemcpyAsync(dst, vals, 8 * (size_t)m->nnz, dev ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, c->stream));
    if (!dev) c->stats.h2d_bytes += 8 * m->nnz;
  }
  if (A.perm) BK_TRY(gather(c, A.val, m->stage, A.perm, m->nnz));
  k_diag<<<sp_grid(c, c->N0), 256, 0, c->stream>>>(A.rowptr, A.col, A.val, m->diag, c->N0);
  c->stats.kernel_launches++;
  BK_CUDA(c, cudaGetLastError());
  m->have_vals = true;
  m->at_vals = false;
  c->pc.jdirty = true;
  if (!dev) BK_CUDA(c, cudaStreamSynchronize(c->stream));  // the caller's host buffer is free again when the call returns
  return BK_OK;
}
