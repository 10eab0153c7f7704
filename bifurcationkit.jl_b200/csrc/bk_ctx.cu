// bk_ctx.cu -- context life cycle, host<->device staging and the S11 vector algebra kernels
// (BorderedArray / VectorInterface methods of src/BorderedArrays.jl:30-35,53-70,79-217 for a
// device-resident state vector).
#include <cstdio>
#include <cstring>
#include <map>
#include <mutex>
#include <new>
#include "bk_common.cuh"
#include "bk_stencil.cuh"

int bk_fail(bk_ctx* c, int code, const char* what, const char* file, int line) {
  if (c) {
    char buf[512];
    snprintf(buf, sizeof buf, "%s (%s:%d)", what, file, line);
    c->err = buf;
  }
  return code;
}

void bk_grant_smem(int device, const void* kern, size_t bytes) {
  static std::mutex mu;
  static std::map<std::pair<int, const void*>, size_t> granted;  // (device, kernel) -> largest size set so far
  std::lock_guard<std::mutex> lk(mu);
  size_t& cur = granted[{device, kern}];
  if (bytes <= cur) return;
  cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
  if (bytes > 48 * 1024) cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
  cur = bytes;
}

bool bk_is_device_ptr(const void* p) {
  cudaPointerAttributes at;
  cudaError_t e = cudaPointerGetAttributes(&at, p);
  if (e != cudaSuccess) {
    cudaGetLastError();
    return false;
  }
  return at.type == cudaMemoryTypeDevice || at.type == cudaMemoryTypeManaged;
}

int bk_stage_in(bk_ctx* c, const double* p, long long n, int slot, bool copy_in, double** dev) {
  BK_CHECK(c, p != nullptr, "null vector argument");
  if (bk_is_device_ptr(p)) {
    *dev = const_cast<double*>(p);
    return BK_OK;
  }
  BK_CHECK(c, slot >= 0 && slot < 16, "bad stage slot");
  if ((int)c->stage.size() <= slot) c->stage.resize(slot + 1, nullptr);
  if (!c->stage[slot]) BK_CUDA(c, cudaMalloc(&c->stage[slot], sizeof(double) * (size_t)c->ld));
  BK_CHECK(c, n <= c->ld, "vector longer than the context's leading dimension");
  if (copy_in) {
    BK_CUDA(c, cudaMemcpyAsync(c->stage[slot], p, sizeof(double) * (size_t)n, cudaMemcpyHostToDevice, c->stream));
    c->stats.h2d_bytes += 8 * n;
  }
  *dev = c->stage[slot];
  return BK_OK;
}

int bk_stage_out(bk_ctx* c, double* p, long long n, const double* dev) {
  if (p == dev) return BK_OK;
  BK_CUDA(c, cudaMemcpyAsync(p, dev, sizeof(double) * (size_t)n, cudaMemcpyDeviceToHost, c->stream));
  BK_CUDA(c, cudaStreamSynchronize(c->stream));
  c->stats.d2h_bytes += 8 * n;
  return BK_OK;
}

int bk_tmp(bk_ctx* c, int slot, double** out) {
  if ((int)c->tmp.size() <= slot) c->tmp.resize(slot + 1, nullptr);
  if (!c->tmp[slot]) BK_CUDA(c, cudaMalloc(&c->tmp[slot], sizeof(double) * (size_t)c->ld));
  *out = c->tmp[slot];
  return BK_OK;
}

extern "C" int32_t bk_ctx_create(int32_t device, int32_t kind, const int64_t dims[3], const double lengths[3],
                                 int32_t krylov_m, bk_ctx** out) {
  if (!out) return BK_ERR_ARG;
  *out = nullptr;
  bk_ctx* c = new (std::nothrow) bk_ctx();
  if (!c) return BK_ERR_ARG;
  *out = c;  // returned even on failure so the caller can read bk_last_error
  c->device = device;
  c->cplx = (kind & BK_COMPLEX) != 0;
  kind &= ~BK_COMPLEX;
  c->kind = kind;
  for (int i = 0; i < 3; ++i) {
    c->dims[i] = dims ? (dims[i] > 0 ? dims[i] : 1) : 1;
    c->lengths[i] = lengths ? lengths[i] : 1.0;
  }
  long long n = 0;
  switch (kind) {
    case BK_CHAN: n = c->dims[0]; break;
    case BK_SH2D: n = c->dims[0] * c->dims[1]; break;
    case BK_SH3D: n = c->dims[0] * c->dims[1] * c->dims[2]; break;
    case BK_CGL2D: n = 2 * c->dims[0] * c->dims[1]; break;
    case BK_POTRAP_CGL2D: n = 2 * c->dims[0] * c->dims[1] * c->dims[2] + 1; break;
    case BK_SPARSE: n = c->dims[0] * c->dims[1] * c->dims[2]; break;
    default: return bk_fail(c, BK_ERR_ARG, "unknown problem kind", __FILE__, __LINE__);
  }
  BK_CHECK(c, n >= 2, "problem too small");
  BK_CHECK(c, krylov_m >= 1 && krylov_m <= 1024, "krylov_m out of range");
  BK_CHECK(c, !(c->cplx && kind == BK_POTRAP_CGL2D), "BK_COMPLEX is not available for the periodic-orbit functional");
  c->N0 = n;
  // a sparse context's operator is the loaded matrix, not a linearisation state: bk_sparse_apply reports a missing one
  c->have_state = (kind == BK_SPARSE);
  if (c->cplx) n *= 2;  // [re; im]
  c->N = n;
  c->m = krylov_m;
  c->ld = ((n + 2 + 31) / 32) * 32;  // >= N + 2: bordered vectors (N+1) keep one zero pad element for even-sized TMA rows
  BK_CUDA(c, cudaSetDevice(device));
  cudaDeviceProp prop;
  BK_CUDA(c, cudaGetDeviceProperties(&prop, device));
  c->nsm = prop.multiProcessorCount;
  BK_CUDA(c, cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
  size_t ld = (size_t)c->ld, m = (size_t)c->m;
  BK_CUDA(c, cudaMalloc(&c->u_state, 8 * ld));
  BK_CUDA(c, cudaMalloc(&c->V, 8 * ld * (m + 1)));
  BK_CUDA(c, cudaMalloc(&c->w, 8 * ld));
  BK_CUDA(c, cudaMalloc(&c->z, 8 * ld));
  BK_CUDA(c, cudaMalloc(&c->r, 8 * ld));
  BK_CUDA(c, cudaMemset(c->u_state, 0, 8 * ld));
  BK_CUDA(c, cudaMemset(c->V, 0, 8 * ld * (m + 1)));
  BK_CUDA(c, cudaMemset(c->w, 0, 8 * ld));
  BK_CUDA(c, cudaMemset(c->z, 0, 8 * ld));
  BK_CUDA(c, cudaMemset(c->r, 0, 8 * ld));
  BK_CUDA(c, cudaMalloc(&c->scales, 8 * (m + 4)));
  BK_CUDA(c, cudaMalloc(&c->gcoef, 8 * (m + 4)));
  BK_CUDA(c, cudaMalloc(&c->hcols, 8 * (m + 1) * (m + 4)));
  BK_CUDA(c, cudaMalloc(&c->hcols2, 8 * (m + 1) * (m + 4)));
  BK_CUDA(c, cudaMemset(c->hcols, 0, 8 * (m + 1) * (m + 4)));
  BK_CUDA(c, cudaMemset(c->hcols2, 0, 8 * (m + 1) * (m + 4)));
  BK_CUDA(c, cudaMallocHost(&c->h_pinned, 2 * 8 * (m + 1) * (m + 4)));
  // number of partial-sum columns: one per CTA of the widest reduction grid
  long long g = (n + 2 + 255) / 256 + 8;  // worst case: one CTA per 256 values
  if (kind == BK_SH2D) {
    // the fused 2-D kernel tiles rows, not the flat vector: a narrow grid (nx << 256) has up to ceil(nx/256) * ny CTAs
    long long gf = ((c->dims[0] + 255) / 256) * c->dims[1] + 8;
    if (gf > g) g = gf;
  }
  if (kind == BK_SH2D || kind == BK_SH3D) {  // first-generation tile kernels (64x32 / 32x8x8 tiles, ragged grids)
    long long gt = kind == BK_SH2D ? sh_num_tiles<2>((int)c->dims[0], (int)c->dims[1], 1)
                                   : sh_num_tiles<3>((int)c->dims[0], (int)c->dims[1], (int)c->dims[2]);
    if (gt + 8 > g) g = gt + 8;
  }
  if (g < 4 * c->nsm) g = 4 * c->nsm;
  c->gmax = (int)g;
  BK_CUDA(c, cudaMalloc(&c->partials, 8 * (m + 4) * (size_t)c->gmax));
  BK_CUDA(c, cudaMalloc(&c->counters, 64 * sizeof(unsigned int)));
  BK_CUDA(c, cudaMemset(c->counters, 0, 64 * sizeof(unsigned int)));
  BK_CUDA(c, cudaMalloc(&c->red_out, 8 * 16));
  BK_CUDA(c, cudaMallocHost(&c->red_pinned, 8 * 16));
  BK_CUDA(c, cudaMallocHost(&c->coef_pinned, 8 * (m + 4)));
  c->events.resize(m + 2);
  for (auto& e : c->events) BK_CUDA(c, cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
  BK_CUDA(c, cudaEventCreate(&c->tev0));
  BK_CUDA(c, cudaEventCreate(&c->tev1));
  if (kind == BK_POTRAP_CGL2D) {
    BK_CUDA(c, cudaMalloc(&c->phi, 8 * ld));
    BK_CUDA(c, cudaMalloc(&c->xpi, 8 * ld));
    BK_CUDA(c, cudaMalloc(&c->fcache, 8 * ld));
    BK_CUDA(c, cudaMemset(c->phi, 0, 8 * ld));
    BK_CUDA(c, cudaMemset(c->xpi, 0, 8 * ld));
  }
  BK_CUDA(c, cudaStreamSynchronize(c->stream));
  return BK_OK;
}

extern "C" int32_t bk_ctx_destroy(bk_ctx* c) {
  if (!c) return BK_OK;
  cudaSetDevice(c->device);
  if (c->stream) cudaStreamSynchronize(c->stream);
  double* bufs[] = {c->u_state, c->V, c->w, c->z, c->r, c->scales, c->gcoef, c->hcols, c->hcols2, c->partials,
                    c->red_out, c->phi, c->xpi, c->fcache, c->pc.work, c->pc.work2, c->pc.tri, c->Q, c->Q2, c->eig_dev};
  for (double* b : bufs)
    if (b) cudaFree(b);
  for (int d = 0; d < 3; ++d) {
    void* tabs[] = {c->pc.lam[d], c->pc.ftw[d], c->pc.fom[d], c->pc.flam2[d], c->pc.gwl[d], c->pc.gph[d]};
    for (void* t : tabs)
      if (t) cudaFree(t);
  }
  for (auto& p : c->pc_pairs) {
    cudaEventDestroy(p.first);
    cudaEventDestroy(p.second);
  }
  if (c->pc.tdft) cudaFree(c->pc.tdft);
  if (c->pc.jpiv) cudaFree(c->pc.jpiv);
  if (c->pc.jflag) cudaFree(c->pc.jflag);
  bk_sparse_free(c);
  if (c->counters) cudaFree(c->counters);
  for (auto& kv : c->vec_live) cudaFree(kv.first);
  for (double* b : c->stage)
    if (b) cudaFree(b);
  for (double* b : c->tmp)
    if (b) cudaFree(b);
  if (c->h_pinned) cudaFreeHost(c->h_pinned);
  if (c->red_pinned) cudaFreeHost(c->red_pinned);
  if (c->coef_pinned) cudaFreeHost(c->coef_pinned);
  if (c->host_pinned) cudaFreeHost(c->host_pinned);
  if (c->eig_pinned) cudaFreeHost(c->eig_pinned);
  for (auto& e : c->events)
    if (e) cudaEventDestroy(e);
  for (auto& p : c->tpairs) {
    cudaEventDestroy(p.first);
    cudaEventDestroy(p.second);
  }
  if (c->tev0) cudaEventDestroy(c->tev0);
  if (c->tev1) cudaEventDestroy(c->tev1);
  if (c->stream) cudaStreamDestroy(c->stream);
  delete c;
  return BK_OK;
}

extern "C" const char* bk_last_error(bk_ctx* c) { return c ? c->err.c_str() : "null context"; }
extern "C" int64_t bk_problem_size(bk_ctx* c) { return c ? c->N : 0; }
extern "C" int64_t bk_state_size(bk_ctx* c) { return c ? c->N0 : 0; }
extern "C" int32_t bk_set_params(bk_ctx* c, const double* p, int32_t n) {
  BK_ENTER(c);
  BK_CHECK(c, p && n >= 0 && n <= BK_MAX_PAR, "bad params");
  for (int i = 0; i < n; ++i) c->par[i] = p[i];
  return BK_OK;
}
// sum the per-application event pairs recorded by bk_precond_apply_dev (timing enabled); the stream must be idle
void bk_harvest_pc_timing(bk_ctx* c) {
  for (size_t i = 0; i < c->pc_pairs_used; ++i) {
    float t = 0;
    if (cudaEventElapsedTime(&t, c->pc_pairs[i].first, c->pc_pairs[i].second) == cudaSuccess) {
      c->stats.total_precond_ms += t;
      c->stats.total_precond_applies++;
    }
  }
  c->pc_pairs_used = 0;
}

extern "C" int32_t bk_get_stats(bk_ctx* c, bk_stats* out) {
  BK_ENTER(c);
  if (!out) return BK_ERR_ARG;
  if (c->pc_pairs_used) {
    BK_CUDA(c, cudaStreamSynchronize(c->stream));
    bk_harvest_pc_timing(c);
  }
  *out = c->stats;
  return BK_OK;
}
extern "C" int32_t bk_set_timing(bk_ctx* c, int32_t on) {
  BK_ENTER(c);
  c->timing = on != 0;
  c->timing_every = on > 1 ? on : 1;  // on = k > 1: time every k-th solve
  c->timing_now = c->timing && c->timing_every == 1;
  return BK_OK;
}
extern "C" int32_t bk_sync(bk_ctx* c) {
  BK_ENTER(c);
  BK_CUDA(c, cudaStreamSynchronize(c->stream));
  return BK_OK;
}
extern "C" void* bk_stream(bk_ctx* c) { return c ? (void*)c->stream : nullptr; }

// ---- vectors -----------------------------------------------------------------------------------
extern "C" int32_t bk_vec_alloc(bk_ctx* c, int64_t n, double** out) {
  BK_ENTER(c);
  if (!out) return BK_ERR_ARG;
  BK_CHECK(c, n > 0, "bad length");
  BK_CUDA(c, cudaSetDevice(c->device));
  size_t len = ((size_t)n + 31) / 32 * 32;
  // pooled: cudaMalloc/cudaFree synchronise the device and cost far more than a continuation-step kernel;
  // freed vectors are recycled in stream order (every kernel of a context runs on its one stream)
  for (size_t i = 0; i < c->vec_pool.size(); ++i) {
    if (c->vec_pool[i].first == len) {
      *out = c->vec_pool[i].second;
      c->vec_pool[i] = c->vec_pool.back();
      c->vec_pool.pop_back();
      BK_CUDA(c, cudaMemsetAsync(*out, 0, 8 * len, c->stream));
      return BK_OK;
    }
  }
  BK_CUDA(c, cudaMalloc(out, 8 * len));
  c->vec_live[*out] = len;
  BK_CUDA(c, cudaMemsetAsync(*out, 0, 8 * len, c->stream));
  return BK_OK;
}
extern "C" int32_t bk_vec_free(bk_ctx* c, double* v) {
  BK_ENTER(c);
  if (v) {
    auto it = c->vec_live.find(v);
    BK_CHECK(c, it != c->vec_live.end(), "bk_vec_free: pointer was not allocated by bk_vec_alloc of this context");
    c->vec_pool.push_back({it->second, v});
  }
  return BK_OK;
}
// pinned host buffers for option-A callers (host-resident state): H2D/D2H at PCIe speed instead of the
// pageable-memory staging path
extern "C" int32_t bk_host_alloc(bk_ctx* c, int64_t n, double** out) {
  BK_ENTER(c);
  if (!out) return BK_ERR_ARG;
  BK_CHECK(c, n > 0, "bad length");
  BK_CUDA(c, cudaSetDevice(c->device));
  BK_CUDA(c, cudaHostAlloc((void**)out, 8 * (size_t)n, cudaHostAllocDefault));
  return BK_OK;
}
extern "C" int32_t bk_host_free(bk_ctx* c, double* p) {
  BK_ENTER(c);
  if (p) {
    BK_CUDA(c, cudaStreamSynchronize(c->stream));
    BK_CUDA(c, cudaFreeHost(p));
  }
  return BK_OK;
}
extern "C" int32_t bk_vec_upload(bk_ctx* c, double* dst, const double* src, int64_t n) {
  BK_ENTER(c);
  BK_CUDA(c, cudaMemcpyAsync(dst, src, 8 * (size_t)n, cudaMemcpyHostToDevice, c->stream));
  BK_CUDA(c, cudaStreamSynchronize(c->stream));
  c->stats.h2d_bytes += 8 * n;
  return BK_OK;
}
extern "C" int32_t bk_vec_download(bk_ctx* c, double* dst, const double* src, int64_t n) {
  BK_ENTER(c);
  BK_CUDA(c, cudaMemcpyAsync(dst, src, 8 * (size_t)n, cudaMemcpyDeviceToHost, c->stream));
  BK_CUDA(c, cudaStreamSynchronize(c->stream));
  c->stats.d2h_bytes += 8 * n;
  return BK_OK;
}

int bk_dev_copy(bk_ctx* c, double* dst, const double* src, long long n) {
  if (dst == src) return BK_OK;
  BK_CUDA(c, cudaMemcpyAsync(dst, src, 8 * (size_t)n, cudaMemcpyDeviceToDevice, c->stream));
  return BK_OK;
}

static __global__ void __launch_bounds__(256) k_axpby(double* __restrict__ y, double a, const double* __restrict__ x,
                                                      double b, long long n) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  long long stride = (long long)gridDim.x * blockDim.x;
  if (b == 0.0) {
    for (; i < n; i += stride) y[i] = a * x[i];
  } else {
    for (; i < n; i += stride) y[i] = a * x[i] + b * y[i];
  }
}
static __global__ void __launch_bounds__(256) k_scale(double* __restrict__ x, double a, long long n) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  long long stride = (long long)gridDim.x * blockDim.x;
  for (; i < n; i += stride) x[i] *= a;
}

static inline int ew_grid(bk_ctx* c, long long n) {
  long long g = (n + 255) / 256;
  long long cap = (long long)c->nsm * 8;
  return (int)(g < cap ? (g > 0 ? g : 1) : cap);
}

int bk_dev_axpby(bk_ctx* c, double* y, double a, const double* x, double b, long long n) {
  k_axpby<<<ew_grid(c, n), 256, 0, c->stream>>>(y, a, x, b, n);
  c->stats.kernel_launches++;
  BK_CUDA(c, cudaGetLastError());
  return BK_OK;
}
int bk_dev_scale(bk_ctx* c, double* x, double a, long long n) {
  k_scale<<<ew_grid(c, n), 256, 0, c->stream>>>(x, a, n);
  c->stats.kernel_launches++;
  BK_CUDA(c, cudaGetLastError());
  return BK_OK;
}

// mode 0: sum x*y ; 1: max |x| ; 2: sum (x - x0)*y
template <int MODE>
static __global__ void __launch_bounds__(256) k_reduce(const double* __restrict__ x, const double* __restrict__ y,
                                                       const double* __restrict__ x0, long long n,
                                                       double* __restrict__ partials, unsigned int* counter,
                                                       double* __restrict__ out) {
  __shared__ double s_w[8];
  __shared__ int s_flag;
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  long long stride = (long long)gridDim.x * blockDim.x;
  double acc = 0.0;
  for (; i < n; i += stride) {
    if (MODE == 0) acc = fma(x[i], y[i], acc);
    if (MODE == 1) acc = bk_nanmax(acc, fabs(x[i]));
    if (MODE == 2) acc = fma(x[i] - x0[i], y[i], acc);
  }
  acc = (MODE == 1) ? bk_warp_max(acc) : bk_warp_sum(acc);
  int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  if (lane == 0) s_w[wid] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = s_w[0];
    for (int k = 1; k < 8; ++k) t = (MODE == 1) ? bk_nanmax(t, s_w[k]) : t + s_w[k];
    partials[blockIdx.x] = t;
  }
  if (bk_last_block(counter, &s_flag)) {
    double t = 0.0;
    for (int k = threadIdx.x; k < (int)gridDim.x; k += blockDim.x) {
      double v = __ldcg(partials + k);
      t = (MODE == 1) ? bk_nanmax(t, v) : t + v;
    }
    t = (MODE == 1) ? bk_warp_max(t) : bk_warp_sum(t);
    if (lane == 0) s_w[wid] = t;
    __syncthreads();
    if (threadIdx.x == 0) {
      double r = s_w[0];
      for (int k = 1; k < 8; ++k) r = (MODE == 1) ? bk_nanmax(r, s_w[k]) : r + s_w[k];
      out[0] = r;
    }
  }
}

template <int MODE>
static int reduce_launch(bk_ctx* c, const double* x, const double* y, const double* x0, long long n, double* out_host) {
  int g = ew_grid(c, n);
  if (g > c->gmax) g = c->gmax;
  k_reduce<MODE><<<g, 256, 0, c->stream>>>(x, y, x0, n, c->partials, c->counters + 8, c->red_out);
  c->stats.kernel_launches++;
  BK_CUDA(c, cudaGetLastError());
  BK_CUDA(c, cudaMemcpyAsync(c->red_pinned, c->red_out, 8, cudaMemcpyDeviceToHost, c->stream));
  BK_CUDA(c, cudaStreamSynchronize(c->stream));
  *out_host = c->red_pinned[0];
  return BK_OK;
}
int bk_dev_dot(bk_ctx* c, const double* x, const double* y, long long n, double* out_host) {
  return reduce_launch<0>(c, x, y, nullptr, n, out_host);
}
int bk_dev_norminf(bk_ctx* c, const double* x, long long n, double* out_host) {
  return reduce_launch<1>(c, x, x, nullptr, n, out_host);
}

#define BK_DEVPTR(c, p) BK_CHECK(c, (p) && bk_is_device_ptr(p), "bk_vec_* needs device pointers from bk_vec_alloc")

extern "C" int32_t bk_vec_copy(bk_ctx* c, double* dst, const double* src, int64_t n) {
  BK_ENTER(c);
  BK_DEVPTR(c, dst);
  BK_DEVPTR(c, src);
  return bk_dev_copy(c, dst, src, n);
}
extern "C" int32_t bk_vec_zero(bk_ctx* c, double* x, int64_t n) {
  BK_ENTER(c);
  BK_DEVPTR(c, x);
  BK_CUDA(c, cudaMemsetAsync(x, 0, 8 * (size_t)n, c->stream));
  return BK_OK;
}
extern "C" int32_t bk_vec_scale(bk_ctx* c, double* x, double a, int64_t n) {
  BK_ENTER(c);
  BK_DEVPTR(c, x);
  return bk_dev_scale(c, x, a, n);
}
extern "C" int32_t bk_vec_axpby(bk_ctx* c, double* y, double a, const double* x, double b, int64_t n) {
  BK_ENTER(c);
  BK_DEVPTR(c, y);
  BK_DEVPTR(c, x);
  return bk_dev_axpby(c, y, a, x, b, n);
}
extern "C" int32_t bk_vec_dot(bk_ctx* c, const double* x, const double* y, int64_t n, double* out) {
  BK_ENTER(c);
  if (!out) return BK_ERR_ARG;
  BK_DEVPTR(c, x);
  BK_DEVPTR(c, y);
  return bk_dev_dot(c, x, y, n, out);
}
extern "C" int32_t bk_vec_norm2(bk_ctx* c, const double* x, int64_t n, double* out) {
  BK_ENTER(c);
  if (!out) return BK_ERR_ARG;
  BK_DEVPTR(c, x);
  double d = 0;
  BK_TRY(bk_dev_dot(c, x, x, n, &d));
  *out = sqrt(d);
  return BK_OK;
}
extern "C" int32_t bk_vec_norminf(bk_ctx* c, const double* x, int64_t n, double* out) {
  BK_ENTER(c);
  if (!out) return BK_ERR_ARG;
  BK_DEVPTR(c, x);
  return bk_dev_norminf(c, x, n, out);
}
extern "C" int32_t bk_vec_diffdot(bk_ctx* c, const double* x, const double* x0, const double* tau, int64_t n, double* out) {
  BK_ENTER(c);
  if (!out) return BK_ERR_ARG;
  BK_DEVPTR(c, x);
  BK_DEVPTR(c, x0);
  BK_DEVPTR(c, tau);
  return reduce_launch<2>(c, x, tau, x0, n, out);
}
