// bk_problems.cu -- K1/K2: residual F(u;p) and Jacobian-vector product a0 v + a1 J(u) v of the
// named PDE stencils as stand-alone kernels, the MatrixFreeBLS bordered map (K2') and the
// trapezoid periodic-orbit functional (K7).  Reference definitions:
//   P1 examples/chan.jl:5-19,85-95        P2 examples/SH2d-fronts.jl:13-34,124-127
//   P3 examples/SH3d.jl:16-53             P4 examples/cGL2d.jl:6-22,262-318
//   P5 src/periodicorbit/PeriodicOrbitTrapeze.jl:209-330,362-386
//   bordered map src/LinearBorderSolver.jl:299-335
#include "bk_common.cuh"
#include "bk_stencil.cuh"
#include "bk_krylov_tma.cuh"

// ------------------------------------------------------------------------------------------ SH
template <int DIM, int MODE>
static __global__ void __launch_bounds__(BK_THREADS) k_sh_apply(OpDesc op, const double* __restrict__ in,
                                                                const double* __restrict__ in_scale_ptr,
                                                                double* __restrict__ out) {
  extern __shared__ double smem[];
  double val[BK_EPT];
  long long off[BK_EPT];
  double s = in_scale_ptr ? __ldg(in_scale_ptr) : 1.0;
  sh_tile_eval<DIM, MODE>(op, in, s, smem, val, off);
#pragma unroll
  for (int e = 0; e < BK_EPT; ++e)
    if (off[e] >= 0) out[off[e]] = val[e];
}

// ------------------------------------------------------------------------------------------ chan
__device__ __forceinline__ double chan_Nl(double x, double b) { return 1.0 + (x + 0.5 * x * x) / (1.0 + b * x * x); }
__device__ __forceinline__ double chan_dNl(double x, double b) {
  double d = 1.0 + b * x * x;
  return (1.0 - b * x * x + 2.0 * 0.5 * x) / (d * d);
}
// MODE 0 JVP, 1 residual
template <int MODE>
static __global__ void __launch_bounds__(256) k_chan_apply(OpDesc op, const double* __restrict__ in,
                                                           const double* __restrict__ in_scale_ptr,
                                                           double* __restrict__ out) {
  const int n = op.nx;
  const double alpha = op.par[0], beta = op.par[1];
  const double s = in_scale_ptr ? __ldg(in_scale_ptr) : 1.0;
  const double h2 = (double)(n - 1) * (double)(n - 1);
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    double v = s * in[i];
    double r;
    if (i == 0 || i == n - 1) {
      r = (MODE == 0) ? v : v - beta;
    } else {
      double lap = (s * in[i - 1] - 2.0 * v + s * in[i + 1]) * h2;
      r = (MODE == 0) ? lap + alpha * chan_dNl(op.u[i], beta) * v : lap + alpha * chan_Nl(v, beta);
    }
    out[i] = (MODE == 0) ? op.a0 * v + op.a1 * r : r;
  }
}

// ------------------------------------------------------------------------------------------ cGL
struct CglPar {
  double r, mu, nu, c3, c5;
};
__device__ __forceinline__ void cgl_nl(const CglPar& p, double u1, double u2, double& f1, double& f2) {
  double ua = u1 * u1 + u2 * u2;
  f1 = p.r * u1 - p.nu * u2 - ua * (p.c3 * u1 - p.mu * u2) - p.c5 * ua * ua * u1;
  f2 = p.r * u2 + p.nu * u1 - ua * (p.c3 * u2 + p.mu * u1) - p.c5 * ua * ua * u2;
}
template <bool TR = false>
__device__ __forceinline__ void cgl_dnl(const CglPar& p, double u1, double u2, double d1, double d2, double& f1,
                                        double& f2) {
  double u12 = u1 * u1, u22 = u2 * u2;
  double a11 = -5 * p.c5 * u12 * u12 + (-6 * p.c5 * u22 - 3 * p.c3) * u12 + 2 * p.mu * u1 * u2 - p.c5 * u22 * u22 -
               p.c3 * u22 + p.r;
  double a12 = -4 * p.c5 * u2 * u12 * u1 + p.mu * u12 + (-4 * p.c5 * u22 * u2 - 2 * p.c3 * u2) * u1 + 3 * u22 * p.mu - p.nu;
  double a21 = -4 * p.c5 * u2 * u12 * u1 - 3 * p.mu * u12 + (-4 * p.c5 * u22 * u2 - 2 * p.c3 * u2) * u1 - u22 * p.mu + p.nu;
  double a22 = -p.c5 * u12 * u12 + (-6 * p.c5 * u22 - p.c3) * u12 - 2 * p.mu * u1 * u2 - 5 * p.c5 * u22 * u22 -
               3 * p.c3 * u22 + p.r;
  f1 = a11 * d1 + (TR ? a21 : a12) * d2;  // TR: J' (the Laplacian is symmetric, only this 2 x 2 block changes)
  f2 = (TR ? a12 : a21) * d1 + a22 * d2;
}
// Dirichlet 5-point Laplacian (zero ghost cells; diagonal -2/h^2 everywhere, examples/cGL2d.jl:12-16)
__device__ __forceinline__ double lap_dirichlet(const double* __restrict__ a, int i, int j, int nx, int ny, double cx,
                                                double cy, double s) {
  long long g = i + (long long)j * nx;
  double c = a[g];
  double xm = i > 0 ? a[g - 1] : 0.0, xp = i < nx - 1 ? a[g + 1] : 0.0;
  double ym = j > 0 ? a[g - nx] : 0.0, yp = j < ny - 1 ? a[g + nx] : 0.0;
  return s * (cx * (xm - 2.0 * c + xp) + cy * (ym - 2.0 * c + yp));
}
// Vector field / JVP at one grid point of one slice: base pointers to the slice's [u1;u2].
template <int MODE, bool TR = false>
__device__ __forceinline__ void cgl_point(const CglPar& p, const double* __restrict__ u, const double* __restrict__ v,
                                          double s, int i, int j, int nx, int ny, double cx, double cy, double& o1,
                                          double& o2) {
  long long n = (long long)nx * ny, g = i + (long long)j * nx;
  if (MODE == 1) {
    double u1 = s * v[g], u2 = s * v[g + n];
    cgl_nl(p, u1, u2, o1, o2);
    o1 += lap_dirichlet(v, i, j, nx, ny, cx, cy, s);
    o2 += lap_dirichlet(v + n, i, j, nx, ny, cx, cy, s);
  } else {
    cgl_dnl<TR>(p, u[g], u[g + n], s * v[g], s * v[g + n], o1, o2);
    o1 += lap_dirichlet(v, i, j, nx, ny, cx, cy, s);
    o2 += lap_dirichlet(v + n, i, j, nx, ny, cx, cy, s);
  }
}
__device__ __forceinline__ CglPar cgl_par(const OpDesc& op) {
  CglPar p;
  p.r = op.par[0];
  p.mu = op.par[1];
  p.nu = op.par[2];
  p.c3 = op.par[3];
  p.c5 = op.par[4];
  return p;
}

template <int MODE>
static __global__ void __launch_bounds__(256) k_cgl_apply(OpDesc op, const double* __restrict__ in,
                                                          const double* __restrict__ in_scale_ptr,
                                                          double* __restrict__ out) {
  const int nx = op.nx, ny = op.ny;
  const long long n = (long long)nx * ny;
  const double s = in_scale_ptr ? __ldg(in_scale_ptr) : 1.0;
  const CglPar p = cgl_par(op);
  for (long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x; g < n; g += (long long)gridDim.x * blockDim.x) {
    int i = (int)(g % nx), j = (int)(g / nx);
    double o1, o2;
    if (MODE == 0 && op.transpose) cgl_point<MODE, true>(p, op.u, in, s, i, j, nx, ny, op.cx, op.cy, o1, o2);
    else cgl_point<MODE>(p, op.u, in, s, i, j, nx, ny, op.cx, op.cy, o1, o2);
    if (MODE == 0) {
      out[g] = op.a0 * s * in[g] + op.a1 * o1;
      out[g + n] = op.a0 * s * in[g + n] + op.a1 * o2;
    } else {
      out[g] = o1;
      out[g + n] = o2;
    }
  }
}

// ------------------------------------------------------------------------------------------ potrap over cGL
// x = [x_1 .. x_M ; T], slice length Ns = 2 nx ny.  Rows i = 1..M-1: (x_i - x_{i-1}) - h/2 (F(x_i) + F(x_{i-1})),
// x_0 == x_{M-1}; row M: x_M - x_1; last: <x - xpi, phi>  (phase condition written by a second kernel).
// MODE 1: residual.  MODE 0: JVP with F(x_i) read from the cache filled at bk_jac_set_state
// (the reference recomputes it on every po_jvp!, PeriodicOrbitTrapeze.jl:310-317; results identical).
template <int MODE>
static __global__ void __launch_bounds__(256) k_potrap_apply(OpDesc op, const double* __restrict__ in,
                                                             const double* __restrict__ in_scale_ptr,
                                                             double* __restrict__ out) {
  const int nx = op.nx, ny = op.ny, M = op.nz;
  const long long n = (long long)nx * ny, Ns = 2 * n;
  const double s = in_scale_ptr ? __ldg(in_scale_ptr) : 1.0;
  const CglPar p = cgl_par(op);
  const double T = (MODE == 1) ? s * in[Ns * M] : op.u[Ns * M];
  const double dT = (MODE == 0) ? s * in[Ns * M] : 0.0;
  const double h2 = 0.5 * T / M, dh2 = 0.5 * dT / M;
  const long long total = n * M;
  for (long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x; q < total; q += (long long)gridDim.x * blockDim.x) {
    long long g = q % n;
    int sl = (int)(q / n);
    int i = (int)(g % nx), j = (int)(g / nx);
    long long o = (long long)sl * Ns + g;
    if (sl == M - 1) {
      double c1 = s * (in[o] - in[g]), c2 = s * (in[o + n] - in[g + n]);
      out[o] = (MODE == 0) ? op.a0 * s * in[o] + op.a1 * c1 : c1;
      out[o + n] = (MODE == 0) ? op.a0 * s * in[o + n] + op.a1 * c2 : c2;
      continue;
    }
    int sp = sl > 0 ? sl - 1 : M - 2;
    const double* vi = in + (long long)sl * Ns;
    const double* vp = in + (long long)sp * Ns;
    double a1, a2, b1, b2;
    if (MODE == 1) {
      cgl_point<1>(p, nullptr, vi, s, i, j, nx, ny, op.cx, op.cy, a1, a2);
      cgl_point<1>(p, nullptr, vp, s, i, j, nx, ny, op.cx, op.cy, b1, b2);
      out[o] = s * (vi[g] - vp[g]) - h2 * (a1 + b1);
      out[o + n] = s * (vi[g + n] - vp[g + n]) - h2 * (a2 + b2);
    } else {
      const double* ui = op.u + (long long)sl * Ns;
      const double* up = op.u + (long long)sp * Ns;
      cgl_point<0>(p, ui, vi, s, i, j, nx, ny, op.cx, op.cy, a1, a2);
      cgl_point<0>(p, up, vp, s, i, j, nx, ny, op.cx, op.cy, b1, b2);
      const double* fi = op.fcache + (long long)sl * Ns;
      const double* fp = op.fcache + (long long)sp * Ns;
      double r1 = s * (vi[g] - vp[g]) - h2 * (a1 + b1) - dh2 * (fi[g] + fp[g]);
      double r2 = s * (vi[g + n] - vp[g + n]) - h2 * (a2 + b2) - dh2 * (fi[g + n] + fp[g + n]);
      out[o] = op.a0 * s * vi[g] + op.a1 * r1;
      out[o + n] = op.a0 * s * vi[g + n] + op.a1 * r2;
    }
  }
}
// F(x_i) for every slice (the cache)
static __global__ void __launch_bounds__(256) k_potrap_fcache(OpDesc op, const double* __restrict__ x, double* __restrict__ f) {
  const int nx = op.nx, ny = op.ny, M = op.nz;
  const long long n = (long long)nx * ny, Ns = 2 * n, total = n * M;
  const CglPar p = cgl_par(op);
  for (long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x; q < total; q += (long long)gridDim.x * blockDim.x) {
    long long g = q % n;
    int sl = (int)(q / n);
    double a1, a2;
    cgl_point<1>(p, nullptr, x + (long long)sl * Ns, 1.0, (int)(g % nx), (int)(g / nx), nx, ny, op.cx, op.cy, a1, a2);
    f[(long long)sl * Ns + g] = a1;
    f[(long long)sl * Ns + g + n] = a2;
  }
}

// ------------------------------------------------------------------------------------------ tail reductions
// out[N_tail] = alpha * sum_i x[i]*(scale) * y[i] + beta0   (+ optional elementwise border fix)
//   potrap phase condition:   out[n] = s * <in, phi> - <xpi, phi>(residual only)
//   bordered map (K2'):       out[i] += xp * a[i] + shift * s * in[i];   out[N] = s * (bscale <b, in> + c in[N])
// mode 0: phase condition; mode 1: border fix.
template <int MODE>
static __global__ void __launch_bounds__(256) k_tail(OpDesc op, const double* __restrict__ in,
                                                     const double* __restrict__ in_scale_ptr, double* __restrict__ out,
                                                     long long n, double beta0, int jvp_mode, double* __restrict__ partials,
                                                     unsigned int* counter) {
  __shared__ double s_w[8];
  __shared__ int s_flag;
  const double s = in_scale_ptr ? __ldg(in_scale_ptr) : 1.0;
  double acc = 0.0;
  const double xp = (MODE == 1) ? s * in[n] : 0.0;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    double v = in[i];
    if (MODE == 0) {
      acc = fma(v, op.phi[i], acc);
    } else {
      acc = fma(v, op.bb[i], acc);
      out[i] += xp * op.ba[i] + op.bshift * s * v;
    }
  }
  acc = bk_warp_sum(acc);
  int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  if (lane == 0) s_w[wid] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0;
    for (int k = 0; k < 8; ++k) t += s_w[k];
    partials[blockIdx.x] = t;
  }
  if (bk_last_block(counter, &s_flag)) {
    double t = 0.0;
    for (int k = threadIdx.x; k < (int)gridDim.x; k += blockDim.x) t += __ldcg(partials + k);
    t = bk_warp_sum(t);
    if (lane == 0) s_w[wid] = t;
    __syncthreads();
    if (threadIdx.x == 0) {
      double r = 0;
      for (int k = 0; k < 8; ++k) r += s_w[k];
      if (MODE == 0) {
        double ph = s * r - beta0;
        out[n] = jvp_mode ? op.a0 * s * in[n] + op.a1 * ph : ph;
      } else {
        out[n] = s * op.bscale * r + op.bc * xp;
      }
    }
  }
}

// two borders (block / tuple MatrixFreeBLSmap, src/LinearBorderSolver.jl:338-389): the same pass with two dot products
static __global__ void __launch_bounds__(256) k_tail2(OpDesc op, const double* __restrict__ in,
                                                      const double* __restrict__ in_scale_ptr, double* __restrict__ out,
                                                      long long n, double* __restrict__ partials, unsigned int* counter) {
  __shared__ double s_w[16];
  __shared__ int s_flag;
  const double s = in_scale_ptr ? __ldg(in_scale_ptr) : 1.0;
  const double xp0 = s * in[n], xp1 = s * in[n + 1];
  double acc0 = 0.0, acc1 = 0.0;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const double v = in[i];
    acc0 = fma(v, op.bb[i], acc0);
    acc1 = fma(v, op.bb2[i], acc1);
    out[i] += xp0 * op.ba[i] + xp1 * op.ba2[i] + op.bshift * s * v;
  }
  acc0 = bk_warp_sum(acc0);
  acc1 = bk_warp_sum(acc1);
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  if (lane == 0) {
    s_w[wid] = acc0;
    s_w[8 + wid] = acc1;
  }
  __syncthreads();
  if (threadIdx.x < 2) {
    double t = 0;
    for (int k = 0; k < 8; ++k) t += s_w[8 * threadIdx.x + k];
    partials[(size_t)threadIdx.x * gridDim.x + blockIdx.x] = t;
  }
  if (bk_last_block(counter, &s_flag)) {
    double t0 = 0.0, t1 = 0.0;
    for (int k = threadIdx.x; k < (int)gridDim.x; k += blockDim.x) {
      t0 += __ldcg(partials + k);
      t1 += __ldcg(partials + gridDim.x + k);
    }
    t0 = bk_warp_sum(t0);
    t1 = bk_warp_sum(t1);
    if (lane == 0) {
      s_w[wid] = t0;
      s_w[8 + wid] = t1;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
      double r0 = 0, r1 = 0;
      for (int k = 0; k < 8; ++k) {
        r0 += s_w[k];
        r1 += s_w[8 + k];
      }
      out[n] = s * op.bscale * r0 + op.bc * xp0 + op.bc01 * xp1;
      out[n + 1] = s * op.bscale * r1 + op.bc10 * xp0 + op.bc11 * xp1;
    }
  }
}

// ------------------------------------------------------------------------------------------ host side
static void fill_grid(bk_ctx* c, OpDesc& op) {
  op.kind = c->kind;
  op.nx = (int)c->dims[0];
  op.ny = (int)c->dims[1];
  op.nz = (int)c->dims[2];
  // h = 2 l / N in every example (SH2d-fronts.jl:14-15, SH3d.jl:18-20, cGL2d.jl:7-8)
  op.cx = 1.0 / ((2 * c->lengths[0] / c->dims[0]) * (2 * c->lengths[0] / c->dims[0]));
  op.cy = 1.0 / ((2 * c->lengths[1] / c->dims[1]) * (2 * c->lengths[1] / c->dims[1]));
  op.cz = (c->kind == BK_SH3D) ? 1.0 / ((2 * c->lengths[2] / c->dims[2]) * (2 * c->lengths[2] / c->dims[2])) : 0.0;
  op.N = c->N;
  op.bordered = 0;
  op.ba = op.bb = nullptr;
  op.bc = op.bshift = 0.0;
  op.bscale = 1.0;
  op.ba2 = op.bb2 = nullptr;
  op.bc01 = op.bc10 = op.bc11 = 0.0;
  op.phi = c->phi;
  op.fcache = c->fcache;
  op.cplx = c->cplx ? 1 : 0;
  op.a0i = c->shift_imag;
  op.transpose = c->transpose ? 1 : 0;
}

OpDesc bk_make_op(bk_ctx* c, double a0, double a1) {
  OpDesc op;
  fill_grid(c, op);
  for (int i = 0; i < BK_MAX_PAR; ++i) op.par[i] = c->jpar[i];
  op.u = c->u_state;
  op.a0 = a0;
  op.a1 = a1;
  return op;
}
OpDesc bk_make_residual_op(bk_ctx* c) {
  OpDesc op;
  fill_grid(c, op);
  for (int i = 0; i < BK_MAX_PAR; ++i) op.par[i] = c->par[i];
  op.u = nullptr;
  op.a0 = 0;
  op.a1 = 1;
  op.N = c->N0;  // F acts on the real state also in a BK_COMPLEX context
  op.cplx = 0;
  op.transpose = 0;
  return op;
}

static inline int lin_grid(bk_ctx* c, long long n) {
  long long g = (n + 255) / 256;
  long long cap = (long long)c->nsm * 8;
  return (int)(g < cap ? (g > 0 ? g : 1) : cap);
}

template <int MODE>
static int launch_kind(bk_ctx* c, const OpDesc& op, const double* in, const double* sp, double* out) {
  switch (op.kind) {
    case BK_SH2D: {
      const bool aligned = (op.nx % 2 == 0) && ((((uintptr_t)in) & 15) == 0);
      static int no_tma = -1;
      if (no_tma < 0) no_tma = getenv("BK_SH2D_NO_TMA") ? 1 : 0;  // diagnostics: the first-generation 64 x 32 tile kernel
      if (aligned && !no_tma) {
        // TMA-staged tile (bk_krylov_tma.cuh): tallest tile that still gives every SM about two CTAs
        const int tiles_x = (op.nx + BK2_ROW - 1) / BK2_ROW;
        int E = BK2_EMAX;
        while (E > 1 && (long long)tiles_x * ((op.ny + E - 1) / E) < 2LL * c->nsm) E >>= 1;
        const int grid = tiles_x * ((op.ny + E - 1) / E);
#define BK2A_GO(EE)                                                                                        \
  do {                                                                                                     \
    const size_t sm = Sh2Scratch<EE>::BYTES;                                                               \
    bk_ensure_smem(c, k2_apply<EE, MODE>, sm);                                                             \
    k2_apply<EE, MODE><<<grid, BK2_THREADS, sm, c->stream>>>(op, in, sp, out);                             \
  } while (0)
        if (E == 8) BK2A_GO(8);
        else if (E == 4) BK2A_GO(4);
        else if (E == 2) BK2A_GO(2);
        else BK2A_GO(1);
#undef BK2A_GO
        break;
      }
      bk_ensure_smem(c, k_sh_apply<2, MODE>, ShSmem<2>::BYTES);
      k_sh_apply<2, MODE><<<sh_num_tiles<2>(op.nx, op.ny, 1), BK_THREADS, ShSmem<2>::BYTES, c->stream>>>(op, in, sp, out);
      break;
    }
    case BK_SH3D: {
      bk_ensure_smem(c, k_sh_apply<3, MODE>, ShSmem<3>::BYTES);
      k_sh_apply<3, MODE><<<sh_num_tiles<3>(op.nx, op.ny, op.nz), BK_THREADS, ShSmem<3>::BYTES, c->stream>>>(op, in, sp, out);
      break;
    }
    case BK_CHAN: k_chan_apply<MODE><<<lin_grid(c, op.nx), 256, 0, c->stream>>>(op, in, sp, out); break;
    case BK_CGL2D: k_cgl_apply<MODE><<<lin_grid(c, (long long)op.nx * op.ny), 256, 0, c->stream>>>(op, in, sp, out); break;
    case BK_POTRAP_CGL2D: {
      long long tot = (long long)op.nx * op.ny * op.nz;
      k_potrap_apply<MODE><<<lin_grid(c, tot), 256, 0, c->stream>>>(op, in, sp, out);
      c->stats.kernel_launches++;
      BK_CUDA(c, cudaGetLastError());
      int g = lin_grid(c, op.N - 1);
      if (g > c->gmax) g = c->gmax;
      k_tail<0><<<g, 256, 0, c->stream>>>(op, in, sp, out, op.N - 1, (MODE == 1) ? c->phi_dot_xpi : 0.0, MODE == 0 ? 1 : 0,
                                          c->partials, c->counters + 9);
      break;
    }
    case BK_SPARSE:
      BK_TRY(MODE == 1 ? bk_fail(c, BK_ERR_ARG, "BK_SPARSE: F is the caller's function, the context has no residual", __FILE__, __LINE__)
                       : bk_sparse_apply(c, op, in, sp, out));
      break;
    default: return bk_fail(c, BK_ERR_ARG, "unknown kind", __FILE__, __LINE__);
  }
  c->stats.kernel_launches++;
  BK_CUDA(c, cudaGetLastError());
  return BK_OK;
}

int bk_launch_residual(bk_ctx* c, const double* u, double* out) {
  OpDesc op = bk_make_residual_op(c);
  return launch_kind<1>(c, op, u, nullptr, out);
}

// imaginary part of the shift on a split complex vector: out_re -= a0i s in_im, out_im += a0i s in_re
static __global__ void __launch_bounds__(256) k_cshift(double* __restrict__ out, const double* __restrict__ in,
                                                       const double* __restrict__ in_scale_ptr, double a0i, long long n0) {
  const double s = (in_scale_ptr ? __ldg(in_scale_ptr) : 1.0) * a0i;
  for (long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x; g < n0; g += (long long)gridDim.x * blockDim.x) {
    const double xr = in[g], xi = in[g + n0];
    out[g] -= s * xi;
    out[g + n0] += s * xr;
  }
}

int bk_launch_apply(bk_ctx* c, const OpDesc& op, const double* in, const double* sp, double* out) {
  if (op.transpose)
    BK_CHECK(c, op.kind == BK_SH2D || op.kind == BK_SH3D || op.kind == BK_CGL2D || op.kind == BK_SPARSE,
             "J' is not available for this problem kind");
  if (op.cplx) {
    // ((a0 + i a0i) I + a1 J)(x + i y): the real operator on both halves, then the cross terms of the imaginary shift
    OpDesc half = op;
    half.cplx = 0;
    half.N = op.N / 2;
    half.bordered = 0;
    BK_TRY(launch_kind<0>(c, half, in, sp, out));
    BK_TRY(launch_kind<0>(c, half, in + half.N, sp, out + half.N));
    if (op.a0i != 0.0) {
      k_cshift<<<lin_grid(c, half.N), 256, 0, c->stream>>>(out, in, sp, op.a0i, half.N);
      c->stats.kernel_launches++;
      BK_CUDA(c, cudaGetLastError());
    }
  } else {
    BK_TRY(launch_kind<0>(c, op, in, sp, out));
  }
  if (op.bordered) {
    int g = lin_grid(c, op.N);
    if (g > c->gmax) g = c->gmax;
    if (op.bordered == 2) k_tail2<<<g, 256, 0, c->stream>>>(op, in, sp, out, op.N, c->partials, c->counters + 9);
    else k_tail<1><<<g, 256, 0, c->stream>>>(op, in, sp, out, op.N, 0.0, 0, c->partials, c->counters + 9);
    c->stats.kernel_launches++;
    BK_CUDA(c, cudaGetLastError());
  }
  return BK_OK;
}

int bk_potrap_refresh_cache(bk_ctx* c) {
  if (c->kind != BK_POTRAP_CGL2D) return BK_OK;
  OpDesc op = bk_make_op(c, 0, 1);
  long long tot = (long long)op.nx * op.ny * op.nz;
  k_potrap_fcache<<<lin_grid(c, tot), 256, 0, c->stream>>>(op, c->u_state, c->fcache);
  c->stats.kernel_launches++;
  BK_CUDA(c, cudaGetLastError());
  return BK_OK;
}

// ------------------------------------------------------------------------------------------ C ABI
extern "C" int32_t bk_residual(bk_ctx* c, const double* u, double* out) {
  BK_ENTER(c);
  BkRange nvtx_range("bk_residual");
  BK_CHECK(c, c->kind != BK_SPARSE, "bk_residual: a BK_SPARSE context has no residual, F is the caller's function");
  double *du, *dout;
  BK_TRY(bk_stage_in(c, u, c->N0, 0, true, &du));
  BK_TRY(bk_stage_in(c, out, c->N0, 1, false, &dout));
  BK_TRY(bk_launch_residual(c, du, dout));
  return bk_stage_out(c, out, c->N0, dout);
}

extern "C" int32_t bk_jac_set_state(bk_ctx* c, const double* u) {
  BK_ENTER(c);
  BK_CHECK(c, u != nullptr, "null state");
  cudaMemcpyKind kind = bk_is_device_ptr(u) ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
  BK_CUDA(c, cudaMemcpyAsync(c->u_state, u, 8 * (size_t)c->N0, kind, c->stream));
  if (kind == cudaMemcpyHostToDevice) c->stats.h2d_bytes += 8 * c->N0;
  for (int i = 0; i < BK_MAX_PAR; ++i) c->jpar[i] = c->par[i];
  c->have_state = true;
  return bk_potrap_refresh_cache(c);
}

extern "C" int32_t bk_jac_set_shift_imag(bk_ctx* c, double a0_imag) {
  BK_ENTER(c);
  BK_CHECK(c, c->cplx || a0_imag == 0.0, "an imaginary shift needs a BK_COMPLEX context");
  c->shift_imag = a0_imag;
  return BK_OK;
}

extern "C" int32_t bk_jac_set_transpose(bk_ctx* c, int32_t on) {
  BK_ENTER(c);
  BK_CHECK(c, !on || c->kind == BK_SH2D || c->kind == BK_SH3D || c->kind == BK_CGL2D || c->kind == BK_SPARSE,
           "J' is not available for this problem kind");
  c->transpose = on != 0;
  return BK_OK;
}

extern "C" int32_t bk_jvp(bk_ctx* c, const double* v, double* out, double a0, double a1) {
  BK_ENTER(c);
  BkRange nvtx_range("bk_jvp");
  BK_CHECK(c, c->have_state, "bk_jac_set_state must be called before bk_jvp");
  double *dv, *dout;
  BK_TRY(bk_stage_in(c, v, c->N, 0, true, &dv));
  BK_TRY(bk_stage_in(c, out, c->N, 1, false, &dout));
  BK_CHECK(c, dv != dout, "bk_jvp: in-place application is not supported");
  OpDesc op = bk_make_op(c, a0, a1);
  BK_TRY(bk_launch_apply(c, op, dv, nullptr, dout));
  return bk_stage_out(c, out, c->N, dout);
}

extern "C" int32_t bk_bls_map(bk_ctx* c, const double* a, const double* b, double bc, int32_t has_shift, double shift,
                              double dotscale, const double* x, double* out) {
  BK_ENTER(c);
  BK_CHECK(c, c->have_state, "bk_jac_set_state must be called first");
  double *da, *db, *dx, *dout;
  BK_TRY(bk_stage_in(c, a, c->N, 2, true, &da));
  BK_TRY(bk_stage_in(c, b, c->N, 3, true, &db));
  BK_TRY(bk_stage_in(c, x, c->N + 1, 0, true, &dx));
  BK_TRY(bk_stage_in(c, out, c->N + 1, 1, false, &dout));
  OpDesc op = bk_make_op(c, 0.0, 1.0);
  op.bordered = 1;
  op.ba = da;
  op.bb = db;
  op.bc = bc;
  op.bshift = has_shift ? shift : 0.0;
  op.bscale = dotscale;
  BK_TRY(bk_launch_apply(c, op, dx, nullptr, dout));
  return bk_stage_out(c, out, c->N + 1, dout);
}

extern "C" int32_t bk_potrap_set_section(bk_ctx* c, const double* phi, const double* xpi) {
  BK_ENTER(c);
  BK_CHECK(c, c->kind == BK_POTRAP_CGL2D, "not a potrap context");
  long long n = c->N - 1;
  cudaMemcpyKind k1 = bk_is_device_ptr(phi) ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
  BK_CUDA(c, cudaMemcpyAsync(c->phi, phi, 8 * (size_t)n, k1, c->stream));
  if (xpi) {
    cudaMemcpyKind k2 = bk_is_device_ptr(xpi) ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
    BK_CUDA(c, cudaMemcpyAsync(c->xpi, xpi, 8 * (size_t)n, k2, c->stream));
  } else {
    BK_CUDA(c, cudaMemsetAsync(c->xpi, 0, 8 * (size_t)n, c->stream));
  }
  return bk_dev_dot(c, c->xpi, c->phi, n, &c->phi_dot_xpi);
}
