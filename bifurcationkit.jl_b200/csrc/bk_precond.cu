// bk_precond.cu -- K6: preconditioners honouring the reference's Pl/Pr contract
// (ldiv!(y, P, x), src/Preconditioner.jl:11-37).
//
// BK_PC_SH_DCT: the examples precondition Swift-Hohenberg with a sparse factorisation of L1 + I
//   (examples/SH2d-fronts.jl:120-122  Pl = lu(par.L1 + I); examples/SH3d.jl:88 cholesky(L1)).  The
//   Neumann-closure Laplacian (SH2d-fronts.jl:13-29) is diagonalised by the DCT-II, so
//   (L1 + shift I)^-1 r = IDCT( DCT(r) / ((1 + lx_i + ly_j [+ lz_k])^2 + shift) )  exactly
//   (identity pinned in tests/test_oracle_palc.py::test_dct_symbol_diagonalises_L1).
//   Power-of-two line lengths 64..2048 run the register-resident FFT kernels of bk_fft_fast.cuh (two lines per complex
//   FFT, the last dimension fused: forward + symbol + inverse, so an application is 3 kernels in 2-D and 5 in 3-D);
//   every other length runs the mixed-radix kernel of bk_fft_gen.cuh.  No library on this path.
// BK_PC_CHAN_TRIDIAG: lu(P) of examples/chan.jl:108-111 (Thomas algorithm, one thread: n = 1e3 plumbing).
// BK_PC_CGL_DST: per-component (a0 I + a1 Lap_dirichlet)^-1 by DST-I (stand-in for the ILU of
//   examples/cGL2d.jl:209-213); for potrap contexts it is applied slice by slice (block Jacobi, cf.
//   jacobian_block_diag, src/periodicorbit/PeriodicOrbitTrapeze.jl:619-643).
// BK_PC_POTRAP_CIRC: block-circulant-in-time linearisation of the Trapeze functional at the trivial state, inverted
//   exactly: DST-I in space, u1 +- i u2, DFT over the M-1 cyclic slices, scalar symbol.
#include <cmath>
#include <cstdlib>
#include <utility>
#include <vector>
#include "bk_common.cuh"

#include "bk_fft_fast.cuh"
#include "bk_fft_gen.cuh"

// divide by the symbol
static __global__ void __launch_bounds__(256) k_sh_symbol_div(double* __restrict__ a, int nx, int ny, int nz,
                                                              const double* __restrict__ lx, const double* __restrict__ ly,
                                                              const double* __restrict__ lz, double shift, double scale) {
  const long long total = (long long)nx * ny * nz;
  for (long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x; q < total; q += (long long)gridDim.x * blockDim.x) {
    int i = (int)(q % nx), j = (int)((q / nx) % ny), k = (int)(q / ((long long)nx * ny));
    double t = 1.0 + lx[i] + ly[j] + (lz ? lz[k] : 0.0);
    a[q] = a[q] * scale / (t * t + shift);
  }
}
static __global__ void __launch_bounds__(256) k_helmholtz_symbol_div(double* __restrict__ a, int nx, int ny, long long nblocks,
                                                                     const double* __restrict__ lx,
                                                                     const double* __restrict__ ly, double a0, double a1) {
  const long long n = (long long)nx * ny, total = n * nblocks;
  for (long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x; q < total; q += (long long)gridDim.x * blockDim.x) {
    long long g = q % n;
    int i = (int)(g % nx), j = (int)(g / nx);
    a[q] = a[q] / (a0 + a1 * (lx[i] + ly[j]));
  }
}

// ---- potrap circulant preconditioner: time direction -------------------------------------------------------------------
// B holds the DST-I coefficients of all 2M slice components (field f = 2*slice + comp, n values each).  One thread per
// spatial mode: w+- = u1 +- i u2 over the K = M-1 cyclic slices, DFT in time, divide by
//   s+-_k = (1 - g_k) - h/2 (1 + g_k)(lambda + r +- i nu),   g_k = exp(-2 pi i k/K),
// inverse DFT, back to (u1, u2).  In place.
#define BK_PO_KMAX 64
static __global__ void __launch_bounds__(128) k_potrap_time(double* __restrict__ B, long long n, int nx, int K,
                                                            const double* __restrict__ lamx, const double* __restrict__ lamy,
                                                            double h, double r, double nu, const double2* __restrict__ tw) {
  const long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= n) return;
  const double lam = lamx[g % nx] + lamy[g / nx];
  double2 wp[BK_PO_KMAX], wm[BK_PO_KMAX];
  for (int i = 0; i < K; ++i) {
    const double a = B[(long long)(2 * i) * n + g], b = B[(long long)(2 * i + 1) * n + g];
    wp[i] = make_double2(a, b);
    wm[i] = make_double2(a, -b);
  }
  double2 yp[BK_PO_KMAX], ym[BK_PO_KMAX];
  const double invK = 1.0 / K;
  for (int k = 0; k < K; ++k) {
    double2 ap = make_double2(0, 0), am = make_double2(0, 0);
    int idx = 0;
    for (int i = 0; i < K; ++i) {
      const double2 t = tw[idx];  // exp(-2 pi i k i / K)
      ap.x += wp[i].x * t.x - wp[i].y * t.y;
      ap.y += wp[i].x * t.y + wp[i].y * t.x;
      am.x += wm[i].x * t.x - wm[i].y * t.y;
      am.y += wm[i].x * t.y + wm[i].y * t.x;
      idx += k;
      if (idx >= K) idx -= K;
    }
    const double2 gk = tw[k];
    // s = (1 - g) - h/2 (1 + g) (lam + r +- i nu)
    const double2 omg = make_double2(1.0 - gk.x, -gk.y), opg = make_double2(1.0 + gk.x, gk.y);
    const double cr = lam + r;
    double2 sp = make_double2(omg.x - 0.5 * h * (opg.x * cr - opg.y * nu), omg.y - 0.5 * h * (opg.x * nu + opg.y * cr));
    double2 sm = make_double2(omg.x - 0.5 * h * (opg.x * cr + opg.y * nu), omg.y - 0.5 * h * (-opg.x * nu + opg.y * cr));
    const double dp = 1.0 / (sp.x * sp.x + sp.y * sp.y), dm = 1.0 / (sm.x * sm.x + sm.y * sm.y);
    yp[k] = make_double2((ap.x * sp.x + ap.y * sp.y) * dp * invK, (ap.y * sp.x - ap.x * sp.y) * dp * invK);
    ym[k] = make_double2((am.x * sm.x + am.y * sm.y) * dm * invK, (am.y * sm.x - am.x * sm.y) * dm * invK);
  }
  for (int i = 0; i < K; ++i) {
    double2 ap = make_double2(0, 0), am = make_double2(0, 0);
    int idx = 0;
    for (int k = 0; k < K; ++k) {
      const double2 t = tw[idx];  // conj -> exp(+2 pi i k i / K)
      ap.x += yp[k].x * t.x + yp[k].y * t.y;
      ap.y += yp[k].y * t.x - yp[k].x * t.y;
      am.x += ym[k].x * t.x + ym[k].y * t.y;
      am.y += ym[k].y * t.x - ym[k].x * t.y;
      idx += i;
      if (idx >= K) idx -= K;
    }
    B[(long long)(2 * i) * n + g] = 0.5 * (ap.x + am.x);      // Re((yp + ym)/2)
    B[(long long)(2 * i + 1) * n + g] = 0.5 * (ap.y - am.y);  // Re((yp - ym)/(2i)) = Im(yp - ym)/2
  }
}
// closure row of the preconditioner: x_M = r_M + x_1; the period entry passes through
static __global__ void __launch_bounds__(256) k_potrap_close(const double* __restrict__ in, double* __restrict__ out,
                                                             long long Ns, int M) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < Ns) out[(long long)(M - 1) * Ns + i] = in[(long long)(M - 1) * Ns + i] + out[i];
  if (i == 0) out[(long long)M * Ns] = in[(long long)M * Ns];
}

// Thomas solve with precomputed factors: tri = [cprime (n) | denom_inv (n) | lower (n)]
static __global__ void k_thomas(const double* __restrict__ tri, const double* __restrict__ in, double* __restrict__ out, int n) {
  if (blockIdx.x != 0 || threadIdx.x != 0) return;
  const double* cp = tri;
  const double* di = tri + n;
  const double* lo = tri + 2 * n;
  double prev = in[0] * di[0];
  out[0] = prev;
  for (int i = 1; i < n; ++i) {
    prev = (in[i] - lo[i] * prev) * di[i];
    out[i] = prev;
  }
  for (int i = n - 2; i >= 0; --i) out[i] -= cp[i] * out[i + 1];
}

// ------------------------------------------------------------------------------------------------ host
static inline int lin_grid(bk_ctx* c, long long n) {
  long long g = (n + 255) / 256, cap = (long long)c->nsm * 8;
  return (int)(g < cap ? (g > 0 ? g : 1) : cap);
}

static int upload(bk_ctx* c, void** dst, const void* src, size_t bytes) {
  if (*dst) cudaFree(*dst);
  *dst = nullptr;
  BK_CUDA(c, cudaMalloc(dst, bytes));
  BK_CUDA(c, cudaMemcpy(*dst, src, bytes, cudaMemcpyHostToDevice));
  return BK_OK;
}

// ---- fast path: one instantiation per (values per thread, line length) -----------------------------------------------------
// Values per thread E = 2^loge of the fast kernels for a line of length n.  Measured on B200: warm, isolated per-kernel times
// (profiles/r02_fft_warm_times.txt) favour E = 32 at n = 1024 (38.9 us per application against 44-48 us for E = 4 / 8 / 16), but
// inside the GMRES loop E = 8 wins (46.6 us per application against 52.7 us for E = 32, bench.py `roofline.preconditioner`):
// more warps per SM hide the latencies that the neighbouring kernels' PDL overlap does not.  n <= 512: E = 4 (18.9 us against
// 32 us for E = 32, too few warps per SM).  BK_FFT_LOGE overrides (2..5).
static int fast_loge(long long n) {
  static int e = -1;
  if (e < 0) {
    const char* a = getenv("BK_FFT_LOGE");
    e = a ? atoi(a) : 0;
    if (e < 2 || e > 5) e = 0;
  }
  if (e) return e;
  return n >= 1024 ? 3 : 2;
}
static int fast_logn(long long n) {
  static int off = -1;
  if (off < 0) off = getenv("BK_FFT_NO_FAST") ? 1 : 0;  // diagnostics: force the general kernel everywhere
  if (off) return 0;
  for (int l = fast_loge(n) + 1; l <= 11; ++l)
    if (l >= 6 && n == (1LL << l)) return l;
  return 0;
}
#define BKF_DISPATCH_N(LE, LOGN, ...)                                                   \
  switch (LOGN) {                                                                      \
    case 6: { using FC = bkf::Cfg<6, LE>; __VA_ARGS__; } break;                        \
    case 7: { using FC = bkf::Cfg<7, LE>; __VA_ARGS__; } break;                        \
    case 8: { using FC = bkf::Cfg<8, LE>; __VA_ARGS__; } break;                        \
    case 9: { using FC = bkf::Cfg<9, LE>; __VA_ARGS__; } break;                        \
    case 10: { using FC = bkf::Cfg<10, LE>; __VA_ARGS__; } break;                      \
    default: { using FC = bkf::Cfg<11, LE>; __VA_ARGS__; } break;                      \
  }
#define BKF_DISPATCH(LOGN, ...)                                                        \
  switch (fast_loge(1LL << (LOGN))) {                                                               \
    case 2: BKF_DISPATCH_N(2, LOGN, __VA_ARGS__) break;                                \
    case 3: BKF_DISPATCH_N(3, LOGN, __VA_ARGS__) break;                                \
    case 4: BKF_DISPATCH_N(4, LOGN, __VA_ARGS__) break;                                \
    default: BKF_DISPATCH_N(5, LOGN, __VA_ARGS__) break;                               \
  }

template <class FC>
static int fast_setup(bk_ctx* c, int d, const double* lam_host) {
  std::vector<double> tw, om, lam2;
  bkf::build_tables<FC>(tw, om, lam2, lam_host);
  Precond& pc = c->pc;
  if (tw.empty()) tw.assign(2, 0.0);
  BK_TRY(upload(c, (void**)&pc.ftw[d], tw.data(), 8 * tw.size()));
  BK_TRY(upload(c, (void**)&pc.fom[d], om.data(), 8 * om.size()));
  BK_TRY(upload(c, (void**)&pc.flam2[d], lam2.data(), 8 * lam2.size()));
  return BK_OK;
}

// mode 0 forward (2 C), 1 inverse (n x), 2 fused forward + symbol + inverse (strided only)
template <class FC>
static int fast_launch(bk_ctx* c, int d, bool strided, int mode, const double* in, double* out, const bkf::Geom& g,
                       const bkf::Symbol* sy) {
  Precond& pc = c->pc;
  bkf::Tables tb{pc.ftw[d], pc.fom[d], pc.flam2[d]};
  bkf::Symbol s0{};
  if (sy) s0 = *sy;
  if (strided) {
    dim3 grid((g.nb + 2 * FC::PP - 1) / (2 * FC::PP), g.nouter);
    if (mode == 0) {
      bk_ensure_smem(c, bkf::k_strided<FC, 0>, FC::SMEM);
      BK_CUDA(c, bk_launch_pdl(bkf::k_strided<FC, 0>, grid, dim3(FC::THREADS), FC::SMEM, c->stream, in, out, g, tb, s0));
    } else if (mode == 1) {
      bk_ensure_smem(c, bkf::k_strided<FC, 1>, FC::SMEM);
      BK_CUDA(c, bk_launch_pdl(bkf::k_strided<FC, 1>, grid, dim3(FC::THREADS), FC::SMEM, c->stream, in, out, g, tb, s0));
    } else {
      bk_ensure_smem(c, bkf::k_strided<FC, 2>, FC::SMEM_FUSED);
      BK_CUDA(c, bk_launch_pdl(bkf::k_strided<FC, 2>, grid, dim3(FC::THREADS), FC::SMEM_FUSED, c->stream, in, out, g, tb, s0));
    }
  } else {
    dim3 grid((unsigned)((g.nb + 2 * FC::PP - 1) / (2 * FC::PP)));
    if (mode == 0) {
      bk_ensure_smem(c, bkf::k_contig<FC, 0>, FC::SMEM);
      BK_CUDA(c, bk_launch_pdl(bkf::k_contig<FC, 0>, grid, dim3(FC::THREADS), FC::SMEM, c->stream, in, out, g, tb));
    } else {
      bk_ensure_smem(c, bkf::k_contig<FC, 1>, FC::SMEM);
      BK_CUDA(c, bk_launch_pdl(bkf::k_contig<FC, 1>, grid, dim3(FC::THREADS), FC::SMEM, c->stream, in, out, g, tb));
    }
  }
  return BK_OK;
}

// ---- general path ----------------------------------------------------------------------------------------------------------
static void factorize(int L, bkg::Plan& pl) {
  pl.npass = 0;
  while (L % 4 == 0 && pl.npass < BKG_MAXPASS) {
    pl.radix[pl.npass++] = 4;
    L /= 4;
  }
  for (int p = 2; L > 1 && pl.npass < BKG_MAXPASS; ++p)
    while (L % p == 0 && pl.npass < BKG_MAXPASS) {
      pl.radix[pl.npass++] = p;
      L /= p;
    }
}
#define BKG_THREADS 512
#define BKG_SMEM_BUDGET (100 * 1024)   // two CTAs per SM
#define BKG_SMEM_MAX (200 * 1024)
static int gen_ppg(int L) {
  long long per = 32LL * L;  // two buffers of L complex values per pair
  int p = (int)(BKG_SMEM_BUDGET / per);
  if (p < 1) p = 1;
  if (p > 8) p = 8;
  return p;
}

// type 0: DCT-II (Neumann), 1: DST-I (Dirichlet)
static int gen_setup(bk_ctx* c, int d, int n, int type) {
  Precond& pc = c->pc;
  bkg::Plan& pl = pc.gplan[d];
  pl.n = n;
  pl.L = type == 0 ? 2 * n : 2 * n + 2;
  BK_CHECK(c, 32LL * pl.L <= BKG_SMEM_MAX, "line too long for the general transform kernel (n <= 3199)");
  factorize(pl.L, pl);
  const long double PI = 3.14159265358979323846264338327950288L;
  std::vector<double> wl(2 * (size_t)pl.L), ph(2 * (size_t)n);
  for (int t = 0; t < pl.L; ++t) {
    wl[2 * t] = (double)cosl(-2.0L * PI * t / pl.L);
    wl[2 * t + 1] = (double)sinl(-2.0L * PI * t / pl.L);
  }
  for (int k = 0; k < n; ++k) {
    ph[2 * k] = (double)cosl(-PI * k / (2.0L * n));
    ph[2 * k + 1] = (double)sinl(-PI * k / (2.0L * n));
  }
  BK_TRY(upload(c, (void**)&pc.gwl[d], wl.data(), 8 * wl.size()));
  BK_TRY(upload(c, (void**)&pc.gph[d], ph.data(), 8 * ph.size()));
  pl.wl = pc.gwl[d];
  pl.ph = pc.gph[d];
  pl.dst_scale = 0.5 * sqrt(2.0 / (n + 1.0));
  return BK_OK;
}

// mode 0 DCT forward (2 C), 1 DCT inverse (n x), 2 DST-I (orthonormal)
static int gen_launch(bk_ctx* c, int d, bool strided, int mode, const double* in, double* out, const bkf::Geom& g) {
  const bkg::Plan& pl = c->pc.gplan[d];
  const int ppg = gen_ppg(pl.L);
  const size_t sm = 32 * (size_t)pl.L * ppg;
  const long long npairs = ((long long)g.nb + 1) / 2;
  dim3 grid((unsigned)((npairs + ppg - 1) / ppg), strided ? g.nouter : 1);
#define BKG_GO(S, M)                                                                                                       \
  do {                                                                                                                     \
    bk_ensure_smem(c, bkg::k_gen<S, M>, sm);                                                                               \
    BK_CUDA(c, bk_launch_pdl(bkg::k_gen<S, M>, grid, dim3(BKG_THREADS), sm, c->stream, in, out, g, pl, ppg));              \
  } while (0)
  if (strided) {
    if (mode == 0) BKG_GO(true, 0);
    else if (mode == 1) BKG_GO(true, 1);
    else BKG_GO(true, 2);
  } else {
    if (mode == 0) BKG_GO(false, 0);
    else if (mode == 1) BKG_GO(false, 1);
    else BKG_GO(false, 2);
  }
#undef BKG_GO
  return BK_OK;
}

// transform tables for dimension d of length n. type 0: DCT-II (Neumann), 1: DST-I (Dirichlet)
static int setup_dim(bk_ctx* c, int d, long long n, double inv_h2, int type, bool even_nx) {
  Precond& pc = c->pc;
  std::vector<double> lam(n);
  const long double PI = 3.14159265358979323846264338327950288L;
  for (long long k = 0; k < n; ++k)
    lam[k] = (type == 0) ? (double)((2.0L * cosl(PI * k / n) - 2.0L)) * inv_h2
                         : (double)(-(2.0L - 2.0L * cosl(PI * (k + 1) / (n + 1)))) * inv_h2;
  BK_TRY(upload(c, (void**)&pc.lam[d], lam.data(), 8 * n));
  pc.ttype[d] = type;
  pc.fast[d] = (type == 0 && even_nx) ? fast_logn(n) : 0;  // 16-byte accesses need an even row length
  if (pc.fast[d]) {
    BKF_DISPATCH(pc.fast[d], BK_TRY(fast_setup<FC>(c, d, lam.data())));
  }
  return gen_setup(c, d, (int)n, type);  // always available: unaligned vectors fall back to it
}

// number of grid dimensions of the DCT preconditioner: SH3d, or a BK_SPARSE context with a 3-D grid shape
static int pc_ndim(const bk_ctx* c) { return (c->kind == BK_SH3D || (c->kind == BK_SPARSE && c->dims[2] > 1)) ? 3 : 2; }

extern "C" int32_t bk_precond_setup(bk_ctx* c, int32_t kind, double a0, double a1) {
  BK_ENTER(c);
  BK_CUDA(c, cudaStreamSynchronize(c->stream));
  Precond& pc = c->pc;
  if (kind == BK_PC_NONE) {
    pc.kind = BK_PC_NONE;
    return BK_OK;
  }
  if (!pc.work) BK_CUDA(c, cudaMalloc(&pc.work, 8 * (size_t)c->ld));
  if (!pc.work2) BK_CUDA(c, cudaMalloc(&pc.work2, 8 * (size_t)c->ld));
  const bool even_nx = (c->dims[0] % 2) == 0;
  if (kind == BK_PC_SH_DCT) {
    BK_CHECK(c, c->kind == BK_SH2D || c->kind == BK_SH3D || (c->kind == BK_SPARSE && c->dims[1] > 1),
             "BK_PC_SH_DCT needs a Swift-Hohenberg context or a grid-shaped BK_SPARSE context");
    int nd = pc_ndim(c);
    for (int d = 0; d < nd; ++d) {
      double h = 2 * c->lengths[d] / c->dims[d];
      BK_TRY(setup_dim(c, d, c->dims[d], 1.0 / (h * h), 0, even_nx));
    }
  } else if (kind == BK_PC_CGL_DST) {
    BK_CHECK(c, c->kind == BK_CGL2D || c->kind == BK_POTRAP_CGL2D || (c->kind == BK_SPARSE && c->dims[1] > 1),
             "BK_PC_CGL_DST needs a cGL context or a grid-shaped BK_SPARSE context");
    for (int d = 0; d < 2; ++d) {
      double h = 2 * c->lengths[d] / c->dims[d];
      BK_TRY(setup_dim(c, d, c->dims[d], 1.0 / (h * h), 1, even_nx));
    }
  } else if (kind == BK_PC_POTRAP_CIRC) {
    BK_CHECK(c, c->kind == BK_POTRAP_CGL2D, "BK_PC_POTRAP_CIRC needs a Trapeze (potrap) context");
    const int K = (int)c->dims[2] - 1;
    BK_CHECK(c, K >= 1 && K <= BK_PO_KMAX, "BK_PC_POTRAP_CIRC supports 2 <= M <= 65 time slices");
    BK_CHECK(c, a0 > 0, "BK_PC_POTRAP_CIRC: a0 must be the period T > 0");
    for (int d = 0; d < 2; ++d) {
      double h = 2 * c->lengths[d] / c->dims[d];
      BK_TRY(setup_dim(c, d, c->dims[d], 1.0 / (h * h), 1, even_nx));
    }
    std::vector<double2> tw(K);
    const long double PI = 3.14159265358979323846264338327950288L;
    for (int j = 0; j < K; ++j) tw[j] = make_double2((double)cosl(-2.0L * PI * j / K), (double)sinl(-2.0L * PI * j / K));
    BK_TRY(upload(c, (void**)&pc.tdft, tw.data(), 16 * (size_t)K));
    pc.po_T = a0;
    pc.po_r = c->par[0];   // (r, mu, nu, c3, c5)
    pc.po_nu = c->par[2];
  } else if (kind == BK_PC_CHAN_TRIDIAG) {
    BK_CHECK(c, c->kind == BK_CHAN, "BK_PC_CHAN_TRIDIAG needs a chan context");
    long long n = c->N0;
    double s = (double)(n - 1) * (double)(n - 1);
    std::vector<double> lo(n, s), di(n, -2 * s), up(n, s), tri(3 * n);
    di[0] = 1;
    up[0] = 0;
    lo[n - 1] = 0;
    di[n - 1] = 1;  // P[1,1:2] = [1,0]; P[end,end-1:end] = [0,1]  (chan.jl:109)
    lo[0] = 0;
    up[n - 1] = 0;
    // forward elimination factors
    double denom = di[0];
    tri[n + 0] = 1.0 / denom;
    tri[0] = up[0] / denom;
    for (long long i = 1; i < n; ++i) {
      denom = di[i] - lo[i] * tri[i - 1];
      tri[n + i] = 1.0 / denom;
      tri[i] = up[i] / denom;
      tri[2 * n + i] = lo[i];
    }
    BK_TRY(upload(c, (void**)&pc.tri, tri.data(), 8 * 3 * n));
  } else if (kind == BK_PC_JACOBI) {
    BK_CHECK(c, c->kind == BK_SPARSE, "BK_PC_JACOBI needs a BK_SPARSE context (the kind with an assembled diagonal)");
    pc.kind = kind;
    pc.a0 = a0;
    pc.a1 = a1;
    pc.jdirty = true;  // no values loaded yet: the pivots are computed (and checked) at the first application
    const int st = (c->sp && c->sp->have_vals) ? bk_jacobi_refresh(c) : BK_OK;
    if (st < 0) pc.kind = BK_PC_NONE;
    return st;
  } else {
    return bk_fail(c, BK_ERR_ARG, "unknown preconditioner kind", __FILE__, __LINE__);
  }
  pc.kind = kind;
  pc.a0 = a0;
  pc.a1 = a1;
  return BK_OK;
}

// one 1-D transform pass along dimension d over fields of nx * ny * nz values.
// mode 0: forward, 1: inverse; fused != NULL (fast path, last dimension): forward + symbol + inverse in one kernel.
// Conventions: DCT forward returns 2 C, DCT inverse returns n x (the caller's symbol carries 1 / prod(2 n_d)); DST-I is orthonormal.
static int transform_pass(bk_ctx* c, int d, int mode, const double* in, double* out, int nx, int ny, int nz, bool aligned,
                          const bkf::Symbol* fused = nullptr) {
  Precond& pc = c->pc;
  bkf::Geom g;
  bool strided = d != 0;
  if (d == 0) {
    g.es = 1;
    g.os = nx;
    g.nb = ny * nz;  // number of lines
    g.nouter = 1;
  } else if (d == 1) {
    g.es = nx;
    g.nb = nx;
    g.os = (long long)nx * ny;
    g.nouter = nz;
  } else {
    g.es = (long long)nx * ny;
    g.nb = nx;
    g.os = nx;
    g.nouter = ny;
  }
  if (pc.fast[d] && aligned) {
    BKF_DISPATCH(pc.fast[d], BK_TRY(fast_launch<FC>(c, d, strided, fused ? 2 : mode, in, out, g, fused)));
  } else {
    BK_CHECK(c, !fused, "internal: fused transform on the general path");
    BK_TRY(gen_launch(c, d, strided, pc.ttype[d] == 1 ? 2 : mode, in, out, g));
  }
  c->stats.kernel_launches++;
  return BK_OK;
}

static inline bool aligned16(const void* a, const void* b) { return ((((uintptr_t)a) | ((uintptr_t)b)) & 15) == 0; }

static int precond_apply_one(bk_ctx* c, const double* in, double* out, long long n);

int bk_precond_apply_dev(bk_ctx* c, const double* in, double* out, long long n) {
  BK_CHECK(c, c->pc.kind != BK_PC_NONE, "no preconditioner set up (bk_precond_setup)");
  BK_CHECK(c, in != out, "preconditioner: in-place application is not supported");
  if (!c->cplx) return precond_apply_one(c, in, out, n);
  // split complex vector: the real preconditioner on both halves (border entries, if any, follow the second half)
  BK_CHECK(c, n >= c->N, "preconditioner: vector shorter than the complexified problem");
  BK_TRY(precond_apply_one(c, in, out, c->N0));
  return precond_apply_one(c, in + c->N0, out + c->N0, n - c->N0);
}

static int precond_apply_one(bk_ctx* c, const double* in, double* out, long long n) {
  Precond& pc = c->pc;
  const long long N = c->N0;
  bool tail_done = false;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  if (c->timing_now) {  // per-application device time for bench.py's breakdown (event pairs are read back in bk_get_stats)
    if (c->pc_pairs_used >= c->pc_pairs.size()) {
      cudaEvent_t a, b;
      cudaEventCreate(&a);
      cudaEventCreate(&b);
      c->pc_pairs.push_back({a, b});
    }
    ev0 = c->pc_pairs[c->pc_pairs_used].first;
    ev1 = c->pc_pairs[c->pc_pairs_used].second;
    c->pc_pairs_used++;
    cudaEventRecord(ev0, c->stream);
  }
  const bool al = aligned16(in, out);
  if (pc.kind == BK_PC_SH_DCT) {
    const int nd = pc_ndim(c);
    const int nx = (int)c->dims[0], ny = (int)c->dims[1], nz = nd == 3 ? (int)c->dims[2] : 1;
    double* A = pc.work;
    double* B = pc.work2;
    const int last = nd - 1;
    double scale = 1.0;
    for (int d = 0; d < nd; ++d) scale /= 2.0 * (double)c->dims[d];
    if (pc.fast[last] && al) {
      // x fwd, [y fwd,] (last dim: fwd + symbol + inverse in one kernel), [y inv,] x inv
      bkf::Symbol sy{pc.lam[0], nd == 3 ? pc.lam[1] : nullptr, pc.a0, scale, nullptr, nullptr, 0};
      if (n > N && n - N <= 32) {  // border entries ride along with the fused kernel
        sy.tail_src = in + N;
        sy.tail_dst = out + N;
        sy.tail_n = (int)(n - N);
        tail_done = true;
      }
      BK_TRY(transform_pass(c, 0, 0, in, A, nx, ny, nz, al));
      if (nd == 3) {
        BK_TRY(transform_pass(c, 1, 0, A, B, nx, ny, nz, true));
        BK_TRY(transform_pass(c, 2, 0, B, A, nx, ny, nz, true, &sy));
        BK_TRY(transform_pass(c, 1, 1, A, B, nx, ny, nz, true));
        BK_TRY(transform_pass(c, 0, 1, B, out, nx, ny, nz, al));
      } else {
        BK_TRY(transform_pass(c, 1, 0, A, B, nx, ny, nz, true, &sy));
        BK_TRY(transform_pass(c, 0, 1, B, out, nx, ny, nz, al));
      }
    } else {
      BK_TRY(transform_pass(c, 0, 0, in, A, nx, ny, nz, al));
      BK_TRY(transform_pass(c, 1, 0, A, B, nx, ny, nz, true));
      double* cur = B;
      double* oth = A;
      if (nd == 3) {
        BK_TRY(transform_pass(c, 2, 0, B, A, nx, ny, nz, true));
        cur = A;
        oth = B;
      }
      k_sh_symbol_div<<<lin_grid(c, N), 256, 0, c->stream>>>(cur, nx, ny, nz, pc.lam[0], pc.lam[1],
                                                            nd == 3 ? pc.lam[2] : nullptr, pc.a0, scale);
      c->stats.kernel_launches++;
      BK_CUDA(c, cudaGetLastError());
      if (nd == 3) {
        BK_TRY(transform_pass(c, 2, 1, cur, oth, nx, ny, nz, true));
        std::swap(cur, oth);
      }
      BK_TRY(transform_pass(c, 1, 1, cur, oth, nx, ny, nz, true));
      BK_TRY(transform_pass(c, 0, 1, oth, out, nx, ny, nz, al));
    }
  } else if (pc.kind == BK_PC_CGL_DST) {
    const int nx = (int)c->dims[0], ny = (int)c->dims[1];
    // components x slices (a grid-shaped BK_SPARSE context: one field per z slice)
    const long long nblk = (c->kind == BK_POTRAP_CGL2D) ? 2 * c->dims[2] : (c->kind == BK_SPARSE ? c->dims[2] : 2);
    double* A = pc.work;
    double* B = pc.work2;
    BK_TRY(transform_pass(c, 0, 0, in, A, nx, ny, (int)nblk, al));
    BK_TRY(transform_pass(c, 1, 0, A, B, nx, ny, (int)nblk, true));
    k_helmholtz_symbol_div<<<lin_grid(c, (long long)nx * ny * nblk), 256, 0, c->stream>>>(B, nx, ny, nblk, pc.lam[0], pc.lam[1],
                                                                                         pc.a0, pc.a1);
    c->stats.kernel_launches++;
    BK_CUDA(c, cudaGetLastError());
    BK_TRY(transform_pass(c, 1, 1, B, A, nx, ny, (int)nblk, true));
    BK_TRY(transform_pass(c, 0, 1, A, out, nx, ny, (int)nblk, al));
    if (c->kind == BK_POTRAP_CGL2D) BK_CUDA(c, cudaMemcpyAsync(out + N - 1, in + N - 1, 8, cudaMemcpyDeviceToDevice, c->stream));
  } else if (pc.kind == BK_PC_POTRAP_CIRC) {
    const int nx = (int)c->dims[0], ny = (int)c->dims[1], M = (int)c->dims[2];
    const long long nn = (long long)nx * ny, Ns = 2 * nn;
    const int nf = 2 * M;
    double* A = pc.work;
    double* Bf = pc.work2;
    // DST-I in space over all 2M slice components (mixed-radix FFT of the odd extension, bk_fft_gen.cuh), the circulant
    // solve in time per spatial mode, DST-I back
    BK_TRY(transform_pass(c, 0, 0, in, A, nx, ny, nf, al));
    BK_TRY(transform_pass(c, 1, 0, A, Bf, nx, ny, nf, true));
    k_potrap_time<<<(unsigned)((nn + 127) / 128), 128, 0, c->stream>>>(Bf, nn, nx, M - 1, pc.lam[0], pc.lam[1], pc.po_T / M,
                                                                    pc.po_r, pc.po_nu, pc.tdft);
    BK_CUDA(c, cudaGetLastError());
    BK_TRY(transform_pass(c, 1, 1, Bf, A, nx, ny, nf, true));
    BK_TRY(transform_pass(c, 0, 1, A, out, nx, ny, nf, al));
    k_potrap_close<<<(unsigned)((Ns + 255) / 256), 256, 0, c->stream>>>(in, out, Ns, M);
    c->stats.kernel_launches += 2;
    BK_CUDA(c, cudaGetLastError());
  } else if (pc.kind == BK_PC_JACOBI) {
    BK_TRY(bk_jacobi_apply(c, in, out));
  } else if (pc.kind == BK_PC_CHAN_TRIDIAG) {
    k_thomas<<<1, 32, 0, c->stream>>>(pc.tri, in, out, (int)N);
    c->stats.kernel_launches++;
    BK_CUDA(c, cudaGetLastError());
  }
  if (n > N && !tail_done)
    BK_CUDA(c, cudaMemcpyAsync(out + N, in + N, 8 * (size_t)(n - N), cudaMemcpyDeviceToDevice, c->stream));
  if (ev1) cudaEventRecord(ev1, c->stream);
  return BK_OK;
}

extern "C" int32_t bk_precond_apply(bk_ctx* c, const double* in, double* out) {
  BK_ENTER(c);
  BkRange nvtx_range("bk_precond_apply");
  double *din, *dout;
  BK_TRY(bk_stage_in(c, in, c->N, 10, true, &din));
  BK_TRY(bk_stage_in(c, out, c->N, 11, false, &dout));
  BK_TRY(bk_precond_apply_dev(c, din, dout, c->N));
  return bk_stage_out(c, out, c->N, dout);
}
