// bk_eigs.cu -- S10 / K5: shift-invert Arnoldi eigensolver for stability detection.
//
// Replaces (eig_si::ShiftInvert)(J, nev) (src/EigSolver.jl:257-266) together with the Krylov package
// behind it (ArnoldiMethod.partialschur / KrylovKit.eigsolve, src/EigSolver.jl:157-160,204-225; the
// hand-rolled equivalent examples/SH3d.jl:103-113 uses krylovdim = max(30, nev+30)):
//   Jmap(rhs) = ls(J, rhs; a0 = -sigma, a1 = 1)[1]   -> one bk_gmres_dev solve per Arnoldi vector,
//   i.e. the same fused JVP+Arnoldi kernels as the corrector;
//   eigenvalues theta of (J - sigma)^-1 of largest magnitude, lambda = sigma + 1/theta, sorted by
//   decreasing real part (src/EigSolver.jl:16-19).
// Outer iteration: explicitly restarted Arnoldi with two classical Gram-Schmidt passes (CGS2) on the
// device (same k_dots / k_update_norm kernels as GMRES); the small Hessenberg eigenproblem is solved
// on the host (complex shifted QR + inverse iteration), like the Givens rotations of GMRES.
#include <algorithm>
#include <cmath>
#include <complex>
#include <vector>
#include "bk_common.cuh"

typedef std::complex<double> cplx;

// Eigenvalues of a real upper-Hessenberg matrix (n x n, column-major H[i + j*ldh]) by the complex
// single-shift QR algorithm with Wilkinson shifts and deflation.  A subdiagonal entry is neglected when it is below eps
// times its two diagonal neighbours.  The retry of hess_eigvals for the matrices on which that alone stalls (`robust`):
// also neglect entries below eps ||H||_F (spectra spread over several decades), and take an isolated trailing 2 x 2 block's
// eigenvalues from its characteristic polynomial (a double eigenvalue: the shifted QR step cannot shrink the subdiagonal of a
// block that is a multiple of the identity plus a nilpotent part).
static bool hess_eigvals_pass(const std::vector<double>& Hr, int n, int ldh, std::vector<cplx>& ev, bool robust) {
  std::vector<cplx> A((size_t)n * n);
  for (int j = 0; j < n; ++j)
    for (int i = 0; i < n; ++i) A[i + (size_t)j * n] = (i <= j + 1) ? cplx(Hr[i + (size_t)j * ldh], 0.0) : cplx(0, 0);
  double hnorm = 0.0;
  if (robust)
    for (const cplx& z : A) hnorm += std::norm(z);
  hnorm = std::sqrt(hnorm);
  ev.assign(n, cplx(0, 0));
  int hi = n - 1, iter = 0;
  const double eps = 2.2e-16;
  std::vector<cplx> cs(n), sn(n);
  while (hi >= 0) {
    if (hi == 0) {
      ev[0] = A[0];
      break;
    }
    int l = hi;
    while (l > 0) {
      double s = std::abs(A[(l - 1) + (size_t)(l - 1) * n]) + std::abs(A[l + (size_t)l * n]);
      if (s == 0.0) s = 1.0;
      const double sub = std::abs(A[l + (size_t)(l - 1) * n]);
      if (sub < eps * s || sub < eps * hnorm) {
        A[l + (size_t)(l - 1) * n] = 0.0;
        break;
      }
      --l;
    }
    if (l == hi) {
      ev[hi] = A[hi + (size_t)hi * n];
      --hi;
      iter = 0;
      continue;
    }
    if (++iter > 60 * n) return false;
    // Wilkinson shift from the trailing 2x2 block
    cplx a = A[(hi - 1) + (size_t)(hi - 1) * n], b = A[(hi - 1) + (size_t)hi * n], c = A[hi + (size_t)(hi - 1) * n],
         d = A[hi + (size_t)hi * n];
    cplx tr = a + d, det = a * d - b * c;
    cplx disc = std::sqrt(tr * tr - 4.0 * det);
    cplx m1 = 0.5 * (tr + disc), m2 = 0.5 * (tr - disc);
    if (robust && l == hi - 1) {  // isolated 2 x 2 block
      ev[hi - 1] = m1;
      ev[hi] = m2;
      hi -= 2;
      iter = 0;
      continue;
    }
    cplx mu = (std::abs(m1 - d) < std::abs(m2 - d)) ? m1 : m2;
    if (iter % 11 == 10) mu += cplx(std::abs(c), 0.37 * std::abs(c));  // exceptional shift
    // QR step on the active block l..hi
    for (int i = l; i <= hi; ++i) A[i + (size_t)i * n] -= mu;
    for (int k = l; k < hi; ++k) {
      cplx x = A[k + (size_t)k * n], y = A[(k + 1) + (size_t)k * n];
      double r = std::sqrt(std::norm(x) + std::norm(y));
      cplx c_, s_;
      if (r == 0.0) {
        c_ = 1.0;
        s_ = 0.0;
      } else {
        c_ = x / r;
        s_ = y / r;
      }
      cs[k] = c_;
      sn[k] = s_;
      // rows k, k+1:  [ conj(c) conj(s); -s c ]
      for (int j = k; j < n; ++j) {
        cplx t1 = A[k + (size_t)j * n], t2 = A[(k + 1) + (size_t)j * n];
        A[k + (size_t)j * n] = std::conj(c_) * t1 + std::conj(s_) * t2;
        A[(k + 1) + (size_t)j * n] = -s_ * t1 + c_ * t2;
      }
    }
    for (int k = l; k < hi; ++k) {
      cplx c_ = cs[k], s_ = sn[k];
      int top = std::min(hi, k + 2);
      for (int i = 0; i <= top; ++i) {
        cplx t1 = A[i + (size_t)k * n], t2 = A[i + (size_t)(k + 1) * n];
        A[i + (size_t)k * n] = t1 * c_ + t2 * s_;
        A[i + (size_t)(k + 1) * n] = -t1 * std::conj(s_) + t2 * std::conj(c_);
      }
    }
    for (int i = l; i <= hi; ++i) A[i + (size_t)i * n] += mu;
  }
  return true;
}
static bool hess_eigvals(const std::vector<double>& Hr, int n, int ldh, std::vector<cplx>& ev) {
  return hess_eigvals_pass(Hr, n, ldh, ev, false) || hess_eigvals_pass(Hr, n, ldh, ev, true);
}

// Eigenvector of the real Hessenberg matrix for eigenvalue theta by inverse iteration (complex LU with
// partial pivoting).  Returns the unit-norm vector y.
static void hess_eigvec(const std::vector<double>& Hr, int n, int ldh, cplx theta, std::vector<cplx>& y) {
  double hn = 0;
  for (int j = 0; j < n; ++j)
    for (int i = 0; i <= std::min(n - 1, j + 1); ++i) hn = std::max(hn, std::fabs(Hr[i + (size_t)j * ldh]));
  if (hn == 0) hn = 1;
  cplx th = theta + cplx(1e-10 * hn, 1e-11 * hn);  // perturb so that the matrix is invertible
  std::vector<cplx> A((size_t)n * n);
  for (int j = 0; j < n; ++j)
    for (int i = 0; i < n; ++i) {
      cplx v = (i <= j + 1) ? cplx(Hr[i + (size_t)j * ldh], 0.0) : cplx(0, 0);
      if (i == j) v -= th;
      A[i + (size_t)j * n] = v;
    }
  std::vector<int> piv(n);
  for (int k = 0; k < n; ++k) {
    int p = k;
    double best = std::abs(A[k + (size_t)k * n]);
    for (int i = k + 1; i < n; ++i)
      if (std::abs(A[i + (size_t)k * n]) > best) {
        best = std::abs(A[i + (size_t)k * n]);
        p = i;
      }
    piv[k] = p;
    if (p != k)
      for (int j = 0; j < n; ++j) std::swap(A[k + (size_t)j * n], A[p + (size_t)j * n]);
    if (std::abs(A[k + (size_t)k * n]) < 1e-300) A[k + (size_t)k * n] = 1e-300;
    for (int i = k + 1; i < n; ++i) {
      cplx f = A[i + (size_t)k * n] / A[k + (size_t)k * n];
      A[i + (size_t)k * n] = f;
      if (f != cplx(0, 0))
        for (int j = k + 1; j < n; ++j) A[i + (size_t)j * n] -= f * A[k + (size_t)j * n];
    }
  }
  y.assign(n, cplx(1.0, 0.0));
  for (int i = 0; i < n; ++i) y[i] = cplx(1.0 / (1.0 + i), 0.3 / (2.0 + i));
  for (int it = 0; it < 3; ++it) {
    for (int k = 0; k < n; ++k)
      if (piv[k] != k) std::swap(y[k], y[piv[k]]);  // whole rows were swapped (getrf style): permute first
    for (int k = 0; k < n; ++k)
      for (int i = k + 1; i < n; ++i) y[i] -= A[i + (size_t)k * n] * y[k];
    for (int k = n - 1; k >= 0; --k) {
      for (int j = k + 1; j < n; ++j) y[k] -= A[k + (size_t)j * n] * y[j];
      y[k] /= A[k + (size_t)k * n];
    }
    double nr = 0;
    for (auto& v : y) nr += std::norm(v);
    nr = std::sqrt(nr);
    for (auto& v : y) v /= nr;
  }
  // fix the phase: largest component real positive
  int im = 0;
  for (int i = 1; i < n; ++i)
    if (std::abs(y[i]) > std::abs(y[im])) im = i;
  cplx ph = std::conj(y[im]) / std::abs(y[im]);
  for (auto& v : y) v *= ph;
}

// Host-only utility (no GPU needed): eigen-decomposition of a real upper-Hessenberg matrix, the small dense
// problem the Arnoldi eigensolver hands to the host.  Exposed so that it can be validated on CPU against
// the reference's golden spectrum (test/linear_solvers/test_linear.jl:595-614).
extern "C" int32_t bk_hessenberg_eig(const double* H, int32_t n, int32_t ldh, double* wr, double* wi, double* vec_re,
                                     double* vec_im) {
  if (!H || n < 1 || ldh < n || !wr || !wi) return BK_ERR_ARG;
  std::vector<double> Hc((size_t)ldh * n);
  for (size_t i = 0; i < Hc.size(); ++i) Hc[i] = H[i];
  std::vector<cplx> ev;
  if (!hess_eigvals(Hc, n, ldh, ev)) return BK_NOT_CONVERGED;
  std::vector<cplx> y;
  for (int q = 0; q < n; ++q) {
    wr[q] = ev[q].real();
    wi[q] = ev[q].imag();
    if (vec_re && vec_im) {
      hess_eigvec(Hc, n, ldh, ev[q], y);
      for (int i = 0; i < n; ++i) {
        vec_re[i + (size_t)q * n] = y[i].real();
        vec_im[i + (size_t)q * n] = y[i].imag();
      }
    }
  }
  return BK_OK;
}

// Symmetric eigen-decomposition by cyclic Jacobi rotations: A (n x n, column-major, overwritten) = S diag(w) S^T.
static void jacobi_eig(std::vector<double>& A, int n, std::vector<double>& w, std::vector<double>& S) {
  S.assign((size_t)n * n, 0.0);
  for (int i = 0; i < n; ++i) S[i + (size_t)i * n] = 1.0;
  for (int sweep = 0; sweep < 60; ++sweep) {
    double off = 0, dg = 0;
    for (int j = 0; j < n; ++j)
      for (int i = 0; i < n; ++i) (i == j ? dg : off) += A[i + (size_t)j * n] * A[i + (size_t)j * n];
    if (off <= 1e-32 * (dg + 1e-300)) break;
    for (int p = 0; p < n - 1; ++p)
      for (int q = p + 1; q < n; ++q) {
        double apq = A[p + (size_t)q * n];
        if (apq == 0.0) continue;
        double app = A[p + (size_t)p * n], aqq = A[q + (size_t)q * n];
        double th = (aqq - app) / (2.0 * apq);
        double t = (th >= 0 ? 1.0 : -1.0) / (fabs(th) + sqrt(th * th + 1.0));
        double cs = 1.0 / sqrt(t * t + 1.0), sn = t * cs;
        for (int k = 0; k < n; ++k) {  // columns p, q
          double akp = A[k + (size_t)p * n], akq = A[k + (size_t)q * n];
          A[k + (size_t)p * n] = cs * akp - sn * akq;
          A[k + (size_t)q * n] = sn * akp + cs * akq;
        }
        for (int k = 0; k < n; ++k) {  // rows p, q
          double apk = A[p + (size_t)k * n], aqk = A[q + (size_t)k * n];
          A[p + (size_t)k * n] = cs * apk - sn * aqk;
          A[q + (size_t)k * n] = sn * apk + cs * aqk;
        }
        for (int k = 0; k < n; ++k) {
          double skp = S[k + (size_t)p * n], skq = S[k + (size_t)q * n];
          S[k + (size_t)p * n] = cs * skp - sn * skq;
          S[k + (size_t)q * n] = sn * skp + cs * skq;
        }
      }
  }
  w.resize(n);
  for (int i = 0; i < n; ++i) w[i] = A[i + (size_t)i * n];
}

static __global__ void k_fill_ones(double* p, int n) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) p[i] = 1.0;
}
// deterministic start vector (the reference uses rand(); any generic vector works)
static __global__ void k_start_vector(double* v, long long n) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    unsigned long long z = (unsigned long long)i * 0x9E3779B97F4A7C15ULL + 0x1234567ULL;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ULL;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBULL;
    z ^= z >> 31;
    v[i] = (double)(z >> 11) * (1.0 / 9007199254740992.0) + 0.05;
  }
}

extern "C" int32_t bk_eigs_shift_invert(bk_ctx* c, double sigma, int32_t nev, int32_t krylovdim, double tol,
                                        int32_t maxrestart, const bk_gmres_opts* inner, const double* v0, double* vals_re,
                                        double* vals_im, double* vecs, int32_t* nconv, int32_t* nops) {
  BK_ENTER(c);
  BkRange nvtx_range("bk_eigs_shift_invert");
  BK_CHECK(c, c->have_state, "bk_jac_set_state must be called first");
  BK_CHECK(c, inner != nullptr && vals_re && vals_im, "null argument");
  const long long n = c->N;
  int m = krylovdim;
  if ((long long)m > n) m = (int)n;
  BK_CHECK(c, nev >= 1 && nev <= m, "need 1 <= nev <= krylovdim <= N");
  if (maxrestart < 1) maxrestart = 1;
  // workspace
  if (c->qcap < m) {
    BK_CUDA(c, cudaStreamSynchronize(c->stream));
    if (c->Q) cudaFree(c->Q);
    if (c->eig_dev) cudaFree(c->eig_dev);
    if (c->eig_pinned) cudaFreeHost(c->eig_pinned);
    c->Q = c->eig_dev = c->eig_pinned = nullptr;
    BK_CUDA(c, cudaMalloc(&c->Q, 8 * (size_t)c->ld * (m + 1)));
    BK_CUDA(c, cudaMalloc(&c->eig_dev, 8 * (size_t)(m + 4) * 6));
    BK_CUDA(c, cudaMallocHost(&c->eig_pinned, 8 * (size_t)(m + 4) * 6));
    c->qcap = m;
    k_fill_ones<<<(m + 4 + 255) / 256, 256, 0, c->stream>>>(c->eig_dev, m + 4);
  }
  // partial-sum buffer must hold m rows
  BK_CHECK(c, m <= c->m, "krylovdim exceeds the context's krylov_m (partial-sum workspace)");
  const int S = m + 4;
  double* ones = c->eig_dev;
  double* hA = c->eig_dev + S;
  double* hB = c->eig_dev + 2 * S;
  double* gco = c->eig_dev + 3 * S;
  double* coef = c->eig_dev + 4 * S;  // 2*S
  double* hp = c->eig_pinned;
  double* x;
  BK_TRY(bk_tmp(c, 3, &x));
  OpDesc op = bk_make_op(c, -sigma, 1.0);  // (a0 I + a1 J) with a0 = -sigma (src/EigSolver.jl:260)

  // start vector
  if (v0) {
    cudaMemcpyKind kd = bk_is_device_ptr(v0) ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
    BK_CUDA(c, cudaMemcpyAsync(x, v0, 8 * (size_t)n, kd, c->stream));
  } else {
    k_start_vector<<<c->nsm * 4, 256, 0, c->stream>>>(x, n);
  }
  int total_ops = 0;
  std::vector<double> H((size_t)(m + 1) * m);
  std::vector<cplx> ev, ritz(nev);
  std::vector<std::vector<cplx>> Y(nev);
  bool converged = false;
  int keff = m;
  // ---------------- symmetric operators (Swift-Hohenberg): thick-restart (Krylov-Schur with Ritz vectors) ----------------
  const bool sym = (c->kind == BK_SH2D || c->kind == BK_SH3D);
  std::vector<double> Ssym, wsym;
  std::vector<int> order;
  if (sym) {
    if (!c->Q2 || c->q2cap < m) {
      BK_CUDA(c, cudaStreamSynchronize(c->stream));
      if (c->Q2) cudaFree(c->Q2);
      BK_CUDA(c, cudaMalloc(&c->Q2, 8 * (size_t)c->ld * (m + 1)));
      c->q2cap = m;
    }
    std::fill(H.begin(), H.end(), 0.0);
    BK_TRY(bk_launch_update(c, c->Q, gco, x, n, 0, c->Q, hA, hB));
    BK_CUDA(c, cudaMemcpyAsync(hp, hA, 8, cudaMemcpyDeviceToHost, c->stream));
    BK_CUDA(c, cudaStreamSynchronize(c->stream));
    BK_CHECK(c, hp[0] > 0, "zero start vector");
    BK_TRY(bk_dev_scale(c, c->Q, 1.0 / hp[0], n));
    int kstart = 0;
    for (int rs = 0; rs < maxrestart && !converged; ++rs) {
      keff = m;
      for (int k = kstart; k < m; ++k) {
        const int j = k + 1;
        int cv = 0, it = 0;
        int st = bk_gmres_dev(c, op, c->Q + (size_t)k * c->ld, x, inner, &cv, &it, nullptr);
        if (st < 0) return st;
        ++total_ops;
        double* qn = c->Q + (size_t)(k + 1) * c->ld;
        BK_TRY(bk_launch_dots(c, c->Q, ones, x, n, j, hA, gco));
        BK_TRY(bk_launch_update(c, c->Q, gco, x, n, j, qn, hA + j, hB + S - 1));
        BK_TRY(bk_launch_dots(c, c->Q, ones, qn, n, j, hB, gco));
        BK_TRY(bk_launch_update(c, c->Q, gco, qn, n, j, qn, hA + j, hB + S - 1));
        BK_CUDA(c, cudaMemcpyAsync(hp, hA, 8 * (size_t)(2 * S), cudaMemcpyDeviceToHost, c->stream));
        BK_CUDA(c, cudaStreamSynchronize(c->stream));
        double cn = 0;
        for (int i = 0; i < j; ++i) {
          H[i + (size_t)k * (m + 1)] = hp[i] + hp[S + i];
          cn = fmax(cn, fabs(H[i + (size_t)k * (m + 1)]));
        }
        double hk1 = hp[j];
        H[j + (size_t)k * (m + 1)] = hk1;
        if (!(hk1 > 1e-14 * fmax(cn, 1e-300))) {
          keff = k + 1;
          break;
        }
        BK_TRY(bk_dev_scale(c, qn, 1.0 / hk1, n));
      }
      // symmetrised projected matrix (exactly symmetric in exact arithmetic)
      std::vector<double> A((size_t)keff * keff);
      for (int jj = 0; jj < keff; ++jj)
        for (int i = 0; i < keff; ++i) {
          double hij = (i <= jj + 1 || jj < kstart) ? H[i + (size_t)jj * (m + 1)] : 0.0;
          double hji = (jj <= i + 1 || i < kstart) ? H[jj + (size_t)i * (m + 1)] : 0.0;
          // below-diagonal entries of Arnoldi columns other than the sub-diagonal are zero; the arrow row of a
          // restarted factorisation is stored in row kstart of the retained columns
          A[i + (size_t)jj * keff] = (i == jj) ? hij : ((i < jj) ? hij : hji);
        }
      for (int jj = 0; jj < keff; ++jj)
        for (int i = jj + 1; i < keff; ++i) A[i + (size_t)jj * keff] = A[jj + (size_t)i * keff];
      jacobi_eig(A, keff, wsym, Ssym);
      order.resize(keff);
      for (int i = 0; i < keff; ++i) order[i] = i;
      std::sort(order.begin(), order.end(), [&](int a, int b) { return fabs(wsym[a]) > fabs(wsym[b]); });
      const double hlast = (keff == m) ? H[m + (size_t)(m - 1) * (m + 1)] : 0.0;
      int nv = std::min<int>(nev, keff);
      bool all = true;
      for (int q = 0; q < nv; ++q) {
        const int iq = order[q];
        ritz[q] = cplx(wsym[iq], 0.0);
        Y[q].assign(keff, cplx(0, 0));
        for (int i = 0; i < keff; ++i) Y[q][i] = cplx(Ssym[i + (size_t)iq * keff], 0.0);
        double resid = fabs(hlast) * fabs(Ssym[(keff - 1) + (size_t)iq * keff]);
        if (resid > tol * fmax(fabs(wsym[iq]), 1e-300)) all = false;
      }
      for (int q = nv; q < nev; ++q) ritz[q] = cplx(0, 0);
      converged = all || keff < m;
      if (!converged && rs + 1 < maxrestart) {
        int pkeep = std::min(keff - 2, nev + std::max(8, (m - nev) / 3));
        if (pkeep < 1) pkeep = 1;
        for (int q = 0; q < pkeep; ++q) {  // Q2_q = Q S[:, order[q]]
          for (int i = 0; i < keff; ++i) hp[i] = Ssym[i + (size_t)order[q] * keff];
          BK_CUDA(c, cudaMemcpyAsync(coef, hp, 8 * (size_t)keff, cudaMemcpyHostToDevice, c->stream));
          BK_TRY(bk_launch_lincomb(c, c->Q, nullptr, c->Q2 + (size_t)q * c->ld, 0.0, n, keff, coef));
          BK_CUDA(c, cudaStreamSynchronize(c->stream));
        }
        BK_TRY(bk_dev_copy(c, c->Q2 + (size_t)pkeep * c->ld, c->Q + (size_t)keff * c->ld, n));  // residual direction q_{m+1}
        BK_CUDA(c, cudaMemcpyAsync(c->Q, c->Q2, 8 * (size_t)c->ld * (pkeep + 1), cudaMemcpyDeviceToDevice, c->stream));
        std::vector<double> bnew(pkeep), thnew(pkeep);
        for (int q = 0; q < pkeep; ++q) {
          thnew[q] = wsym[order[q]];
          bnew[q] = hlast * Ssym[(keff - 1) + (size_t)order[q] * keff];
        }
        std::fill(H.begin(), H.end(), 0.0);
        for (int q = 0; q < pkeep; ++q) {
          H[q + (size_t)q * (m + 1)] = thnew[q];
          H[pkeep + (size_t)q * (m + 1)] = bnew[q];
        }
        kstart = pkeep;
      }
    }
  }
  for (int rs = 0; !sym && rs < maxrestart && !converged; ++rs) {
    std::fill(H.begin(), H.end(), 0.0);
    // Q_0 = x / ||x||
    BK_TRY(bk_launch_update(c, c->Q, gco, x, n, 0, c->Q, hA, hB));
    BK_CUDA(c, cudaMemcpyAsync(hp, hA, 8, cudaMemcpyDeviceToHost, c->stream));
    BK_CUDA(c, cudaStreamSynchronize(c->stream));
    BK_CHECK(c, hp[0] > 0, "zero start vector");
    BK_TRY(bk_dev_scale(c, c->Q, 1.0 / hp[0], n));
    keff = m;
    for (int k = 0; k < m; ++k) {
      const int j = k + 1;
      int cv = 0, it = 0;
      int st = bk_gmres_dev(c, op, c->Q + (size_t)k * c->ld, x, inner, &cv, &it, nullptr);
      if (st < 0) return st;
      ++total_ops;
      double* qn = c->Q + (size_t)(k + 1) * c->ld;
      BK_TRY(bk_launch_dots(c, c->Q, ones, x, n, j, hA, gco));
      BK_TRY(bk_launch_update(c, c->Q, gco, x, n, j, qn, hA + j, hB + S - 1));
      BK_TRY(bk_launch_dots(c, c->Q, ones, qn, n, j, hB, gco));
      BK_TRY(bk_launch_update(c, c->Q, gco, qn, n, j, qn, hA + j, hB + S - 1));
      BK_CUDA(c, cudaMemcpyAsync(hp, hA, 8 * (size_t)(2 * S), cudaMemcpyDeviceToHost, c->stream));
      BK_CUDA(c, cudaStreamSynchronize(c->stream));
      double cn = 0;
      for (int i = 0; i < j; ++i) {
        H[i + (size_t)k * (m + 1)] = hp[i] + hp[S + i];
        cn = fmax(cn, fabs(H[i + (size_t)k * (m + 1)]));
      }
      double hk1 = hp[j];
      H[j + (size_t)k * (m + 1)] = hk1;
      if (!(hk1 > 1e-14 * fmax(cn, 1e-300))) {  // invariant subspace found
        keff = k + 1;
        break;
      }
      BK_TRY(bk_dev_scale(c, qn, 1.0 / hk1, n));
    }
    // Ritz values / vectors of H(keff x keff)
    BK_CHECK(c, hess_eigvals(H, keff, m + 1, ev), "QR iteration on the Hessenberg matrix did not converge");
    std::sort(ev.begin(), ev.end(), [](const cplx& a, const cplx& b) {
      double da = std::abs(a), db = std::abs(b);
      if (da != db) return da > db;
      return a.imag() > b.imag();
    });
    int nv = std::min<int>(nev, keff);
    double hlast = (keff == m) ? H[m + (size_t)(m - 1) * (m + 1)] : 0.0;
    bool all = true;
    for (int q = 0; q < nv; ++q) {
      ritz[q] = ev[q];
      hess_eigvec(H, keff, m + 1, ev[q], Y[q]);
      double resid = fabs(hlast) * std::abs(Y[q][keff - 1]);
      if (resid > tol * fmax(std::abs(ev[q]), 1e-300)) all = false;
    }
    for (int q = nv; q < nev; ++q) ritz[q] = cplx(0, 0);
    converged = all || keff < m;
    if (!converged && rs + 1 < maxrestart) {
      // restart vector = sum of the real parts of the wanted Ritz vectors
      for (int i = 0; i < keff; ++i) {
        double s = 0;
        for (int q = 0; q < nv; ++q) s += Y[q][i].real();
        hp[i] = s;
      }
      BK_CUDA(c, cudaMemcpyAsync(coef, hp, 8 * (size_t)keff, cudaMemcpyHostToDevice, c->stream));
      BK_TRY(bk_launch_lincomb(c, c->Q, nullptr, x, 0.0, n, keff, coef));
      BK_CUDA(c, cudaStreamSynchronize(c->stream));
    }
  }
  // map back, sort by decreasing real part (ties: decreasing imaginary part)
  int nv = std::min<int>(nev, keff);
  std::vector<int> idx(nv);
  std::vector<cplx> lam(nv);
  for (int q = 0; q < nv; ++q) {
    idx[q] = q;
    lam[q] = sigma + 1.0 / ritz[q];
  }
  std::sort(idx.begin(), idx.end(), [&](int a, int b) {
    if (lam[a].real() != lam[b].real()) return lam[a].real() > lam[b].real();
    return lam[a].imag() > lam[b].imag();
  });
  for (int q = 0; q < nev; ++q) {
    vals_re[q] = q < nv ? lam[idx[q]].real() : NAN;
    vals_im[q] = q < nv ? lam[idx[q]].imag() : NAN;
  }
  if (vecs) {
    // column q = Re(Q y_q) for real eigenvalues and for the member of a pair with Im >= 0; Im(Q y_q) for Im < 0
    double* tmpv;
    BK_TRY(bk_tmp(c, 4, &tmpv));
    const bool dev_out = bk_is_device_ptr(vecs);
    for (int q = 0; q < nv; ++q) {
      const std::vector<cplx>& y = Y[idx[q]];
      bool use_im = lam[idx[q]].imag() < 0;
      for (int i = 0; i < keff; ++i) hp[i] = use_im ? y[i].imag() : y[i].real();
      BK_CUDA(c, cudaMemcpyAsync(coef, hp, 8 * (size_t)keff, cudaMemcpyHostToDevice, c->stream));
      double* dst = dev_out ? vecs + (size_t)q * n : tmpv;
      BK_TRY(bk_launch_lincomb(c, c->Q, nullptr, dst, 0.0, n, keff, coef));
      if (!dev_out) {
        BK_CUDA(c, cudaMemcpyAsync(vecs + (size_t)q * n, tmpv, 8 * (size_t)n, cudaMemcpyDeviceToHost, c->stream));
        c->stats.d2h_bytes += 8 * n;
      }
      BK_CUDA(c, cudaStreamSynchronize(c->stream));
    }
  }
  BK_CUDA(c, cudaStreamSynchronize(c->stream));
  if (nconv) *nconv = converged ? nv : 0;
  if (nops) *nops = total_ops;
  return converged ? BK_OK : BK_NOT_CONVERGED;
}
